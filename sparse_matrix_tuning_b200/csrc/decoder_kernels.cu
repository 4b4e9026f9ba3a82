// Elementwise work of a LLaMA decoder layer: RMSNorm (optionally fused with the residual add before it), rotary
// position embedding of q and k, and the SwiGLU gate, forward and backward.
//
// Every kernel is memory-bound: 128-bit loads and stores, fp32 arithmetic, no atomics and a fixed reduction order, so a
// recomputed forward (activation checkpointing) reproduces the first one bit for bit.  The forward kernels round where
// the HF modules round (one bf16 rounding per PyTorch op they replace); see include/smt_b200.h for each formula.
#include "common.cuh"

namespace smt {
namespace {

constexpr int kRowMaxVec = 4;        // uint4 (8 bf16) per thread and row tensor in the norm kernels
constexpr int kFlatThreads = 256;

__device__ __forceinline__ float bf16r(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float (&f)[8]) { unpack8<SMT_BF16>(u, f); }

__device__ __forceinline__ uint4 pack_bf16x8(const float (&f)[8]) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]),
                    pack_bf16x2(f[6], f[7]));
}

// ---- RMSNorm ---------------------------------------------------------------------------------------------------
// One CTA per row; each thread keeps up to kRowMaxVec 16-byte vectors of the row in registers between the reduction
// and the output pass.

template <bool RESIDUAL>
__global__ void __launch_bounds__(1024) rmsnorm_fwd_kernel(const uint4* __restrict__ a, const uint4* __restrict__ res,
                                                           const uint4* __restrict__ w, int nvec, float inv_n, float eps,
                                                           uint4* __restrict__ h_out, uint4* __restrict__ y,
                                                           float* __restrict__ rstd_out) {
  __shared__ float scratch[32];
  const int64_t row = blockIdx.x;
  const uint4* ar = a + row * nvec;
  uint4 xv[kRowMaxVec];
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < kRowMaxVec; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
      uint4 u = ld_stream_u4(ar + v);
      float f[8];
      unpack_bf16x8(u, f);
      if (RESIDUAL) {
        float r[8];
        unpack_bf16x8(ld_stream_u4(res + row * nvec + v), r);
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = bf16r(r[e] + f[e]);      // h = bf16(res + a)
        u = pack_bf16x8(f);
        h_out[row * nvec + v] = u;
      }
      xv[i] = u;
#pragma unroll
      for (int e = 0; e < 8; ++e) ss += __fmul_rn(f[e], f[e]);       // pow(2) rounds each square to fp32
    }
  }
  const float total = block_sum(ss, scratch);
  if (threadIdx.x == 0) scratch[0] = rsqrtf(__fadd_rn(__fmul_rn(total, inv_n), eps));   // mean, + eps: two roundings
  __syncthreads();
  const float rstd = scratch[0];
  if (threadIdx.x == 0) rstd_out[row] = rstd;
#pragma unroll
  for (int i = 0; i < kRowMaxVec; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
      float f[8], wf[8];
      unpack_bf16x8(xv[i], f);
      unpack_bf16x8(w[v], wf);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] = wf[e] * bf16r(__fmul_rn(f[e], rstd));   // w * bf16(x * rstd), rounded below
      y[row * nvec + v] = pack_bf16x8(f);
    }
  }
}

// dx = rstd * (g - xhat * mean(g * xhat)) [+ dres],  g = dy * w,  xhat = x * rstd; one rounding to bf16.
template <bool DRES>
__global__ void __launch_bounds__(1024) rmsnorm_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ w,
                                                           const float* __restrict__ rstd_in,
                                                           const uint4* __restrict__ dy, const uint4* __restrict__ dres,
                                                           int nvec, float inv_n, uint4* __restrict__ dx) {
  __shared__ float scratch[32];
  const int64_t row = blockIdx.x;
  const float rstd = rstd_in[row];
  uint4 xv[kRowMaxVec], gv[kRowMaxVec];
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < kRowMaxVec; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
      xv[i] = ld_stream_u4(x + row * nvec + v);
      gv[i] = ld_stream_u4(dy + row * nvec + v);
      float xf[8], gf[8], wf[8];
      unpack_bf16x8(xv[i], xf);
      unpack_bf16x8(gv[i], gf);
      unpack_bf16x8(w[v], wf);
#pragma unroll
      for (int e = 0; e < 8; ++e) dot += (gf[e] * wf[e]) * (xf[e] * rstd);
    }
  }
  const float total = block_sum(dot, scratch);
  if (threadIdx.x == 0) scratch[0] = total * inv_n;
  __syncthreads();
  const float mean_gx = scratch[0];
#pragma unroll
  for (int i = 0; i < kRowMaxVec; ++i) {
    const int v = threadIdx.x + i * blockDim.x;
    if (v < nvec) {
      float xf[8], gf[8], wf[8], o[8];
      unpack_bf16x8(xv[i], xf);
      unpack_bf16x8(gv[i], gf);
      unpack_bf16x8(w[v], wf);
      float rf[8];
      if (DRES) unpack_bf16x8(ld_stream_u4(dres + row * nvec + v), rf);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        o[e] = rstd * (gf[e] * wf[e] - (xf[e] * rstd) * mean_gx);
        if (DRES) o[e] += rf[e];
      }
      dx[row * nvec + v] = pack_bf16x8(o);
    }
  }
}

int row_threads(int nvec) {
  int t = (nvec + kRowMaxVec - 1) / kRowMaxVec;
  t = (t + 31) / 32 * 32;
  return t < 32 ? 32 : t;
}

// ---- rotary position embedding ---------------------------------------------------------------------------------
// Rows of 128 (head_dim) elements; work item j (0..7) of a row owns elements [8j, 8j+8) and their rotation partners
// [64+8j, 64+8j+8).  q rows come first, then k rows; row r of q belongs to token r / Hq (token = b*S + s).
//   forward  out[d]  = bf16(bf16(x[d]*cos[d]) + bf16(rot(x)[d]*sin[d])),  rot(x) = (-x[64:], x[:64])
//   backward dx[d]   = bf16(bf16(g[d]*cos[d]) + t[d]),  t[:64] = bf16(g[64:]*sin[64:]),  t[64:] = -bf16(g[:64]*sin[:64])
// which are PyTorch's per-op roundings of apply_rotary_pos_emb and of its autograd graph.
constexpr int kHeadDim = 128;

template <bool BWD>
__global__ void __launch_bounds__(kFlatThreads) rope_kernel(const uint4* __restrict__ q, const uint4* __restrict__ k,
                                                            const uint4* __restrict__ cos_, const uint4* __restrict__ sin_,
                                                            int S, int Hq, int Hk, int64_t rows_q, int64_t rows_k,
                                                            int64_t cs_bstride_vec, uint4* __restrict__ q_out,
                                                            uint4* __restrict__ k_out) {
  constexpr int VPR = kHeadDim / 8;       // 16-byte vectors per row
  const int64_t items = (rows_q + rows_k) * 8;
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = it >> 3;
    const int j = (int)(it & 7);
    const uint4* src;
    uint4* dst;
    int64_t tok;
    if (row < rows_q) {
      src = q + row * VPR;
      dst = q_out + row * VPR;
      tok = row / Hq;
    } else {
      row -= rows_q;
      src = k + row * VPR;
      dst = k_out + row * VPR;
      tok = row / Hk;
    }
    const int64_t b = tok / S, s = tok - b * S;
    const uint4* cr = cos_ + b * cs_bstride_vec + s * VPR;
    const uint4* sr = sin_ + b * cs_bstride_vec + s * VPR;
    float x1[8], x2[8], c1[8], c2[8], s1[8], s2[8], o1[8], o2[8];
    unpack_bf16x8(ld_stream_u4(src + j), x1);
    unpack_bf16x8(ld_stream_u4(src + 8 + j), x2);
    unpack_bf16x8(cr[j], c1);
    unpack_bf16x8(cr[8 + j], c2);
    unpack_bf16x8(sr[j], s1);
    unpack_bf16x8(sr[8 + j], s2);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      if (!BWD) {
        o1[e] = bf16r(x1[e] * c1[e]) + bf16r(-x2[e] * s1[e]);
        o2[e] = bf16r(x2[e] * c2[e]) + bf16r(x1[e] * s2[e]);
      } else {
        o1[e] = bf16r(x1[e] * c1[e]) + bf16r(x2[e] * s2[e]);
        o2[e] = bf16r(x2[e] * c2[e]) - bf16r(x1[e] * s1[e]);
      }
    }
    dst[j] = pack_bf16x8(o1);
    dst[8 + j] = pack_bf16x8(o2);
  }
}

// ---- per-head RMSNorm of q and k followed by RoPE (Qwen3 attention) ---------------------------------------------
// rope_kernel's layout: 8 work items per 128-element head row, item j holding vectors j and 8 + j.  The row sums run
// over the 8 items with xor shuffles in a fixed order, so every item of a row gets the same bits and the result
// depends on the row alone (a checkpointed recomputation reproduces the first forward).
//   forward   rstd = rsqrt(mean(x^2) + eps),  y = bf16(w * bf16(x * rstd)),  out = rope_kernel<false>(y)
//   backward  dy = rope_kernel<true>(g)  (bf16, as autograd produces it),  gw = dy * w,  xhat = x * rstd,
//             dx = bf16(rstd * (gw - xhat * mean(gw * xhat)))       (rmsnorm_bwd_kernel's formula; w is frozen)
// Forward reads `a` = (q, k) and writes rstd; backward reads `a` = (dq_out, dk_out), `x` = (q, k) and rstd.
__device__ __forceinline__ float sum8_rows(float v, unsigned mask) {
  v += __shfl_xor_sync(mask, v, 4);
  v += __shfl_xor_sync(mask, v, 2);
  v += __shfl_xor_sync(mask, v, 1);
  return v;
}

template <bool BWD>
__global__ void __launch_bounds__(kFlatThreads) qk_norm_rope_kernel(
    const uint4* __restrict__ a_q, const uint4* __restrict__ a_k, const uint4* __restrict__ x_q,
    const uint4* __restrict__ x_k, const uint4* __restrict__ wq, const uint4* __restrict__ wk, float eps_q, float eps_k,
    const uint4* __restrict__ cos_, const uint4* __restrict__ sin_, int S, int Hq, int Hk, int64_t rows_q,
    int64_t rows_k, int64_t cs_bstride_vec, float* __restrict__ rstd_q, float* __restrict__ rstd_k,
    uint4* __restrict__ out_q, uint4* __restrict__ out_k) {
  constexpr int VPR = kHeadDim / 8;
  constexpr float kInvD = 1.0f / kHeadDim;
  const int64_t items = (rows_q + rows_k) * 8;
  // the 8 items of a row are 8 aligned lanes of one warp (block size and grid stride are multiples of 32), and they
  // enter and leave the loop together
  const unsigned mask = 0xffu << (threadIdx.x & 24);
  for (int64_t it = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
    int64_t row = it >> 3;
    const int j = (int)(it & 7);
    const uint4 *src, *xs, *w;
    uint4* dst;
    float* rstd_p;
    float eps;
    int64_t tok;
    if (row < rows_q) {
      src = a_q + row * VPR;
      xs = BWD ? x_q + row * VPR : nullptr;
      dst = out_q + row * VPR;
      rstd_p = rstd_q + row;
      w = wq;
      eps = eps_q;
      tok = row / Hq;
    } else {
      row -= rows_q;
      src = a_k + row * VPR;
      xs = BWD ? x_k + row * VPR : nullptr;
      dst = out_k + row * VPR;
      rstd_p = rstd_k + row;
      w = wk;
      eps = eps_k;
      tok = row / Hk;
    }
    const int64_t b = tok / S, s = tok - b * S;
    const uint4* cr = cos_ + b * cs_bstride_vec + s * VPR;
    const uint4* sr = sin_ + b * cs_bstride_vec + s * VPR;
    float a1[8], a2[8], c1[8], c2[8], s1[8], s2[8], w1[8], w2[8], o1[8], o2[8];
    unpack_bf16x8(ld_stream_u4(src + j), a1);
    unpack_bf16x8(ld_stream_u4(src + 8 + j), a2);
    unpack_bf16x8(cr[j], c1);
    unpack_bf16x8(cr[8 + j], c2);
    unpack_bf16x8(sr[j], s1);
    unpack_bf16x8(sr[8 + j], s2);
    unpack_bf16x8(w[j], w1);
    unpack_bf16x8(w[8 + j], w2);
    if (!BWD) {
      float ss = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) ss += __fmul_rn(a1[e], a1[e]);
#pragma unroll
      for (int e = 0; e < 8; ++e) ss += __fmul_rn(a2[e], a2[e]);
      const float rstd = rsqrtf(__fadd_rn(__fmul_rn(sum8_rows(ss, mask), kInvD), eps));
      if (j == 0) *rstd_p = rstd;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float y1 = bf16r(w1[e] * bf16r(__fmul_rn(a1[e], rstd)));
        const float y2 = bf16r(w2[e] * bf16r(__fmul_rn(a2[e], rstd)));
        o1[e] = bf16r(y1 * c1[e]) + bf16r(-y2 * s1[e]);
        o2[e] = bf16r(y2 * c2[e]) + bf16r(y1 * s2[e]);
      }
    } else {
      const float rstd = *rstd_p;
      float x1[8], x2[8];
      unpack_bf16x8(ld_stream_u4(xs + j), x1);
      unpack_bf16x8(ld_stream_u4(xs + 8 + j), x2);
      float dot = 0.f;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float d1 = bf16r(bf16r(a1[e] * c1[e]) + bf16r(a2[e] * s2[e]));
        const float d2 = bf16r(bf16r(a2[e] * c2[e]) - bf16r(a1[e] * s1[e]));
        a1[e] = d1 * w1[e];                     // gw, in place of the incoming gradient
        a2[e] = d2 * w2[e];
        x1[e] *= rstd;                          // xhat
        x2[e] *= rstd;
        dot += a1[e] * x1[e];
        dot += a2[e] * x2[e];
      }
      const float mean_gx = sum8_rows(dot, mask) * kInvD;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        o1[e] = rstd * (a1[e] - x1[e] * mean_gx);
        o2[e] = rstd * (a2[e] - x2[e] * mean_gx);
      }
    }
    dst[j] = pack_bf16x8(o1);
    dst[8 + j] = pack_bf16x8(o2);
  }
}

// ---- SwiGLU ----------------------------------------------------------------------------------------------------
// silu and its derivative are written as in PyTorch's CUDA kernels (exp and division at full precision), so the
// forward matches torch's `silu(g) * u` bit for bit.

__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(kFlatThreads) swiglu_fwd_kernel(const uint4* __restrict__ g, const uint4* __restrict__ u,
                                                                  int64_t nvec, uint4* __restrict__ h) {
  for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
    float gf[8], uf[8];
    unpack_bf16x8(ld_stream_u4(g + v), gf);
    unpack_bf16x8(ld_stream_u4(u + v), uf);
#pragma unroll
    for (int e = 0; e < 8; ++e) gf[e] = bf16r(silu_f(gf[e])) * uf[e];
    h[v] = pack_bf16x8(gf);
  }
}

// du = bf16(dh * bf16(silu(g))),  dg = silu'(g) * bf16(dh * u)  (torch's silu_backward formula)
__global__ void __launch_bounds__(kFlatThreads) swiglu_bwd_kernel(const uint4* __restrict__ g, const uint4* __restrict__ u,
                                                                  const uint4* __restrict__ dh, int64_t nvec,
                                                                  uint4* __restrict__ dg, uint4* __restrict__ du) {
  for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < nvec; v += (int64_t)gridDim.x * blockDim.x) {
    float gf[8], uf[8], df[8], og[8], ou[8];
    unpack_bf16x8(ld_stream_u4(g + v), gf);
    unpack_bf16x8(ld_stream_u4(u + v), uf);
    unpack_bf16x8(ld_stream_u4(dh + v), df);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float x = gf[e];
      const float sig = 1.0f / (1.0f + expf(-x));
      ou[e] = df[e] * bf16r(x / (1.0f + expf(-x)));
      const float dy = bf16r(df[e] * uf[e]);
      og[e] = dy * sig * (1.0f + x * (1.0f - sig));
    }
    dg[v] = pack_bf16x8(og);
    du[v] = pack_bf16x8(ou);
  }
}

int flat_grid(int64_t items) {
  const int64_t want = (items + kFlatThreads - 1) / kFlatThreads;
  const int64_t cap = (int64_t)sm_count() * 16;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace
}  // namespace smt

using smt::aligned16;

extern "C" SMT_API int smt_rmsnorm_forward(const void* a, const void* res, const void* w, int64_t T, int H, float eps,
                                           void* h_out, void* y, float* rstd, void* stream) {
  SMT_CHECK_ARG(T >= 0 && H > 0 && H % 8 == 0 && H / 8 <= smt::kRowMaxVec * 1024,
                "smt_rmsnorm_forward: H = %d must be a positive multiple of 8 and <= %d", H, smt::kRowMaxVec * 8192);
  if (T == 0) return SMT_OK;
  SMT_CHECK_ARG(a && w && y && rstd && (!res || h_out), "smt_rmsnorm_forward: null pointer");
  SMT_CHECK_ARG(aligned16(a) && aligned16(w) && aligned16(y) && (!res || (aligned16(res) && aligned16(h_out))) &&
                    (uintptr_t)rstd % 4 == 0,
                "smt_rmsnorm_forward: tensors must be 16-byte aligned (rstd: 4-byte)");
  const int nvec = H / 8;
  const int threads = smt::row_threads(nvec);
  const float inv_n = 1.0f / (float)H;
  if (res)
    smt::rmsnorm_fwd_kernel<true><<<(unsigned)T, threads, 0, (cudaStream_t)stream>>>(
        (const uint4*)a, (const uint4*)res, (const uint4*)w, nvec, inv_n, eps, (uint4*)h_out, (uint4*)y, rstd);
  else
    smt::rmsnorm_fwd_kernel<false><<<(unsigned)T, threads, 0, (cudaStream_t)stream>>>(
        (const uint4*)a, nullptr, (const uint4*)w, nvec, inv_n, eps, nullptr, (uint4*)y, rstd);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_rmsnorm_backward(const void* x, const void* w, const float* rstd, const void* dy,
                                            const void* dres, int64_t T, int H, void* dx, void* stream) {
  SMT_CHECK_ARG(T >= 0 && H > 0 && H % 8 == 0 && H / 8 <= smt::kRowMaxVec * 1024,
                "smt_rmsnorm_backward: H = %d must be a positive multiple of 8 and <= %d", H, smt::kRowMaxVec * 8192);
  if (T == 0) return SMT_OK;
  SMT_CHECK_ARG(x && w && rstd && dy && dx, "smt_rmsnorm_backward: null pointer");
  SMT_CHECK_ARG(aligned16(x) && aligned16(w) && aligned16(dy) && aligned16(dx) && (!dres || aligned16(dres)) &&
                    (uintptr_t)rstd % 4 == 0,
                "smt_rmsnorm_backward: tensors must be 16-byte aligned (rstd: 4-byte)");
  const int nvec = H / 8;
  const int threads = smt::row_threads(nvec);
  const float inv_n = 1.0f / (float)H;
  if (dres)
    smt::rmsnorm_bwd_kernel<true><<<(unsigned)T, threads, 0, (cudaStream_t)stream>>>(
        (const uint4*)x, (const uint4*)w, rstd, (const uint4*)dy, (const uint4*)dres, nvec, inv_n, (uint4*)dx);
  else
    smt::rmsnorm_bwd_kernel<false><<<(unsigned)T, threads, 0, (cudaStream_t)stream>>>(
        (const uint4*)x, (const uint4*)w, rstd, (const uint4*)dy, nullptr, nvec, inv_n, (uint4*)dx);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

static int rope_launch(bool bwd, const void* q, const void* k, const void* cos_, const void* sin_, int B, int S, int Hq,
                       int Hk, int64_t cs_bstride, void* q_out, void* k_out, void* stream, const char* who) {
  SMT_CHECK_ARG(B >= 0 && S >= 0 && Hq >= 0 && Hk >= 0 && cs_bstride >= 0 && cs_bstride % 8 == 0,
                "%s: bad shape (B %d, S %d, Hq %d, Hk %d, cos/sin batch stride %lld)", who, B, S, Hq, Hk,
                (long long)cs_bstride);
  const int64_t rows_q = (int64_t)B * S * Hq, rows_k = (int64_t)B * S * Hk;
  if (rows_q + rows_k == 0) return SMT_OK;
  SMT_CHECK_ARG(cos_ && sin_ && (!rows_q || (q && q_out)) && (!rows_k || (k && k_out)), "%s: null pointer", who);
  SMT_CHECK_ARG(aligned16(cos_) && aligned16(sin_) && aligned16(q) && aligned16(k) && aligned16(q_out) &&
                    aligned16(k_out),
                "%s: tensors must be 16-byte aligned", who);
  const int grid = smt::flat_grid((rows_q + rows_k) * 8);
  auto kern = bwd ? smt::rope_kernel<true> : smt::rope_kernel<false>;
  kern<<<grid, smt::kFlatThreads, 0, (cudaStream_t)stream>>>((const uint4*)q, (const uint4*)k, (const uint4*)cos_,
                                                             (const uint4*)sin_, S, Hq > 0 ? Hq : 1, Hk > 0 ? Hk : 1,
                                                             rows_q, rows_k, cs_bstride / 8, (uint4*)q_out,
                                                             (uint4*)k_out);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_rope_forward(const void* q, const void* k, const void* cos_, const void* sin_, int B, int S,
                                        int Hq, int Hk, int64_t cs_bstride, void* q_out, void* k_out, void* stream) {
  return rope_launch(false, q, k, cos_, sin_, B, S, Hq, Hk, cs_bstride, q_out, k_out, stream, "smt_rope_forward");
}

extern "C" SMT_API int smt_rope_backward(const void* dq_out, const void* dk_out, const void* cos_, const void* sin_,
                                         int B, int S, int Hq, int Hk, int64_t cs_bstride, void* dq, void* dk,
                                         void* stream) {
  return rope_launch(true, dq_out, dk_out, cos_, sin_, B, S, Hq, Hk, cs_bstride, dq, dk, stream, "smt_rope_backward");
}

static int qk_norm_rope_launch(bool bwd, const void* a_q, const void* a_k, const void* x_q, const void* x_k,
                               const void* wq, const void* wk, float eps_q, float eps_k, const void* cos_,
                               const void* sin_, int B, int S, int Hq, int Hk, int64_t cs_bstride, float* rstd_q,
                               float* rstd_k, void* out_q, void* out_k, void* stream, const char* who) {
  SMT_CHECK_ARG(B >= 0 && S >= 0 && Hq >= 0 && Hk >= 0 && cs_bstride >= 0 && cs_bstride % 8 == 0,
                "%s: bad shape (B %d, S %d, Hq %d, Hk %d, cos/sin batch stride %lld)", who, B, S, Hq, Hk,
                (long long)cs_bstride);
  const int64_t rows_q = (int64_t)B * S * Hq, rows_k = (int64_t)B * S * Hk;
  if (rows_q + rows_k == 0) return SMT_OK;
  SMT_CHECK_ARG(cos_ && sin_ && (!rows_q || (a_q && wq && rstd_q && out_q && (!bwd || x_q))) &&
                    (!rows_k || (a_k && wk && rstd_k && out_k && (!bwd || x_k))),
                "%s: null pointer", who);
  SMT_CHECK_ARG(aligned16(cos_) && aligned16(sin_) && aligned16(a_q) && aligned16(a_k) && aligned16(x_q) &&
                    aligned16(x_k) && aligned16(wq) && aligned16(wk) && aligned16(out_q) && aligned16(out_k) &&
                    (uintptr_t)rstd_q % 4 == 0 && (uintptr_t)rstd_k % 4 == 0,
                "%s: tensors must be 16-byte aligned (rstd: 4-byte)", who);
  const int grid = smt::flat_grid((rows_q + rows_k) * 8);
  auto kern = bwd ? smt::qk_norm_rope_kernel<true> : smt::qk_norm_rope_kernel<false>;
  kern<<<grid, smt::kFlatThreads, 0, (cudaStream_t)stream>>>(
      (const uint4*)a_q, (const uint4*)a_k, (const uint4*)x_q, (const uint4*)x_k, (const uint4*)wq, (const uint4*)wk,
      eps_q, eps_k, (const uint4*)cos_, (const uint4*)sin_, S, Hq > 0 ? Hq : 1, Hk > 0 ? Hk : 1, rows_q, rows_k,
      cs_bstride / 8, rstd_q, rstd_k, (uint4*)out_q, (uint4*)out_k);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_qk_norm_rope_forward(const void* q, const void* k, const void* wq, const void* wk,
                                                float eps_q, float eps_k, const void* cos_, const void* sin_, int B,
                                                int S, int Hq, int Hk, int64_t cs_bstride, void* q_out, void* k_out,
                                                float* rstd_q, float* rstd_k, void* stream) {
  return qk_norm_rope_launch(false, q, k, nullptr, nullptr, wq, wk, eps_q, eps_k, cos_, sin_, B, S, Hq, Hk,
                             cs_bstride, rstd_q, rstd_k, q_out, k_out, stream, "smt_qk_norm_rope_forward");
}

extern "C" SMT_API int smt_qk_norm_rope_backward(const void* q, const void* k, const void* wq, const void* wk,
                                                 const float* rstd_q, const float* rstd_k, const void* cos_,
                                                 const void* sin_, const void* dq_out, const void* dk_out, int B,
                                                 int S, int Hq, int Hk, int64_t cs_bstride, void* dq, void* dk,
                                                 void* stream) {
  return qk_norm_rope_launch(true, dq_out, dk_out, q, k, wq, wk, 0.f, 0.f, cos_, sin_, B, S, Hq, Hk, cs_bstride,
                             const_cast<float*>(rstd_q), const_cast<float*>(rstd_k), dq, dk, stream,
                             "smt_qk_norm_rope_backward");
}

extern "C" SMT_API int smt_swiglu_forward(const void* g, const void* u, int64_t n, void* h, void* stream) {
  SMT_CHECK_ARG(n >= 0 && n % 8 == 0, "smt_swiglu_forward: n = %lld must be a multiple of 8", (long long)n);
  if (n == 0) return SMT_OK;
  SMT_CHECK_ARG(g && u && h, "smt_swiglu_forward: null pointer");
  SMT_CHECK_ARG(aligned16(g) && aligned16(u) && aligned16(h), "smt_swiglu_forward: tensors must be 16-byte aligned");
  smt::swiglu_fwd_kernel<<<smt::flat_grid(n / 8), smt::kFlatThreads, 0, (cudaStream_t)stream>>>(
      (const uint4*)g, (const uint4*)u, n / 8, (uint4*)h);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_swiglu_backward(const void* g, const void* u, const void* dh, int64_t n, void* dg, void* du,
                                           void* stream) {
  SMT_CHECK_ARG(n >= 0 && n % 8 == 0, "smt_swiglu_backward: n = %lld must be a multiple of 8", (long long)n);
  if (n == 0) return SMT_OK;
  SMT_CHECK_ARG(g && u && dh && dg && du, "smt_swiglu_backward: null pointer");
  SMT_CHECK_ARG(aligned16(g) && aligned16(u) && aligned16(dh) && aligned16(dg) && aligned16(du),
                "smt_swiglu_backward: tensors must be 16-byte aligned");
  smt::swiglu_bwd_kernel<<<smt::flat_grid(n / 8), smt::kFlatThreads, 0, (cudaStream_t)stream>>>(
      (const uint4*)g, (const uint4*)u, (const uint4*)dh, n / 8, (uint4*)dg, (uint4*)du);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}
