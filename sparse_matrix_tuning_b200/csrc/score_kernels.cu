// Warm-up scoring kernels (HBM-bound): elementwise fp32 accumulation of gradients, per-block
// signed-sum accumulation, block-score reduction with the four reference strategies, the factored
// block sums of a frozen-weight warm-up (token block sums + their outer product), and the
// activation (channel) scoring pair.
//
// Reference call sites replaced (paths relative to the reference root):
//   deepspeed/fine_tune.py:716-768   D2H copy + CPU `+=` of every q/k/v(/MLP) gradient
//   deepspeed/smt/smt_helper.py:55-78, 233-251   reshape to [R/b, b, C/b, b] and reduce dims (1,3)
//   (smt_token_block_sums + smt_block_outer_accumulate replace both of the above for `mean_abs`
//    without the weight gradient ever being formed)
//   deepspeed/fine_tune.py:649-678   activation hook (|x|, allreduce, D2H, `+=`)
//   deepspeed/smt/smt_helper.py:168-183   channel scores
#include "common.cuh"

namespace smt {
namespace {

constexpr int kThreads = 256;

// ---- acc += grad ---------------------------------------------------------------------------

constexpr int kScoreUnroll = 2;     // vec8 groups in flight per thread (measured best of {1, 2, 4}: profiles/r01_kernels.md)
constexpr int kScoreCtas = 4;       // grid cap in CTAs per SM for the streaming kernels (2 x 4 measured best: 6 125 GB/s)

template <int DT>
__device__ __forceinline__ void load_grad8(const void* __restrict__ grad, int64_t i, float (&g)[8]) {
  if (DT == SMT_F32) {
    const float4 a = ld_stream_f4(reinterpret_cast<const float4*>(grad) + 2 * i);
    const float4 b = ld_stream_f4(reinterpret_cast<const float4*>(grad) + 2 * i + 1);
    g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w;
    g[4] = b.x; g[5] = b.y; g[6] = b.z; g[7] = b.w;
  } else {
    unpack8<DT>(ld_stream_u4(reinterpret_cast<const uint4*>(grad) + i), g);
  }
}

template <int DT>
__global__ void __launch_bounds__(kThreads) score_accumulate_vec_kernel(
    float* __restrict__ acc, const void* __restrict__ grad, int64_t n_vec8) {
  // one "vec8" = 8 consecutive elements: 32 B of fp32 accumulator, 16 B (16-bit) or 32 B (fp32) of grad
  constexpr int U = kScoreUnroll;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + (U - 1) * stride < n_vec8; i += U * stride) {
    float g[U][8];
    float4 a0[U], a1[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {                       // all loads first: U x 48 B in flight per thread
      load_grad8<DT>(grad, i + u * stride, g[u]);
      const float4* ap = reinterpret_cast<const float4*>(acc) + 2 * (i + u * stride);
      a0[u] = ap[0];
      a1[u] = ap[1];
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float4* ap = reinterpret_cast<float4*>(acc) + 2 * (i + u * stride);
      a0[u].x += g[u][0]; a0[u].y += g[u][1]; a0[u].z += g[u][2]; a0[u].w += g[u][3];
      a1[u].x += g[u][4]; a1[u].y += g[u][5]; a1[u].z += g[u][6]; a1[u].w += g[u][7];
      ap[0] = a0[u];
      ap[1] = a1[u];
    }
  }
  for (; i < n_vec8; i += stride) {                     // remainder
    float g[8];
    load_grad8<DT>(grad, i, g);
    float4* ap = reinterpret_cast<float4*>(acc) + 2 * i;
    float4 a0 = ap[0], a1 = ap[1];
    a0.x += g[0]; a0.y += g[1]; a0.z += g[2]; a0.w += g[3];
    a1.x += g[4]; a1.y += g[5]; a1.z += g[6]; a1.w += g[7];
    ap[0] = a0;
    ap[1] = a1;
  }
}

template <int DT>
__global__ void __launch_bounds__(kThreads) score_accumulate_scalar_kernel(
    float* __restrict__ acc, const void* __restrict__ grad, int64_t begin, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    acc[i] += load_as_float<DT>(grad, i);
}

// ---- per-block reductions --------------------------------------------------------------------
// One CTA per b x b block.  A row of the block is contiguous (b*sizeof(T) bytes), so a group of
// b/VEC threads reads one row with 128-bit loads and the CTA walks down the rows.

enum { kSigned = 0, kAbs = 1, kSquare = 2 };

template <int MODE>
__device__ __forceinline__ float term(float x) {
  if (MODE == kSigned) return x;
  if (MODE == kAbs) return fabsf(x);
  return x * x;
}

template <int B, int DT, int MODE>
__device__ __forceinline__ float block_partial(const void* __restrict__ src, int64_t ld, int brow,
                                               int bcol) {
  constexpr int VEC = (DT == SMT_F32) ? 4 : 8;          // elements per 128-bit load
  constexpr int TPR = B / VEC;                          // threads per row
  constexpr int RPP = kThreads / TPR;                   // rows per pass
  constexpr int PASSES = B / RPP;
  constexpr int UNROLL = PASSES >= 4 ? 4 : PASSES;
  static_assert(kThreads % TPR == 0 && B % RPP == 0 && PASSES % UNROLL == 0, "tiling");
  const int tcol = threadIdx.x % TPR, trow = threadIdx.x / TPR;
  const char* base = reinterpret_cast<const char*>(src) +
                     ((int64_t)(brow * B + trow) * ld + (int64_t)bcol * B + tcol * VEC) *
                         (DT == SMT_F32 ? 4 : 2);
  const int64_t pass_stride = (int64_t)RPP * ld * (DT == SMT_F32 ? 4 : 2);
  float s0 = 0.f, s1 = 0.f;
#pragma unroll 1
  for (int p = 0; p < PASSES; p += UNROLL) {
    uint4 u[UNROLL];
#pragma unroll
    for (int j = 0; j < UNROLL; ++j) u[j] = ld_stream_u4(base + (int64_t)(p + j) * pass_stride);
#pragma unroll
    for (int j = 0; j < UNROLL; ++j) {
      if (DT == SMT_F32) {
        s0 += term<MODE>(__uint_as_float(u[j].x)) + term<MODE>(__uint_as_float(u[j].y));
        s1 += term<MODE>(__uint_as_float(u[j].z)) + term<MODE>(__uint_as_float(u[j].w));
      } else {
        float f[8];
        unpack8<DT>(u[j], f);
        s0 += (term<MODE>(f[0]) + term<MODE>(f[1])) + (term<MODE>(f[2]) + term<MODE>(f[3]));
        s1 += (term<MODE>(f[4]) + term<MODE>(f[5])) + (term<MODE>(f[6]) + term<MODE>(f[7]));
      }
    }
  }
  return s0 + s1;
}

template <int B, int MODE>
__global__ void __launch_bounds__(kThreads) block_score_reduce_kernel(
    const float* __restrict__ acc, int64_t ld, int strategy, float* __restrict__ scores) {
  __shared__ float scratch[32];
  const int bcol = blockIdx.x, brow = blockIdx.y;
  float s = block_partial<B, SMT_F32, MODE>(acc, ld, brow, bcol);
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) {
    const float cnt = (float)(B * B);
    float r;
    if (strategy == SMT_MEAN_ABS) r = fabsf(s / cnt);
    else if (strategy == SMT_ABS_MEAN) r = s / cnt;
    else if (strategy == SMT_L1) r = s;
    else r = sqrtf(s);
    scores[(int64_t)brow * gridDim.x + bcol] = r;
  }
}

template <int B, int DT>
__global__ void __launch_bounds__(kThreads) block_sum_accumulate_kernel(
    float* __restrict__ sums, const void* __restrict__ grad, int64_t ld) {
  __shared__ float scratch[32];
  const int bcol = blockIdx.x, brow = blockIdx.y;
  float s = block_partial<B, DT, kSigned>(grad, ld, brow, bcol);
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) sums[(int64_t)brow * gridDim.x + bcol] += s;
}

__global__ void block_sum_finalize_kernel(const float* __restrict__ sums, float* __restrict__ scores,
                                          int64_t n, float cnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) scores[i] = fabsf(sums[i] / cnt);
}

// ---- activation scoring ------------------------------------------------------------------------

template <int DT>
__global__ void __launch_bounds__(kThreads) act_score_accumulate_kernel(
    float* __restrict__ acc, const void* __restrict__ x, int batch, int64_t sc_vec8) {
  // sc_vec8 = S*C/8 vectors per batch entry
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < sc_vec8; i += stride) {
    float s[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = 0; b < batch; ++b) {
      float g[8];
      if (DT == SMT_F32) {
        const float4* p = reinterpret_cast<const float4*>(x) + 2 * ((int64_t)b * sc_vec8 + i);
        const float4 a = ld_stream_f4(p), c = ld_stream_f4(p + 1);
        g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w;
        g[4] = c.x; g[5] = c.y; g[6] = c.z; g[7] = c.w;
      } else {
        const uint4 u = ld_stream_u4(reinterpret_cast<const uint4*>(x) + (int64_t)b * sc_vec8 + i);
        unpack8<DT>(u, g);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) s[j] += fabsf(g[j]);
    }
    float4* ap = reinterpret_cast<float4*>(acc) + 2 * i;
    float4 a0 = ap[0], a1 = ap[1];
    a0.x += s[0]; a0.y += s[1]; a0.z += s[2]; a0.w += s[3];
    a1.x += s[4]; a1.y += s[5]; a1.z += s[6]; a1.w += s[7];
    ap[0] = a0;
    ap[1] = a1;
  }
}

// out[c] over rows of acc[S, C]; CTA = 32 column-quads x 8 row lanes.
__global__ void __launch_bounds__(kThreads) channel_score_reduce_kernel(
    const float* __restrict__ acc, int seq, int channels, int strategy, float* __restrict__ out) {
  __shared__ float4 part[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c4 = blockIdx.x * 32 + tx;  // column quad
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 * 4 < channels) {
    for (int r = ty; r < seq; r += 8) {
      const float4 v = *reinterpret_cast<const float4*>(acc + (int64_t)r * channels + c4 * 4);
      if (strategy == SMT_L2) {
        s.x += v.x * v.x; s.y += v.y * v.y; s.z += v.z * v.z; s.w += v.w * v.w;
      } else if (strategy == SMT_ABS_MEAN) {
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      } else {
        s.x += fabsf(v.x); s.y += fabsf(v.y); s.z += fabsf(v.z); s.w += fabsf(v.w);
      }
    }
  }
  part[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c4 * 4 < channels) {
    float4 t = part[0][tx];
#pragma unroll
    for (int j = 1; j < 8; ++j) {
      t.x += part[j][tx].x; t.y += part[j][tx].y; t.z += part[j][tx].z; t.w += part[j][tx].w;
    }
    const float cnt = (float)seq;
    if (strategy == SMT_MEAN_ABS) { t.x /= cnt; t.y /= cnt; t.z /= cnt; t.w /= cnt; }
    else if (strategy == SMT_ABS_MEAN) {
      t.x = fabsf(t.x / cnt); t.y = fabsf(t.y / cnt); t.z = fabsf(t.z / cnt); t.w = fabsf(t.w / cnt);
    } else if (strategy == SMT_L2) {
      t.x = sqrtf(t.x); t.y = sqrtf(t.y); t.z = sqrtf(t.z); t.w = sqrtf(t.w);
    }
    *reinterpret_cast<float4*>(out + c4 * 4) = t;
  }
}

// ---- factored block sums (frozen-weight warm-up) -------------------------------------------------
// For y = x W^T the signed sum of block (r, c) of dW factors over tokens:
//   sum_{o in r, k in c} dW[o, k] = sum_t Dy[t, r] * X[t, c],  Dy / X = per-token segment sums of dy / x.
// token_block_sums_kernel makes Dy and X (one read of the activation), block_outer_* contracts them.

constexpr int kTbsUnroll = 4;       // segment groups in flight per thread

// out[t, j] = sum_{k < B} src[t, j*B + k].  L lanes of a warp share one segment (L = min(vectors per segment, 32)),
// each lane loads P = vectors / L 128-bit vectors of it; the lane sums run in a fixed order, then an xor butterfly over
// the L lanes.  The arithmetic of a segment never depends on which warp handles it, so any grid gives the same bits.
template <int B, int DT>
__global__ void __launch_bounds__(kThreads) token_block_sums_kernel(
    const void* __restrict__ src, int64_t ld, int64_t T, int seg_per_row, float* __restrict__ out) {
  constexpr int ES = DT == SMT_F32 ? 4 : 2;
  constexpr int VEC = 16 / ES;                          // elements per 128-bit vector
  constexpr int NV = B / VEC;                           // vectors per segment: 8 .. 64
  constexpr int L = NV < 32 ? NV : 32;                  // lanes per segment
  constexpr int P = NV / L;                             // vectors per lane per segment
  constexpr int SPW = 32 / L;                           // segments per warp and group
  constexpr int U = kTbsUnroll;
  const int lane = threadIdx.x & 31, sub = lane / L, l = lane % L;
  const int64_t n_seg = T * seg_per_row;
  const int64_t n_groups = (n_seg + SPW - 1) / SPW;
  const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
  const char* base = reinterpret_cast<const char*>(src);
  for (int64_t g0 = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g0 < n_groups; g0 += U * warps) {
    uint4 v[U][P];
#pragma unroll
    for (int u = 0; u < U; ++u) {                       // all loads first: U x P x 16 B in flight per lane
      const int64_t s = (g0 + u * warps) * SPW + sub;
      const bool ok = s < n_seg;
      int64_t t = 0, j = 0;
      if (ok && n_seg <= 0xffffffffll) {                 // 32-bit division is far cheaper than 64-bit
        t = (uint32_t)s / (uint32_t)seg_per_row;
        j = (uint32_t)s - (uint32_t)t * (uint32_t)seg_per_row;
      } else if (ok) {
        t = s / seg_per_row;
        j = s - t * seg_per_row;
      }
      const char* p = base + (t * ld + j * B) * ES + (int64_t)l * 16;
#pragma unroll
      for (int q = 0; q < P; ++q) v[u][q] = ok ? ld_stream_u4(p + q * L * 16) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      float acc = 0.f;
#pragma unroll
      for (int q = 0; q < P; ++q) {
        if (DT == SMT_F32) {
          acc += (__uint_as_float(v[u][q].x) + __uint_as_float(v[u][q].y)) +
                 (__uint_as_float(v[u][q].z) + __uint_as_float(v[u][q].w));
        } else {
          float f[8];
          unpack8<DT>(v[u][q], f);
          acc += ((f[0] + f[1]) + (f[2] + f[3])) + ((f[4] + f[5]) + (f[6] + f[7]));
        }
      }
#pragma unroll
      for (int o = L / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      const int64_t s = (g0 + u * warps) * SPW + sub;
      if (l == 0 && s < n_seg) out[s] = acc;
    }
  }
}

// Tokens per partial of block_outer_accumulate: a fixed partition of T (independent of the device), so the sums are
// bit-identical on every GPU and from run to run.  (Chunks of 512 tokens with four fma chains measured slower: 25-27 us
// against 15-19 us at T = 8 192, fewer CTAs each waiting on two staging rounds.)
constexpr int kOuterChunk = 128;
constexpr int kOuterTile = 16;                          // 16 x 16 outputs per CTA, one per thread

// part[k, r, c] = sum over the tokens of chunk k of dy[t, r] * x[t, c], tokens in increasing order.
__global__ void __launch_bounds__(kThreads) block_outer_partial_kernel(
    const float* __restrict__ dy, const float* __restrict__ x, int64_t T, int rb, int cb, float* __restrict__ part) {
  __shared__ float sdy[kOuterChunk][kOuterTile];
  __shared__ float sx[kOuterChunk][kOuterTile];
  const int64_t t0 = (int64_t)blockIdx.x * kOuterChunk;
  const int c0 = blockIdx.y * kOuterTile, r0 = blockIdx.z * kOuterTile;
  for (int i = threadIdx.x; i < kOuterChunk * kOuterTile; i += kThreads) {
    const int tt = i / kOuterTile, k = i % kOuterTile;
    const int64_t t = t0 + tt;
    sdy[tt][k] = (t < T && r0 + k < rb) ? dy[t * rb + r0 + k] : 0.f;
    sx[tt][k] = (t < T && c0 + k < cb) ? x[t * cb + c0 + k] : 0.f;
  }
  __syncthreads();
  const int ty = threadIdx.x / kOuterTile, tx = threadIdx.x % kOuterTile;
  float acc = 0.f;
#pragma unroll 8
  for (int tt = 0; tt < kOuterChunk; ++tt) acc = fmaf(sdy[tt][ty], sx[tt][tx], acc);
  const int r = r0 + ty, c = c0 + tx;
  if (r < rb && c < cb) part[((int64_t)blockIdx.x * rb + r) * cb + c] = acc;
}

// block_sums[i] += sum_k part[k, i], k in increasing order (loads issued 8 at a time, the sum stays sequential).
__global__ void __launch_bounds__(kThreads) block_outer_reduce_kernel(
    const float* __restrict__ part, int64_t n_chunks, int64_t n, float* __restrict__ block_sums) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  int64_t k = 0;
  for (; k + 8 <= n_chunks; k += 8) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = part[(k + j) * n + i];
#pragma unroll
    for (int j = 0; j < 8; ++j) s += v[j];
  }
  for (; k < n_chunks; ++k) s += part[k * n + i];
  block_sums[i] += s;
}

// One wave: at most as many CTAs as can be resident, so no CTA of a second partial wave runs its grid-stride loop
// after the others have finished (the launches are 10-60 us long, so a tail wave is a large fraction of them).
template <int B, int DT>
void launch_token_block_sums(const void* src, int64_t ld, int64_t T, int seg_per_row, float* out, int64_t want,
                             cudaStream_t st) {
  static int per_sm = 0;
  if (per_sm == 0) {
    int o = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, token_block_sums_kernel<B, DT>, kThreads, 0) != cudaSuccess ||
        o <= 0)
      o = 4;
    per_sm = o;
  }
  const int64_t cap = (int64_t)sm_count() * per_sm;
  const int grid = (int)(want < cap ? want : cap);
  token_block_sums_kernel<B, DT><<<grid, kThreads, 0, st>>>(src, ld, T, seg_per_row, out);
}

inline int streaming_grid(int64_t work_items) {
  // enough CTAs for ~8 resident per SM, capped by the work
  int64_t want = (work_items + kThreads - 1) / kThreads;
  int64_t cap = (int64_t)sm_count() * kScoreCtas;
  return (int)(want < cap ? (want < 1 ? 1 : want) : cap);
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API int smt_score_accumulate(float* acc, const void* grad, int grad_dtype, int64_t n,
                                    void* stream) {
  SMT_CHECK_ARG(acc && grad, "smt_score_accumulate: null pointer");
  SMT_CHECK_ARG(n >= 0, "smt_score_accumulate: n < 0");
  SMT_CHECK_ARG(grad_dtype >= SMT_F32 && grad_dtype <= SMT_F16, "smt_score_accumulate: bad dtype %d",
                grad_dtype);
  if (n == 0) return SMT_OK;
  cudaStream_t st = (cudaStream_t)stream;
  int64_t n_vec = (aligned16(acc) && aligned16(grad)) ? n / 8 : 0;
  if (n_vec > 0) {
    int grid = streaming_grid(n_vec);
    if (grad_dtype == SMT_F32) score_accumulate_vec_kernel<SMT_F32><<<grid, kThreads, 0, st>>>(acc, grad, n_vec);
    else if (grad_dtype == SMT_BF16) score_accumulate_vec_kernel<SMT_BF16><<<grid, kThreads, 0, st>>>(acc, grad, n_vec);
    else score_accumulate_vec_kernel<SMT_F16><<<grid, kThreads, 0, st>>>(acc, grad, n_vec);
    SMT_CHECK_LAUNCH();
  }
  if (n_vec * 8 < n) {
    int grid = streaming_grid(n - n_vec * 8);
    if (grad_dtype == SMT_F32) score_accumulate_scalar_kernel<SMT_F32><<<grid, kThreads, 0, st>>>(acc, grad, n_vec * 8, n);
    else if (grad_dtype == SMT_BF16) score_accumulate_scalar_kernel<SMT_BF16><<<grid, kThreads, 0, st>>>(acc, grad, n_vec * 8, n);
    else score_accumulate_scalar_kernel<SMT_F16><<<grid, kThreads, 0, st>>>(acc, grad, n_vec * 8, n);
    SMT_CHECK_LAUNCH();
  }
  return SMT_OK;
}

namespace {
int check_blocked(const char* who, const void* p, int rows, int cols, int64_t ld, int block, int elem_bytes) {
  SMT_CHECK_ARG(p != nullptr, "%s: null pointer", who);
  SMT_CHECK_ARG(block_ok(block), "%s: block size %d not in {64,128,256}", who, block);
  SMT_CHECK_ARG(rows > 0 && cols > 0 && rows % block == 0 && cols % block == 0,
                "%s: matrix %dx%d is not a multiple of block %d", who, rows, cols, block);
  SMT_CHECK_ARG(ld >= cols, "%s: ld %lld < cols %d", who, (long long)ld, cols);
  SMT_CHECK_ARG(aligned16(p) && (ld * elem_bytes) % 16 == 0, "%s: matrix must be 16-byte aligned (ptr and row pitch)", who);
  SMT_CHECK_ARG(rows / block <= 65535, "%s: too many block rows", who);
  return SMT_OK;
}
}  // namespace

extern "C" SMT_API int smt_block_score_reduce(const float* acc, int rows, int cols, int64_t ld, int block,
                                      int strategy, float* scores, void* stream) {
  if (int rc = check_blocked("smt_block_score_reduce", acc, rows, cols, ld, block, 4)) return rc;
  SMT_CHECK_ARG(scores != nullptr, "smt_block_score_reduce: null scores");
  SMT_CHECK_ARG(strategy >= SMT_MEAN_ABS && strategy <= SMT_L2, "smt_block_score_reduce: unknown strategy %d", strategy);
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(cols / block, rows / block);
  const int mode = strategy == SMT_MEAN_ABS ? kSigned : (strategy == SMT_L2 ? kSquare : kAbs);
#define SMT_LAUNCH_REDUCE(B)                                                                       \
  do {                                                                                             \
    if (mode == kSigned) block_score_reduce_kernel<B, kSigned><<<grid, kThreads, 0, st>>>(acc, ld, strategy, scores); \
    else if (mode == kAbs) block_score_reduce_kernel<B, kAbs><<<grid, kThreads, 0, st>>>(acc, ld, strategy, scores);  \
    else block_score_reduce_kernel<B, kSquare><<<grid, kThreads, 0, st>>>(acc, ld, strategy, scores);                 \
  } while (0)
  if (block == 256) SMT_LAUNCH_REDUCE(256);
  else if (block == 128) SMT_LAUNCH_REDUCE(128);
  else SMT_LAUNCH_REDUCE(64);
#undef SMT_LAUNCH_REDUCE
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_block_sum_accumulate(float* block_sums, const void* grad, int grad_dtype, int rows,
                                        int cols, int64_t ld, int block, void* stream) {
  SMT_CHECK_ARG(grad_dtype >= SMT_F32 && grad_dtype <= SMT_F16, "smt_block_sum_accumulate: bad dtype %d", grad_dtype);
  if (int rc = check_blocked("smt_block_sum_accumulate", grad, rows, cols, ld, block, dtype_bytes(grad_dtype))) return rc;
  SMT_CHECK_ARG(block_sums != nullptr, "smt_block_sum_accumulate: null block_sums");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(cols / block, rows / block);
#define SMT_LAUNCH_BS(B)                                                                                      \
  do {                                                                                                        \
    if (grad_dtype == SMT_F32) block_sum_accumulate_kernel<B, SMT_F32><<<grid, kThreads, 0, st>>>(block_sums, grad, ld);   \
    else if (grad_dtype == SMT_BF16) block_sum_accumulate_kernel<B, SMT_BF16><<<grid, kThreads, 0, st>>>(block_sums, grad, ld); \
    else block_sum_accumulate_kernel<B, SMT_F16><<<grid, kThreads, 0, st>>>(block_sums, grad, ld);            \
  } while (0)
  if (block == 256) SMT_LAUNCH_BS(256);
  else if (block == 128) SMT_LAUNCH_BS(128);
  else SMT_LAUNCH_BS(64);
#undef SMT_LAUNCH_BS
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_block_sum_finalize(const float* block_sums, float* scores, int64_t n, int block,
                                      void* stream) {
  SMT_CHECK_ARG(block_sums && scores, "smt_block_sum_finalize: null pointer");
  SMT_CHECK_ARG(block_ok(block), "smt_block_sum_finalize: bad block %d", block);
  if (n <= 0) return SMT_OK;
  int grid = (int)((n + 255) / 256);
  block_sum_finalize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(block_sums, scores, n, (float)(block * block));
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_token_block_sums(const void* src, int dtype, int64_t T, int F, int64_t ld, int block,
                                            float* out, void* stream) {
  SMT_CHECK_ARG(T >= 0 && F >= 0, "smt_token_block_sums: negative size (T = %lld, F = %d)", (long long)T, F);
  SMT_CHECK_ARG(dtype >= SMT_F32 && dtype <= SMT_F16, "smt_token_block_sums: bad dtype %d", dtype);
  SMT_CHECK_ARG(block_ok(block), "smt_token_block_sums: block size %d not in {64,128,256}", block);
  SMT_CHECK_ARG(F % block == 0, "smt_token_block_sums: F = %d is not a multiple of block %d", F, block);
  if (T == 0 || F == 0) return SMT_OK;
  SMT_CHECK_ARG(src && out, "smt_token_block_sums: null pointer");
  SMT_CHECK_ARG(ld >= F, "smt_token_block_sums: ld %lld < F %d", (long long)ld, F);
  SMT_CHECK_ARG(aligned16(src) && (ld * dtype_bytes(dtype)) % 16 == 0,
                "smt_token_block_sums: src must be 16-byte aligned (ptr and row pitch)");
  SMT_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 3u) == 0, "smt_token_block_sums: out must be 4-byte aligned");
  const int seg_per_row = F / block;
  const int vec = dtype == SMT_F32 ? 4 : 8;
  const int lanes = block / vec < 32 ? block / vec : 32;
  const int64_t groups = (T * seg_per_row + 32 / lanes - 1) / (32 / lanes);   // one warp per group
  const int64_t want = (groups + (kThreads / 32) * kTbsUnroll - 1) / ((kThreads / 32) * kTbsUnroll);
  cudaStream_t st = (cudaStream_t)stream;
#define SMT_LAUNCH_TBS(B)                                                                                            \
  do {                                                                                                               \
    if (dtype == SMT_F32) launch_token_block_sums<B, SMT_F32>(src, ld, T, seg_per_row, out, want, st);              \
    else if (dtype == SMT_BF16) launch_token_block_sums<B, SMT_BF16>(src, ld, T, seg_per_row, out, want, st);       \
    else launch_token_block_sums<B, SMT_F16>(src, ld, T, seg_per_row, out, want, st);                               \
  } while (0)
  if (block == 256) SMT_LAUNCH_TBS(256);
  else if (block == 128) SMT_LAUNCH_TBS(128);
  else SMT_LAUNCH_TBS(64);
#undef SMT_LAUNCH_TBS
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API size_t smt_block_outer_accumulate_workspace_bytes(int64_t T, int rb, int cb) {
  if (T <= 0 || rb <= 0 || cb <= 0) return 0;
  return (size_t)((T + kOuterChunk - 1) / kOuterChunk) * (size_t)rb * (size_t)cb * sizeof(float);
}

extern "C" SMT_API int smt_block_outer_accumulate(float* block_sums, const float* dy_sums, const float* x_sums,
                                                  int64_t T, int rb, int cb, void* workspace, size_t workspace_bytes,
                                                  void* stream) {
  SMT_CHECK_ARG(T >= 0 && rb >= 0 && cb >= 0, "smt_block_outer_accumulate: negative size (T = %lld, rb = %d, cb = %d)",
                (long long)T, rb, cb);
  if (T == 0 || rb == 0 || cb == 0) return SMT_OK;
  SMT_CHECK_ARG(block_sums && dy_sums && x_sums && workspace, "smt_block_outer_accumulate: null pointer");
  SMT_CHECK_ARG(((reinterpret_cast<uintptr_t>(block_sums) | reinterpret_cast<uintptr_t>(dy_sums) |
                  reinterpret_cast<uintptr_t>(x_sums) | reinterpret_cast<uintptr_t>(workspace)) & 3u) == 0,
                "smt_block_outer_accumulate: pointers must be 4-byte aligned");
  const int64_t n_chunks = (T + kOuterChunk - 1) / kOuterChunk;
  const size_t need = smt_block_outer_accumulate_workspace_bytes(T, rb, cb);
  if (workspace_bytes < need) {
    ::smt::set_error("smt_block_outer_accumulate: workspace %zu B < %zu B", workspace_bytes, need);
    return SMT_ERR_WORKSPACE;
  }
  const int tiles_c = (cb + kOuterTile - 1) / kOuterTile, tiles_r = (rb + kOuterTile - 1) / kOuterTile;
  SMT_CHECK_ARG(n_chunks <= 0x7fffffff && tiles_c <= 65535 && tiles_r <= 65535, "smt_block_outer_accumulate: too large");
  cudaStream_t st = (cudaStream_t)stream;
  float* part = static_cast<float*>(workspace);
  block_outer_partial_kernel<<<dim3((unsigned)n_chunks, tiles_c, tiles_r), kThreads, 0, st>>>(dy_sums, x_sums, T, rb,
                                                                                               cb, part);
  SMT_CHECK_LAUNCH();
  const int64_t n = (int64_t)rb * cb;
  block_outer_reduce_kernel<<<(unsigned)((n + kThreads - 1) / kThreads), kThreads, 0, st>>>(part, n_chunks, n,
                                                                                           block_sums);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_act_score_accumulate(float* acc, const void* x, int x_dtype, int batch, int seq,
                                        int channels, void* stream) {
  SMT_CHECK_ARG(acc && x, "smt_act_score_accumulate: null pointer");
  SMT_CHECK_ARG(x_dtype >= SMT_F32 && x_dtype <= SMT_F16, "smt_act_score_accumulate: bad dtype %d", x_dtype);
  SMT_CHECK_ARG(batch > 0 && seq > 0 && channels > 0, "smt_act_score_accumulate: empty input");
  SMT_CHECK_ARG(channels % 8 == 0 && aligned16(acc) && aligned16(x), "smt_act_score_accumulate: channels must be a multiple of 8 and pointers 16-byte aligned");
  const int64_t sc_vec8 = (int64_t)seq * channels / 8;
  int grid = streaming_grid(sc_vec8);
  cudaStream_t st = (cudaStream_t)stream;
  if (x_dtype == SMT_F32) act_score_accumulate_kernel<SMT_F32><<<grid, kThreads, 0, st>>>(acc, x, batch, sc_vec8);
  else if (x_dtype == SMT_BF16) act_score_accumulate_kernel<SMT_BF16><<<grid, kThreads, 0, st>>>(acc, x, batch, sc_vec8);
  else act_score_accumulate_kernel<SMT_F16><<<grid, kThreads, 0, st>>>(acc, x, batch, sc_vec8);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_channel_score_reduce(const float* acc, int seq, int channels, int strategy,
                                        float* out, void* stream) {
  SMT_CHECK_ARG(acc && out, "smt_channel_score_reduce: null pointer");
  SMT_CHECK_ARG(seq > 0 && channels > 0 && channels % 4 == 0, "smt_channel_score_reduce: channels must be a positive multiple of 4");
  SMT_CHECK_ARG(aligned16(acc) && aligned16(out), "smt_channel_score_reduce: pointers must be 16-byte aligned");
  SMT_CHECK_ARG(strategy >= SMT_MEAN_ABS && strategy <= SMT_L2, "smt_channel_score_reduce: unknown strategy %d", strategy);
  int grid = (channels / 4 + 31) / 32;
  channel_score_reduce_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(acc, seq, channels, strategy, out);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}
