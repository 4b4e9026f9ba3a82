// Causal-LM cross-entropy over rows of bf16 logits, with the gradient written over the logits (the loss of
// transformers' ForCausalLMLoss for one chunk of rows, and the input gradient its autograd graph would produce).
//
// One CTA per row, two passes over the row:
//   1. online (max, sum of exp) per thread, merged across the CTA in a fixed order;
//   2. g = scale * exp(x - lse) - scale * [v == y], written in place.
// A row is V * 2 bytes (256 KB at V = 128 256).  The CTAs resident at one time (2 per SM) hold about 76 MB of rows, well
// under the 126 MB L2, so the second pass is meant to read the row from L2: each logit crosses HBM once in and once out.
// No atomics and a fixed reduction order: results are identical run to run and do not depend on how the rows are
// chunked.  The fp32 steps copy ATen's log_softmax forward and backward epilogues (out = (x - m) - log(s),
// g = gO - exp(out) * sum(gO)), with `_rn` intrinsics where contraction would change bits.  The two exponentials per
// logit use `__expf` (ex2.approx after one multiply, about 1e-6 relative at the arguments that matter) rather than
// ATen's full-precision expf: with expf the kernel was instruction-bound at 0.52 of HBM peak
// (profiles/r04_causal_lm_loss.md), and the difference is far below the one bf16 rounding of the gradient.
#include "common.cuh"

namespace smt {
namespace {

constexpr int kCeThreads = 512;
constexpr int kCeUnroll = 4;         // 16-byte vectors in flight per thread and iteration

__device__ __forceinline__ void merge_ms(float& m, float& s, float m2, float s2) {
  const float mn = fmaxf(m, m2);
  if (mn == -INFINITY) return;       // both empty (or all -inf): keep (-inf, 0)
  s = s * expf(m - mn) + s2 * expf(m2 - mn);
  m = mn;
}

__global__ void __launch_bounds__(kCeThreads, 2) ce_rows_kernel(uint16_t* __restrict__ logits, int64_t ldl, int V,
                                                                 const int64_t* __restrict__ labels, int64_t ignore_index,
                                                                 const float* __restrict__ scale_p,
                                                                 float* __restrict__ loss_rows) {
  __shared__ float red_m[kCeThreads / 32], red_s[kCeThreads / 32];
  __shared__ float row_stat[2];      // the row's max and log(sum of exp)
  const int64_t row = blockIdx.x;
  uint4* xr = reinterpret_cast<uint4*>(logits + row * ldl);
  const int nvec = V / 8;
  const int64_t y = labels[row];

  if (y == ignore_index) {           // whole row 0, loss 0; the logits are never read
    for (int v = threadIdx.x; v < nvec; v += kCeThreads) xr[v] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) loss_rows[row] = 0.f;
    return;
  }
  const bool bad = y < 0 || y >= V;

  // ---- pass 1: online max / sum of exp ----
  float m = -INFINITY, s = 0.f;
  for (int v0 = threadIdx.x; v0 < nvec; v0 += kCeUnroll * kCeThreads) {
    uint4 u[kCeUnroll];
#pragma unroll
    for (int i = 0; i < kCeUnroll; ++i) {
      const int v = v0 + i * kCeThreads;
      if (v < nvec) u[i] = xr[v];
    }
#pragma unroll
    for (int i = 0; i < kCeUnroll; ++i) {
      if (v0 + i * kCeThreads < nvec) {
        float f[8];
        unpack8<SMT_BF16>(u[i], f);
        float vm = f[0];
#pragma unroll
        for (int e = 1; e < 8; ++e) vm = fmaxf(vm, f[e]);
        if (vm > m) {
          s = (m == -INFINITY) ? 0.f : s * expf(m - vm);
          m = vm;
        }
        if (m != -INFINITY) {
#pragma unroll
          for (int e = 0; e < 8; ++e) s += __expf(__fsub_rn(f[e], m));
        }
      }
    }
  }
  // fixed-order merge: butterfly within the warp, then warp 0 over the warps in index order
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    merge_ms(m, s, m2, s2);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    red_m[warp] = m;
    red_s[warp] = s;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float mt = red_m[0], st = red_s[0];
    for (int w = 1; w < kCeThreads / 32; ++w) merge_ms(mt, st, red_m[w], red_s[w]);
    const float logs = logf(st);
    row_stat[0] = mt;
    row_stat[1] = logs;
    // x[y] is read before any thread of this CTA overwrites the row (the barrier below orders it)
    const float xy = bad ? 0.f : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(logits)[row * ldl + y]);
    const float out_y = __fsub_rn(__fsub_rn(xy, mt), logs);                 // log_softmax(x)[y]
    loss_rows[row] = bad ? __int_as_float(0x7fc00000) : -out_y;
  }
  __syncthreads();

  // ---- pass 2: g = scale * exp(out) - scale * [v == y], in place ----
  const float mt = row_stat[0], logs = row_stat[1];
  const float scale = bad ? __int_as_float(0x7fc00000) : *scale_p;
  const float neg_scale = -scale;
  const int yi = bad ? -1 : (int)y;
  for (int v0 = threadIdx.x; v0 < nvec; v0 += kCeUnroll * kCeThreads) {
    uint4 u[kCeUnroll];
#pragma unroll
    for (int i = 0; i < kCeUnroll; ++i) {
      const int v = v0 + i * kCeThreads;
      if (v < nvec) u[i] = xr[v];
    }
#pragma unroll
    for (int i = 0; i < kCeUnroll; ++i) {
      const int v = v0 + i * kCeThreads;
      if (v < nvec) {
        float f[8];
        unpack8<SMT_BF16>(u[i], f);
        const int c0 = v * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float out = __fsub_rn(__fsub_rn(f[e], mt), logs);
          const float go = (c0 + e == yi) ? neg_scale : 0.f;                // nll_loss backward: -scale at the label
          f[e] = __fmaf_rn(-__expf(out), neg_scale, go);                    // gO - exp(out) * sum(gO), sum(gO) = -scale
        }
        xr[v] = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]),
                           pack_bf16x2(f[6], f[7]));
      }
    }
  }
}

}  // namespace
}  // namespace smt

extern "C" SMT_API int smt_cross_entropy_rows(void* logits, int64_t ldl, int64_t T, int V, const int64_t* labels,
                                              int64_t ignore_index, const float* scale, float* loss_rows,
                                              void* stream) {
  SMT_CHECK_ARG(V > 0 && V % 8 == 0, "smt_cross_entropy_rows: V = %d must be a positive multiple of 8", V);
  SMT_CHECK_ARG(T >= 0 && T < (1ll << 31), "smt_cross_entropy_rows: bad row count %lld", (long long)T);
  SMT_CHECK_ARG(ldl >= V && ldl % 8 == 0, "smt_cross_entropy_rows: row pitch %lld must be >= V and a multiple of 8",
                (long long)ldl);
  if (T == 0) return SMT_OK;
  SMT_CHECK_ARG(logits && labels && scale && loss_rows, "smt_cross_entropy_rows: null pointer");
  SMT_CHECK_ARG((reinterpret_cast<uintptr_t>(logits) & 15u) == 0, "smt_cross_entropy_rows: logits must be 16-byte aligned");
  smt::ce_rows_kernel<<<(unsigned)T, smt::kCeThreads, 0, (cudaStream_t)stream>>>(
      (uint16_t*)logits, ldl, V, labels, ignore_index, scale, loss_rows);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}
