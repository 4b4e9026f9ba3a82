// Compact AdamW step fused with gradient clipping and dense write-back, plus the deterministic
// sum-of-squares reduction that feeds the clip.  HBM-bound: 28 B/element with bf16 grads and bf16 W
// (grad 2 + master 4r/4w + m 4r/4w + v 4r/4w + W 2w), 30 B when a compact bf16 copy is also written.
//
// Reference call sites replaced:
//   deepspeed/fine_tune.py:352-363, 379-384, 773   FusedAdam(betas=(0.9,0.95)) stepped by the DeepSpeed
//       engine (bf16 params, fp32 masters, gradient_clipping 1.0 — helpers/deepspeed_helpers.py:87).
//       DeepSpeed itself is not vendored in the reference; the arithmetic below restates the published
//       multi_tensor_adam "adam_w_mode" update (see oracle/smt_oracle.py: adamw_fused_step).
//   deepspeed/smt/smt.py:332-341   the per-forward scatter of updated blocks into the dense weight —
//       done here, once per step, by the same kernel that produced the values.
//   deepspeed/smt/smt.py:208-211   the same for channel sparsity (weight columns here, see smt_column_scatter):
//       compact_adam_columns_kernel, the same per-element arithmetic (adam_update) with a column write-back.
//
// All floating-point operations use the *_rn intrinsics so nvcc cannot contract them into FMAs: the
// fp32 state after a step is bit-identical to the numpy restatement in oracle/.
#include "common.cuh"

namespace smt {
namespace {

constexpr int kAdamThreads = 256;
constexpr int kSqPartials = 1024;  // stage-1 partial sums (<= 4 KiB of floats)

template <int GDT>
__device__ __forceinline__ void load8(const void* p, int64_t vec, float (&g)[8]) {
  if (GDT == SMT_F32) {
    const float4 a = ld_stream_f4(reinterpret_cast<const float4*>(p) + 2 * vec);
    const float4 b = ld_stream_f4(reinterpret_cast<const float4*>(p) + 2 * vec + 1);
    g[0] = a.x; g[1] = a.y; g[2] = a.z; g[3] = a.w;
    g[4] = b.x; g[5] = b.y; g[6] = b.z; g[7] = b.w;
  } else {
    unpack8<GDT>(ld_stream_u4(reinterpret_cast<const uint4*>(p) + vec), g);
  }
}

struct AdamArgs {
  float lr, beta1, beta2, eps, wd, bc1, bc2, grad_scale, max_norm;
};

constexpr int kAdamMinBlocks = 5;   // resident CTAs per SM the register allocation is tuned for: measured best of {3,4,5,6,8} (profiles/r01_kernels.md)
constexpr int kAdamVec = 4;         // elements per thread per iteration (4 or 8); 4 x 5 CTAs/SM beat 8 x 4 by 12 %

constexpr int kAdamColumnsMinBlocks = 4;   // the column table entry costs registers: 5 CTAs/SM would spill


template <int GDT, int N>
__device__ __forceinline__ void load_grad(const void* p, int64_t e, float (&g)[N]) {
  if (GDT == SMT_F32) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q) {
      const float4 a = ld_stream_f4(reinterpret_cast<const float*>(p) + e + 4 * q);
      g[4 * q] = a.x; g[4 * q + 1] = a.y; g[4 * q + 2] = a.z; g[4 * q + 3] = a.w;
    }
  } else if (N == 8) {
    float t[8];
    unpack8<GDT>(ld_stream_u4(reinterpret_cast<const uint16_t*>(p) + e), t);
#pragma unroll
    for (int j = 0; j < N; ++j) g[j] = t[j];
  } else {
    uint2 u;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(u.x), "=r"(u.y)
                 : "l"(reinterpret_cast<const uint16_t*>(p) + e));
    if (GDT == SMT_BF16) {
      g[0] = __uint_as_float(u.x << 16); g[1] = __uint_as_float(u.x & 0xffff0000u);
      g[2] = __uint_as_float(u.y << 16); g[3] = __uint_as_float(u.y & 0xffff0000u);
    } else {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      g[0] = a.x; g[1] = a.y; g[2] = b.x; g[3] = b.y;
    }
  }
}

template <int N>
__device__ __forceinline__ void load_state(const float* p, int64_t e, float (&s)[N]) {
#pragma unroll
  for (int q = 0; q < N / 4; ++q) {
    const float4 a = *reinterpret_cast<const float4*>(p + e + 4 * q);   // plain loads: the state is rewritten below
    s[4 * q] = a.x; s[4 * q + 1] = a.y; s[4 * q + 2] = a.z; s[4 * q + 3] = a.w;
  }
}

template <int ODT, int N>
__device__ __forceinline__ void store_vals(void* base, int64_t e, const float (&p)[N]) {
  if (ODT == SMT_F32) {
#pragma unroll
    for (int q = 0; q < N / 4; ++q)
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + e + 4 * q) =
          make_float4(p[4 * q], p[4 * q + 1], p[4 * q + 2], p[4 * q + 3]);
  } else {
    uint32_t w[N / 2];
#pragma unroll
    for (int q = 0; q < N / 2; ++q)
      w[q] = ODT == SMT_BF16 ? pack_bf16x2(p[2 * q], p[2 * q + 1]) : pack_f16x2(p[2 * q], p[2 * q + 1]);
    uint16_t* o = reinterpret_cast<uint16_t*>(base) + e;
    if (N == 8) *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
    else *reinterpret_cast<uint2*>(o) = make_uint2(w[0], w[1]);
  }
}

// Gradient multiplier of a step: grad_scale, times the clip coefficient when a norm is given.  Every thread of the CTA
// must call it (the partial-sum form reduces across the block).
__device__ __forceinline__ float clip_grad_scale(const AdamArgs& a, const float* __restrict__ sqnorm, int n_sq,
                                                 float* sq_scratch, float* sq_total) {
  // clip coefficient (uniform): deepspeed clip = max_norm / (norm + 1e-6), applied when < 1
  float gscale = a.grad_scale;
  if (sqnorm != nullptr && a.max_norm > 0.f) {
    float total;
    if (n_sq == 1) {
      total = *sqnorm;
    } else {
      // partial sums (GEMM epilogue slots / per-chunk norms): every CTA adds them in the same fixed order
      // (thread-strided, then the block tree), so the coefficient is identical in all CTAs and run to run
      float t = 0.f;
      for (int i = threadIdx.x; i < n_sq; i += kAdamThreads) t = __fadd_rn(t, sqnorm[i]);
      t = block_sum(t, sq_scratch);
      if (threadIdx.x == 0) *sq_total = t;
      __syncthreads();
      total = *sq_total;
    }
    const float norm = __fmul_rn(__fsqrt_rn(total), a.grad_scale);
    const float coef = __fdiv_rn(a.max_norm, __fadd_rn(norm, 1e-6f));
    if (coef < 1.f) gscale = __fmul_rn(a.grad_scale, coef);
  }
  return gscale;
}

// The AdamW update of N elements in registers: g is the raw gradient, p / m / v are updated in place.  Both Adam kernels
// call this, so they produce bit-identical state from the same inputs.
template <int N>
__device__ __forceinline__ void adam_update(const AdamArgs& a, float gscale, const float (&g)[N], float (&p)[N],
                                            float (&m)[N], float (&v)[N]) {
  const float omb1 = __fsub_rn(1.f, a.beta1), omb2 = __fsub_rn(1.f, a.beta2);
#pragma unroll
  for (int j = 0; j < N; ++j) {
    const float gj = __fmul_rn(g[j], gscale);
    m[j] = __fadd_rn(__fmul_rn(a.beta1, m[j]), __fmul_rn(omb1, gj));
    v[j] = __fadd_rn(__fmul_rn(a.beta2, v[j]), __fmul_rn(__fmul_rn(omb2, gj), gj));
    const float mhat = __fdiv_rn(m[j], a.bc1);
    const float vhat = __fdiv_rn(v[j], a.bc2);
    const float denom = __fadd_rn(__fsqrt_rn(vhat), a.eps);
    const float update = __fadd_rn(__fdiv_rn(mhat, denom), __fmul_rn(a.wd, p[j]));
    p[j] = __fsub_rn(p[j], __fmul_rn(a.lr, update));
  }
}

template <int GDT, int CDT, int WDT>
__global__ void __launch_bounds__(kAdamThreads, kAdamMinBlocks) compact_adam_kernel(
    float* __restrict__ master, float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq,
    const void* __restrict__ grad, int64_t n_vec, AdamArgs a, const float* __restrict__ sqnorm, int n_sq,
    void* __restrict__ compact_out, const smt_block_ref* __restrict__ table, int block_shift) {
  constexpr int N = kAdamVec;
  __shared__ float sq_scratch[32];
  __shared__ float sq_total;
  const float gscale = clip_grad_scale(a, sqnorm, n_sq, sq_scratch, &sq_total);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t vec = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; vec < n_vec; vec += stride) {
    const int64_t e = vec * N;
    float g[N], p[N], m[N], v[N];
    load_grad<GDT, N>(grad, e, g);
    load_state<N>(master, e, p);
    load_state<N>(exp_avg, e, m);
    load_state<N>(exp_avg_sq, e, v);
    adam_update<N>(a, gscale, g, p, m, v);
    store_vals<SMT_F32, N>(master, e, p);
    store_vals<SMT_F32, N>(exp_avg, e, m);
    store_vals<SMT_F32, N>(exp_avg_sq, e, v);
    if (compact_out != nullptr) store_vals<CDT, N>(compact_out, e, p);
    if (table != nullptr) {
      // element e lives in block e >> (2*block_shift), at (row, col) inside it
      const int64_t bi = e >> (2 * block_shift);
      const int within = (int)(e & (((int64_t)1 << (2 * block_shift)) - 1));
      const int r = within >> block_shift, c = within & ((1 << block_shift) - 1);
      const smt_block_ref ref = table[bi];
      const int64_t off = ((int64_t)ref.row << block_shift) * ref.ldw + ((int64_t)ref.col << block_shift) +
                          (int64_t)r * ref.ldw + c;
      store_vals<WDT, N>(reinterpret_cast<void*>(ref.w_ptr), off, p);
    }
  }
}

// The same step over the arena rows of selected weight COLUMNS (channel sparsity).  A CTA takes kColGroup consecutive
// table entries (channels, normally of one weight) and walks their arena rows in tiles of kColRows elements:
//   state phase      warp w owns entry w, its lanes read / update / write kAdamVec contiguous arena elements each (the
//                    state traffic stays coalesced), and the updated masters go to a shared-memory tile;
//   write-back phase the tile is written to the weights transposed: the lanes of a warp cover the kColGroup columns of
//                    four weight rows, so the 2-byte stores of one row leave together and the CTAs working on the same
//                    row tile of a weight (launched side by side) fill its sectors in L2.
// Entries that are not inside [0, n_elems) with 8-aligned `off` and `n_out`, or whose column is outside [0, ldw), are
// skipped (the host builds the table from checked values: ops.make_column_table).
constexpr int kColGroup = kAdamThreads / 32;      // entries per CTA: one warp each in the state phase
constexpr int kColRows = 32 * kAdamVec;           // arena elements of an entry per tile
static_assert(kColRows == kAdamVec * (kAdamThreads / kColGroup), "write-back: kAdamVec rows per thread cover the tile");

template <int GDT, int CDT, int WDT>
__global__ void __launch_bounds__(kAdamThreads, kAdamColumnsMinBlocks) compact_adam_columns_kernel(
    float* __restrict__ master, float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq,
    const void* __restrict__ grad, int64_t n_elems, AdamArgs a, const float* __restrict__ sqnorm, int n_sq,
    void* __restrict__ compact_out, const smt_column_ref* __restrict__ columns, int n_columns) {
  constexpr int N = kAdamVec;
  __shared__ float sq_scratch[32];
  __shared__ float sq_total;
  __shared__ smt_column_ref refs[kColGroup];
  __shared__ float tile[kColGroup][kColRows + 1];
  const float gscale = clip_grad_scale(a, sqnorm, n_sq, sq_scratch, &sq_total);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int g0 = blockIdx.x * kColGroup; g0 < n_columns; g0 += gridDim.x * kColGroup) {
    __syncthreads();                                   // the previous group's write-back is done with refs / tile
    if (threadIdx.x < kColGroup) {
      smt_column_ref ref{};
      if (g0 + (int)threadIdx.x < n_columns) {
        ref = columns[g0 + threadIdx.x];
        if (ref.off < 0 || ref.n_out <= 0 || ((ref.off | (int64_t)ref.n_out) & 7) != 0 || ref.off + ref.n_out > n_elems ||
            ref.col < 0 || ref.col >= ref.ldw)
          ref.n_out = 0;                               // skipped
      }
      refs[threadIdx.x] = ref;
    }
    __syncthreads();
    int rows = 0;
#pragma unroll
    for (int c = 0; c < kColGroup; ++c) rows = refs[c].n_out > rows ? refs[c].n_out : rows;
    for (int o0 = 0; o0 < rows; o0 += kColRows) {
      const int o = o0 + lane * N;
      if (o < refs[warp].n_out) {
        const int64_t e = refs[warp].off + o;
        float g[N], p[N], m[N], v[N];
        load_grad<GDT, N>(grad, e, g);
        load_state<N>(master, e, p);
        load_state<N>(exp_avg, e, m);
        load_state<N>(exp_avg_sq, e, v);
        adam_update<N>(a, gscale, g, p, m, v);
        store_vals<SMT_F32, N>(master, e, p);
        store_vals<SMT_F32, N>(exp_avg, e, m);
        store_vals<SMT_F32, N>(exp_avg_sq, e, v);
        if (compact_out != nullptr) store_vals<CDT, N>(compact_out, e, p);
#pragma unroll
        for (int j = 0; j < N; ++j) tile[warp][lane * N + j] = p[j];
      }
      __syncthreads();
      const int c = threadIdx.x % kColGroup;
      const smt_column_ref& ref = refs[c];
#pragma unroll
      for (int k = 0; k < N; ++k) {
        const int r = (int)threadIdx.x / kColGroup + k * (kAdamThreads / kColGroup);
        if (o0 + r < ref.n_out)
          store_from_float<WDT>(reinterpret_cast<void*>(ref.w_ptr), (int64_t)(o0 + r) * ref.ldw + ref.col, tile[c][r]);
      }
      __syncthreads();
    }
  }
}

// ---- deterministic sum of squares -----------------------------------------------------------------

template <int GDT>
__global__ void __launch_bounds__(kAdamThreads) sqnorm_stage1_kernel(const void* __restrict__ grad,
                                                                     int64_t n, float* __restrict__ partials) {
  __shared__ float scratch[32];
  // fixed assignment of contiguous chunks to CTAs => summation order independent of scheduling
  const int64_t n_vec8 = n / 8;
  const int64_t per_cta = (n_vec8 + gridDim.x - 1) / gridDim.x;
  const int64_t v0 = (int64_t)blockIdx.x * per_cta;
  const int64_t v1 = v0 + per_cta < n_vec8 ? v0 + per_cta : n_vec8;
  float s = 0.f;
  // four independent 128-bit loads in flight per thread (the single-load version sat at 0.52 of the HBM peak on the
  // 114 MB buffer of LLaMA-3-8B at 0.71 %: latency-bound); the order of the additions is still fixed
  int64_t vec = v0 + threadIdx.x;
  for (; vec + 3 * (int64_t)blockDim.x < v1; vec += 4 * (int64_t)blockDim.x) {
    float g0[8], g1[8], g2[8], g3[8];
    load8<GDT>(grad, vec, g0);
    load8<GDT>(grad, vec + blockDim.x, g1);
    load8<GDT>(grad, vec + 2 * (int64_t)blockDim.x, g2);
    load8<GDT>(grad, vec + 3 * (int64_t)blockDim.x, g3);
    float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      t0 += g0[j] * g0[j]; t1 += g1[j] * g1[j]; t2 += g2[j] * g2[j]; t3 += g3[j] * g3[j];
    }
    s += (t0 + t1) + (t2 + t3);
  }
  for (; vec < v1; vec += blockDim.x) {
    float g[8];
    load8<GDT>(grad, vec, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) s += g[j] * g[j];
  }
  if (blockIdx.x == gridDim.x - 1) {  // scalar tail
    for (int64_t i = n_vec8 * 8 + threadIdx.x; i < n; i += blockDim.x) {
      const float x = load_as_float<GDT>(grad, i);
      s += x * x;
    }
  }
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

__global__ void __launch_bounds__(kAdamThreads) sqnorm_stage2_kernel(const float* __restrict__ partials,
                                                                     int n_partials, float* __restrict__ out) {
  __shared__ float scratch[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n_partials; i += blockDim.x) s += partials[i];
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) out[0] = s;
}

// Arguments of one launch of either Adam kernel: `columns` != NULL selects the column write-back kernel (n = n_elems),
// otherwise the block / compact kernel runs (n = number of kAdamVec vectors).
struct AdamLaunch {
  float *master, *m, *v;
  const void* grad;
  int64_t n;
  AdamArgs a;
  const float* sqnorm;
  int n_sq;
  void* compact_out;
  const smt_block_ref* table;
  int shift;
  const smt_column_ref* columns;
  int n_columns;
};

template <int GDT, int CDT, int WDT>
void launch_adam_kernel(const AdamLaunch& L, int grid, cudaStream_t st) {
  if (L.columns != nullptr)
    compact_adam_columns_kernel<GDT, CDT, WDT><<<grid, kAdamThreads, 0, st>>>(
        L.master, L.m, L.v, L.grad, L.n, L.a, L.sqnorm, L.n_sq, L.compact_out, L.columns, L.n_columns);
  else
    compact_adam_kernel<GDT, CDT, WDT><<<grid, kAdamThreads, 0, st>>>(
        L.master, L.m, L.v, L.grad, L.n, L.a, L.sqnorm, L.n_sq, L.compact_out, L.table, L.shift);
}

template <int GDT, int CDT>
int launch_adam_w(int w_dtype, int grid, cudaStream_t st, const AdamLaunch& L) {
  if (w_dtype == SMT_F32) launch_adam_kernel<GDT, CDT, SMT_F32>(L, grid, st);
  else if (w_dtype == SMT_BF16) launch_adam_kernel<GDT, CDT, SMT_BF16>(L, grid, st);
  else launch_adam_kernel<GDT, CDT, SMT_F16>(L, grid, st);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

template <int GDT>
int launch_adam_c(int c_dtype, int w_dtype, int grid, cudaStream_t st, const AdamLaunch& L) {
  if (c_dtype == SMT_F32) return launch_adam_w<GDT, SMT_F32>(w_dtype, grid, st, L);
  if (c_dtype == SMT_BF16) return launch_adam_w<GDT, SMT_BF16>(w_dtype, grid, st, L);
  return launch_adam_w<GDT, SMT_F16>(w_dtype, grid, st, L);
}

int launch_adam(int grad_dtype, int c_dtype, int w_dtype, int grid, cudaStream_t st, const AdamLaunch& L) {
  if (grad_dtype == SMT_F32) return launch_adam_c<SMT_F32>(c_dtype, w_dtype, grid, st, L);
  if (grad_dtype == SMT_BF16) return launch_adam_c<SMT_BF16>(c_dtype, w_dtype, grid, st, L);
  return launch_adam_c<SMT_F16>(c_dtype, w_dtype, grid, st, L);
}

// Checks shared by both Adam entry points; fills `a`.
int check_adam_args(const char* who, float* master, float* exp_avg, float* exp_avg_sq, const void* grad,
                    int grad_dtype, int64_t n_elems, float lr, float beta1, float beta2, float eps, float weight_decay,
                    float bias_correction1, float bias_correction2, float grad_scale, const float* sqnorm, int n_sqnorm,
                    float max_norm, void* compact_out, int* compact_dtype, AdamArgs* a) {
  SMT_CHECK_ARG(master != nullptr, "%s: null pointer (master)", who);
  SMT_CHECK_ARG(exp_avg != nullptr, "%s: null pointer (exp_avg)", who);
  SMT_CHECK_ARG(exp_avg_sq != nullptr, "%s: null pointer (exp_avg_sq)", who);
  SMT_CHECK_ARG(grad != nullptr, "%s: null pointer (grad)", who);
  SMT_CHECK_ARG(grad_dtype >= SMT_F32 && grad_dtype <= SMT_F16, "%s: bad grad dtype %d", who, grad_dtype);
  SMT_CHECK_ARG(n_elems % 8 == 0, "%s: n_elems must be a multiple of 8", who);
  SMT_CHECK_ARG(aligned16(master) && aligned16(exp_avg) && aligned16(exp_avg_sq) && aligned16(grad) &&
                    (compact_out == nullptr || aligned16(compact_out)),
                "%s: state pointers must be 16-byte aligned", who);
  SMT_CHECK_ARG(bias_correction1 > 0.f && bias_correction2 > 0.f, "%s: bias corrections must be > 0", who);
  SMT_CHECK_ARG(sqnorm == nullptr || n_sqnorm >= 1, "%s: n_sqnorm must be >= 1 when sqnorm is given", who);
  if (compact_out != nullptr)
    SMT_CHECK_ARG(*compact_dtype >= SMT_F32 && *compact_dtype <= SMT_F16, "%s: bad compact dtype %d", who,
                  *compact_dtype);
  else
    *compact_dtype = SMT_BF16;
  *a = AdamArgs{lr, beta1, beta2, eps, weight_decay, bias_correction1, bias_correction2, grad_scale, max_norm};
  return SMT_OK;
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API size_t smt_grad_sqnorm_workspace_bytes(void) { return kSqPartials * sizeof(float); }

extern "C" SMT_API int smt_grad_sqnorm(const void* grad, int grad_dtype, int64_t n, float* out_sqnorm,
                               void* workspace, size_t workspace_bytes, void* stream) {
  SMT_CHECK_ARG(grad_dtype >= SMT_F32 && grad_dtype <= SMT_F16, "smt_grad_sqnorm: bad dtype %d", grad_dtype);
  SMT_CHECK_ARG(n >= 0, "smt_grad_sqnorm: n < 0");
  // n = 0 needs no gradient pointer (an empty tensor's data_ptr() is 0), but still writes 0 to out_sqnorm: the clip
  // of smt_compact_adam reads it
  SMT_CHECK_ARG(grad != nullptr || n == 0, "smt_grad_sqnorm: null pointer (grad)");
  SMT_CHECK_ARG(out_sqnorm != nullptr, "smt_grad_sqnorm: null pointer (out_sqnorm)");
  SMT_CHECK_ARG(aligned16(grad), "smt_grad_sqnorm: grad must be 16-byte aligned");
  if (workspace == nullptr || workspace_bytes < smt_grad_sqnorm_workspace_bytes()) {
    set_error("smt_grad_sqnorm: workspace too small");
    return SMT_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  float* partials = reinterpret_cast<float*>(workspace);
  // grid depends only on n (not on the device), so the result is reproducible across GPUs
  int64_t want = (n / 8 + kAdamThreads * 4 - 1) / (kAdamThreads * 4);
  int grid = (int)(want < 1 ? 1 : (want > kSqPartials ? kSqPartials : want));
  if (grad_dtype == SMT_F32) sqnorm_stage1_kernel<SMT_F32><<<grid, kAdamThreads, 0, st>>>(grad, n, partials);
  else if (grad_dtype == SMT_BF16) sqnorm_stage1_kernel<SMT_BF16><<<grid, kAdamThreads, 0, st>>>(grad, n, partials);
  else sqnorm_stage1_kernel<SMT_F16><<<grid, kAdamThreads, 0, st>>>(grad, n, partials);
  SMT_CHECK_LAUNCH();
  sqnorm_stage2_kernel<<<1, kAdamThreads, 0, st>>>(partials, grid, out_sqnorm);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_compact_adam(float* master, float* exp_avg, float* exp_avg_sq, const void* grad,
                                int grad_dtype, int64_t n_elems, float lr, float beta1, float beta2,
                                float eps, float weight_decay, float bias_correction1,
                                float bias_correction2, float grad_scale, const float* sqnorm, int n_sqnorm,
                                float max_norm, void* compact_out, int compact_dtype,
                                const smt_block_ref* table, int n_blocks, int block, int w_dtype,
                                void* stream) {
  SMT_CHECK_ARG(n_elems >= 0, "smt_compact_adam: n_elems < 0");
  if (n_elems == 0) return SMT_OK;
  AdamArgs a;
  if (int rc = check_adam_args("smt_compact_adam", master, exp_avg, exp_avg_sq, grad, grad_dtype, n_elems, lr, beta1,
                               beta2, eps, weight_decay, bias_correction1, bias_correction2, grad_scale, sqnorm,
                               n_sqnorm, max_norm, compact_out, &compact_dtype, &a))
    return rc;
  int shift = 0;
  if (table != nullptr) {
    SMT_CHECK_ARG(block_ok(block), "smt_compact_adam: block size %d not in {64,128,256}", block);
    SMT_CHECK_ARG((int64_t)n_blocks * block * block == n_elems, "smt_compact_adam: n_blocks*b*b != n_elems");
    SMT_CHECK_ARG(w_dtype >= SMT_F32 && w_dtype <= SMT_F16, "smt_compact_adam: bad W dtype %d", w_dtype);
    shift = block == 256 ? 8 : (block == 128 ? 7 : 6);
  } else {
    w_dtype = SMT_BF16;
  }
  const int64_t n_vec = n_elems / kAdamVec;        // vectors of kAdamVec elements (n_elems is a multiple of 8)
  int64_t want = (n_vec + kAdamThreads - 1) / kAdamThreads;
  const int64_t cap = (int64_t)sm_count() * kAdamMinBlocks * 2;
  const int grid = (int)(want < cap ? want : cap);
  const AdamLaunch L{master, exp_avg, exp_avg_sq, grad, n_vec, a, sqnorm, n_sqnorm, compact_out, table, shift,
                     nullptr, 0};
  return launch_adam(grad_dtype, compact_dtype, w_dtype, grid, (cudaStream_t)stream, L);
}

extern "C" SMT_API int smt_compact_adam_columns(float* master, float* exp_avg, float* exp_avg_sq, const void* grad,
                                                int grad_dtype, int64_t n_elems, float lr, float beta1, float beta2,
                                                float eps, float weight_decay, float bias_correction1,
                                                float bias_correction2, float grad_scale, const float* sqnorm,
                                                int n_sqnorm, float max_norm, void* compact_out, int compact_dtype,
                                                const smt_column_ref* columns, int n_columns, int w_dtype,
                                                void* stream) {
  SMT_CHECK_ARG(n_elems >= 0 && n_columns >= 0, "smt_compact_adam_columns: negative size");
  if (n_elems == 0 || n_columns == 0) return SMT_OK;
  AdamArgs a;
  if (int rc = check_adam_args("smt_compact_adam_columns", master, exp_avg, exp_avg_sq, grad, grad_dtype, n_elems, lr,
                               beta1, beta2, eps, weight_decay, bias_correction1, bias_correction2, grad_scale, sqnorm,
                               n_sqnorm, max_norm, compact_out, &compact_dtype, &a))
    return rc;
  SMT_CHECK_ARG(columns != nullptr, "smt_compact_adam_columns: null column table");
  SMT_CHECK_ARG(w_dtype >= SMT_F32 && w_dtype <= SMT_F16, "smt_compact_adam_columns: bad W dtype %d", w_dtype);
  const int64_t groups = (n_columns + kColGroup - 1) / kColGroup;
  const int64_t cap = (int64_t)sm_count() * kAdamColumnsMinBlocks * 2;
  const int grid = (int)(groups < cap ? groups : cap);
  const AdamLaunch L{master, exp_avg, exp_avg_sq, grad, n_elems, a, sqnorm, n_sqnorm, compact_out, nullptr, 0,
                     columns, n_columns};
  return launch_adam(grad_dtype, compact_dtype, w_dtype, grid, (cudaStream_t)stream, L);
}
