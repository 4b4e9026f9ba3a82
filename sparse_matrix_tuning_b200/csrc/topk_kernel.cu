// Segmented, bit-exact top-k over block scores.
//
// Replaces the Python min-heap of deepspeed/smt/smt_helper.py:102-146 (`no_restriction`: one global
// top-n, one `.item()` + heap op per block) and the per-matrix argsort of smt_helper.py:81-100
// (`norm_dist`).  The reference's total order is Python tuple order on
// (score, ((module_name, layer), i, j)); the host ranks the (name, layer, i, j) tuples once and the
// kernel orders 64-bit keys  key = orderable(score) << 32 | rank,  so indices are exact whenever the
// scores are identical, ties included.
//
// One CTA per segment: 8-pass MSB radix select of the k-th largest key, compaction of the k winners,
// bitonic sort (shared memory up to 8192 keys, global workspace beyond).  This is latency-scale work
// (12 288 - 98 304 keys); no roofline is claimed for it.
#include "common.cuh"

namespace smt {
namespace {

constexpr int kTopkThreads = 1024;
constexpr int kSmemKeys = 8192;  // 64 KiB of dynamic shared memory

__device__ __forceinline__ uint32_t orderable(float f) {
  uint32_t u = __float_as_uint(f);
  if ((u << 1) == 0u) u = 0u;  // -0.0 == +0.0 in the reference's float comparison
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ uint64_t make_key(const float* scores, const uint32_t* rank, int64_t i) {
  const uint32_t r = rank ? rank[i] : (uint32_t)i;
  return ((uint64_t)orderable(scores[i]) << 32) | r;
}

// In-place descending bitonic sort of `n_pow2` keys (shared or global memory), whole CTA.
__device__ void bitonic_sort_desc(uint64_t* keys, int n_pow2) {
  for (int size = 2; size <= n_pow2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < (n_pow2 >> 1); t += blockDim.x) {
        const int lo = 2 * t - (t & (stride - 1));
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = keys[lo], b = keys[hi];
        if ((a < b) == desc) {
          keys[lo] = b;
          keys[hi] = a;
        }
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kTopkThreads) topk_blocks_kernel(
    const float* __restrict__ scores, const uint32_t* __restrict__ rank,
    const uint32_t* __restrict__ inv_rank, const int32_t* __restrict__ seg_offsets,
    const int32_t* __restrict__ seg_k, const int32_t* __restrict__ out_offsets,
    int32_t* __restrict__ out_idx, uint64_t* __restrict__ ws_keys) {
  extern __shared__ uint64_t s_keys[];
  __shared__ uint32_t hist[256];
  __shared__ uint64_t s_prefix;
  __shared__ uint32_t s_need;
  __shared__ uint32_t s_count;

  const int seg = blockIdx.x;
  const int64_t begin = seg_offsets[seg], end = seg_offsets[seg + 1];
  const int64_t len = end - begin;
  int64_t k = seg_k[seg];
  if (k > len) k = len;
  if (k <= 0) return;

  // ---- radix select: find the k-th largest key, MSB digit first --------------------------------
  if (threadIdx.x == 0) {
    s_prefix = 0;
    s_need = (uint32_t)k;
  }
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    for (int b = threadIdx.x; b < 256; b += blockDim.x) hist[b] = 0;
    __syncthreads();
    const uint64_t prefix = s_prefix;
    const uint64_t himask = pass == 0 ? 0ull : (~0ull << (shift + 8));
    for (int64_t i = begin + threadIdx.x; i < end; i += blockDim.x) {
      const uint64_t key = make_key(scores, rank, i);
      if ((key & himask) == prefix) atomicAdd(&hist[(uint32_t)(key >> shift) & 0xffu], 1u);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t need = s_need, cum = 0;
      int d = 255;
      for (; d > 0; --d) {
        if (cum + hist[d] >= need) break;
        cum += hist[d];
      }
      s_need = need - cum;  // still wanted inside digit d
      s_prefix = prefix | ((uint64_t)d << shift);
    }
    __syncthreads();
  }
  const uint64_t threshold = s_prefix;  // exactly k keys are >= threshold (keys are unique)

  // ---- compact the winners and sort them ----------------------------------------------------------
  int n_pow2 = 1;
  while (n_pow2 < k) n_pow2 <<= 1;
  // shared memory when the padded winners fit, else this segment's private slice of the global
  // workspace: it starts at 2*begin and holds 2*len >= n_pow2 keys (n_pow2 < 2k <= 2*len).
  uint64_t* buf = (n_pow2 <= kSmemKeys) ? s_keys : (ws_keys + 2 * begin);
  if (threadIdx.x == 0) s_count = 0;
  __syncthreads();
  for (int64_t i = begin + threadIdx.x; i < end; i += blockDim.x) {
    const uint64_t key = make_key(scores, rank, i);
    if (key >= threshold) {
      const uint32_t slot = atomicAdd(&s_count, 1u);
      if (slot < (uint32_t)n_pow2) buf[slot] = key;  // (overflow only if ranks were not unique)
    }
  }
  __syncthreads();
  for (int i = (int)k + threadIdx.x; i < n_pow2; i += blockDim.x) buf[i] = 0ull;  // pads sort last
  bitonic_sort_desc(buf, n_pow2);

  int32_t* out = out_idx + out_offsets[seg];
  for (int i = threadIdx.x; i < (int)k; i += blockDim.x) {
    const uint32_t r = (uint32_t)(buf[i] & 0xffffffffull);
    out[i] = (int32_t)(inv_rank ? inv_rank[r] : r);
  }
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API size_t smt_topk_workspace_bytes(int64_t n_scores) {
  if (n_scores < 0) n_scores = 0;
  // every segment may need its keys padded to the next power of two (< 2x its length)
  return (size_t)(2 * n_scores + 2) * sizeof(uint64_t);
}

extern "C" SMT_API int smt_topk_blocks(const float* scores, const uint32_t* tiebreak_rank,
                               const uint32_t* inv_rank, int64_t n_scores,
                               const int32_t* seg_offsets, const int32_t* seg_k,
                               const int32_t* out_offsets, int num_segments, int32_t* out_idx,
                               void* workspace, size_t workspace_bytes, void* stream) {
  SMT_CHECK_ARG(num_segments >= 0, "smt_topk_blocks: num_segments < 0");
  if (num_segments == 0 || n_scores == 0) return SMT_OK;
  SMT_CHECK_ARG(scores != nullptr, "smt_topk_blocks: null pointer (scores)");
  SMT_CHECK_ARG(seg_offsets != nullptr, "smt_topk_blocks: null pointer (seg_offsets)");
  SMT_CHECK_ARG(seg_k != nullptr, "smt_topk_blocks: null pointer (seg_k)");
  SMT_CHECK_ARG(out_offsets != nullptr, "smt_topk_blocks: null pointer (out_offsets)");
  SMT_CHECK_ARG(out_idx != nullptr, "smt_topk_blocks: null pointer (out_idx)");
  SMT_CHECK_ARG((tiebreak_rank == nullptr) == (inv_rank == nullptr), "smt_topk_blocks: tiebreak_rank and inv_rank must be given together");
  SMT_CHECK_ARG(n_scores < (1ll << 31), "smt_topk_blocks: too many scores");
  if (workspace_bytes < smt_topk_workspace_bytes(n_scores) || workspace == nullptr) {
    set_error("smt_topk_blocks: workspace too small (%zu < %zu)", workspace_bytes, smt_topk_workspace_bytes(n_scores));
    return SMT_ERR_WORKSPACE;
  }
  const int smem = kSmemKeys * (int)sizeof(uint64_t);
  SMT_CHECK_CUDA(cudaFuncSetAttribute(topk_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  topk_blocks_kernel<<<num_segments, kTopkThreads, smem, (cudaStream_t)stream>>>(
      scores, tiebreak_rank, inv_rank, seg_offsets, seg_k, out_offsets, out_idx,
      reinterpret_cast<uint64_t*>(workspace));
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}
