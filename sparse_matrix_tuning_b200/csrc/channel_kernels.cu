// Channel (input-column) movement for the channel-sparsity layer.
//
// Reference call sites replaced:
//   deepspeed/smt/smt.py:240-247   linearChannel.forward: partial_input[:, :, i] = input[:, :, index]  (n slice copies)
//   deepspeed/smt/smt.py:198-200   LinearLayer_ChannelSparsity.__init__: selected_weight[i, :] = weight[index, :]
//   deepspeed/smt/smt.py:208-211   LinearLayer_ChannelSparsity.forward: weight[index, :] = selected_weight[i, :]
// The reference copies weight ROWS although its indices are input channels and its gradient (smt.py:283-284) is the
// gradient of weight COLUMNS; that only type-checks for square weights and trains the wrong entries there.  These
// kernels implement the consistent version: channel i owns column idx[i] of W, stored as row i of the compact
// [n, out_features] parameter (so the compact gradient is exactly the reference's partial_input^T @ grad_output).
#include "common.cuh"

namespace smt {
namespace {

constexpr int kTile = 32;

// out[t, i] = x[t, idx[i]] (0 where idx[i] < 0): consecutive threads walk i (coalesced writes; reads stay inside one
// row of x).
template <typename E>
__global__ void __launch_bounds__(256) channel_gather_kernel(const E* __restrict__ x, int64_t ldx, int64_t T,
                                                             const int32_t* __restrict__ idx, int n,
                                                             E* __restrict__ out) {
  const int64_t total = T * (int64_t)n;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = e / n;
    const int i = (int)(e - t * n);
    const int c = idx[i];
    out[e] = c >= 0 ? x[t * ldx + c] : E(0);      // idx < 0: padding column (keeps the row pitch a multiple of 16 B)
  }
}

// 32 x 32 tile through shared memory: the compact side [n, out_features] is read / written along out_features, the
// dense side along the channel list (scattered columns of one row of W).
template <typename E, bool GATHER>
__global__ void __launch_bounds__(kTile * 8) column_copy_kernel(E* __restrict__ W, int64_t ldw, int out_features,
                                                                const int32_t* __restrict__ idx, int n,
                                                                E* __restrict__ compact) {
  __shared__ E tile[kTile][kTile + 1];
  const int o0 = blockIdx.x * kTile, i0 = blockIdx.y * kTile;
  const int tx = threadIdx.x & (kTile - 1), ty = threadIdx.x / kTile;   // 8 rows of 32 threads
  if (GATHER) {
    const int i = i0 + tx;
    const int col = i < n ? idx[i] : 0;
    for (int r = ty; r < kTile; r += 8) {
      const int o = o0 + r;
      if (o < out_features && i < n) tile[r][tx] = W[(int64_t)o * ldw + col];
    }
    __syncthreads();
    for (int r = ty; r < kTile; r += 8) {
      const int ii = i0 + r, o = o0 + tx;
      if (ii < n && o < out_features) compact[(int64_t)ii * out_features + o] = tile[tx][r];
    }
  } else {
    for (int r = ty; r < kTile; r += 8) {
      const int ii = i0 + r, o = o0 + tx;
      if (ii < n && o < out_features) tile[tx][r] = compact[(int64_t)ii * out_features + o];
    }
    __syncthreads();
    const int i = i0 + tx;
    const int col = i < n ? idx[i] : 0;
    for (int r = ty; r < kTile; r += 8) {
      const int o = o0 + r;
      if (o < out_features && i < n) W[(int64_t)o * ldw + col] = tile[r][tx];
    }
  }
}

template <typename E>
int launch_column_copy(bool gather, void* W, int64_t ldw, int out_features, const int32_t* idx, int n, void* compact,
                       cudaStream_t st) {
  dim3 grid((out_features + kTile - 1) / kTile, (n + kTile - 1) / kTile);
  if (gather)
    column_copy_kernel<E, true><<<grid, kTile * 8, 0, st>>>((E*)W, ldw, out_features, idx, n, (E*)compact);
  else
    column_copy_kernel<E, false><<<grid, kTile * 8, 0, st>>>((E*)W, ldw, out_features, idx, n, (E*)compact);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

int column_copy(bool gather, void* W, int64_t ldw, int out_features, int in_features, const int32_t* idx, int n,
                int elem_bytes, void* compact, void* stream, const char* who) {
  SMT_CHECK_ARG(n >= 0 && out_features >= 0, "%s: negative size", who);
  if (n == 0 || out_features == 0) return SMT_OK;
  SMT_CHECK_ARG(W != nullptr, "%s: null pointer (W)", who);
  SMT_CHECK_ARG(idx != nullptr, "%s: null pointer (idx)", who);
  SMT_CHECK_ARG(compact != nullptr, "%s: null pointer (compact)", who);
  SMT_CHECK_ARG(elem_bytes == 2 || elem_bytes == 4, "%s: elem_bytes must be 2 or 4", who);
  SMT_CHECK_ARG(ldw >= in_features && in_features > 0, "%s: bad leading dimension", who);
  SMT_CHECK_ARG((n + kTile - 1) / kTile <= 65535, "%s: too many channels", who);
  return elem_bytes == 2 ? launch_column_copy<uint16_t>(gather, W, ldw, out_features, idx, n, compact, (cudaStream_t)stream)
                         : launch_column_copy<uint32_t>(gather, W, ldw, out_features, idx, n, compact, (cudaStream_t)stream);
}

}  // namespace
}  // namespace smt

extern "C" SMT_API int smt_channel_gather(const void* x, int64_t T, int64_t ldx, const int32_t* idx, int n,
                                          int elem_bytes, void* out, void* stream) {
  SMT_CHECK_ARG(T >= 0 && n >= 0, "smt_channel_gather: negative size");
  if (T == 0 || n == 0) return SMT_OK;
  SMT_CHECK_ARG(x != nullptr, "smt_channel_gather: null pointer (x)");
  SMT_CHECK_ARG(idx != nullptr, "smt_channel_gather: null pointer (idx)");
  SMT_CHECK_ARG(out != nullptr, "smt_channel_gather: null pointer (out)");
  SMT_CHECK_ARG(elem_bytes == 2 || elem_bytes == 4, "smt_channel_gather: elem_bytes must be 2 or 4");
  SMT_CHECK_ARG(ldx > 0, "smt_channel_gather: bad leading dimension");
  const int64_t total = T * (int64_t)n;
  const int64_t want = (total + 255) / 256;
  const int grid = (int)(want < (int64_t)smt::sm_count() * 16 ? want : (int64_t)smt::sm_count() * 16);
  if (elem_bytes == 2)
    smt::channel_gather_kernel<uint16_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)x, ldx, T, idx, n,
                                                                                 (uint16_t*)out);
  else
    smt::channel_gather_kernel<uint32_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)x, ldx, T, idx, n,
                                                                                 (uint32_t*)out);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

extern "C" SMT_API int smt_column_gather(const void* W, int64_t ldw, int out_features, int in_features,
                                         const int32_t* idx, int n, int elem_bytes, void* compact, void* stream) {
  return smt::column_copy(true, const_cast<void*>(W), ldw, out_features, in_features, idx, n, elem_bytes, compact,
                          stream, "smt_column_gather");
}

extern "C" SMT_API int smt_column_scatter(void* W, int64_t ldw, int out_features, int in_features, const int32_t* idx,
                                          int n, int elem_bytes, const void* compact, void* stream) {
  return smt::column_copy(false, W, ldw, out_features, in_features, idx, n, elem_bytes, const_cast<void*>(compact),
                          stream, "smt_column_scatter");
}
