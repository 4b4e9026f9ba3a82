// Table-driven movement of selected b x b blocks between dense weights and compact storage.
//
// Reference call sites replaced:
//   deepspeed/smt/smt.py:317-325   gather at LinearLayer_MatrixSparsity.__init__ (n slice copies)
//   deepspeed/smt/smt.py:332-341   scatter at the start of EVERY forward (n slice copies per module)
//   deepspeed/smt/smt.py:427-439   scatter inside convert_matrix_sparsity_to_linear_layer
// One launch moves every block of every module named in the table (HBM-bound, 2*n*b*b*elem bytes).
#include "common.cuh"

namespace smt {
namespace {

constexpr int kCopyThreads = 256;
constexpr int kRowSplit = 4;  // CTAs per block (row quarters) for parallelism at small n

template <bool GATHER>
__global__ void __launch_bounds__(kCopyThreads) block_copy_kernel(
    const smt_block_ref* __restrict__ table, int block, int row_bytes, char* __restrict__ compact) {
  const smt_block_ref ref = table[blockIdx.x];
  const int vec_per_row = row_bytes / 16;
  const int rows_per_cta = block / kRowSplit;
  const int row0 = blockIdx.y * rows_per_cta;
  const int elem_bytes = row_bytes / block;
  char* w = reinterpret_cast<char*>(ref.w_ptr) +
            ((int64_t)ref.row * block * ref.ldw + (int64_t)ref.col * block) * elem_bytes;
  char* c = compact + (int64_t)blockIdx.x * block * row_bytes;
  const int64_t w_pitch = ref.ldw * elem_bytes;
  const int total = rows_per_cta * vec_per_row;
  for (int i = threadIdx.x; i < total; i += kCopyThreads) {
    const int r = row0 + i / vec_per_row, v = i % vec_per_row;
    uint4* wp = reinterpret_cast<uint4*>(w + (int64_t)r * w_pitch) + v;
    uint4* cp = reinterpret_cast<uint4*>(c + (int64_t)r * row_bytes) + v;
    if (GATHER) *cp = *wp;
    else *wp = *cp;
  }
}

int launch_copy(bool gather, const smt_block_ref* table, int n_blocks, int block, int elem_bytes,
                void* compact, void* stream, const char* who) {
  SMT_CHECK_ARG(n_blocks >= 0, "%s: n_blocks < 0", who);
  if (n_blocks == 0) return SMT_OK;
  SMT_CHECK_ARG(table && compact, "%s: null pointer", who);
  SMT_CHECK_ARG(block_ok(block), "%s: block size %d not in {64,128,256}", who, block);
  SMT_CHECK_ARG(elem_bytes == 2 || elem_bytes == 4, "%s: elem_bytes must be 2 or 4", who);
  SMT_CHECK_ARG(aligned16(compact), "%s: compact must be 16-byte aligned", who);
  dim3 grid(n_blocks, kRowSplit);
  const int row_bytes = block * elem_bytes;
  if (gather)
    block_copy_kernel<true><<<grid, kCopyThreads, 0, (cudaStream_t)stream>>>(table, block, row_bytes, (char*)compact);
  else
    block_copy_kernel<false><<<grid, kCopyThreads, 0, (cudaStream_t)stream>>>(table, block, row_bytes, (char*)compact);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

}  // namespace
}  // namespace smt

extern "C" SMT_API int smt_block_gather(const smt_block_ref* table, int n_blocks, int block, int elem_bytes,
                                void* compact, void* stream) {
  return smt::launch_copy(true, table, n_blocks, block, elem_bytes, compact, stream, "smt_block_gather");
}

extern "C" SMT_API int smt_block_scatter(const smt_block_ref* table, int n_blocks, int block, int elem_bytes,
                                 const void* compact, void* stream) {
  return smt::launch_copy(false, table, n_blocks, block, elem_bytes, const_cast<void*>(compact), stream,
                          "smt_block_scatter");
}
