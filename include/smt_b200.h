/*
 * smt_b200.h — C-ABI of the B200-native SMT (Sparse Matrix Tuning) hot path.
 *
 * The reference (yudaohai666/Sparse_Matrix_Tuning) has no native interface: its
 * hot path is eager PyTorch inside `deepspeed/smt/smt.py`, `deepspeed/smt/smt_helper.py`
 * and three snippets of `deepspeed/fine_tune.py`.  Each entry point below replaces one
 * of those Python call sites (cited per function, paths relative to the reference root)
 * and is what a maintainer would bind with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a `cudaStream_t` passed as `void*` (NULL = legacy default stream);
 *   - return value: 0 = ok, negative = error; `smt_last_error()` returns a thread-local
 *     message for the calling thread (forward runs on the caller thread, backward on the
 *     autograd worker thread, so nothing here keeps cross-thread mutable state);
 *   - no allocation inside: workspaces are sized by the `*_workspace_bytes` twins;
 *   - matrices are row-major, `ld*` are leading dimensions in ELEMENTS;
 *   - a weight matrix is `W[out_features, in_features]`; block (r, c) covers
 *     `W[r*b:(r+1)*b, c*b:(c+1)*b]` (reference smt.py:319-325), b in {64, 128, 256};
 *   - "compact" storage stacks block i at rows [i*b, (i+1)*b) of an `[n*b, b]` matrix,
 *     i.e. at flat element offset i*b*b (reference smt.py:312-325).
 */
#ifndef SMT_B200_H_
#define SMT_B200_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define SMT_API __attribute__((visibility("default")))
#else
#define SMT_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* element types */
enum { SMT_F32 = 0, SMT_BF16 = 1, SMT_F16 = 2 };

/* block-score strategies (reference smt_helper.py:233-251) */
enum { SMT_MEAN_ABS = 0,  /* |mean(g)|   smt_helper.py:233 */
       SMT_ABS_MEAN = 1,  /* mean(|g|)   smt_helper.py:238 */
       SMT_L1       = 2,  /* sum(|g|)    smt_helper.py:243 */
       SMT_L2       = 3   /* sqrt(sum g^2) smt_helper.py:249 */ };

/* error codes */
enum { SMT_OK = 0, SMT_ERR_ARG = -1, SMT_ERR_CUDA = -2, SMT_ERR_UNSUPPORTED = -3,
       SMT_ERR_WORKSPACE = -4 };

/* One selected block of one weight matrix.  A table of these describes a whole model's
 * selection: entry i owns compact flat offset i*b*b. */
typedef struct smt_block_ref {
  uint64_t w_ptr;   /* device address of the dense weight W this block lives in        */
  int64_t  ldw;     /* leading dimension of W, elements                                */
  int32_t  row;     /* block row    (out_features / b index)                           */
  int32_t  col;     /* block column (in_features  / b index)                           */
} smt_block_ref;

SMT_API const char* smt_last_error(void);
SMT_API int  smt_version(void);
/* number of kernels the last smt_block_grad_gemm* call on this thread launched (1, or 2 with a separate reduce) */
SMT_API int  smt_last_launch_count(void);
/* sm_count / compute capability of the current device. */
SMT_API int  smt_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host);

/* ---- warm-up scoring ------------------------------------------------------------- */

/* acc[i] += (float)grad[i]   — replaces the D2H copy + CPU `+=` of fine_tune.py:724-740,751-765. */
SMT_API int smt_score_accumulate(float* acc, const void* grad, int grad_dtype, int64_t n, void* stream);

/* block_sums[R/b, C/b] += sum over each b x b tile of grad[R, C] (signed sums).
 * Linear in g, hence valid for SMT_MEAN_ABS only (= what q/k/v always use, fine_tune.py:306-313). */
SMT_API int smt_block_sum_accumulate(float* block_sums, const void* grad, int grad_dtype,
                             int rows, int cols, int64_t ld, int block, void* stream);

/* scores[i] = |block_sums[i]| / b^2  (mean_abs from accumulated signed block sums). */
SMT_API int smt_block_sum_finalize(const float* block_sums, float* scores, int64_t n, int block, void* stream);

/* scores[R/b, C/b] = strategy over each b x b tile of acc[R, C] — smt_helper.py:55-78, 233-251. */
SMT_API int smt_block_score_reduce(const float* acc, int rows, int cols, int64_t ld, int block,
                           int strategy, float* scores, void* stream);

/* Factored block sums for a frozen-weight warm-up — replace fine_tune.py:716-768 (capture of every q/k/v(/MLP)
 * weight gradient) and smt_helper.py:55-78 (its reduction to b x b blocks) for `mean_abs`, without forming dW.
 * For y = x W^T:  sum_{o in r, k in c} dW[o, k] = sum_t Dy[t, r] * X[t, c],  with Dy, X the per-token block sums of
 * dy and x below.  Both calls are deterministic (fixed reduction order, no atomics, nothing depends on the SM count)
 * and no-ops for T = 0, even with NULL pointers.
 *
 * out[t, j] = sum_{k < b} src[t, j*b + k]  (fp32).  src: [T, F] row-major, `dtype` (F32 / BF16 / F16), row pitch `ld`
 * elements, unit column stride, 16-byte aligned base and pitch; F % b == 0; out: contiguous [T, F/b] fp32. */
SMT_API int smt_token_block_sums(const void* src, int dtype, int64_t T, int F, int64_t ld, int block, float* out,
                                 void* stream);
/* block_sums[r, c] += sum_t dy_sums[t, r] * x_sums[t, c]  — contiguous fp32 [rb, cb], [T, rb], [T, cb].
 * T is split into fixed chunks of 128 tokens whose partial products go to `workspace`, then added in chunk order. */
SMT_API size_t smt_block_outer_accumulate_workspace_bytes(int64_t T, int rb, int cb);
SMT_API int smt_block_outer_accumulate(float* block_sums, const float* dy_sums, const float* x_sums, int64_t T,
                                       int rb, int cb, void* workspace, size_t workspace_bytes, void* stream);

/* acc[S, C] += sum_b |x[b, S, C]|  — the activation hook of fine_tune.py:649-678 reduced over the
 * batch dimension, which is all smt_helper.py:170 consumes. */
SMT_API int smt_act_score_accumulate(float* acc, const void* x, int x_dtype, int batch, int seq, int channels,
                             void* stream);

/* out[C] = strategy over the S rows of acc[S, C]  — smt_helper.py:172-183 (acc is already >= 0). */
SMT_API int smt_channel_score_reduce(const float* acc, int seq, int channels, int strategy, float* out,
                             void* stream);

/* ---- top-k selection ---------------------------------------------------------------- */

/* Segmented top-k over `scores[N]`.  Segment s covers [seg_offsets[s], seg_offsets[s+1]) and keeps
 * its k_s = min(seg_k[s], length) best entries, written best-first as flat indices into [0, N) at
 * out_idx[out_offsets[s] ...].  Order: descending score; equal scores are ordered by descending
 * `tiebreak_rank` (unique within a segment; NULL = the flat index).  This is Python's tuple order on
 * (score, ((module, layer), i, j)) used by the heap in smt_helper.py:111-130 once the host has
 * ranked the tuples.  `inv_rank[rank] = flat index` (NULL when tiebreak_rank is NULL).
 * One segment = `no_restriction` (smt_helper.py:102-146); one segment per matrix = `norm_dist`
 * (smt_helper.py:81-100).  NaN scores are not supported (the reference's order is unspecified). */
SMT_API size_t smt_topk_workspace_bytes(int64_t n_scores);
SMT_API int smt_topk_blocks(const float* scores, const uint32_t* tiebreak_rank, const uint32_t* inv_rank,
                    int64_t n_scores, const int32_t* seg_offsets, const int32_t* seg_k,
                    const int32_t* out_offsets, int num_segments, int32_t* out_idx,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ---- compact <-> dense block movement ------------------------------------------------ */

/* compact[i] <- W_i[block]  — LinearLayer_MatrixSparsity.__init__, smt.py:317-325. */
SMT_API int smt_block_gather(const smt_block_ref* table, int n_blocks, int block, int elem_bytes,
                     void* compact, void* stream);
/* W_i[block] <- compact[i]  — the scatter loop of forward, smt.py:332-341, and
 * convert_matrix_sparsity_to_linear_layer, smt.py:427-439. */
SMT_API int smt_block_scatter(const smt_block_ref* table, int n_blocks, int block, int elem_bytes,
                      const void* compact, void* stream);

/* ---- channel (input-column) movement for the channel-sparsity layer -------------------- */

/* out[t, i] <- x[t, idx[i]], t in [0, T), i in [0, n): the packed copy of the selected input channels that
 * linearChannel.forward saves for backward (smt.py:240-247, n strided slice copies there).  `ldx` in elements. */
SMT_API int smt_channel_gather(const void* x, int64_t T, int64_t ldx, const int32_t* idx, int n, int elem_bytes,
                       void* out, void* stream);
/* compact[i, o] <- W[o, idx[i]]  (LinearLayer_ChannelSparsity.__init__, smt.py:198-200) and
 * W[o, idx[i]] <- compact[i, o]  (its forward, smt.py:208-211), o in [0, out_features).  The reference copies weight
 * ROW idx[i] although idx are input channels and its gradient (smt.py:283-284) is that of weight COLUMN idx[i]; the
 * column form here is the consistent one (identical gradient formula, works for non-square weights).
 * `compact` is a contiguous [n, out_features] array; idx must not repeat for the scatter. */
SMT_API int smt_column_gather(const void* W, int64_t ldw, int out_features, int in_features, const int32_t* idx,
                      int n, int elem_bytes, void* compact, void* stream);
SMT_API int smt_column_scatter(void* W, int64_t ldw, int out_features, int in_features, const int32_t* idx, int n,
                       int elem_bytes, const void* compact, void* stream);

/* ---- block-gradient contraction (linearZ.backward, smt.py:386-404) -------------------- */

/* G[i*b + o, k] (+)= sum_t dy[t, row_i*b + o] * x[t, col_i*b + k],  t in [0, T).
 * x: [T, in_features] (ldx), dy: [T, out_features] (lddy), both `in_dtype`.
 * bf16/f16 inputs run the TMA-fed tcgen05/TMEM grouped kernel with fp32 accumulation over all T
 * (one rounding, to `out_dtype`); f32 inputs run an fp32 FMA kernel (exact-order-free, 1e-5 class).
 * `block_rc` is a device int32 [n_blocks][2] table of (row, col).
 * `accumulate` != 0 adds into G instead of overwriting it.
 * Workspace contract: the buffer must be ZERO-initialised once when it is allocated and must not be shared with other
 * entry points or with launches running concurrently on other streams: its first 16 KiB hold split-K arrival counters
 * that the kernel re-arms itself (all-zero again when the launch completes). */
SMT_API size_t smt_block_grad_gemm_workspace_bytes(int n_blocks, int block, int64_t T, int in_dtype);
SMT_API int smt_block_grad_gemm(const void* x, int64_t ldx, int in_features,
                        const void* dy, int64_t lddy, int out_features,
                        int64_t T, int in_dtype,
                        const int32_t* block_rc, int n_blocks, int block,
                        void* G, int out_dtype, int accumulate,
                        void* workspace, size_t workspace_bytes, void* stream);
/* Grouped form: the blocks of SEVERAL (x, dy) problems (e.g. every module whose backward ran since the last
 * flush) in one launch.  `maps` is a device array of 128-byte TMA descriptors produced on the host by
 * smt_encode_operand_map (one per distinct x or dy operand, all with the same T and dtype); `items` is a device
 * array with one entry per block: which dy / x descriptor, which block (row, col), and where its b x b result goes
 * (`out_off` = element offset from `out_base`, a multiple of 8).  Same arithmetic and determinism as the
 * single-problem call.
 * Item order is execution order.  A launch of b = 256 blocks large enough to need no split-K runs on SM pairs
 * (tcgen05 cta_group::2): items (2c, 2c+1) go to CTA pair c, which loads the dy strip once when the two items have the
 * same `map_dy` and `row` - so callers should place row-sharing blocks on such positions (ops.BlockGradBatch does).
 * SMT_GEMM_2SM=0 in the environment selects the single-CTA kernel (bit-identical results). */
typedef struct smt_gemm_item {
  uint32_t map_dy;   /* index into maps: descriptor of the dy operand   */
  uint32_t map_x;    /* index into maps: descriptor of the x operand    */
  int32_t  row;      /* block row    (out_features / b index)            */
  int32_t  col;      /* block column (in_features  / b index)            */
  int64_t  out_off;  /* element offset of this block's [b, b] output     */
  uint32_t flags;    /* SMT_ITEM_* bits                                   */
  int32_t  sq_slot;  /* >= 0: sq_partials[sq_slot], [sq_slot + 1] receive the sum of squares of the values STORED for
                        this block (after accumulation and rounding to out_dtype; upper / lower half of the rows for
                        b = 256, [total, 0] for smaller blocks); < 0: none                                            */
} smt_gemm_item;
/* item flag: overwrite this block's output even when the launch-level `accumulate` is set (first micro-batch after a
 * lazy zero_grad: no memset of the gradient buffer, no read-modify-write in the epilogue) */
enum { SMT_ITEM_OVERWRITE = 1 };
/* `block` = the block size of the launch the descriptor will be used in (it fixes the TMA box height). */
SMT_API int smt_encode_operand_map(void* map_host, const void* base, int64_t features, int64_t T, int64_t ld,
                                   int dtype, int block);
SMT_API size_t smt_block_grad_gemm_grouped_workspace_bytes(int n_items, int block, int64_t T);
/* 1 when a grouped launch of this shape runs the cta_group::2 kernel, 0 when it runs single-CTA tiles (introspection
 * for tests and reports; depends on the planner and on SMT_GEMM_2SM). */
SMT_API int smt_block_grad_gemm_grouped_uses_2sm(int n_items, int block, int64_t T);
/* `sq_partials` (device, fp32, may be NULL): per-block sums of squares, see smt_gemm_item.sq_slot.  They are produced by
 * the launches that need no split-K (smt_block_grad_gemm_grouped_emits_sq tells); the sums are deterministic (fixed
 * order inside each CTA) and feed the clip of smt_compact_adam without a separate pass over the gradient buffer. */
SMT_API int smt_block_grad_gemm_grouped_emits_sq(int n_items, int block, int64_t T);
/* `ld_out`: row pitch of every output tile in elements; 0 = compact storage (pitch = block).  A larger pitch lets the
 * tiles of one launch assemble a plain row-major matrix (item (r, c) -> out_off = r*b*ld_out + c*b): the channel-sparsity
 * gradient `partial_input^T @ grad_output` (smt.py:283-284) runs through this form, with the `dy` operand = the packed
 * selected input channels [T, n] (TMA zero-fills the columns past n) and the `x` operand = grad_output. */
SMT_API int smt_block_grad_gemm_grouped(const void* maps, const smt_gemm_item* items, int n_items,
                                        int64_t T, int block, int in_dtype, void* out_base, int out_dtype,
                                        int accumulate, int64_t ld_out, float* sq_partials, void* workspace,
                                        size_t workspace_bytes, void* stream);
/* Strip-sharing form of the single-problem call: a tile is a RUN - one block row and up to
 * smt_block_grad_gemm_run_width(block) (4 / 2 / 2 for b = 64 / 128 / 256) of its selected block columns - so the dy strip
 * is fetched once per run and the x strips form one wide UMMA operand (b = 256: one 128-row half of the block row per
 * run, `half`).  Same arithmetic as smt_block_grad_gemm (fp32 accumulation over all T, one rounding; deterministic).
 * The caller forms the runs (ops.block_grad_gemm does, from the Python index list) and passes them as a DEVICE array;
 * `out_blk[j]` is the position of block (row, cols[j]) in the index list, i.e. its result goes to G + out_blk[j]*b*b. */
typedef struct smt_gemm_run {
  int32_t row;         /* block row (dy strip)                                        */
  int32_t half;        /* b = 256: 0 / 1 = rows [0,128) / [128,256) of the block; else 0 */
  int32_t ncols;       /* 1 .. run width                                               */
  int32_t cols[4];     /* block columns (x strips)                                     */
  int32_t out_blk[4];  /* index of (row, cols[j]) in the caller's block list           */
  int32_t pad_;
} smt_gemm_run;
SMT_API int smt_block_grad_gemm_run_width(int block);
SMT_API size_t smt_block_grad_gemm_runs_workspace_bytes(int n_runs, int block, int64_t T);
SMT_API int smt_block_grad_gemm_runs(const void* x, int64_t ldx, int in_features,
                                     const void* dy, int64_t lddy, int out_features,
                                     int64_t T, int in_dtype, const smt_gemm_run* runs, int n_runs, int block,
                                     void* G, int out_dtype, int accumulate,
                                     void* workspace, size_t workspace_bytes, void* stream);
/* debug: register a device buffer of 8*max_ctas uint64; each CTA of smt_block_grad_gemm stamps %globaltimer at its
 * phase boundaries (tools/trace_gemm.py). NULL switches tracing off. Not for production use. */
SMT_API int smt_debug_set_gemm_trace(void* dev_buf, int max_ctas);
/* introspection for tests/bench: split-K factor and CTA count the launch above would use. */
SMT_API int smt_block_grad_gemm_plan(int n_blocks, int block, int64_t T, int in_dtype,
                             int* splits_host, int* ctas_host);

/* ---- dense side of linearZ, fused over modules that share their input (q, k, v of a decoder layer) ------------- */

/* forward:  y_j[T, N_j] = x[T, K] . W_j[N_j, K]^T  for j < n_seg (<= 3)   — linearZ.forward, smt.py:366, once instead of
 *           once per module; x is read once, the N tiles of [W_0; W_1; W_2] are walked as one weight.
 * dgrad:    dx[T, K]   = sum_j dy_j[T, N_j] . W_j[N_j, K]                 — linearZ.backward's grad_input, smt.py:406,
 *           for all modules at once: the reduction runs through the n_seg (dy_j, W_j) pairs into one accumulator, so
 *           the elementwise adds autograd inserts between three separate results disappear.
 * Hand-written persistent tcgen05 kernel (cta_group::2, 256 x 256 tiles, TMA-fed, double-buffered TMEM accumulators),
 * fp32 accumulation, one rounding to `dtype` (bf16 / f16 = the dtype of every operand and result).
 * Constraints (smt_fused_linear_supported tells): K % 64 == 0; N_j % 64 == 0, and N_j % 256 == 0 for forward (an N tile
 * must not straddle two modules); 16-byte aligned pointers and row pitches; any T (edge tiles are clipped).
 * `*_host` arrays live in HOST memory (n_seg entries); all matrices are device pointers, row-major, `ld*` in elements. */
SMT_API int smt_fused_linear_supported(int n_seg, const int* N_host, int K, int dtype, int dgrad);
SMT_API int smt_fused_linear_forward(const void* x, int64_t ldx, int64_t T, int K, int n_seg,
                                     const void* const* W_host, const int64_t* ldw_host, const int* N_host,
                                     void* const* y_host, const int64_t* ldy_host, int dtype, void* stream);
SMT_API int smt_fused_linear_dgrad(const void* const* dy_host, const int64_t* lddy_host, int64_t T, int K, int n_seg,
                                   const void* const* W_host, const int64_t* ldw_host, const int* N_host,
                                   void* dx, int64_t lddx, int dtype, void* stream);

/* ---- elementwise work of a LLaMA decoder layer (bf16, fp32 arithmetic, deterministic) -------------------------------
 * All tensors are contiguous bf16 (rstd: fp32) with 16-byte aligned storage.  The forward kernels reproduce the
 * roundings of the HF modules they replace (transformers' LlamaRMSNorm, apply_rotary_pos_emb, LlamaMLP's
 * `act_fn(gate) * up`), one bf16 rounding per PyTorch op. */

/* RMSNorm over rows of H elements (H % 8 == 0, H <= 32768), T rows:
 *   res == NULL:  x = a
 *   res != NULL:  x = bf16(res + a), written to h_out       (the residual add in front of the norm)
 *   rstd[t] = rsqrt(mean(x^2) + eps)   (fp32, kept for backward)
 *   y = bf16(w * bf16(x * rstd))       (HF's two roundings; only the order of the row sum differs) */
SMT_API int smt_rmsnorm_forward(const void* a, const void* res, const void* w, int64_t T, int H, float eps,
                                void* h_out, void* y, float* rstd, void* stream);
/* Input gradient of the norm above for a frozen weight (no dw):
 *   g = dy * w,  xhat = x * rstd,  dx = bf16(rstd * (g - xhat * mean(g * xhat)) [+ dres])
 * `dres` (optional) is the gradient that reaches x along the residual stream; adding it here replaces autograd's
 * separate bf16 add at the fork.  `x` is the norm's input (h_out of a residual forward). */
SMT_API int smt_rmsnorm_backward(const void* x, const void* w, const float* rstd, const void* dy,
                                 const void* dres, int64_t T, int H, void* dx, void* stream);
/* Rotary position embedding of q [B, S, Hq, 128] and k [B, S, Hk, 128] in one launch (the memory layout of the
 * q/k projections' outputs).  cos / sin: [*, S, 128], batch stride `cs_bstride` elements (0 = shared by the batch).
 *   forward   out = bf16(bf16(x * cos) + bf16(rotate_half(x) * sin)),  rotate_half(x) = (-x[64:], x[:64])
 *   backward  the transpose with autograd's roundings:
 *             dx = bf16(bf16(g * cos) + t),  t[:64] = bf16(g[64:] * sin[64:]),  t[64:] = -bf16(g[:64] * sin[:64])
 * Outputs are separate tensors of the inputs' shape. */
SMT_API int smt_rope_forward(const void* q, const void* k, const void* cos_, const void* sin_, int B, int S, int Hq,
                             int Hk, int64_t cs_bstride, void* q_out, void* k_out, void* stream);
SMT_API int smt_rope_backward(const void* dq_out, const void* dk_out, const void* cos_, const void* sin_, int B, int S,
                              int Hq, int Hk, int64_t cs_bstride, void* dq, void* dk, void* stream);
/* SwiGLU over n elements (n % 8 == 0):
 *   forward   h  = bf16(bf16(silu(g)) * u)
 *   backward  du = bf16(dh * bf16(silu(g))),  dg = bf16(silu'(g) * bf16(dh * u))   (torch's silu_backward formula) */
SMT_API int smt_swiglu_forward(const void* g, const void* u, int64_t n, void* h, void* stream);
SMT_API int smt_swiglu_backward(const void* g, const void* u, const void* dh, int64_t n, void* dg, void* du,
                                void* stream);

/* ---- causal-LM loss --------------------------------------------------------------------- */

/* Causal-LM cross-entropy over rows of bf16 logits (transformers' ForCausalLMLoss for one chunk of rows), with the
 * gradient written over the logits:
 *   lse_t   = m_t + log(sum_v exp(x[t,v] - m_t))                          (fp32)
 *   loss[t] = lse_t - x[t, y_t]   (0 where y_t == ignore_index; NaN where y_t is outside [0, V))
 *   x[t,v] <- bf16(scale * (exp(x[t,v] - lse_t) - [v == y_t]))            (the whole row 0 where y_t == ignore_index,
 *                                                                          NaN where y_t is outside [0, V))
 * scale: device fp32 scalar (1 / number of valid labels, or 1 / num_items_in_batch), read on the device (no host sync).
 * V % 8 == 0, ldl % 8 == 0, 16-byte aligned logits; int64 labels.  Deterministic (no atomics). */
SMT_API int smt_cross_entropy_rows(void* logits, int64_t ldl, int64_t T, int V, const int64_t* labels,
                                   int64_t ignore_index, const float* scale, float* loss_rows, void* stream);

/* ---- compact optimizer ---------------------------------------------------------------- */

/* out_sqnorm[0] = sum grad[i]^2 (fp32, deterministic two-stage tree). workspace: 4 KiB floats. */
SMT_API size_t smt_grad_sqnorm_workspace_bytes(void);
SMT_API int smt_grad_sqnorm(const void* grad, int grad_dtype, int64_t n, float* out_sqnorm,
                    void* workspace, size_t workspace_bytes, void* stream);

/* AdamW step (DeepSpeed FusedAdam adam_w_mode, fine_tune.py:352-363) over the flat compact state,
 * fused with global-norm clipping (deepspeed_helpers.py:87) and with the write-back of the updated
 * blocks into the dense weights (smt.py:332-341), so no scatter is needed in forward.
 *   g      = grad * grad_scale * clip,   clip = min(1, max_norm / (grad_scale*sqrt(S) + 1e-6)),
 *            S = sqnorm[0] + ... + sqnorm[n_sqnorm-1] summed in a fixed order inside the kernel (n_sqnorm = 1: the
 *            scalar of smt_grad_sqnorm; > 1: the per-block partials of the GEMM epilogue or per-chunk partials of a
 *            data-parallel exchange);  clip = 1 when sqnorm == NULL or max_norm <= 0
 *   m      = b1*m + (1-b1)*g ;  v = b2*v + (1-b2)*g*g
 *   update = (m/bc1) / (sqrt(v/bc2) + eps) + wd*p ;  p -= lr*update        (p = fp32 master)
 * then compact_out[i] (optional) and W blocks (optional, via `table`) receive p rounded to their
 * dtype.  bias corrections bc1/bc2 are passed by the host (1 - beta^step, computed in double). */
SMT_API int smt_compact_adam(float* master, float* exp_avg, float* exp_avg_sq,
                     const void* grad, int grad_dtype, int64_t n_elems,
                     float lr, float beta1, float beta2, float eps, float weight_decay,
                     float bias_correction1, float bias_correction2,
                     float grad_scale, const float* sqnorm, int n_sqnorm, float max_norm,
                     void* compact_out, int compact_dtype,
                     const smt_block_ref* table, int n_blocks, int block, int w_dtype,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* SMT_B200_H_ */
