// Strip-sharing tiles for the block-gradient contraction of linearZ.backward (reference deepspeed/smt/smt.py:386-404):
//
//     G[i*b + o, k] = sum_t dy[t, row_i*b + o] * x[t, col_i*b + k]
//
// A tile of the plain kernel (block_grad_gemm.cu) is ONE selected block: per pipeline stage it fills b features of dy and
// b features of x into shared memory for b*b MACs per token, i.e. b/2 flop per byte - 32 (b = 64) and 64 (b = 128)
// against the 128 of a 256-block, which is why those sizes sat at 1/4 and 1/2 of the whole-block rate (round-1 profile,
// section 1c/1d).  Blocks of one block ROW share their dy strip, so here a tile is a RUN: one block row and up to
// kRunWidth(b) of its selected block columns.  The dy strip is loaded once per stage and the x strips of the run sit side by
// side in shared memory, forming one UMMA B operand of N = ncols*b columns:
//
//     b = 64   up to 4 blocks per tile   1 + 4 TMA boxes of 96 tokens per stage, 3 stages   M = 128 (upper half unused), N <= 256
//     b = 128  up to 2 blocks per tile   2 + 4 boxes of 64 tokens, 4 stages                 M = 128, N <= 256
//
// There is no b = 256 form: a run of two 256-blocks needs 80 KiB per 64-token stage, and two such stages cannot hide HBM
// latency (measured 37.8 us against 29.6 us for the plain kernel's whole-block tiles on 12 clustered blocks).
//
// Split-K over tokens for few tiles: one wave of CTAs, cooperative launch, partial tiles in an fp32 workspace, reduced in
// the kernel by the split-K reduction that the plain kernel also calls (fused_splitk_reduce in gemm_epilogue.cuh: every
// sibling CTA sums its slice in the fixed order 0..splits-1; deterministic, no atomics on data).  The host
// (ops.block_grad_gemm) forms the runs from the Python index list, keeps the device copy cached per list, and takes this
// path when enough blocks share a row.
#include <cuda.h>
#include <string.h>

#include "common.cuh"
#include "umma_ptx.cuh"
#include "gemm_epilogue.cuh"
#include "tma_host.cuh"

namespace smt {
namespace {

constexpr int kRunThreads = 64 + 32 * 8;        // warp 0 TMA, warp 1 MMA + TMEM, warps 2-9 epilogue
constexpr int kRunEpiWarps = 8;

// Tokens per pipeline stage for b = 64 / 128 (measured: profiles/r02_runs_variants_raw.txt).  A launch whose strips
// come from HBM needs >= 3 stages to hide the load latency, and every TMA box costs the producer ~70 clk whatever its
// height - so the tallest box that still leaves 3-4 stages wins: b = 64: 96 tokens (5 boxes, 60 KiB, 3 stages: 115.6 us
// on 716 blocks x T 8192, against 140.0 with 64-token and 119.6 with 80-token stages); b = 128: 64 tokens (6 boxes,
// 48 KiB, 4 stages; 80 tokens x 3 stages measured the same).  128-token stages (two stages only) were no better than
// the plain kernel.
constexpr int kRunKTile64 = 96;
constexpr int kRunKTile128 = 64;

template <int B>
struct RunCfg {
  static_assert(B == 64 || B == 128, "run tiles exist for b = 64 / 128 only");
  static constexpr int NW = B == 64 ? 4 : 2;                 // blocks per run
  static constexpr int KT = B == 128 ? kRunKTile128 : kRunKTile64;   // tokens per pipeline stage
  static constexpr int CHUNK = KT * 128;                     // one {64 features x KT tokens} TMA box
  static constexpr int A_LOAD = B == 64 ? 1 : 2;             // dy chunks (the M = 128 operand of b = 64 aliases the next chunk)
  static constexpr int B_PER_BLOCK = B / 64;
  static constexpr int B_MAX = NW * B_PER_BLOCK;             // 4, 4
  static constexpr int STAGE_BYTES = (A_LOAD + B_MAX) * CHUNK;   // 60 / 48 KiB
  static constexpr int STAGES = (200 * 1024) / STAGE_BYTES;      // 3 / 4
  static constexpr int TILE_ROWS = B == 64 ? 64 : 128;       // output rows of one block that a tile produces
  static constexpr int SLOT = TILE_ROWS * B;                 // elements of one block's part of a tile
  static constexpr int TMEM_COLS = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;
  static_assert(STAGES * STAGE_BYTES >= kRunEpiWarps * 32 * kStageRow * 4, "epilogue staging must fit");
};

struct RunParams {
  const smt_gemm_run* runs;
  void* out;
  float* ws;             // fp32 partial slots when splits > 1: [(run * splits + split) * NW + j][SLOT]
  int* counters;         // 2 self-resetting ints per run (splits > 1)
  int splits;
  int kt_total, kt_per_split;
  int out_dtype;
  int accumulate;
  int in_fmt;
};

template <int B>
__global__ void __launch_bounds__(kRunThreads, 1) block_grad_runs_kernel(const __grid_constant__ CUtensorMap tmap_x,
                                                                         const __grid_constant__ CUtensorMap tmap_dy,
                                                                         const RunParams p) {
  using C = RunCfg<B>;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[C::STAGES];
  __shared__ __align__(8) uint64_t empty_bar[C::STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x, split = blockIdx.y;
  const smt_gemm_run run = p.runs[tile];
  const int ncols = run.ncols;
  const int kt_begin = split * p.kt_per_split;
  const int kt_end = min(kt_begin + p.kt_per_split, p.kt_total);
  const int n_kt = kt_end - kt_begin;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  auto a_addr = [&](int stage) { return smem_base + stage * C::STAGE_BYTES; };
  auto b_addr = [&](int stage) { return smem_base + stage * C::STAGE_BYTES + C::A_LOAD * C::CHUNK; };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmap_x);
    prefetch_tmap(&tmap_dy);
    for (int s = 0; s < C::STAGES; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_slot), C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===== TMA producer: the dy strip once, then the x strip of every block of the run =====
    if (lane == 0) {
      const int a_col0 = run.row * B;
      const uint32_t tx = (uint32_t)((C::A_LOAD + ncols * C::B_PER_BLOCK) * C::CHUNK);
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % C::STAGES;
        const uint32_t phase = (uint32_t)(it / C::STAGES) & 1u;
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
        const uint32_t fb = smem_u32(&full_bar[stage]);
        mbar_expect_tx(fb, tx);
        const int t0 = (kt_begin + it) * C::KT;
#pragma unroll
        for (int c = 0; c < C::A_LOAD; ++c) tma_load_2d(a_addr(stage) + c * C::CHUNK, &tmap_dy, fb, a_col0 + c * 64, t0);
        for (int j = 0; j < ncols; ++j) {
          const int col = run.cols[j] * B;
#pragma unroll
          for (int c = 0; c < C::B_PER_BLOCK; ++c)
            tma_load_2d(b_addr(stage) + (j * C::B_PER_BLOCK + c) * C::CHUNK, &tmap_x, fb, col + c * 64, t0);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: ONE instruction over all the run's columns =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(p.in_fmt, 128, ncols * B);
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % C::STAGES;
        const uint32_t phase = (uint32_t)(it / C::STAGES) & 1u;
        mbar_wait(smem_u32(&full_bar[stage]), phase);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < C::KT / 16; ++k) {
          const uint64_t adesc = make_desc_mn_sw128(a_addr(stage) + k * 2048, C::CHUNK, 1024);
          const uint64_t bdesc = make_desc_mn_sw128(b_addr(stage) + k * 2048, C::CHUNK, 1024);
          umma_f16(tmem_base, adesc, bdesc, idesc, (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(smem_u32(&empty_bar[stage]));
      }
      umma_commit(smem_u32(&tmem_full_bar));
    }
  } else {
    // ===== epilogue: every block of the run, TMEM -> registers -> smem transpose -> coalesced stores =====
    const int ew = warp - 2, q = warp & 3, par = ew >> 2;
    mbar_wait(smem_u32(&tmem_full_bar), 0);
    tc_fence_after();
    if (q * 32 < C::TILE_ROWS) {
      float* stage = reinterpret_cast<float*>(smem_gen) + ew * 32 * kStageRow;
      const bool final_out = (p.splits == 1);
      const int row_in_block = q * 32;
#pragma unroll 1
      for (int j = 0; j < ncols; ++j) {
        float* part = p.ws + (((int64_t)tile * p.splits + split) * C::NW + j) * C::SLOT;
        const int64_t out0 = (int64_t)run.out_blk[j] * B * B + (int64_t)row_in_block * B;
#pragma unroll 1
        for (int cc = par; cc < B / 32; cc += kRunEpiWarps / 4) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * B + cc * 32), r);
          tmem_ld_wait();
          if (!final_out)
            store_subtile<SMT_F32, false>(stage, r, lane, part, (int64_t)(q * 32) * B + cc * 32, B);
          else
            store_subtile_any(p.out_dtype, p.accumulate != 0, stage, r, lane, p.out, out0 + cc * 32, B);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }

  if (p.counters != nullptr) {
    // a split's partial of the run is one tile of NW slots; element e lives in slot e / SLOT of the run
    fused_splitk_reduce(p.counters + 2 * tile, split, p.splits, p.ws + (int64_t)tile * p.splits * C::NW * C::SLOT,
                        C::NW * C::SLOT, ncols * C::SLOT, p.out, p.out_dtype, p.accumulate != 0,
                        [&](int e) { return (int64_t)run.out_blk[e / C::SLOT] * B * B + e % C::SLOT; },
                        "smt_block_grad_gemm_runs");
  }
}

// ---- host side ------------------------------------------------------------------------------------------

int encode_strip_map(CUtensorMap* map, const void* base, int64_t features, int64_t T, int64_t ld, int in_dtype, int ktile) {
  return encode_2d_sw128(map, base, features, T, ld, in_dtype, ktile, "smt_block_grad_gemm_runs");
}

struct RunPlan {
  int splits, kt_total, kt_per_split;
};

int run_ktile(int block) { return block == 128 ? kRunKTile128 : kRunKTile64; }
int run_width(int block) { return block == 64 ? 4 : 2; }
bool runs_block_ok(int block) { return block == 64 || block == 128; }
int run_slot(int block) { return (block == 64 ? 64 : 128) * block; }

// One wave: the token range is split so that n_runs * splits CTAs fill the SMs once (the reduction is fused into the
// kernel, which needs all CTAs resident); at least 512 tokens per split; more tiles than SMs => no split, several waves.
RunPlan make_run_plan(int n_runs, int block, int64_t T) {
  RunPlan pl{};
  const int kt = run_ktile(block);
  pl.kt_total = (int)((T + kt - 1) / kt);
  int s = n_runs > 0 ? sm_count() / n_runs : 1;
  const int max_s = (int)(T / 512);
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  pl.kt_per_split = (pl.kt_total + s - 1) / s;
  pl.splits = (pl.kt_total + pl.kt_per_split - 1) / pl.kt_per_split;
  return pl;
}

size_t run_workspace_bytes(int n_runs, int block, const RunPlan& pl) {
  if (pl.splits <= 1) return 0;
  return kSplitCounterBytes + (size_t)n_runs * run_width(block) * pl.splits * run_slot(block) * sizeof(float);
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API int smt_block_grad_gemm_run_width(int block) { return runs_block_ok(block) ? run_width(block) : 0; }

extern "C" SMT_API size_t smt_block_grad_gemm_runs_workspace_bytes(int n_runs, int block, int64_t T) {
  if (n_runs <= 0 || T <= 0 || !runs_block_ok(block)) return 0;
  return run_workspace_bytes(n_runs, block, make_run_plan(n_runs, block, T));
}

extern "C" SMT_API int smt_block_grad_gemm_runs(const void* x, int64_t ldx, int in_features, const void* dy, int64_t lddy,
                                                int out_features, int64_t T, int in_dtype, const smt_gemm_run* runs,
                                                int n_runs, int block, void* G, int out_dtype, int accumulate,
                                                void* workspace, size_t workspace_bytes, void* stream) {
  SMT_CHECK_ARG(n_runs >= 0 && T > 0, "smt_block_grad_gemm_runs: needs T > 0 and n_runs >= 0");
  if (n_runs == 0) return SMT_OK;
  SMT_CHECK_ARG(runs_block_ok(block), "smt_block_grad_gemm_runs: block size %d not in {64,128} (b = 256 has no run tiles)",
                block);
  SMT_CHECK_ARG(x && dy && G && runs, "smt_block_grad_gemm_runs: null pointer");
  SMT_CHECK_ARG((in_dtype == SMT_BF16 || in_dtype == SMT_F16) && out_dtype >= SMT_F32 && out_dtype <= SMT_F16,
                "smt_block_grad_gemm_runs: 16-bit inputs only");
  SMT_CHECK_ARG(in_features > 0 && out_features > 0 && in_features % block == 0 && out_features % block == 0,
                "smt_block_grad_gemm_runs: features (%d in, %d out) must be multiples of block %d", in_features,
                out_features, block);
  SMT_CHECK_ARG(ldx >= in_features && lddy >= out_features && aligned16(x) && aligned16(dy) && aligned16(G) &&
                    (ldx * 2) % 16 == 0 && (lddy * 2) % 16 == 0,
                "smt_block_grad_gemm_runs: operands must be 16-byte aligned (pointer and row pitch)");
  SMT_CHECK_ARG(T < (1ll << 31) - 256, "smt_block_grad_gemm_runs: T too large");
  const RunPlan pl = make_run_plan(n_runs, block, T);
  int* counters;
  float* partials;
  if (int rc = carve_split_workspace("smt_block_grad_gemm_runs", workspace, workspace_bytes,
                                     run_workspace_bytes(n_runs, block, pl), &counters, &partials))
    return rc;
  SMT_CHECK_ARG(counters == nullptr || (size_t)n_runs * 2 * sizeof(int) <= kSplitCounterBytes,
                "smt_block_grad_gemm_runs: too many runs for a split launch");
  CUtensorMap mx, mdy;
  if (int rc = encode_strip_map(&mx, x, in_features, T, ldx, in_dtype, run_ktile(block))) return rc;
  if (int rc = encode_strip_map(&mdy, dy, out_features, T, lddy, in_dtype, run_ktile(block))) return rc;
  RunParams rp{};
  rp.runs = runs;
  rp.out = G;
  rp.ws = partials;
  rp.counters = counters;
  rp.splits = pl.splits;
  rp.kt_total = pl.kt_total;
  rp.kt_per_split = pl.kt_per_split;
  rp.out_dtype = out_dtype;
  rp.accumulate = accumulate;
  rp.in_fmt = in_dtype == SMT_BF16 ? 1 : 0;
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid(n_runs, pl.splits);
  const bool coop = counters != nullptr;
  const int rc = block == 128
                     ? launch_tiles(block_grad_runs_kernel<128>, grid, kRunThreads, RunCfg<128>::SMEM_BYTES, coop, st, mx, mdy, rp)
                     : launch_tiles(block_grad_runs_kernel<64>, grid, kRunThreads, RunCfg<64>::SMEM_BYTES, coop, st, mx, mdy, rp);
  if (rc) return rc;
  set_launch_count(1);
  return SMT_OK;
}
