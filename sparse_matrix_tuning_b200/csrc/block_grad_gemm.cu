// Block-gradient contraction of linearZ.backward (reference deepspeed/smt/smt.py:386-404):
//
//     G[i*b + o, k] = sum_t dy[t, row_i*b + o] * x[t, col_i*b + k]          for every selected block i
//
// The reference issues, per block, a batched cuBLAS bmm ([B,b,S]x[B,S,b]), a reduction over the batch and
// a slice copy (3 launches per block, results rounded to bf16 per batch entry).  Here ONE grouped launch
// covers every block of a module — or, through the grouped entry point, of every module whose backward ran
// since the last flush: a TMA-fed tcgen05/TMEM GEMM with fp32 accumulation over all T tokens and a single
// final rounding.
//
// Operand layout.  The reduction dimension is the token index t, the SLOW dimension of both row-major
// inputs, so both UMMA operands are "MN-major": A[m,k] = dy[k, row*b+m] has m contiguous, B[k,n] =
// x[k, col*b+n] has n contiguous.  A TMA box of {64 features, K_TILE tokens} with 128-byte swizzle lands
// in shared memory exactly as the canonical MN-major SWIZZLE_128B UMMA layout
// ((8,n),(8,k)):((1,LBO),(8,SBO)) [units of 16 B]: 8 token rows of 128 B form one 1024-B swizzle atom
// (SBO = 1024 B between 8-token groups) and consecutive 64-feature chunks are LBO = K_TILE*128 B apart.
//
// Work decomposition.  Work item = (tile, K-split); one CTA per item with 10 warps: TMA producer, MMA
// issuer / TMEM owner, 8 epilogue warps.  For b = 256 a tile is either the whole block (MH = 2: two M=128
// accumulators share one x strip, N = 256, all 512 TMEM columns, 256 flop per byte of shared-memory fill)
// or half a block (MH = 1: used when there are few blocks, it halves the split-K partial traffic).  With few
// tiles per launch the token range is split across CTAs and partial tiles go to an fp32 workspace.  When the
// grid fits in one wave the kernel is launched cooperatively and the reduction is fused: after a per-tile
// arrival counter, each sibling CTA sums its slice of the tile over all partials in the fixed order 0..splits-1.
// Larger grids use a second kernel (programmatic dependent launch hides its launch latency).  Either way the
// sum order is fixed: deterministic, no atomics on data.  The epilogue transposes 32x32 accumulator sub-tiles
// through shared memory so that every global store instruction writes whole 128-byte rows.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "umma_ptx.cuh"
#include "gemm_epilogue.cuh"
#include "tma_host.cuh"

namespace smt {
namespace {

// Tokens per pipeline stage (multiples of 16, <= 256 = the tallest TMA box), per block size.  Every stage carries a
// fixed cost (~100-150 clk per TMA box plus the barrier round trip) that a whole-block b = 256 tile hides behind
// 1 024 clk of UMMA work; the small tiles do not, so they take 128-token stages (half as many boxes and barrier
// round trips per token; +23-56 % on B200, profiles/r01_kernels.md section 1c).
constexpr int kKTile256 = 64;
constexpr int kKTile128 = 128;
constexpr int kKTile64 = 256;
constexpr int kMaxStages = 8;
constexpr int ktile_for(int block) {
  return block == 256 ? kKTile256 : block == 128 ? kKTile128 : kKTile64;
}
constexpr int kMaxKTile = 256;                // TMA box height limit
static_assert(ktile_for(256) % 16 == 0 && ktile_for(128) % 16 == 0 && ktile_for(64) % 16 == 0, "K tile");
static_assert(ktile_for(256) <= kMaxKTile && ktile_for(128) <= kMaxKTile && ktile_for(64) <= kMaxKTile, "K tile");
constexpr int kEpiWarps = 8;                  // multiple of 4 (one TMEM lane quarter per warp % 4)
constexpr int kGemmThreads = 64 + 32 * kEpiWarps;   // warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2-9 epilogue
constexpr int kSmemBudget = 200 * 1024;       // pipeline stages (dynamic smem), leaves room for barriers
constexpr int kMinTokensPerSplit = 256;

template <int B, int MH_>
struct Cfg {
  static constexpr int MH = MH_;                              // M=128 accumulators per CTA
  static constexpr int KT = ktile_for(B);                     // tokens per pipeline stage
  static constexpr int CHUNK_BYTES = KT * 128;                // one {64 features x KT tokens} TMA box of 16-bit data
  // dy chunks fetched per stage.  An M=128 MMA always spans two 64-row chunks.  For b = 64 only the first is loaded;
  // the second half of the operand aliases the x chunk that follows it in the stage (initialised shared memory; it
  // feeds accumulator rows 64..127, which are never read) instead of owning a slot.
  static constexpr int A_LOAD = B >= 128 ? 2 * MH : 1;
  static constexpr int B_LOAD = B / 64;                       // N = B
  static constexpr int TILES_PER_BLOCK = (B == 256 && MH == 1) ? 2 : 1;
  static constexpr int TILE_ROWS = B >= 128 ? 128 * MH : B;   // output rows one CTA produces
  static constexpr int TILE_ELEMS = TILE_ROWS * B;
  static constexpr int STAGE_BYTES = (A_LOAD + B_LOAD) * CHUNK_BYTES;
  static constexpr int STAGES_RAW = kSmemBudget / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > kMaxStages ? kMaxStages : STAGES_RAW;
  static constexpr int TX_BYTES = (A_LOAD + B_LOAD) * CHUNK_BYTES;
  static constexpr int TMEM_COLS = MH * B < 32 ? 32 : MH * B;  // 512 / 256 / 128 / 64 (powers of two)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024;  // + alignment slack
  static_assert(STAGES * STAGE_BYTES >= kEpiWarps * 32 * kStageRow * 4, "epilogue staging must fit in the pipeline smem");
};

// ---- the tcgen05 kernel ----------------------------------------------------------------------------

struct GemmParams {
  const int32_t* block_rc;        // single problem: [n_blocks][2] (row, col)
  const smt_gemm_item* items;     // grouped: one entry per block
  const CUtensorMap* maps;        // grouped: tensor maps in global memory (indexed by the items)
  void* out;                      // G base (single problem: block i at i*b*b; grouped: items[i].out_off)
  float* ws;                      // fp32 partial tiles when splits > 1
  float* sq;                      // grouped, no split-K: per-block sum-of-squares slots (items[i].sq_slot), or NULL
  int* counters;                  // fused reduction: 2 self-resetting ints per tile (NULL = separate reduce kernel)
  int64_t ld_out;                 // row pitch of an output tile in elements (== block for compact storage)
  int splits;
  int kt_total;                   // number of K tiles = ceil(T / ktile_for(block))
  int kt_per_split;
  int out_dtype;                  // of G; the workspace is always fp32
  int accumulate;
  int in_fmt;                     // 0 = f16, 1 = bf16
};

template <int B, int MH, bool GROUPED>
__global__ void __launch_bounds__(kGemmThreads, 1) block_grad_umma_kernel(
    const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy,
    const GemmParams p) {
  using C = Cfg<B, MH>;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[C::STAGES];
  __shared__ __align__(8) uint64_t empty_bar[C::STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_slot;
  __shared__ float sq_warp[kEpiWarps][2];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x, split = blockIdx.y;
  const int blk = tile / C::TILES_PER_BLOCK, half = tile % C::TILES_PER_BLOCK;
  const int kt_begin = split * p.kt_per_split;
  const int kt_end = min(kt_begin + p.kt_per_split, p.kt_total);
  const int n_kt = kt_end - kt_begin;  // >= 1 by construction of the plan

  // 1024-byte aligned pipeline buffers (SWIZZLE_128B atoms are 1024 B)
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  auto a_addr = [&](int stage) { return smem_base + stage * C::STAGE_BYTES; };
  auto b_addr = [&](int stage) { return smem_base + stage * C::STAGE_BYTES + C::A_LOAD * C::CHUNK_BYTES; };

  int row, col;
  const CUtensorMap* map_x = &tmap_x;
  const CUtensorMap* map_dy = &tmap_dy;
  int64_t out_off;                       // element offset of this tile's first output row
  bool acc_out = p.accumulate != 0;      // add into the output (an item may ask for a plain overwrite instead)
  int sq_slot = -1;
  if (GROUPED) {
    const smt_gemm_item item = p.items[blk];
    row = item.row; col = item.col;
    map_x = p.maps + item.map_x;
    map_dy = p.maps + item.map_dy;
    out_off = item.out_off + (int64_t)half * 128 * p.ld_out;
    if (item.flags & SMT_ITEM_OVERWRITE) acc_out = false;
    if (p.sq != nullptr && p.splits == 1) sq_slot = item.sq_slot;
  } else {
    row = p.block_rc[2 * blk]; col = p.block_rc[2 * blk + 1];
    out_off = (int64_t)tile * C::TILE_ELEMS;
  }

  if (warp == 0 && lane == 0) {
    prefetch_tmap(map_x);
    prefetch_tmap(map_dy);
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
  if (threadIdx.x == 0) pdl_launch_dependents();   // the split-K reduce grid may get scheduled (it waits for us)

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      const int a_col0 = row * B + half * 128;
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % C::STAGES;
        const uint32_t phase = (uint32_t)(it / C::STAGES) & 1u;
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
        const uint32_t fb = smem_u32(&full_bar[stage]);
        mbar_expect_tx(fb, C::TX_BYTES);
        const int t0 = (kt_begin + it) * C::KT;
#pragma unroll
        for (int c = 0; c < C::A_LOAD; ++c)
          tma_load_2d(a_addr(stage) + c * C::CHUNK_BYTES, map_dy, fb, a_col0 + c * 64, t0);
#pragma unroll
        for (int c = 0; c < C::B_LOAD; ++c)
          tma_load_2d(b_addr(stage) + c * C::CHUNK_BYTES, map_x, fb, col * B + c * 64, t0);
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      const uint32_t idesc = make_idesc(p.in_fmt, 128, B);
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % C::STAGES;
        const uint32_t phase = (uint32_t)(it / C::STAGES) & 1u;
        mbar_wait(smem_u32(&full_bar[stage]), phase);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < C::KT / 16; ++k) {
          // 16 tokens = two 8-row swizzle atoms = 2048 B further down every chunk
          const uint64_t bdesc = make_desc_mn_sw128(b_addr(stage) + k * 2048, C::CHUNK_BYTES, 1024);
#pragma unroll
          for (int mh = 0; mh < MH; ++mh) {
            const uint64_t adesc =
                make_desc_mn_sw128(a_addr(stage) + mh * 2 * C::CHUNK_BYTES + k * 2048, C::CHUNK_BYTES, 1024);
            umma_f16(tmem_base + mh * B, adesc, bdesc, idesc, (it > 0 || k > 0) ? 1u : 0u);
          }
        }
        umma_commit(smem_u32(&empty_bar[stage]));  // frees the smem stage when these MMAs retire
      }
      umma_commit(smem_u32(&tmem_full_bar));       // accumulators complete
    }
  } else {
    // ===== epilogue: TMEM -> registers -> smem transpose -> coalesced global stores =====
    const int ew = warp - 2;            // 0..7
    const int q = warp & 3;             // TMEM lane quarter this warp may access
    const int par = ew >> 2;            // kEpiWarps / 4 warps per quarter, interleaved over the column chunks
    constexpr int ROWS_PER_MH = B < 128 ? B : 128;
    mbar_wait(smem_u32(&tmem_full_bar), 0);
    tc_fence_after();
    float sq0 = 0.f, sq1 = 0.f;
    if (q * 32 < ROWS_PER_MH) {
      // all MMAs have retired => the pipeline buffers are dead; reuse them as transpose staging
      float* stage = reinterpret_cast<float*>(smem_gen) + ew * 32 * kStageRow;
      const bool final_out = (p.splits == 1);
      float* part = p.ws + ((int64_t)tile * p.splits + split) * C::TILE_ELEMS;
#pragma unroll 1
      for (int mh = 0; mh < MH; ++mh) {
#pragma unroll 1
        for (int cc = par; cc < B / 32; cc += kEpiWarps / 4) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mh * B + cc * 32), r);
          tmem_ld_wait();
          const int64_t off_in_tile = (int64_t)(mh * 128 + q * 32) * B + cc * 32;
          if (!final_out) {
            store_subtile<SMT_F32, false>(stage, r, lane, part, off_in_tile, B);
          } else {
            const int64_t off_out = out_off + (int64_t)(mh * 128 + q * 32) * p.ld_out + cc * 32;
            const float sv = store_subtile_any(p.out_dtype, acc_out, stage, r, lane, p.out, off_out, (int)p.ld_out);
            if (mh == 0) sq0 += sv; else sq1 += sv;
          }
        }
      }
    }
    if (sq_slot >= 0) {
      const float s0 = warp_sum(sq0), s1 = warp_sum(sq1);
      if (lane == 0) { sq_warp[ew][0] = s0; sq_warp[ew][1] = s1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
  if (sq_slot >= 0 && threadIdx.x == 0) {
    // fixed-order sum over the epilogue warps: deterministic.  Slot layout: [rows 0-127, rows 128-255] of a b = 256
    // block, [total, 0] for smaller blocks.
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int w = 0; w < kEpiWarps; ++w) { t0 += sq_warp[w][0]; t1 += sq_warp[w][1]; }
    if (C::TILES_PER_BLOCK == 2) {
      p.sq[sq_slot + half] = t0;
    } else {
      p.sq[sq_slot] = t0;
      p.sq[sq_slot + 1] = t1;
    }
  }

  if (p.counters != nullptr) {
    // element e of the (row-major, pitch B) tile lives at row e / B, column e % B of the output (pitch ld_out)
    fused_splitk_reduce(p.counters + 2 * tile, split, p.splits, p.ws + (int64_t)tile * p.splits * C::TILE_ELEMS,
                        C::TILE_ELEMS, C::TILE_ELEMS, p.out, p.out_dtype, acc_out,
                        [&](int e) { return out_off + (int64_t)(e / B) * p.ld_out + e % B; }, "smt_block_grad_gemm");
  }
}

// ---- 2-SM (cta_group::2) kernel: two whole b = 256 blocks per CTA pair ---------------------------------
//
// A cluster of two CTAs (one SM pair) works on TWO grouped work items.  Every UMMA is a `cta_group::2` instruction with
// M = 256 (CTA r owns dy rows [128 r, 128 r + 128) of the block and accumulator lanes for those rows) and N = 256 whose
// x operand is SPLIT across the pair (CTA r loads x columns [128 r, 128 r + 128) of the block): per 64-token stage a CTA
// fills  A0 (16 KiB) + B0 half (16 KiB) + A1 (16 KiB) + B1 half (16 KiB) = 64 KiB for the same UMMA work per SM as the
// single-CTA whole-block tile -- and only 48 KiB (4 instead of 3 stages) when the two items share their dy strip
// (same operand, same block row: the host places such pairs on positions (2c, 2c+1)), because A1 == A0 is then not
// loaded at all.  Fewer TMA boxes and bytes per unit of tensor work is what the single-CTA tile is short of
// (profiles/r01_kernels.md section 1b).
// Protocol (the CUTLASS sm100 2-SM scheme): both CTAs run a TMA producer that loads ITS halves with
// `cp.async.bulk.tensor...cta_group::2` signalling the LEADER's (cluster rank 0) full barrier, which expects the bytes
// of both CTAs; only the leader issues UMMAs; stage-free and accumulators-ready commits are multicast to both CTAs.

constexpr int k2smStageChunks = 8;                                   // A0, B0, A1, B1: two 64-feature chunks each
constexpr int k2smKTile = ktile_for(256);
constexpr int k2smChunkBytes = k2smKTile * 128;
constexpr int k2smMaxStages = 4;
constexpr int k2smSmemBytes = 3 * k2smStageChunks * k2smChunkBytes + 1024;   // 3 x 64 KiB = 4 x 48 KiB

__global__ void __launch_bounds__(kGemmThreads, 1) block_grad_umma_2sm_kernel(const GemmParams p, int n_items) {
  constexpr int B = 256, KT = k2smKTile, CB = k2smChunkBytes;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[k2smMaxStages];
  __shared__ __align__(8) uint64_t empty_bar[k2smMaxStages];
  __shared__ __align__(8) uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_slot;
  __shared__ float sq_warp[kEpiWarps][2];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();               // 0 = leader (issues the UMMAs)
  const int pair = blockIdx.x >> 1;
  const smt_gemm_item it0 = p.items[2 * pair];
  const bool has2 = 2 * pair + 1 < n_items;
  const smt_gemm_item it1 = has2 ? p.items[2 * pair + 1] : it0;
  const bool shared_a = has2 && it1.map_dy == it0.map_dy && it1.row == it0.row;
  // stage layout: [A0 | B0 | B1] (shared dy strip, 48 KiB, 4 stages) or [A0 | B0 | A1 | B1] (64 KiB, 3 stages)
  const int stage_bytes = (shared_a ? 6 : 8) * CB;
  const int n_stages = shared_a ? 4 : 3;
  const uint32_t off_b0 = 2 * CB, off_a1 = 4 * CB, off_b1 = shared_a ? 4 * CB : 6 * CB;
  const uint32_t my_bytes = (uint32_t)((has2 ? (shared_a ? 6 : 8) : 4) * CB);
  const int n_kt = p.kt_total;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  if (warp == 0 && lane == 0) {
    prefetch_tmap(p.maps + it0.map_x);
    prefetch_tmap(p.maps + it0.map_dy);
    for (int s = 0; s < k2smMaxStages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&tmem_full_bar), 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(smem_u32(&tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                  // both CTAs' barriers and TMEM exist before anything crosses the pair
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): my 128 dy rows and my 128 x columns of each block =====
    if (lane == 0) {
      const CUtensorMap* mdy0 = p.maps + it0.map_dy;
      const CUtensorMap* mx0 = p.maps + it0.map_x;
      const CUtensorMap* mdy1 = p.maps + it1.map_dy;
      const CUtensorMap* mx1 = p.maps + it1.map_x;
      const int a0 = it0.row * B + (int)rank * 128, b0 = it0.col * B + (int)rank * 128;
      const int a1 = it1.row * B + (int)rank * 128, b1 = it1.col * B + (int)rank * 128;
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % n_stages;
        const uint32_t phase = (uint32_t)(it / n_stages) & 1u;
        mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
        const uint32_t fb = smem_u32(&full_bar[stage]);
        if (rank == 0) mbar_expect_tx(fb, 2u * my_bytes);          // the leader's barrier counts both CTAs' bytes
        const uint32_t st = smem_base + (uint32_t)(stage * stage_bytes);
        const int t0 = it * KT;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          tma_load_2d_2sm(st + c * CB, mdy0, fb, a0 + c * 64, t0);
          tma_load_2d_2sm(st + off_b0 + c * CB, mx0, fb, b0 + c * 64, t0);
        }
        if (has2) {
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (!shared_a) tma_load_2d_2sm(st + off_a1 + c * CB, mdy1, fb, a1 + c * 64, t0);
            tma_load_2d_2sm(st + off_b1 + c * CB, mx1, fb, b1 + c * 64, t0);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== UMMA issuer: one thread of the leader CTA, on behalf of both SMs =====
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(p.in_fmt, 256, B);
      for (int it = 0; it < n_kt; ++it) {
        const int stage = it % n_stages;
        const uint32_t phase = (uint32_t)(it / n_stages) & 1u;
        mbar_wait(smem_u32(&full_bar[stage]), phase);
        tc_fence_after();
        const uint32_t st = smem_base + (uint32_t)(stage * stage_bytes);
#pragma unroll
        for (int k = 0; k < KT / 16; ++k) {
          const uint32_t acc = (it > 0 || k > 0) ? 1u : 0u;
          const uint64_t a0d = make_desc_mn_sw128(st + k * 2048, CB, 1024);
          umma2_f16(tmem_base, a0d, make_desc_mn_sw128(st + off_b0 + k * 2048, CB, 1024), idesc, acc);
          if (has2) {
            const uint64_t a1d = shared_a ? a0d : make_desc_mn_sw128(st + off_a1 + k * 2048, CB, 1024);
            umma2_f16(tmem_base + B, a1d, make_desc_mn_sw128(st + off_b1 + k * 2048, CB, 1024), idesc, acc);
          }
        }
        umma2_commit_multicast(smem_u32(&empty_bar[stage]), (uint16_t)0x3);   // frees the stage in both CTAs
      }
      umma2_commit_multicast(smem_u32(&tmem_full_bar), (uint16_t)0x3);        // accumulators complete, both CTAs
    }
  } else {
    // ===== epilogue (both CTAs): my 128 rows of each block =====
    const int ew = warp - 2, q = warp & 3, par = ew >> 2;
    mbar_wait(smem_u32(&tmem_full_bar), 0);
    tc_fence_after();
    float* stage = reinterpret_cast<float*>(smem_gen) + ew * 32 * kStageRow;   // pipeline buffers are dead by now
    float sq0 = 0.f, sq1 = 0.f;
#pragma unroll 1
    for (int blk = 0; blk < (has2 ? 2 : 1); ++blk) {
      const smt_gemm_item& item = blk == 0 ? it0 : it1;
      const int64_t out0 = item.out_off + (int64_t)((int)rank * 128 + q * 32) * p.ld_out;
      const bool acc_out = p.accumulate != 0 && !(item.flags & SMT_ITEM_OVERWRITE);
#pragma unroll 1
      for (int cc = par; cc < B / 32; cc += kEpiWarps / 4) {
        uint32_t r[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * B + cc * 32), r);
        tmem_ld_wait();
        const float sv = store_subtile_any(p.out_dtype, acc_out, stage, r, lane, p.out, out0 + cc * 32, (int)p.ld_out);
        if (blk == 0) sq0 += sv; else sq1 += sv;
      }
    }
    if (p.sq != nullptr) {
      const float s0 = warp_sum(sq0), s1 = warp_sum(sq1);
      if (lane == 0) { sq_warp[ew][0] = s0; sq_warp[ew][1] = s1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                  // nobody leaves (or frees TMEM) while the pair may still touch it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
  if (p.sq != nullptr && threadIdx.x == 0) {
    // this CTA stored rows [128 rank, 128 rank + 128) of both blocks: slot `rank` of each; fixed-order sum over the warps
    float t0 = 0.f, t1 = 0.f;
#pragma unroll
    for (int w = 0; w < kEpiWarps; ++w) { t0 += sq_warp[w][0]; t1 += sq_warp[w][1]; }
    if (it0.sq_slot >= 0) p.sq[it0.sq_slot + (int)rank] = t0;
    if (has2 && it1.sq_slot >= 0) p.sq[it1.sq_slot + (int)rank] = t1;
  }
}

// ---- split-K reduction: G = sum_s partial[s] (fixed order) -----------------------------------------

template <int ODT>
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ ws, void* __restrict__ out,
                                                            const smt_gemm_item* __restrict__ items,
                                                            int tile_elems, int tiles_per_block, int block,
                                                            int64_t ldo, int splits, int64_t n_vec8,
                                                            int accumulate_all) {
  pdl_wait();  // programmatic dependent launch: the GEMM grid's partial tiles are complete and visible
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t vec = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; vec < n_vec8; vec += stride) {
    const int64_t e = vec * 8;
    const int64_t tile = e / tile_elems;
    const int within = (int)(e - tile * tile_elems);
    float acc[8];
    sum_partials8<ld_stream_f4>(ws + tile * splits * tile_elems + within, splits, tile_elems, acc);
    int64_t o = e;
    int accumulate = accumulate_all;
    if (items != nullptr) {
      const smt_gemm_item& item = items[tile / tiles_per_block];
      o = item.out_off + ((int64_t)(tile % tiles_per_block) * 128 + within / block) * ldo + within % block;
      if (item.flags & SMT_ITEM_OVERWRITE) accumulate = 0;
    }
    if (ODT == SMT_F32) {
      float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + o);
      float4 v0 = make_float4(acc[0], acc[1], acc[2], acc[3]), v1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
      if (accumulate) {
        const float4 o0 = op[0], o1 = op[1];
        v0.x += o0.x; v0.y += o0.y; v0.z += o0.z; v0.w += o0.w;
        v1.x += o1.x; v1.y += o1.y; v1.z += o1.z; v1.w += o1.w;
      }
      op[0] = v0;
      op[1] = v1;
    } else {
      uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(out) + o);
      if (accumulate) {
        float old[8];
        unpack8<ODT>(*op, old);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] += old[j];
      }
      uint4 u;
      if (ODT == SMT_BF16) {
        u.x = pack_bf16x2(acc[0], acc[1]); u.y = pack_bf16x2(acc[2], acc[3]);
        u.z = pack_bf16x2(acc[4], acc[5]); u.w = pack_bf16x2(acc[6], acc[7]);
      } else {
        u.x = pack_f16x2(acc[0], acc[1]); u.y = pack_f16x2(acc[2], acc[3]);
        u.z = pack_f16x2(acc[4], acc[5]); u.w = pack_f16x2(acc[6], acc[7]);
      }
      *op = u;
    }
  }
}

// ---- fp32 path (parity configuration: fp32 models) --------------------------------------------------
// 64x64 output tile per CTA, 16-token slabs staged in shared memory, 4x4 register micro-tile per thread.

template <int ODT>
__global__ void __launch_bounds__(256) block_grad_f32_kernel(const float* __restrict__ x, int64_t ldx,
                                                             const float* __restrict__ dy, int64_t lddy,
                                                             int64_t T, const int32_t* __restrict__ block_rc,
                                                             int block, void* __restrict__ out, int accumulate) {
  __shared__ float sa[16][64 + 4];  // dy slab  [t][m]
  __shared__ float sb[16][64 + 4];  // x slab   [t][n]
  const int blk = blockIdx.x;
  const int tiles = block / 64;
  const int tm = blockIdx.y / tiles, tn = blockIdx.y % tiles;
  const int row = block_rc[2 * blk], col = block_rc[2 * blk + 1];
  const float* a0 = dy + (int64_t)row * block + tm * 64;
  const float* b0 = x + (int64_t)col * block + tn * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16 threads, 4 x 4 each
  const int lt = threadIdx.x >> 4, lc = (threadIdx.x & 15) * 4;  // loader: token lt, features lc..lc+3
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int64_t t0 = 0; t0 < T; t0 += 16) {
    float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
    if (t0 + lt < T) {
      va = *reinterpret_cast<const float4*>(a0 + (t0 + lt) * lddy + lc);
      vb = *reinterpret_cast<const float4*>(b0 + (t0 + lt) * ldx + lc);
    }
    __syncthreads();
    *reinterpret_cast<float4*>(&sa[lt][lc]) = va;
    *reinterpret_cast<float4*>(&sb[lt][lc]) = vb;
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 16; ++t) {
      const float4 a = *reinterpret_cast<const float4*>(&sa[t][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&sb[t][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t off = ((int64_t)blk * block + tm * 64 + ty * 4 + i) * block + tn * 64 + tx * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v = acc[i][j];
      if (accumulate) v += load_as_float<ODT>(out, off + j);
      store_from_float<ODT>(out, off + j, v);
    }
  }
}

// ---- host side ------------------------------------------------------------------------------------------

struct Plan {
  int mh;             // M=128 accumulators per CTA (2 = whole 256-block per CTA)
  int tiles;          // CTAs along x
  int splits;         // CTAs along y (K splits)
  int kt_total, kt_per_split;
  int tile_elems;
};

int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

// Picks the tile shape and the split-K factor by minimising a small cost model (microseconds):
//
//     cost = 4 + waves * (5 + kt * c_kt + epilogue) + [splits > 1] * (8 + partial_bytes / 4 MB/us)
//
// fitted on B200 over a plan sweep (profiles/r01_plan_sweep_raw.txt; typical error < 8 %; DESIGN.md section 3.1).  c_kt is the
// measured time per 64-token K tile: 0.64 us for a whole 256-block per CTA (two M=128 UMMAs per K step, 84 % of the
// UMMA issue rate), 0.41 us for a half block, 0.27 / 0.22 us for b = 128 / 64 with their taller stages.  Splitting K costs a
// second (reduce) kernel plus writing and re-reading the fp32 partial tiles, so small launches prefer half-block
// tiles (half the partial bytes for the same CTA count) and one wave of CTAs.
Plan make_plan(int n_blocks, int block, int64_t T) {
  const int sms = sm_count();
  Plan best{};
  const int ktile = ktile_for(block);
  const int kt_total = (int)((T + ktile - 1) / ktile);
  double best_cost = 1e30;
  for (int mh = 1; mh <= (block == 256 ? 2 : 1); ++mh) {
    const int tpb = (block == 256 && mh == 1) ? 2 : 1;
    const int tiles = n_blocks * tpb;
    const int tile_rows = block >= 128 ? 128 * mh : block;
    const double tile_bytes = 4.0 * tile_rows * block;                 // fp32 tile
    // fitted per 64 tokens (b = 128 / 64: with 128-token stages)
    const double c_kt = (block == 256 ? (mh == 2 ? 0.64 : 0.41) : block == 128 ? 0.27 : 0.22) * ktile / 64.0;
    int max_splits = (int)(T / kMinTokensPerSplit);
    if (max_splits < 1) max_splits = 1;
    if (max_splits > 64) max_splits = 64;
    for (int s = 1; s <= max_splits; ++s) {
      const int kt = (kt_total + s - 1) / s;
      const int s_eff = (kt_total + kt - 1) / kt;
      const long ctas = (long)tiles * s_eff;
      const long waves = (ctas + sms - 1) / sms;
      const double epi = tile_bytes / 131072.0 * (s_eff > 1 ? 2.0 : 1.0);
      double cost = 4.0 + waves * (5.0 + kt * c_kt + epi);
      // one wave => the reduction is fused into the GEMM kernel (cooperative launch); else a second kernel
      if (s_eff > 1) cost += (ctas <= sms ? 3.0 : 8.0) + (double)ctas * tile_bytes / 4.0e6;
      if (cost < best_cost) {
        best_cost = cost;
        best.mh = mh; best.tiles = tiles; best.splits = s_eff; best.kt_total = kt_total; best.kt_per_split = kt;
        best.tile_elems = tile_rows * block;
      }
    }
  }
  return best;
}

// 2-D map over a row-major [T, features] 16-bit matrix; box = {64 features, ktile tokens}, 128B swizzle.
int encode_operand_map(CUtensorMap* map, const void* base, int64_t features, int64_t T, int64_t ld, int in_dtype,
                       int ktile) {
  return encode_2d_sw128(map, base, features, T, ld, in_dtype, ktile, "smt_block_grad_gemm");
}

template <int B, int MH, bool GROUPED>
int launch_umma_cfg(const CUtensorMap& mx, const CUtensorMap& mdy, const GemmParams& gp, const Plan& pl, cudaStream_t st) {
  return launch_tiles(block_grad_umma_kernel<B, MH, GROUPED>, dim3(pl.tiles, pl.splits), kGemmThreads,
                      Cfg<B, MH>::SMEM_BYTES, gp.counters != nullptr, st, mx, mdy, gp);
}

template <bool GROUPED>
int launch_umma(int block, const CUtensorMap& mx, const CUtensorMap& mdy, const GemmParams& gp, const Plan& pl,
                cudaStream_t st) {
  if (block == 256) {
    if (pl.mh == 2) return launch_umma_cfg<256, 2, GROUPED>(mx, mdy, gp, pl, st);
    return launch_umma_cfg<256, 1, GROUPED>(mx, mdy, gp, pl, st);
  }
  if (block == 128) return launch_umma_cfg<128, 1, GROUPED>(mx, mdy, gp, pl, st);
  return launch_umma_cfg<64, 1, GROUPED>(mx, mdy, gp, pl, st);
}

// Two whole blocks per CTA pair, cta_group::2 UMMAs (grouped launches of b = 256 blocks that need no split-K).
int launch_umma_2sm(const GemmParams& gp, int n_items, cudaStream_t st) {
  SMT_CHECK_CUDA(cudaFuncSetAttribute(block_grad_umma_2sm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      k2smSmemBytes));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(2 * ((n_items + 1) / 2)));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = k2smSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  SMT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, block_grad_umma_2sm_kernel, gp, n_items));
  return SMT_OK;
}

// split-K reduce, launched with programmatic stream serialization so that its launch overlaps the GEMM
int launch_reduce(const float* ws, void* out, const smt_gemm_item* items, int block, int64_t ldo, const Plan& pl,
                  int n_blocks, int out_dtype, int accumulate, cudaStream_t st) {
  const int64_t n_out = (int64_t)n_blocks * block * block;
  const int64_t n_vec8 = n_out / 8;
  int64_t want = (n_vec8 + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(want < cap ? want : cap));
  cfg.blockDim = dim3(256);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  const int tpb = pl.tiles / n_blocks;
  if (out_dtype == SMT_F32)
    SMT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, splitk_reduce_kernel<SMT_F32>, ws, out, items, pl.tile_elems, tpb, block, ldo, pl.splits, n_vec8, accumulate));
  else if (out_dtype == SMT_BF16)
    SMT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, splitk_reduce_kernel<SMT_BF16>, ws, out, items, pl.tile_elems, tpb, block, ldo, pl.splits, n_vec8, accumulate));
  else
    SMT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, splitk_reduce_kernel<SMT_F16>, ws, out, items, pl.tile_elems, tpb, block, ldo, pl.splits, n_vec8, accumulate));
  return SMT_OK;
}

size_t plan_workspace_bytes(const Plan& pl) {
  return pl.splits > 1 ? kSplitCounterBytes + (size_t)pl.tiles * pl.splits * pl.tile_elems * sizeof(float) : 0;
}

// The fused (in-kernel) reduction needs every CTA resident at once: one CTA per SM (shared memory), one wave.
bool use_fused_reduce(const Plan& pl) {
  if (pl.splits <= 1 || env_int("SMT_GEMM_NO_FUSED_REDUCE", 0)) return false;
  static int coop = -1;
  if (coop < 0) {
    int dev = 0, v = 0;
    coop = (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&v, cudaDevAttrCooperativeLaunch, dev) == cudaSuccess && v) ? 1 : 0;
  }
  return coop == 1 && (long)pl.tiles * pl.splits <= sm_count() && (size_t)pl.tiles * 2 * sizeof(int) <= kSplitCounterBytes;
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API int smt_block_grad_gemm_plan(int n_blocks, int block, int64_t T, int in_dtype, int* splits_host,
                                        int* ctas_host) {
  SMT_CHECK_ARG(block_ok(block), "smt_block_grad_gemm_plan: block size %d not in {64,128,256}", block);
  SMT_CHECK_ARG(n_blocks >= 0 && T >= 0, "smt_block_grad_gemm_plan: negative size");
  int splits = 1, ctas = 0;
  if (n_blocks > 0 && T > 0) {
    if (in_dtype == SMT_F32) {
      ctas = n_blocks * (block / 64) * (block / 64);
    } else {
      Plan pl = make_plan(n_blocks, block, T);
      splits = pl.splits;
      ctas = pl.tiles * pl.splits;
    }
  }
  if (splits_host) *splits_host = splits;
  if (ctas_host) *ctas_host = ctas;
  return SMT_OK;
}

extern "C" SMT_API size_t smt_block_grad_gemm_workspace_bytes(int n_blocks, int block, int64_t T, int in_dtype) {
  if (n_blocks <= 0 || T <= 0 || !block_ok(block) || in_dtype == SMT_F32) return 0;
  return plan_workspace_bytes(make_plan(n_blocks, block, T));
}

extern "C" SMT_API int smt_block_grad_gemm(const void* x, int64_t ldx, int in_features, const void* dy, int64_t lddy,
                                   int out_features, int64_t T, int in_dtype, const int32_t* block_rc,
                                   int n_blocks, int block, void* G, int out_dtype, int accumulate,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  SMT_CHECK_ARG(n_blocks >= 0 && T >= 0, "smt_block_grad_gemm: negative size");
  if (n_blocks == 0) return SMT_OK;
  SMT_CHECK_ARG(block_ok(block), "smt_block_grad_gemm: block size %d not in {64,128,256}", block);
  SMT_CHECK_ARG(G && block_rc, "smt_block_grad_gemm: null pointer");
  SMT_CHECK_ARG(in_dtype >= SMT_F32 && in_dtype <= SMT_F16 && out_dtype >= SMT_F32 && out_dtype <= SMT_F16,
                "smt_block_grad_gemm: bad dtype");
  SMT_CHECK_ARG(in_features > 0 && out_features > 0 && in_features % block == 0 && out_features % block == 0,
                "smt_block_grad_gemm: features (%d in, %d out) must be multiples of block %d", in_features,
                out_features, block);
  SMT_CHECK_ARG(aligned16(G), "smt_block_grad_gemm: G must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n_out = (int64_t)n_blocks * block * block;
  if (T == 0) {  // empty token range: the sum is zero
    if (!accumulate) SMT_CHECK_CUDA(cudaMemsetAsync(G, 0, (size_t)n_out * dtype_bytes(out_dtype), st));
    return SMT_OK;
  }
  SMT_CHECK_ARG(x && dy, "smt_block_grad_gemm: null pointer");
  SMT_CHECK_ARG(ldx >= in_features && lddy >= out_features, "smt_block_grad_gemm: leading dimension too small");
  const int in_bytes = dtype_bytes(in_dtype);
  SMT_CHECK_ARG(aligned16(x) && aligned16(dy) && (ldx * in_bytes) % 16 == 0 && (lddy * in_bytes) % 16 == 0,
                "smt_block_grad_gemm: x and dy must be 16-byte aligned (pointer and row pitch)");

  if (in_dtype == SMT_F32) {
    dim3 grid(n_blocks, (block / 64) * (block / 64));
    const float* xf = reinterpret_cast<const float*>(x);
    const float* dyf = reinterpret_cast<const float*>(dy);
    if (out_dtype == SMT_F32) block_grad_f32_kernel<SMT_F32><<<grid, 256, 0, st>>>(xf, ldx, dyf, lddy, T, block_rc, block, G, accumulate);
    else if (out_dtype == SMT_BF16) block_grad_f32_kernel<SMT_BF16><<<grid, 256, 0, st>>>(xf, ldx, dyf, lddy, T, block_rc, block, G, accumulate);
    else block_grad_f32_kernel<SMT_F16><<<grid, 256, 0, st>>>(xf, ldx, dyf, lddy, T, block_rc, block, G, accumulate);
    SMT_CHECK_LAUNCH();
    set_launch_count(1);
    return SMT_OK;
  }

  SMT_CHECK_ARG(T < (1ll << 31) - kMaxKTile, "smt_block_grad_gemm: T too large");
  const Plan pl = make_plan(n_blocks, block, T);
  int* counters;
  float* partials;
  if (int rc = carve_split_workspace("smt_block_grad_gemm", workspace, workspace_bytes, plan_workspace_bytes(pl),
                                     &counters, &partials))
    return rc;

  CUtensorMap mx, mdy;
  if (int rc = encode_operand_map(&mx, x, in_features, T, ldx, in_dtype, ktile_for(block))) return rc;
  if (int rc = encode_operand_map(&mdy, dy, out_features, T, lddy, in_dtype, ktile_for(block))) return rc;

  GemmParams gp{};
  gp.block_rc = block_rc;
  gp.out = G;
  gp.ws = partials;
  gp.counters = use_fused_reduce(pl) ? counters : nullptr;
  gp.splits = pl.splits;
  gp.kt_total = pl.kt_total;
  gp.kt_per_split = pl.kt_per_split;
  gp.out_dtype = out_dtype;
  gp.accumulate = accumulate;
  gp.ld_out = block;
  gp.in_fmt = in_dtype == SMT_BF16 ? 1 : 0;
  if (int rc = launch_umma<false>(block, mx, mdy, gp, pl, st)) return rc;
  set_launch_count(1);
  if (pl.splits > 1 && gp.counters == nullptr) {
    set_launch_count(2);
    return launch_reduce(gp.ws, G, nullptr, block, block, pl, n_blocks, out_dtype, accumulate, st);
  }
  return SMT_OK;
}

// ---- grouped entry point: blocks of several (x, dy) problems in one launch ----------------------------------

extern "C" SMT_API int smt_encode_operand_map(void* map_host, const void* base, int64_t features, int64_t T,
                                              int64_t ld, int dtype, int block) {
  SMT_CHECK_ARG(block_ok(block), "smt_encode_operand_map: block size %d not in {64,128,256}", block);
  SMT_CHECK_ARG(map_host && base, "smt_encode_operand_map: null pointer");
  SMT_CHECK_ARG(dtype == SMT_BF16 || dtype == SMT_F16, "smt_encode_operand_map: 16-bit operands only");
  SMT_CHECK_ARG((reinterpret_cast<uintptr_t>(map_host) & 63u) == 0, "smt_encode_operand_map: map must be 64-byte aligned");
  SMT_CHECK_ARG(features > 0 && T > 0 && ld >= features && (ld * 2) % 16 == 0 && aligned16(base),
                "smt_encode_operand_map: bad operand geometry");
  static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
  return encode_operand_map(reinterpret_cast<CUtensorMap*>(map_host), base, features, T, ld, dtype, ktile_for(block));
}

namespace {
// Large grouped launches of b = 256 blocks (no split-K, whole-block tiles) run on SM pairs (cta_group::2): bit-identical
// to the single-CTA kernel and 3-5 % faster alone / ~1 % in bench.py (profiles/r01_kernels.md section 1b).
// SMT_GEMM_2SM=0 switches back to the single-CTA kernel.  (A cta_group::1 variant that TMA-multicast the shared dy strip
// inside a 2-CTA cluster was measured no faster than single CTAs and removed; numbers in the same section.)
bool use_2sm(int n_items, int block, int64_t T) {
  if (block != 256 || n_items < 2 || !env_int("SMT_GEMM_2SM", 1)) return false;
  const Plan pl = make_plan(n_items, block, T);
  return pl.splits == 1 && pl.mh == 2;
}
}  // namespace

extern "C" SMT_API int smt_block_grad_gemm_grouped_uses_2sm(int n_items, int block, int64_t T) {
  return (n_items > 0 && T > 0 && block_ok(block) && use_2sm(n_items, block, T)) ? 1 : 0;
}

extern "C" SMT_API size_t smt_block_grad_gemm_grouped_workspace_bytes(int n_items, int block, int64_t T) {
  if (n_items <= 0 || T <= 0 || !block_ok(block)) return 0;
  return plan_workspace_bytes(make_plan(n_items, block, T));
}

extern "C" SMT_API int smt_block_grad_gemm_grouped_emits_sq(int n_items, int block, int64_t T) {
  if (n_items <= 0 || T <= 0 || !block_ok(block)) return 0;
  return (use_2sm(n_items, block, T) || make_plan(n_items, block, T).splits == 1) ? 1 : 0;
}

extern "C" SMT_API int smt_block_grad_gemm_grouped(const void* maps, const smt_gemm_item* items, int n_items,
                                                   int64_t T, int block, int in_dtype, void* out_base,
                                                   int out_dtype, int accumulate, int64_t ld_out, float* sq_partials,
                                                   void* workspace, size_t workspace_bytes, void* stream) {
  SMT_CHECK_ARG(n_items >= 0 && T >= 0, "smt_block_grad_gemm_grouped: negative size");
  if (n_items == 0 || T == 0) return SMT_OK;
  SMT_CHECK_ARG(block_ok(block), "smt_block_grad_gemm_grouped: block size %d not in {64,128,256}", block);
  SMT_CHECK_ARG(maps && items && out_base, "smt_block_grad_gemm_grouped: null pointer");
  SMT_CHECK_ARG((in_dtype == SMT_BF16 || in_dtype == SMT_F16) && out_dtype >= SMT_F32 && out_dtype <= SMT_F16,
                "smt_block_grad_gemm_grouped: bad dtype");
  SMT_CHECK_ARG((reinterpret_cast<uintptr_t>(maps) & 63u) == 0 && aligned16(out_base),
                "smt_block_grad_gemm_grouped: maps must be 64-byte and out_base 16-byte aligned");
  SMT_CHECK_ARG(T < (1ll << 31) - kMaxKTile, "smt_block_grad_gemm_grouped: T too large");
  SMT_CHECK_ARG(ld_out == 0 || (ld_out >= block && ld_out % 8 == 0 && ld_out < (1ll << 31)),
                "smt_block_grad_gemm_grouped: ld_out must be 0 (compact tiles) or a multiple of 8 that is >= block");
  const Plan pl = make_plan(n_items, block, T);
  int* counters;
  float* partials;
  if (int rc = carve_split_workspace("smt_block_grad_gemm_grouped", workspace, workspace_bytes,
                                     plan_workspace_bytes(pl), &counters, &partials))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int launches = 0;
  GemmParams gp{};
  gp.maps = reinterpret_cast<const CUtensorMap*>(maps);
  gp.out = out_base;
  gp.out_dtype = out_dtype;
  gp.accumulate = accumulate;
  gp.sq = sq_partials;
  gp.ld_out = ld_out > 0 ? ld_out : block;
  gp.in_fmt = in_dtype == SMT_BF16 ? 1 : 0;
  gp.kt_total = (int)((T + ktile_for(block) - 1) / ktile_for(block));

  if (use_2sm(n_items, block, T)) {
    gp.items = items;
    gp.splits = 1;
    gp.kt_per_split = gp.kt_total;
    if (int rc = launch_umma_2sm(gp, n_items, st)) return rc;
    set_launch_count(1);
    return SMT_OK;
  }
  gp.items = items;
  gp.ws = partials;
  gp.counters = use_fused_reduce(pl) ? counters : nullptr;
  gp.splits = pl.splits;
  gp.kt_total = pl.kt_total;
  gp.kt_per_split = pl.kt_per_split;
  CUtensorMap dummy;
  memset(&dummy, 0, sizeof(dummy));
  if (int rc = launch_umma<true>(block, dummy, dummy, gp, pl, st)) return rc;
  ++launches;
  if (pl.splits > 1 && gp.counters == nullptr) {
    ++launches;
    if (int rc = launch_reduce(gp.ws, out_base, gp.items, block, gp.ld_out, pl, n_items, out_dtype, accumulate, st)) return rc;
  }
  set_launch_count(launches);
  return SMT_OK;
}
