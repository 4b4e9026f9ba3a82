// Dense side of linearZ, fused over the modules that share an input (SURVEY.md section 8f row 2):
//
//   forward   y_j[T, N_j] = x[T, K] . W_j[N_j, K]^T            for j = q, k, v      (reference smt.py:366, three calls)
//   dgrad     dx[T, K]    = sum_j dy_j[T, N_j] . W_j[N_j, K]                        (reference smt.py:406, three calls
//                                                                                    + the two adds autograd inserts)
//
// The reference runs one cuBLAS GEMM per module and direction: q, k and v of a decoder layer read the same x three
// times and produce three dx that autograd then sums with two elementwise kernels.  Here ONE persistent tcgen05 kernel
// does each direction: forward walks the N tiles of [Wq; Wk; Wv] as if they were one 6144-row weight (three B
// descriptors, three output pointers), dgrad runs the reduction over K = 4096 + 1024 + 1024 through the three dy / W
// pairs into one accumulator, so the adds disappear.
//
// Kernel shape (both directions): CTA pairs (cta_group::2), tile 256 x 256 per pair (M = 256 across the pair, each CTA
// owns 128 rows and loads half of the B tile), K step 64 per pipeline stage (32 KiB per CTA and stage, 6 stages),
// two 256-column TMEM accumulators so that the epilogue of tile i overlaps the main loop of tile i + 1, static
// persistent schedule rasterised in groups of 16 M tiles for L2 reuse of the weights.  Warp 0 = TMA producer (both CTAs),
// warp 1 = UMMA issuer (leader CTA), warps 2-5 = epilogue (TMEM -> registers -> bf16 -> per-warp shared-memory transpose
// -> 128-byte row stores).  A is always K-major; B is K-major in forward (W[n, k], k contiguous) and MN-major in dgrad
// (W[k, n], n contiguous): same TMA boxes / UMMA descriptors as the block-gradient kernel for the MN-major side.
#include <cuda.h>
#include <string.h>

#include "common.cuh"
#include "umma_ptx.cuh"
#include "tma_host.cuh"

namespace smt {
namespace {

constexpr int kDenseBK = 64;                           // K elements per stage (one 128-byte swizzle row)
constexpr int kDenseTileM = 256, kDenseTileN = 256;    // per CTA pair
constexpr int kDenseStageBytes = 2 * 128 * kDenseBK * 2;   // A: 128 rows x 64, B half: 128 n x 64  = 32 KiB
constexpr int kDenseStages = 6;                        // 4 stages measured 2 % slower, 5 the same (profiles/r02_fused_qkv.md)
// M tiles per raster group: 16 measured fastest of 2 / 4 / 8 / 16 / 32 (profiles/r02_fused_qkv.md)
constexpr int kDenseGroupM = 16;
constexpr int kDenseEpiWarps = 4;
constexpr int kDenseThreads = 64 + 32 * kDenseEpiWarps;
constexpr int kDenseStagingPitch = 144;                // bytes per staged row: 128 B of bf16 + 16 B pad (conflict-free v4)
constexpr int kDenseStagingBytes = kDenseEpiWarps * 32 * kDenseStagingPitch;
constexpr int kDenseSmemBytes = kDenseStages * kDenseStageBytes + kDenseStagingBytes + 1024;
constexpr int kMaxSeg = 3;

struct DenseParams {
  int T;                       // rows of A and of the outputs (tokens)
  int n_seg;
  int seg_len[kMaxSeg];        // forward: N_j (output features of segment j); dgrad: N_j (reduction length of segment j)
  int seg_tile0[kMaxSeg + 1];  // forward: first N tile of segment j (prefix sums of N_j / 256)
  int k_or_n;                  // forward: K (reduction length); dgrad: width of dx (in_features)
  void* out[kMaxSeg];          // forward: y_j; dgrad: out[0] = dx
  long long ld_out[kMaxSeg];   // elements
  int m_tiles, n_tiles;
  int group_m;                 // M tiles per raster group
  int in_fmt;                  // 0 = f16, 1 = bf16
};

struct DenseMaps {
  CUtensorMap a[kMaxSeg];      // forward: a[0] = x; dgrad: a[j] = dy_j          (K-major, box {64, 128})
  CUtensorMap b[kMaxSeg];      // W_j: forward box {64 k, 128 n}; dgrad box {64 n, 64 k}
};

// tile index -> (m tile, n tile): groups of `group_m` M tiles are swept N-major, so that the CTA pairs running at the same
// time share a handful of weight tiles and a handful of activation tiles in L2
__device__ __forceinline__ void tile_coords(int t, const DenseParams& p, int& m, int& n) {
  const int per_group = p.group_m * p.n_tiles;
  const int g = t / per_group;
  const int m0 = g * p.group_m;
  const int rows = min(p.group_m, p.m_tiles - m0);
  const int r = t - g * per_group;
  m = m0 + r % rows;
  n = r / rows;
}

template <bool DGRAD>
__global__ void __launch_bounds__(kDenseThreads, 1) fused_dense_umma_2sm_kernel(const __grid_constant__ DenseMaps maps,
                                                                                const DenseParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[kDenseStages];
  __shared__ __align__(8) uint64_t empty_bar[kDenseStages];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];      // the LEADER's instance collects both CTAs' epilogue warps
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int n_tiles_total = p.m_tiles * p.n_tiles;

  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));

  // K blocks per tile
  int kb_total;
  if (DGRAD) {
    kb_total = 0;
    for (int s = 0; s < p.n_seg; ++s) kb_total += p.seg_len[s] / kDenseBK;
  } else {
    kb_total = p.k_or_n / kDenseBK;
  }

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.n_seg; ++s) {
      prefetch_tmap(&maps.b[s]);
      if (DGRAD || s == 0) prefetch_tmap(&maps.a[s]);
    }
    for (int s = 0; s < kDenseStages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), 2 * kDenseEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm(smem_u32(&tmem_slot), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                  // both CTAs' barriers and TMEM exist before anything crosses the pair
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): my 128 rows of A and my half of the B tile =====
    if (lane == 0) {
      int it = 0;
      for (int t = pair; t < n_tiles_total; t += n_pairs) {
        int m, n;
        tile_coords(t, p, m, n);
        const int row0 = m * kDenseTileM + (int)rank * 128;
        if (!DGRAD) {
          int seg = 0;
          while (seg + 1 < p.n_seg && n >= p.seg_tile0[seg + 1]) ++seg;
          const int n0 = (n - p.seg_tile0[seg]) * kDenseTileN + (int)rank * 128;
          const CUtensorMap* mb = &maps.b[seg];
          for (int kb = 0; kb < kb_total; ++kb, ++it) {
            const int stage = it % kDenseStages;
            const uint32_t phase = (uint32_t)(it / kDenseStages) & 1u;
            mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
            const uint32_t fb = smem_u32(&full_bar[stage]);
            if (rank == 0) mbar_expect_tx(fb, 2u * kDenseStageBytes);      // the leader's barrier counts both CTAs' bytes
            const uint32_t st = smem_base + (uint32_t)(stage * kDenseStageBytes);
            tma_load_2d_2sm(st, &maps.a[0], fb, kb * kDenseBK, row0);
            tma_load_2d_2sm(st + 128 * kDenseBK * 2, mb, fb, kb * kDenseBK, n0);
          }
        } else {
          const int n0 = n * kDenseTileN + (int)rank * 128;
          for (int seg = 0; seg < p.n_seg; ++seg) {
            const int kbs = p.seg_len[seg] / kDenseBK;
            for (int kb = 0; kb < kbs; ++kb, ++it) {
              const int stage = it % kDenseStages;
              const uint32_t phase = (uint32_t)(it / kDenseStages) & 1u;
              mbar_wait(smem_u32(&empty_bar[stage]), phase ^ 1u);
              const uint32_t fb = smem_u32(&full_bar[stage]);
              if (rank == 0) mbar_expect_tx(fb, 2u * kDenseStageBytes);
              const uint32_t st = smem_base + (uint32_t)(stage * kDenseStageBytes);
              tma_load_2d_2sm(st, &maps.a[seg], fb, kb * kDenseBK, row0);
              // B is MN-major: two {64 n, 64 k} chunks of 8 KiB
              tma_load_2d_2sm(st + 16384, &maps.b[seg], fb, n0, kb * kDenseBK);
              tma_load_2d_2sm(st + 16384 + 8192, &maps.b[seg], fb, n0 + 64, kb * kDenseBK);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== UMMA issuer: one thread of the leader CTA, on behalf of both SMs =====
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = make_idesc_major(p.in_fmt, 256, kDenseTileN, 0, DGRAD ? 1 : 0);
      int it = 0, lt = 0;
      for (int t = pair; t < n_tiles_total; t += n_pairs, ++lt) {
        const int buf = lt & 1;
        mbar_wait(smem_u32(&tmem_empty_bar[buf]), (uint32_t)((lt >> 1) & 1) ^ 1u);   // both CTAs drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < kb_total; ++kb, ++it) {
          const int stage = it % kDenseStages;
          const uint32_t phase = (uint32_t)(it / kDenseStages) & 1u;
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t st = smem_base + (uint32_t)(stage * kDenseStageBytes);
#pragma unroll
          for (int k = 0; k < kDenseBK / 16; ++k) {
            const uint64_t adesc = make_desc_k_sw128(st + k * 32);
            const uint64_t bdesc = DGRAD ? make_desc_mn_sw128(st + 16384 + k * 2048, 8192, 1024)
                                         : make_desc_k_sw128(st + 16384 + k * 32);
            umma2_f16(tmem_base + buf * kDenseTileN, adesc, bdesc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma2_commit_multicast(smem_u32(&empty_bar[stage]), (uint16_t)0x3);      // frees the stage in both CTAs
        }
        umma2_commit_multicast(smem_u32(&tmem_full_bar[buf]), (uint16_t)0x3);      // accumulator complete, both CTAs
      }
    }
  } else {
    // ===== epilogue (both CTAs, 4 warps = the 4 TMEM lane quarters): my 128 rows of every tile of this pair =====
    const int ew = warp - 2, q = warp & 3;
    uint8_t* stg = smem_gen + kDenseStages * kDenseStageBytes + ew * 32 * kDenseStagingPitch;
    const uint32_t empty0 = mapa_rank0(smem_u32(&tmem_empty_bar[0]));
    const uint32_t empty1 = mapa_rank0(smem_u32(&tmem_empty_bar[1]));
    int lt = 0;
    for (int t = pair; t < n_tiles_total; t += n_pairs, ++lt) {
      const int buf = lt & 1;
      int m, n;
      tile_coords(t, p, m, n);
      int seg = 0, col0;
      if (!DGRAD) {
        while (seg + 1 < p.n_seg && n >= p.seg_tile0[seg + 1]) ++seg;
        col0 = (n - p.seg_tile0[seg]) * kDenseTileN;
      } else {
        col0 = n * kDenseTileN;
      }
      const int width = DGRAD ? p.k_or_n : p.seg_len[seg];
      uint16_t* out = reinterpret_cast<uint16_t*>(p.out[seg]);
      const long long ldo = p.ld_out[seg];
      const int row_base = m * kDenseTileM + (int)rank * 128 + q * 32;
      mbar_wait(smem_u32(&tmem_full_bar[buf]), (uint32_t)((lt >> 1) & 1));
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < kDenseTileN / 64; ++cc) {
        if (col0 + cc * 64 < width) {                     // (widths are multiples of 64: whole chunks in or out)
          uint32_t r0[32], r1[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kDenseTileN + cc * 64), r0);
          tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * kDenseTileN + cc * 64 + 32), r1);
          tmem_ld_wait();
          // lane = row: 64 fp32 -> 64 16-bit values = 128 B into my staging row
          uint4* mine = reinterpret_cast<uint4*>(stg + lane * kDenseStagingPitch);
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            uint4 u;
            if (p.in_fmt == 1) {
              u.x = pack_bf16x2(__uint_as_float(r0[8 * v]), __uint_as_float(r0[8 * v + 1]));
              u.y = pack_bf16x2(__uint_as_float(r0[8 * v + 2]), __uint_as_float(r0[8 * v + 3]));
              u.z = pack_bf16x2(__uint_as_float(r0[8 * v + 4]), __uint_as_float(r0[8 * v + 5]));
              u.w = pack_bf16x2(__uint_as_float(r0[8 * v + 6]), __uint_as_float(r0[8 * v + 7]));
            } else {
              u.x = pack_f16x2(__uint_as_float(r0[8 * v]), __uint_as_float(r0[8 * v + 1]));
              u.y = pack_f16x2(__uint_as_float(r0[8 * v + 2]), __uint_as_float(r0[8 * v + 3]));
              u.z = pack_f16x2(__uint_as_float(r0[8 * v + 4]), __uint_as_float(r0[8 * v + 5]));
              u.w = pack_f16x2(__uint_as_float(r0[8 * v + 6]), __uint_as_float(r0[8 * v + 7]));
            }
            mine[v] = u;
          }
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            uint4 u;
            if (p.in_fmt == 1) {
              u.x = pack_bf16x2(__uint_as_float(r1[8 * v]), __uint_as_float(r1[8 * v + 1]));
              u.y = pack_bf16x2(__uint_as_float(r1[8 * v + 2]), __uint_as_float(r1[8 * v + 3]));
              u.z = pack_bf16x2(__uint_as_float(r1[8 * v + 4]), __uint_as_float(r1[8 * v + 5]));
              u.w = pack_bf16x2(__uint_as_float(r1[8 * v + 6]), __uint_as_float(r1[8 * v + 7]));
            } else {
              u.x = pack_f16x2(__uint_as_float(r1[8 * v]), __uint_as_float(r1[8 * v + 1]));
              u.y = pack_f16x2(__uint_as_float(r1[8 * v + 2]), __uint_as_float(r1[8 * v + 3]));
              u.z = pack_f16x2(__uint_as_float(r1[8 * v + 4]), __uint_as_float(r1[8 * v + 5]));
              u.w = pack_f16x2(__uint_as_float(r1[8 * v + 6]), __uint_as_float(r1[8 * v + 7]));
            }
            mine[4 + v] = u;
          }
          __syncwarp();
          // 8 lanes cover one 128-byte row: every store instruction writes 4 whole rows
          const int sub = lane >> 3, cv = lane & 7;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int row = i * 4 + sub;
            const uint4 u = *reinterpret_cast<const uint4*>(stg + row * kDenseStagingPitch + cv * 16);
            const int grow = row_base + row;
            if (grow < p.T)
              *reinterpret_cast<uint4*>(out + (long long)grow * ldo + col0 + cc * 64 + cv * 8) = u;
          }
          __syncwarp();
        }
      }
      tc_fence_before();                 // my TMEM reads are ordered before the release below
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(buf ? empty1 : empty0);
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                    // nobody leaves (or frees TMEM) while the pair may still touch it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// ---- host side -------------------------------------------------------------------------------------------------

// 2-D map over a row-major [rows, cols] 16-bit matrix (cols contiguous); box = {64 cols, box_rows}, 128-byte swizzle,
// out-of-bounds elements read as zero.
int encode_dense_map(CUtensorMap* map, const void* base, int64_t cols, int64_t rows, int64_t ld, int dtype, int box_rows) {
  return encode_2d_sw128(map, base, cols, rows, ld, dtype, box_rows, "smt_fused_linear");
}

template <bool DGRAD>
int launch_dense(const DenseMaps& maps, const DenseParams& p, cudaStream_t st) {
  auto kern = fused_dense_umma_2sm_kernel<DGRAD>;
  SMT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kDenseSmemBytes));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)sm_count());
  cfg.blockDim = dim3(kDenseThreads);
  cfg.dynamicSmemBytes = kDenseSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  static int max_pairs[2] = {0, 0};             // CTA pairs that can be resident at once on this device
  if (max_pairs[DGRAD] == 0) {
    int n = 0;
    SMT_CHECK_CUDA(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
    max_pairs[DGRAD] = n > 0 ? n : 1;
  }
  const int tiles = p.m_tiles * p.n_tiles;
  const int pairs = tiles < max_pairs[DGRAD] ? tiles : max_pairs[DGRAD];
  cfg.gridDim = dim3((unsigned)(2 * pairs));
  SMT_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, p));
  return SMT_OK;
}

int check_common(const char* who, int64_t T, int n_seg, const void* const* W, const int64_t* ldw, const int* N, int K,
                 int dtype) {
  SMT_CHECK_ARG(n_seg >= 1 && n_seg <= kMaxSeg, "%s: 1..3 segments, got %d", who, n_seg);
  SMT_CHECK_ARG(dtype == SMT_BF16 || dtype == SMT_F16, "%s: 16-bit operands only", who);
  SMT_CHECK_ARG(T >= 0 && T < (1ll << 31) - 512, "%s: token count %lld outside [0, 2^31 - 512)", who, (long long)T);
  SMT_CHECK_ARG(K > 0 && K % 64 == 0, "%s: in_features %d must be a multiple of 64", who, K);
  SMT_CHECK_ARG(W && ldw && N, "%s: null pointer", who);
  for (int j = 0; j < n_seg; ++j) {
    SMT_CHECK_ARG(W[j] && aligned16(W[j]) && ldw[j] >= K && (ldw[j] * 2) % 16 == 0,
                  "%s: weight %d must be 16-byte aligned with a row pitch >= in_features", who, j);
    SMT_CHECK_ARG(N[j] > 0 && N[j] % 64 == 0, "%s: out_features %d of segment %d must be a multiple of 64", who, N[j], j);
  }
  return SMT_OK;
}

}  // namespace
}  // namespace smt

using namespace smt;

extern "C" SMT_API int smt_fused_linear_supported(int n_seg, const int* N_host, int K, int dtype, int dgrad) {
  if (n_seg < 1 || n_seg > kMaxSeg || !N_host || K <= 0 || K % 64 != 0) return 0;
  if (dtype != SMT_BF16 && dtype != SMT_F16) return 0;
  for (int j = 0; j < n_seg; ++j) {
    if (N_host[j] <= 0 || N_host[j] % 64 != 0) return 0;
    if (!dgrad && N_host[j] % kDenseTileN != 0) return 0;      // forward: an N tile must not straddle two modules
  }
  return 1;
}

extern "C" SMT_API int smt_fused_linear_forward(const void* x, int64_t ldx, int64_t T, int K, int n_seg,
                                                const void* const* W_host, const int64_t* ldw_host, const int* N_host,
                                                void* const* y_host, const int64_t* ldy_host, int dtype, void* stream) {
  if (int rc = check_common("smt_fused_linear_forward", T, n_seg, W_host, ldw_host, N_host, K, dtype)) return rc;
  if (T == 0) return SMT_OK;
  // every argument is checked before the first map is encoded, so a rejection never depends on the driver
  SMT_CHECK_ARG(x && aligned16(x) && ldx >= K && (ldx * 2) % 16 == 0,
                "smt_fused_linear_forward: x must be 16-byte aligned with a 16-byte row pitch >= in_features");
  SMT_CHECK_ARG(y_host && ldy_host, "smt_fused_linear_forward: null pointer");
  for (int j = 0; j < n_seg; ++j) {
    SMT_CHECK_ARG(N_host[j] % kDenseTileN == 0,
                  "smt_fused_linear_forward: out_features %d of segment %d must be a multiple of %d", N_host[j], j,
                  kDenseTileN);
    SMT_CHECK_ARG(y_host[j] && aligned16(y_host[j]) && ldy_host[j] >= N_host[j] && (ldy_host[j] * 2) % 16 == 0,
                  "smt_fused_linear_forward: output %d must be 16-byte aligned with a 16-byte row pitch >= out_features",
                  j);
  }
  DenseMaps maps;
  memset(&maps, 0, sizeof(maps));
  DenseParams p{};
  p.T = (int)T;
  p.n_seg = n_seg;
  p.k_or_n = K;
  p.in_fmt = dtype == SMT_BF16 ? 1 : 0;
  if (int rc = encode_dense_map(&maps.a[0], x, K, T, ldx, dtype, 128)) return rc;
  int tiles = 0;
  for (int j = 0; j < n_seg; ++j) {
    if (int rc = encode_dense_map(&maps.b[j], W_host[j], K, N_host[j], ldw_host[j], dtype, 128)) return rc;
    p.seg_len[j] = N_host[j];
    p.seg_tile0[j] = tiles;
    tiles += N_host[j] / kDenseTileN;
    p.out[j] = y_host[j];
    p.ld_out[j] = ldy_host[j];
  }
  p.seg_tile0[n_seg] = tiles;
  p.n_tiles = tiles;
  p.m_tiles = (int)((T + kDenseTileM - 1) / kDenseTileM);
  p.group_m = kDenseGroupM;
  if (int rc = launch_dense<false>(maps, p, (cudaStream_t)stream)) return rc;
  set_launch_count(1);
  return SMT_OK;
}

extern "C" SMT_API int smt_fused_linear_dgrad(const void* const* dy_host, const int64_t* lddy_host, int64_t T, int K,
                                              int n_seg, const void* const* W_host, const int64_t* ldw_host,
                                              const int* N_host, void* dx, int64_t lddx, int dtype, void* stream) {
  if (int rc = check_common("smt_fused_linear_dgrad", T, n_seg, W_host, ldw_host, N_host, K, dtype)) return rc;
  if (T == 0) return SMT_OK;
  // every argument is checked before the first map is encoded, so a rejection never depends on the driver
  SMT_CHECK_ARG(dy_host && lddy_host, "smt_fused_linear_dgrad: null pointer");
  for (int j = 0; j < n_seg; ++j)
    SMT_CHECK_ARG(dy_host[j] && aligned16(dy_host[j]) && lddy_host[j] >= N_host[j] && (lddy_host[j] * 2) % 16 == 0,
                  "smt_fused_linear_dgrad: dy %d must be 16-byte aligned with a 16-byte row pitch >= out_features", j);
  SMT_CHECK_ARG(dx && aligned16(dx) && lddx >= K && (lddx * 2) % 16 == 0,
                "smt_fused_linear_dgrad: dx must be 16-byte aligned with a 16-byte row pitch >= in_features");
  DenseMaps maps;
  memset(&maps, 0, sizeof(maps));
  DenseParams p{};
  p.T = (int)T;
  p.n_seg = n_seg;
  p.k_or_n = K;
  p.in_fmt = dtype == SMT_BF16 ? 1 : 0;
  for (int j = 0; j < n_seg; ++j) {
    if (int rc = encode_dense_map(&maps.a[j], dy_host[j], N_host[j], T, lddy_host[j], dtype, 128)) return rc;
    if (int rc = encode_dense_map(&maps.b[j], W_host[j], K, N_host[j], ldw_host[j], dtype, 64)) return rc;
    p.seg_len[j] = N_host[j];
  }
  p.out[0] = dx;
  p.ld_out[0] = lddx;
  p.n_tiles = (K + kDenseTileN - 1) / kDenseTileN;
  p.m_tiles = (int)((T + kDenseTileM - 1) / kDenseTileM);
  p.group_m = kDenseGroupM;
  if (int rc = launch_dense<true>(maps, p, (cudaStream_t)stream)) return rc;
  set_launch_count(1);
  return SMT_OK;
}
