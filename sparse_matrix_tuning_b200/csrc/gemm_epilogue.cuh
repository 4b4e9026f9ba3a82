// Epilogue helpers shared by the block-gradient kernels: accumulator sub-tile -> global memory through a per-warp
// shared-memory transpose (every store instruction writes whole rows), and the split-K reduction of partial tiles
// (device side and the host's workspace layout and launch).
#pragma once

#include "common.cuh"

namespace smt {
namespace {

constexpr int kStageRow = 36;                 // floats per row of the epilogue transpose buffer (32 + 4 pad)

// Stores 4 values (optionally added to what is there) and returns the sum of squares of the values as STORED, i.e.
// after the rounding to the output type (the clip norm is defined on the gradient buffer's contents).
template <int ODT, bool ACC>
__device__ __forceinline__ float store4(void* out_base, int64_t off, float4 v) {
  if (ODT == SMT_F32) {
    float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(out_base) + off);
    if (ACC) {
      const float4 old = *o;
      v.x += old.x; v.y += old.y; v.z += old.z; v.w += old.w;
    }
    *o = v;
    return (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  } else {
    uint2* o = reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(out_base) + off);
    if (ACC) {
      const uint2 old = *o;
      if (ODT == SMT_BF16) {
        v.x += __uint_as_float(old.x << 16); v.y += __uint_as_float(old.x & 0xffff0000u);
        v.z += __uint_as_float(old.y << 16); v.w += __uint_as_float(old.y & 0xffff0000u);
      } else {
        const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&old.x));
        const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&old.y));
        v.x += a.x; v.y += a.y; v.z += b.x; v.w += b.y;
      }
    }
    uint2 u;
    float4 w;
    if (ODT == SMT_BF16) {
      u.x = pack_bf16x2(v.x, v.y); u.y = pack_bf16x2(v.z, v.w);
      w = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u),
                      __uint_as_float(u.y << 16), __uint_as_float(u.y & 0xffff0000u));
    } else {
      u.x = pack_f16x2(v.x, v.y); u.y = pack_f16x2(v.z, v.w);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      w = make_float4(a.x, a.y, b.x, b.y);
    }
    *o = u;
    return (w.x * w.x + w.y * w.y) + (w.z * w.z + w.w * w.w);
  }
}

// One 32x32 fp32 accumulator sub-tile (lane = row, r[] = 32 columns) -> global, transposed through a per-warp
// shared-memory buffer so that each store instruction covers 4 rows x 128 B (fp32) / 64 B (16-bit).
template <int ODT, bool ACC>
__device__ __forceinline__ float store_subtile(float* stage, const uint32_t (&r)[32], int lane, void* out_base,
                                               int64_t off00, int ld) {
  float4* mine = reinterpret_cast<float4*>(stage + lane * kStageRow);
#pragma unroll
  for (int q = 0; q < 8; ++q)
    mine[q] = make_float4(__uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), __uint_as_float(r[4 * q + 2]),
                          __uint_as_float(r[4 * q + 3]));
  __syncwarp();
  const int sub = lane >> 3, cv = (lane & 7) * 4;
  float sq = 0.f;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int row = it * 4 + sub;
    const float4 v = *reinterpret_cast<const float4*>(stage + row * kStageRow + cv);
    sq += store4<ODT, ACC>(out_base, off00 + (int64_t)row * ld + cv, v);
  }
  __syncwarp();
  return sq;
}

// Dispatch on (output type, accumulate) for one sub-tile; returns the thread's sum of squares of the stored values.
__device__ __forceinline__ float store_subtile_any(int out_dtype, bool acc, float* stage, const uint32_t (&r)[32],
                                                   int lane, void* out_base, int64_t off, int ld) {
  if (out_dtype == SMT_F32)
    return acc ? store_subtile<SMT_F32, true>(stage, r, lane, out_base, off, ld)
               : store_subtile<SMT_F32, false>(stage, r, lane, out_base, off, ld);
  if (out_dtype == SMT_BF16)
    return acc ? store_subtile<SMT_BF16, true>(stage, r, lane, out_base, off, ld)
               : store_subtile<SMT_BF16, false>(stage, r, lane, out_base, off, ld);
  return acc ? store_subtile<SMT_F16, true>(stage, r, lane, out_base, off, ld)
             : store_subtile<SMT_F16, false>(stage, r, lane, out_base, off, ld);
}

__device__ __forceinline__ float4 ld_cg_f4(const float* p) {   // L2-coherent load (data written by other CTAs of this grid)
  float4 r;
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- split-K: fp32 partial tiles in a workspace, summed in the fixed split order ----------------------------------

// acc = sum over s = 0..splits-1, in that order, of the 8 floats at src + s * stride.  Every split-K reduction (fused
// and separate) sums through this loop, which is what makes their results bit-identical.  LOAD is ld_cg_f4 for
// partials written by sibling CTAs of the same grid, ld_stream_f4 for partials of an earlier grid.
template <auto LOAD>
__device__ __forceinline__ void sum_partials8(const float* src, int splits, int64_t stride, float (&acc)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  // unrolled 4 deep: left to itself the compiler unrolls 8 deep, +18 registers in the b = 64 block kernels
#pragma unroll 4
  for (int s = 0; s < splits; ++s) {
    const float4 a = LOAD(src + s * stride), b = LOAD(src + s * stride + 4);
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
  }
}

template <int ODT, class OutOff>
__device__ __forceinline__ void fused_reduce_slice(const float* part0, int64_t stride, int splits, int e_begin, int e_end,
                                                   void* out, bool acc_out, const OutOff& out_off) {
  for (int e = e_begin + (int)threadIdx.x * 8; e < e_end; e += (int)blockDim.x * 8) {
    float acc[8];
    sum_partials8<ld_cg_f4>(part0 + e, splits, stride, acc);
    const int64_t o = out_off(e);
    const float4 v0 = make_float4(acc[0], acc[1], acc[2], acc[3]), v1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
    if (acc_out) {
      store4<ODT, true>(out, o, v0);
      store4<ODT, true>(out, o + 4, v1);
    } else {
      store4<ODT, false>(out, o, v0);
      store4<ODT, false>(out, o + 4, v1);
    }
  }
}

// Fused split-K reduction, called by every CTA of a tile once its epilogue has stored the CTA's fp32 partial.  CTAs
// wait on their siblings, so the grid must have been launched cooperatively (all CTAs resident).  When the tile's
// arrival counter reaches `splits`, CTA `split` sums its slice of the tile's `total` elements over all partials
// (partial s at part0 + s * stride) and stores element e at out_off(e) of `out`; out_off must map 8 consecutive
// elements to 8 consecutive outputs.  The last CTA to finish re-arms the tile's two counters, so the counters are all
// zero again when the kernel ends.  `who` names the kernel's entry point in the timeout message; the callers' grids
// are (tile, split).
template <class OutOff>
__device__ __forceinline__ void fused_splitk_reduce(int* counters, int split, int splits, const float* part0,
                                                    int64_t stride, int total, void* out, int out_dtype, bool acc_out,
                                                    const OutOff& out_off, const char* who) {
  __threadfence();                     // this thread's partial-tile stores are visible device-wide ...
  __syncthreads();                     // ... for every thread of the CTA, before the CTA announces itself
  if (threadIdx.x == 0) {
    atomicAdd(counters, 1);
    const long long t0 = clock64();
    while (ld_acquire_gpu(counters) < splits) {
      __nanosleep(64);
      if (clock64() - t0 > 4000000000ll) {
        printf("%s: split-K arrival wait timed out (tile %d split %d)\n", who, (int)blockIdx.x, split);
        __trap();
      }
    }
  }
  __syncthreads();
  const int chunk = ((total / 8 + splits - 1) / splits) * 8;
  const int e_begin = split * chunk, e_end = min(e_begin + chunk, total);
  if (out_dtype == SMT_F32) fused_reduce_slice<SMT_F32>(part0, stride, splits, e_begin, e_end, out, acc_out, out_off);
  else if (out_dtype == SMT_BF16) fused_reduce_slice<SMT_BF16>(part0, stride, splits, e_begin, e_end, out, acc_out, out_off);
  else fused_reduce_slice<SMT_F16>(part0, stride, splits, e_begin, e_end, out, acc_out, out_off);
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(counters + 1, 1) == splits - 1) {   // every sibling has passed its wait: safe to re-arm
      counters[0] = 0;
      counters[1] = 0;
    }
  }
}

// Head of a split-K workspace: 2 self-resetting arrival counters per tile (zero when the workspace is handed over).
constexpr size_t kSplitCounterBytes = 16384;

// Checks the workspace of a launch that needs `need` bytes of it (0: no split) and splits it into the arrival
// counters and the fp32 partials that follow them.
inline int carve_split_workspace(const char* who, void* workspace, size_t workspace_bytes, size_t need, int** counters,
                                 float** partials) {
  *counters = nullptr;
  *partials = nullptr;
  if (need == 0) return SMT_OK;
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("%s: workspace too small (%zu < %zu)", who, workspace_bytes, need);
    return SMT_ERR_WORKSPACE;
  }
  SMT_CHECK_ARG(aligned16(workspace), "%s: workspace must be 16-byte aligned", who);
  *counters = static_cast<int*>(workspace);
  *partials = reinterpret_cast<float*>(static_cast<char*>(workspace) + kSplitCounterBytes);
  return SMT_OK;
}

// Launches a grid of tile CTAs: cooperatively when they run fused_splitk_reduce (which is only safe when the whole grid
// is resident), with <<<>>> otherwise.
template <class... Args>
int launch_tiles(void (*kern)(Args...), dim3 grid, int threads, int smem_bytes, bool cooperative, cudaStream_t st,
                 const Args&... args) {
  SMT_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  if (cooperative) {
    void* argv[] = {const_cast<Args*>(&args)...};
    SMT_CHECK_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(kern), grid, dim3(threads), argv,
                                               (size_t)smem_bytes, st));
    return SMT_OK;
  }
  kern<<<grid, threads, smem_bytes, st>>>(args...);
  SMT_CHECK_LAUNCH();
  return SMT_OK;
}

}  // namespace
}  // namespace smt
