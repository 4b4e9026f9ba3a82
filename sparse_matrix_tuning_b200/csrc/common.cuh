// Shared helpers for the SMT sm_100a kernels: error plumbing, dtype dispatch, 128-bit loads,
// warp/block reductions.  Everything here is header-only except the thread-local error buffer
// (defined in capi.cu).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/smt_b200.h"

namespace smt {

void set_error(const char* fmt, ...);
void set_launch_count(int n);   // kernels launched by the last GEMM entry point on this thread

#define SMT_CHECK_ARG(cond, ...)                    \
  do {                                              \
    if (!(cond)) {                                  \
      ::smt::set_error(__VA_ARGS__);                \
      return SMT_ERR_ARG;                           \
    }                                               \
  } while (0)

#define SMT_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      ::smt::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, \
                       __LINE__);                                                         \
      return SMT_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define SMT_CHECK_LAUNCH() SMT_CHECK_CUDA(cudaGetLastError())

inline int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      return 148;
    cached = n;
  }
  return cached;
}

inline bool block_ok(int b) { return b == 64 || b == 128 || b == 256; }
inline int dtype_bytes(int dt) { return dt == SMT_F32 ? 4 : 2; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- device helpers ------------------------------------------------------------------------

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum; result valid in thread 0.  `scratch` needs >= 32 floats of shared memory.
__device__ __forceinline__ float block_sum(float v, float* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  const int nwarps = (blockDim.x + 31) >> 5;
  float r = 0.f;
  if (warp == 0) {
    r = lane < nwarps ? scratch[lane] : 0.f;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

// streaming 128-bit global load that does not pollute L1
__device__ __forceinline__ uint4 ld_stream_u4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const void* p) {
  uint4 r = ld_stream_u4(p);
  return make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z),
                     __uint_as_float(r.w));
}

// Unpack 8 16-bit floats held in a uint4 into 8 fp32.
template <int DT>
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (DT == SMT_BF16) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    } else {
      __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
      float2 t = __half22float2(h);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
}

template <int DT>
__device__ __forceinline__ float load_as_float(const void* p, int64_t i) {
  if (DT == SMT_F32) return reinterpret_cast<const float*>(p)[i];
  if (DT == SMT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
  return __half2float(reinterpret_cast<const __half*>(p)[i]);
}

template <int DT>
__device__ __forceinline__ void store_from_float(void* p, int64_t i, float v) {
  if (DT == SMT_F32) reinterpret_cast<float*>(p)[i] = v;
  else if (DT == SMT_BF16) reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
  else reinterpret_cast<__half*>(p)[i] = __float2half_rn(v);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 t = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}

}  // namespace smt
