// Process-wide pieces of the C-ABI: thread-local error text, version, device info.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace smt {
namespace {
thread_local char g_err[512] = "";
thread_local int g_launches = 0;
}
void set_launch_count(int n) { g_launches = n; }
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace smt

extern "C" SMT_API const char* smt_last_error(void) { return smt::g_err; }

extern "C" SMT_API int smt_last_launch_count(void) { return smt::g_launches; }

extern "C" SMT_API int smt_version(void) { return 210; /* 0.2.1: + decoder-layer elementwise kernels (RMSNorm, RoPE, SwiGLU) */ }

extern "C" SMT_API int smt_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host) {
  int dev = 0;
  SMT_CHECK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  SMT_CHECK_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sm_count_host) *sm_count_host = prop.multiProcessorCount;
  if (cc_major_host) *cc_major_host = prop.major;
  if (cc_minor_host) *cc_minor_host = prop.minor;
  return SMT_OK;
}
