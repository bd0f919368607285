// api.cu -- version, status strings and the thread-local error detail.
#include <stdarg.h>

#include "common.cuh"

namespace d2b {
static thread_local char g_err[512] = "";
void set_last_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
bool pdl_enabled(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return cs == cudaStreamCaptureStatusNone;
}
static unsigned long long g_launches = 0;
void count_launch() { __atomic_fetch_add(&g_launches, 1ull, __ATOMIC_RELAXED); }
}  // namespace d2b

extern "C" uint64_t d2b_kernel_launch_count(void) { return __atomic_load_n(&d2b::g_launches, __ATOMIC_RELAXED); }

extern "C" int d2b_version(void) { return 100; /* 0.1.0 */ }

extern "C" const char* d2b_status_string(int s) {
  switch (s) {
    case D2B_OK: return "ok";
    case D2B_EINVAL: return "invalid argument";
    case D2B_EWORKSPACE: return "workspace too small or NULL";
    case D2B_ECUDA: return "CUDA error";
    case D2B_EUNSUPPORTED: return "unsupported configuration";
    default: return "unknown status";
  }
}

extern "C" const char* d2b_last_error(void) { return d2b::g_err; }
