// Library-level C-ABI entry points: version, error strings, launch counter.
#include "common.cuh"

namespace recmv {
unsigned long long g_launch_count = 0;
}

extern "C" int recmv_version(void) { return 102; }  // 0.1.2: + recmv_points_*

extern "C" int64_t recmv_launch_count(void) { return (int64_t)recmv::g_launch_count; }

extern "C" const char* recmv_error_string(int status) {
  switch (status) {
    case RECMV_OK: return "ok";
    case RECMV_E_NULL: return "required pointer is NULL";
    case RECMV_E_DTYPE: return "unknown dtype / layout / mode flag";
    case RECMV_E_SHAPE: return "non-positive, misaligned or inconsistent extent";
    case RECMV_E_RANGE: return "size exceeds an implementation limit";
    case RECMV_E_UNSUPPORTED: return "not supported by this build";
    case RECMV_E_DEVICE: return "a previous tcgen05 launch aborted on a bounded mbarrier wait (recmv_check_async_errors)";
    default: break;
  }
  if (status > 0) return cudaGetErrorString((cudaError_t)status);
  return "unknown recmv status";
}
