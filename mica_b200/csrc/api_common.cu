// Error plumbing and bookkeeping entry points of the C ABI.
#include <stdarg.h>
#include <stdlib.h>

#include "common.cuh"

namespace mica {
thread_local char g_last_error[512] = "";
std::atomic<int64_t> g_launches{0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return MICA_OK;
  int code = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? MICA_ERR_NO_DEVICE : MICA_ERR_CUDA;
  return set_error(code, "%s: %s", what, cudaGetErrorString(e));
}
long long peer_timeout_cycles() {
  long long ms = 60000;
  if (const char* env = getenv("MICA_PEER_TIMEOUT_MS")) {
    const long long v = atoll(env);
    if (v > 0) ms = v;
  }
  return ms * 2000000LL;   // clock64 runs at <= 1.97 GHz on a B200
}
TensorMapEncodeFn tensor_map_encode_fn() {
  // looked up once; a function-local static is initialised once even when several threads call at the same time
  static const TensorMapEncodeFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    const bool found = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
                       q == cudaDriverEntryPointSuccess;
    return found ? (TensorMapEncodeFn)p : nullptr;
  }();
  return fn;
}
}  // namespace mica

extern "C" {
int mica_version(void) { return 100; }
const char* mica_last_error(void) { return mica::g_last_error; }
int mica_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    mica::set_error(MICA_ERR_NO_DEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    return MICA_ERR_NO_DEVICE;
  }
  return n;
}
int64_t mica_launch_count(void) { return mica::g_launches.load(); }
}
