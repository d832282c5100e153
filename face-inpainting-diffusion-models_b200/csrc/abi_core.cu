// Error plumbing and device probing for the C ABI (include/fidm_b200.h).
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace fidm {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace fidm

extern "C" int fidm_abi_version(void) { return FIDM_ABI_VERSION; }
extern "C" const char* fidm_last_error_string(void) { return fidm::g_err; }

extern "C" int fidm_device_supported(int dev) {
  cudaDeviceProp p;
  FIDM_CUDA(cudaGetDeviceProperties(&p, dev));
  FIDM_REQUIRE(p.major == 10, FIDM_E_BADARG, "device %d is sm_%d%d; this library is sm_100a only", dev,
               p.major, p.minor);
  return 0;
}
