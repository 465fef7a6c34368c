// Error reporting, device checks and library identity for libvitk.
#include <stdarg.h>
#include <string.h>

#include <atomic>

#include "common.cuh"

namespace vitk {

static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_error(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return static_cast<int>(e);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int num_sms() {
  static thread_local int cached_dev = -1;
  static thread_local int cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

}  // namespace vitk

extern "C" VITK_API int vitk_version(void) { return VITK_VERSION; }

extern "C" VITK_API int64_t vitk_launch_count(void) { return vitk::g_launches.load(std::memory_order_relaxed); }

extern "C" VITK_API const char* vitk_last_error(void) { return vitk::g_err; }

extern "C" VITK_API int vitk_check_device(int dev) {
  int major = 0, minor = 0;
  VITK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  VITK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  VITK_REQUIRE(major == 10, VITK_EDEVICE, "device %d is sm_%d%d; libvitk is built for sm_100a only", dev, major, minor);
  return 0;
}
