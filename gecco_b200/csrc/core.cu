// Library-wide state of the C ABI: error text, device checks.
#include "common.cuh"

#include <string.h>

namespace gecco {

namespace {
thread_local char g_err[512] = "";
int g_sms = 0;
}  // namespace

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  if (g_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_sms <= 0) g_sms = 148;
  }
  return g_sms;
}

int resolve_driver();

thread_local long long g_launches = 0;

}  // namespace gecco

extern "C" int64_t gecco_launch_count(int32_t reset) {
  const long long n = gecco::g_launches;
  if (reset) gecco::g_launches = 0;
  return n;
}

extern "C" int gecco_abi_version(void) { return GECCO_ABI_VERSION; }

extern "C" const char* gecco_last_error(void) { return gecco::g_err; }

extern "C" int gecco_init(int device) {
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return gecco::fail_cuda(e, "cudaGetDeviceProperties");
  if (prop.major != 10) {
    gecco::set_error("device %d is sm_%d%d; gecco_b200 is built for sm_100a only and has no fallback", device,
                     prop.major, prop.minor);
    return GECCO_ERR_DEVICE;
  }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return gecco::fail_cuda(e, "cudaSetDevice");
  return gecco::resolve_driver();
}
