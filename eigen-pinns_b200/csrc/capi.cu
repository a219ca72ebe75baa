// Library-level entry points: version, last-error string, device query.
#include <string.h>
#include "ep_common.cuh"

namespace ep {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static int cached = 0;
  if (cached > 0) return cached;
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  cached = n;
  return cached;
}

static int g_tune[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
int tune_flag(int key) { return (key >= 0 && key < 16) ? g_tune[key] : 0; }
void set_tune_flag(int key, int value) { if (key >= 0 && key < 16) g_tune[key] = value; }

}  // namespace ep

extern "C" {

int ep_version(void) { return 10000 * 0 + 100 * 3 + 0; }

const char* ep_last_error_string(void) { return ep::g_err; }

int ep_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  EP_CUDA_CHECK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  EP_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return EP_OK;
}

}  // extern "C"
