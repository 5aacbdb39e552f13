// api.cu - library-level entry points: version, status strings, device query.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace dlmcq {

static thread_local char g_last_error[256] = "";

int set_cuda_error(cudaError_t e) {
  strncpy(g_last_error, cudaGetErrorString(e), sizeof(g_last_error) - 1);
  g_last_error[sizeof(g_last_error) - 1] = 0;
  return DLMCQ_ECUDA;
}

int num_sms() {
  // per-device cache; the attribute query costs microseconds, the launch path must not
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kNumSmFallback;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSmFallback;
    cached[dev] = n;
  }
  return cached[dev];
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("DLMCQ_NO_PDL");
    return !(e && e[0] == '1');
  }();
  return on;
}

}  // namespace dlmcq

extern "C" int dlmcq_version(void) { return DLMCQ_VERSION; }

extern "C" const char* dlmcq_status_string(int status) {
  switch (status) {
    case DLMCQ_OK: return "ok";
    case DLMCQ_EINVAL: return "invalid argument";
    case DLMCQ_EALIGN: return "pointer not aligned to its element size";
    case DLMCQ_EWORKSPACE: return "workspace too small";
    case DLMCQ_ECUDA: return "CUDA error (see dlmcq_last_cuda_error)";
    case DLMCQ_EUNSUPPORTED: return "unsupported configuration";
  }
  return "unknown status";
}

extern "C" const char* dlmcq_last_cuda_error(void) { return dlmcq::g_last_error; }
