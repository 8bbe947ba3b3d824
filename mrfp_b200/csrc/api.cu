// Library-level entry points: version, error strings, device info cache.
#include "common.cuh"
#include <mutex>

namespace mrfp {
int get_device_info(DeviceInfo* out) {
  static DeviceInfo cache[64];
  static bool filled[64] = {};
  static std::mutex mu;
  int dev = 0;
  MRFP_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return MRFP_ERR_UNSUPPORTED;
  std::lock_guard<std::mutex> lock(mu);
  if (!filled[dev]) {
    DeviceInfo d;
    d.device = dev;
    MRFP_CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev));
    MRFP_CUDA_TRY(cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cache[dev] = d;
    filled[dev] = true;
  }
  *out = cache[dev];
  return MRFP_OK;
}
}  // namespace mrfp

extern "C" int mrfp_version(void) { return 101; }

extern "C" const char* mrfp_strerror(int rc) {
  switch (rc) {
    case MRFP_OK: return "success";
    case MRFP_ERR_NULL_POINTER: return "mrfp: required pointer is NULL";
    case MRFP_ERR_BAD_SHAPE: return "mrfp: invalid shape argument";
    case MRFP_ERR_WORKSPACE: return "mrfp: workspace/saved buffer too small or misaligned";
    case MRFP_ERR_UNSUPPORTED: return "mrfp: unsupported math mode or channel count";
    case MRFP_ERR_BAD_PLAN: return "mrfp: invalid plan handle";
    case MRFP_ERR_DRIVER: return "mrfp: cuTensorMapEncodeTiled unavailable or failed";
    default: break;
  }
  if (rc > 0) return cudaGetErrorString((cudaError_t)rc);
  return "mrfp: unknown error";
}
