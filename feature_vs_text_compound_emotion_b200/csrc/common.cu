#include "common.h"

namespace cer {
static thread_local std::string g_last_error;
int set_error(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
static thread_local const char* g_head_variant = "none";
void set_head_variant(const char* name) { g_head_variant = name; }
}  // namespace cer

extern "C" const char* cer_last_error(void) { return cer::g_last_error.c_str(); }
extern "C" int cer_version(void) { return 104; }
extern "C" const char* cer_head_last_variant(void) { return cer::g_head_variant; }

extern "C" int cer_check_device(void) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cer::set_error(CER_ERR_CUDA, std::string("cudaGetDevice: ") + cudaGetErrorString(e));
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) return cer::set_error(CER_ERR_CUDA, std::string("cudaDeviceGetAttribute: ") + cudaGetErrorString(e));
  if (major != 10) return cer::set_error(CER_ERR_ARCH, "device is not compute capability 10.x (sm_100a kernels only)");
  return CER_OK;
}
