// Error plumbing shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <string>
#include "../../include/cer_b200.h"

namespace cer {
int set_error(int code, const std::string& msg);   // records msg for cer_last_error(), returns code
void set_head_variant(const char* name);           // records the kernel a head launch site ran (cer_head_last_variant)
}

#define CER_CUDA(expr)                                                                              \
  do {                                                                                              \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess)                                                                          \
      return ::cer::set_error(CER_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));    \
  } while (0)

namespace cer {
// Kernel attributes (max dynamic shared memory) belong to a device context: one-time setup must
// run once per DEVICE, not once per process.  `mask` is a static bitmask owned by the call site.
inline bool first_use_on_device(unsigned long long* mask) {
  int dev = 0;
  cudaGetDevice(&dev);
  const unsigned long long bit = 1ull << (dev & 63);
  if (*mask & bit) return false;
  *mask |= bit;
  return true;
}
}  // namespace cer
