// dyn_smem.hpp -- the dynamic shared-memory opt-in of the kernel launchers (host code; kept out of
// device.cuh, which the host-only CPU emulation compiles as well).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>

namespace bart {

// Lets `Kernel` launch with `bytes` of dynamic shared memory: past the 48 KB default the limit is
// raised, once per kernel and larger size.  Returns false when the attribute call fails; the caller
// then launches nothing, and the error stays for the launch check to report.
template <auto Kernel>
bool allow_dyn_smem(size_t bytes) {
  static size_t configured = 0;
  if (bytes > 48 * 1024 && bytes > configured) {
    if (cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
      return false;
    configured = bytes;
  }
  return true;
}

}  // namespace bart
