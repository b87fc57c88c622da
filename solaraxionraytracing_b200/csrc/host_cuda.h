// host_cuda.h — the CUDA runtime helpers of the C-ABI layer (api.cu, comm.cu): error reporting and device switching.
#pragma once
#include <cuda_runtime.h>

#include "sart_internal.h"

namespace sart {

// Records "what: CUDA error" for sart_last_error() and returns SART_ERR_CUDA.
inline int cuda_fail(cudaError_t e, const char* what) {
  return fail(SART_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

#define SART_CUDA(call)                                  \
  do {                                                   \
    cudaError_t e__ = (call);                            \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

// Makes `dev` the current device for the guard's scope and puts the previous one back at its end.
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace sart
