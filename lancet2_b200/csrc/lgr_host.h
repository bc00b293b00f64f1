// lgr_host.h — host-only helpers of the three CUDA libraries (lgr_gpu.cu, lgr_format.cu, lgr_repeat.cu): the
// CUDA error check of the entry points and the grow-only device buffer.  No device code here: lgr_format.cu is
// compiled with -fmad=false and includes this header too.
#ifndef LANCET2_B200_LGR_HOST_H_
#define LANCET2_B200_LGR_HOST_H_

#include <cuda_runtime.h>

#include <cstddef>
#include <string>

#include "../../include/lancet_gpu_realign.h"

// a failed CUDA call: the call and the runtime's message go to (ctx)->err, the entry point returns LGR_E_CUDA
#define LGR_CUDA(ctx, call)                                            \
  do {                                                                 \
    cudaError_t e_ = (call);                                           \
    if (e_ != cudaSuccess) {                                           \
      (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_); \
      return LGR_E_CUDA;                                               \
    }                                                                  \
  } while (0)

// One cudaMalloc block that only grows, freed with its owner (whose destroy function has selected the device).
struct DeviceBuffer {
  void* p = nullptr;
  size_t cap = 0;

  DeviceBuffer() = default;
  DeviceBuffer(const DeviceBuffer&) = delete;
  DeviceBuffer& operator=(const DeviceBuffer&) = delete;
  ~DeviceBuffer() {
    if (p) cudaFree(p);
  }

  // At least `bytes` (256 at least).  A regrow allocates half as much again, because cudaFree / cudaMalloc
  // synchronise the device, or exactly `bytes` when `exact` (a reservation).  On failure the buffer is empty, err
  // says why, and the runtime's last error is cleared so that it cannot fail the next call on this thread.
  int ensure(size_t bytes, bool exact, std::string& err) {
    if (bytes < 256) bytes = 256;
    if (cap >= bytes) return LGR_OK;
    if (p) cudaFree(p);
    p = nullptr, cap = 0;
    const size_t want = exact ? bytes : bytes + bytes / 2;
    const cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      p = nullptr;
      err = "cudaMalloc(" + std::to_string(want) + "): " + cudaGetErrorString(e);
      (void)cudaGetLastError();
      return LGR_E_NOMEM;
    }
    cap = want;
    return LGR_OK;
  }
};

#endif  // LANCET2_B200_LGR_HOST_H_
