// Owner of the CUDA resources one initialised handle acquires (context.cu, road.cu): device and pinned host
// allocations, streams and events.  Each is recorded as it is acquired, and the destructor releases all of them, so
// that Finish, destroy and a failed Initialize release everything the handle holds.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <vector>

namespace isx {

class CudaResources {
 public:
  explicit CudaResources(int device) : device_(device) {}
  CudaResources(const CudaResources &) = delete;
  CudaResources &operator=(const CudaResources &) = delete;

  // Waits for all work on the device (work of the handle may still be queued, and a host function it enqueued may
  // still run on a driver thread), then releases everything in the reverse order of acquisition.
  ~CudaResources() {
    cudaSetDevice(device_);
    cudaDeviceSynchronize();
    for (auto it = items_.rbegin(); it != items_.rend(); ++it) {
      switch (it->kind) {
        case kDevice: cudaFree(it->p); break;
        case kHost: cudaFreeHost(it->p); break;
        case kStream: cudaStreamDestroy(static_cast<cudaStream_t>(it->p)); break;
        case kEvent: cudaEventDestroy(static_cast<cudaEvent_t>(it->p)); break;
      }
    }
  }

  template <typename T>
  cudaError_t device(T **out, size_t bytes) {
    const cudaError_t e = cudaMalloc(out, bytes);
    return keep(e, kDevice, *out);
  }
  template <typename T>
  cudaError_t host(T **out, size_t bytes, unsigned flags = cudaHostAllocDefault) {
    const cudaError_t e = cudaHostAlloc(out, bytes, flags);
    return keep(e, kHost, *out);
  }
  // A non-blocking stream; priority 0 is the default priority.
  cudaError_t stream(cudaStream_t *out, int priority = 0) {
    const cudaError_t e = cudaStreamCreateWithPriority(out, cudaStreamNonBlocking, priority);
    return keep(e, kStream, *out);
  }
  cudaError_t event(cudaEvent_t *out, unsigned flags = cudaEventDisableTiming) {
    const cudaError_t e = cudaEventCreateWithFlags(out, flags);
    return keep(e, kEvent, *out);
  }

 private:
  enum Kind { kDevice, kHost, kStream, kEvent };
  struct Item {
    Kind kind;
    void *p;
  };
  // Records what a successful call acquired; clears the error of a failed one, which the caller gets returned.
  cudaError_t keep(cudaError_t e, Kind kind, void *p) {
    if (e == cudaSuccess) items_.push_back(Item{kind, p});
    else cudaGetLastError();   // a later cudaGetLastError (behind a kernel launch) must not report it again
    return e;
  }

  int device_;
  std::vector<Item> items_;
};

}  // namespace isx
