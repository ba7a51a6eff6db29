// growbuf.cuh -- grow-only host-side allocations of the context and the solver (host code only)
#pragma once
#include <cuda_runtime.h>

namespace srb {

enum class Mem { DEVICE, PINNED, MAPPED };

// A buffer that is reallocated only when asked for more bytes than it holds (its contents are then lost).  A failed
// allocation leaves it empty.  MAPPED is pinned host memory the kernels address directly (zero-copy), 64 KB at least.
// Freed when it goes out of scope, on the device current at that time.
template <Mem K>
class GrowBuf {
 public:
  GrowBuf() = default;
  GrowBuf(const GrowBuf&) = delete;
  GrowBuf& operator=(const GrowBuf&) = delete;
  ~GrowBuf() { release(); }

  cudaError_t reserve(size_t bytes) {
    if (bytes <= bytes_) return cudaSuccess;
    release();
    if (K == Mem::MAPPED && bytes < (64u << 10)) bytes = 64u << 10;
    const cudaError_t e = K == Mem::DEVICE ? cudaMalloc(&p_, bytes)
                                           : cudaHostAlloc(&p_, bytes, K == Mem::MAPPED ? cudaHostAllocMapped : 0);
    if (e != cudaSuccess) p_ = nullptr;
    else bytes_ = bytes;
    return e;
  }
  void release() {
    if (p_) (void)(K == Mem::DEVICE ? cudaFree(p_) : cudaFreeHost(p_));
    p_ = nullptr;
    bytes_ = 0;
  }
  template <class T>
  T* as() const { return static_cast<T*>(p_); }

 private:
  void* p_ = nullptr;
  size_t bytes_ = 0;
};

using DeviceBuf = GrowBuf<Mem::DEVICE>;
using PinnedBuf = GrowBuf<Mem::PINNED>;
using MappedBuf = GrowBuf<Mem::MAPPED>;

}  // namespace srb
