// Grow-only scratch memory, freed with its owner: device memory, or (Staging) pinned host memory with a
// device twin of the same size.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>

template <bool kPinned>
class ScratchBuffer {
 public:
  ScratchBuffer() = default;
  ScratchBuffer(const ScratchBuffer&) = delete;
  ScratchBuffer& operator=(const ScratchBuffer&) = delete;
  ~ScratchBuffer() { release(); }

  // Makes the buffer hold at least `bytes`.  A buffer too small is replaced after `stream` has finished with
  // it, by one of bytes + bytes / 4 + 256 (headroom for the next, slightly larger call).  On failure the
  // buffer is empty, the CUDA last error is cleared and the caller reports the error.
  bool grow(size_t bytes, cudaStream_t stream) {
    if (cap_ && bytes <= cap_) return true;
    if (cap_) cudaStreamSynchronize(stream);
    release();
    const size_t want = bytes + bytes / 4 + 256;
    if (cudaMalloc(&d_, want) != cudaSuccess || (kPinned && cudaMallocHost(&h_, want) != cudaSuccess)) {
      release();
      cudaGetLastError();
      return false;
    }
    cap_ = want;
    return true;
  }
  // cudaMalloc's pointer itself: 256-byte aligned, which the kernels' vector loads and the callers' 256-byte
  // sub-buffer layouts rely on
  void* d() const { return d_; }
  void* h() const {
    static_assert(kPinned, "a device buffer has no host side");
    return h_;
  }

 private:
  void release() {
    if (h_) cudaFreeHost(h_);
    if (d_) cudaFree(d_);
    h_ = d_ = nullptr;
    cap_ = 0;
  }
  void* d_ = nullptr;
  void* h_ = nullptr;
  size_t cap_ = 0;
};

using DeviceScratch = ScratchBuffer<false>;
using Staging = ScratchBuffer<true>;
