// device_buffer.hpp — owning handles for the device memory, pinned host memory, events and stream of a context (engine.cu).
#pragma once
#include <cuda_runtime.h>
#include <memory>
#include <utility>

// size() elements of T from Alloc, handed to Free when the array is destroyed or reallocated; move-only
template <typename T, cudaError_t (*Alloc)(void**, size_t), cudaError_t (*Free)(void*)>
class CudaArray {
 public:
  CudaArray() = default;
  CudaArray(CudaArray&& o) noexcept : p_(std::move(o.p_)), n_(std::exchange(o.n_, 0)) {}
  CudaArray& operator=(CudaArray&& o) noexcept { p_ = std::move(o.p_); n_ = std::exchange(o.n_, 0); return *this; }
  // frees the current elements, then allocates n uninitialised ones; the array is left empty if that fails
  cudaError_t alloc(size_t n) {
    p_.reset();
    void* p = nullptr;
    const cudaError_t err = Alloc(&p, n * sizeof(T));
    p_.reset(err == cudaSuccess ? static_cast<T*>(p) : nullptr);
    n_ = err == cudaSuccess ? n : 0;
    return err;
  }
  T* get() const { return p_.get(); }
  size_t size() const { return n_; }

 private:
  struct Deleter { void operator()(T* p) const { Free(p); } };
  std::unique_ptr<T, Deleter> p_;
  size_t n_ = 0;
};
template <typename T> using DeviceArray = CudaArray<T, cudaMalloc, cudaFree>;
template <typename T> using PinnedArray = CudaArray<T, cudaMallocHost, cudaFreeHost>;

template <typename H, cudaError_t (*Destroy)(H)>
struct CudaDestroy { void operator()(H h) const { Destroy(h); } };
using Event = std::unique_ptr<CUevent_st, CudaDestroy<cudaEvent_t, cudaEventDestroy>>;
using OwnedStream = std::unique_ptr<CUstream_st, CudaDestroy<cudaStream_t, cudaStreamDestroy>>;
