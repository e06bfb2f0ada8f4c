// Owners of the CUDA resources of the library's handles (solver.cu, qp.cu): deleting a handle releases all of them.  An owner converts
// to the raw pointer / stream / event.  ensure() creates the resource only while the owner is empty and returns the CUDA error for the
// caller's fail: an array keeps the size of its first ensure(), so a caller that needs another size starts from a new owner.
#pragma once
#include <cuda_runtime.h>
#include <memory>
#include <type_traits>

namespace mpcdev {

template <class P, cudaError_t (*Release)(P)> struct CudaRelease { void operator()(P p) const { Release(p); } };

// T[count] in device memory, or in pinned host memory with PINNED
template <class T, bool PINNED = false>
struct CudaArray : std::unique_ptr<T, std::conditional_t<PINNED, CudaRelease<void *, cudaFreeHost>, CudaRelease<void *, cudaFree>>> {
  operator T *() const { return this->get(); }
  cudaError_t ensure(size_t count) {
    void *p = nullptr;
    const cudaError_t e = *this ? cudaSuccess : PINNED ? cudaMallocHost(&p, count * sizeof(T)) : cudaMalloc(&p, count * sizeof(T));
    if (p) this->reset(static_cast<T *>(p));
    return e;
  }
};

// a stream or an event, created with `flags`
template <class P, cudaError_t (*Create)(P *, unsigned), cudaError_t (*Destroy)(P)>
struct CudaObject : std::unique_ptr<std::remove_pointer_t<P>, CudaRelease<P, Destroy>> {
  operator P() const { return this->get(); }
  cudaError_t ensure(unsigned flags) {
    P p = nullptr;
    const cudaError_t e = *this ? cudaSuccess : Create(&p, flags);
    if (p) this->reset(p);
    return e;
  }
};
using CudaStream = CudaObject<cudaStream_t, cudaStreamCreateWithFlags, cudaStreamDestroy>;
using CudaEvent = CudaObject<cudaEvent_t, cudaEventCreateWithFlags, cudaEventDestroy>;

} // namespace mpcdev
