// Owning handles for the CUDA memory, events and streams that a context or a per-device record keeps.  Each releases
// what it holds in its destructor, and allocating or creating into one releases what it held first, so no release
// routine has to list them.  Move-only, host code only.  Each converts to the plain pointer or handle, which is what
// launches and copies take.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include <algorithm>
#include <utility>

// One handle of type H (null: none), released with Release.
template <class H, auto Release>
class CudaOwned {
public:
    CudaOwned() = default;
    CudaOwned(CudaOwned &&o) noexcept : h_(std::exchange(o.h_, nullptr)) {}
    CudaOwned &operator=(CudaOwned o) noexcept { std::swap(h_, o.h_); return *this; }
    ~CudaOwned() { reset(); }

    void reset()
    {
        if (h_) Release(h_);
        h_ = nullptr;
    }
    operator H() const { return h_; }

protected:
    cudaError_t made(cudaError_t e)   // the result of a call that allocates or creates into h_
    {
        if (e) h_ = nullptr;
        return e;
    }
    H h_ = nullptr;
};

// An array of T in device memory: max(count, 1) elements plus 64 bytes of slack past the end.
template <class T>
class DeviceArray : public CudaOwned<T *, cudaFree> {
public:
    cudaError_t alloc(size_t count)
    {
        this->reset();
        n_ = count;
        return this->made(cudaMalloc((void **)&this->h_, std::max<size_t>(count, 1) * sizeof(T) + 64));
    }
    cudaError_t lazy(size_t count) { return this->h_ ? cudaSuccess : alloc(count); }                  // first call only
    cudaError_t grow(size_t count) { return this->h_ && count <= n_ ? cudaSuccess : alloc(count); }   // contents not kept
    size_t size() const { return this->h_ ? n_ : 0; }
    T *get() const { return this->h_; }

private:
    size_t n_ = 0;
};

// An array of T in pinned host memory, exactly count elements; cudaHostAllocWriteCombined suits a buffer that the host
// only writes and the copy engine only reads.
template <class T>
class PinnedArray : public CudaOwned<T *, cudaFreeHost> {
public:
    cudaError_t alloc(size_t count, unsigned flags = cudaHostAllocDefault)
    {
        this->reset();
        return this->made(cudaHostAlloc((void **)&this->h_, count * sizeof(T), flags));
    }
};

class CudaEvent : public CudaOwned<cudaEvent_t, cudaEventDestroy> {
public:
    cudaError_t create(unsigned flags = cudaEventDefault)
    {
        reset();
        return made(cudaEventCreateWithFlags(&h_, flags));
    }
};

// A stream the holder created, destroyed with it, or one it was lent, which it never destroys.
class CudaStream : public CudaOwned<cudaStream_t, cudaStreamDestroy> {
public:
    cudaError_t create(unsigned flags, int priority = 0)
    {
        borrow(nullptr);
        return made(cudaStreamCreateWithPriority(&h_, flags, priority));
    }
    void borrow(cudaStream_t s)
    {
        reset();
        lent_ = s;
    }
    operator cudaStream_t() const { return h_ ? h_ : lent_; }

private:
    cudaStream_t lent_ = nullptr;
};
