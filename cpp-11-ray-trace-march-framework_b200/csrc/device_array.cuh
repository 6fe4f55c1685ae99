// Owning arrays of device and page-locked host memory, and a stream drain for the temporaries of a call.
#pragma once

#include <utility>
#include <cuda_runtime.h>

namespace rtm
{

// size() elements of device memory (kPinned: page-locked host memory, allocated with kHostFlags); move-only.  The
// memory is freed, ignoring errors, on the device that was current at alloc(), and the current device stays as it is.
template <class T, bool kPinned, unsigned kHostFlags>
class OwnedArray
{
public:
    OwnedArray() = default;
    OwnedArray(OwnedArray&& o) noexcept { swap(o); }
    OwnedArray& operator=(OwnedArray&& o) noexcept { OwnedArray(std::move(o)).swap(*this); return *this; }
    ~OwnedArray() { release(); }

    T *get() const { return p_; }
    size_t size() const { return n_; }

    // Frees what the array holds and allocates n elements on the current device (none, when that fails)
    cudaError_t alloc(size_t n)
    {
        release();
        void *p = nullptr;
        cudaError_t e = cudaGetDevice(&dev_);
        if (e == cudaSuccess)
            e = kPinned ? cudaHostAlloc(&p, n * sizeof(T), kHostFlags) : cudaMalloc(&p, n * sizeof(T));
        if (e == cudaSuccess)
        {
            p_ = static_cast<T *>(p);
            n_ = n;
        }
        return e;
    }

    // alloc(n), discarding the contents, only when the array holds fewer than n elements; then sets *grown
    cudaError_t grow(size_t n, bool *grown = nullptr)
    {
        if (n <= n_)
            return cudaSuccess;
        if (grown)
            *grown = true;
        return alloc(n);
    }

    void release()
    {
        if (p_)
        {
            int cur = dev_;
            cudaGetDevice(&cur);
            if (cur != dev_) cudaSetDevice(dev_);
            kPinned ? cudaFreeHost(p_) : cudaFree(p_);
            if (cur != dev_) cudaSetDevice(cur);
        }
        p_ = nullptr;
        n_ = 0;
    }

private:
    void swap(OwnedArray& o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); std::swap(dev_, o.dev_); }
    T *p_ = nullptr;
    size_t n_ = 0;
    int dev_ = 0;
};

template <class T>
using DeviceArray = OwnedArray<T, false, 0>;
template <class T, unsigned kHostFlags = cudaHostAllocDefault>
using PinnedArray = OwnedArray<T, true, kHostFlags>;

// Synchronises the stream at the end of the scope unless sync() did.  Declared after the temporaries a call enqueues
// work on, it makes every return, failures included, release them only once that work is done.
class StreamDrain
{
public:
    explicit StreamDrain(cudaStream_t s) : s_(s) {}
    ~StreamDrain() { if (pending_) cudaStreamSynchronize(s_); }
    cudaError_t sync() { pending_ = false; return cudaStreamSynchronize(s_); }

private:
    cudaStream_t s_;
    bool pending_ = true;
};

} // namespace rtm
