// devbuf.h -- owners of the device memory and events of a plan (host side only).
// A plan struct holds these instead of raw pointers: it is value-initialised, its destroy is a plain delete, and a create
// that fails part-way releases whatever it allocated when it deletes the unfinished plan.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>

template <typename T>
class DevBuf {
public:
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    ~DevBuf() { reset(); }

    // n elements, replacing what the buffer held
    cudaError_t alloc(size_t n)
    {
        reset();
        const cudaError_t e = cudaMalloc(&p_, n * sizeof(T));
        if (e != cudaSuccess) { p_ = nullptr; return e; }
        n_ = n;
        return cudaSuccess;
    }
    // grow-only scratch: keeps the buffer while it holds n elements, else frees it before allocating n
    cudaError_t ensure(size_t n) { return n_ >= n ? cudaSuccess : alloc(n); }

    void reset()
    {
        if (p_) cudaFree(p_);
        p_ = nullptr;
        n_ = 0;
    }
    T *get() const { return p_; }
    operator T *() const { return p_; }

private:
    T     *p_ = nullptr;
    size_t n_ = 0;
};

// an event without timing (what every plan records), created on first use
class DevEvent {
public:
    DevEvent() = default;
    DevEvent(const DevEvent &) = delete;
    DevEvent &operator=(const DevEvent &) = delete;
    DevEvent(DevEvent &&o) noexcept : e_(o.e_) { o.e_ = nullptr; }
    ~DevEvent() { if (e_) cudaEventDestroy(e_); }

    cudaError_t ensure() { return e_ ? cudaSuccess : cudaEventCreateWithFlags(&e_, cudaEventDisableTiming); }
    operator cudaEvent_t() const { return e_; }

private:
    cudaEvent_t e_ = nullptr;
};
