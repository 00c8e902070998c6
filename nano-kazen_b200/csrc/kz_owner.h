/* kz_owner.h -- move-only owners of the CUDA resources of a context (kz_api.cu) and of the arrays an accel build returns
 * (kz_lbvh.cuh).  Each releases what it holds when it is destroyed or reassigned, so an early return frees whatever was made
 * before it.  They are host-side only: kernels take the plain pointers they hold.
 */
#ifndef KZ_OWNER_H
#define KZ_OWNER_H
#include <cuda_runtime.h>
#include <algorithm>
#include <cstddef>

/* cudaMalloc memory: long-lived buffers (scene tables, accel, path pools, scratch) */
struct DevMem {
    void *p = nullptr;
    size_t bytes = 0;
    DevMem() = default;
    DevMem(DevMem &&o) noexcept : p(o.p), bytes(o.bytes) { o.p = nullptr; o.bytes = 0; }
    DevMem &operator=(DevMem &&o) noexcept {
        if (this != &o) { reset(); p = o.p; bytes = o.bytes; o.p = nullptr; o.bytes = 0; }
        return *this;
    }
    ~DevMem() { reset(); }
    void reset() {
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
    }
    /* frees what is held, then allocates max(n, 16) bytes; holds nothing if the allocation fails */
    cudaError_t alloc(size_t n) {
        reset();
        n = std::max<size_t>(n, 16);
        const cudaError_t e = cudaMalloc(&p, n);
        if (e == cudaSuccess) bytes = n;
        else p = nullptr;
        return e;
    }
    /* grow-only: keeps the buffer if it holds at least n bytes, else replaces it by one of max(n, at_least) bytes */
    cudaError_t ensure(size_t n, size_t at_least = 16) { return bytes >= n ? cudaSuccess : alloc(std::max(n, at_least)); }
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

/* cudaMallocAsync memory: short-lived buffers from the device's stream-ordered pool, freed with cudaFreeAsync on the stream
 * they were allocated on */
struct AsyncMem {
    void *p = nullptr;
    cudaStream_t s = nullptr;
    AsyncMem() = default;
    AsyncMem(const AsyncMem &) = delete;
    AsyncMem &operator=(const AsyncMem &) = delete;
    ~AsyncMem() { reset(); }
    void reset() {
        if (p) cudaFreeAsync(p, s);
        p = nullptr;
    }
    cudaError_t alloc(size_t n, cudaStream_t st) {
        reset();
        s = st;
        const cudaError_t e = cudaMallocAsync(&p, std::max<size_t>(n, 16), st);
        if (e != cudaSuccess) p = nullptr;
        return e;
    }
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

/* a stream or an event; converts to the raw handle, so it can be passed wherever one is expected */
template <typename H, cudaError_t (*Destroy)(H)> struct CudaHandle {
    H h = nullptr;
    CudaHandle() = default;
    CudaHandle(CudaHandle &&o) noexcept : h(o.h) { o.h = nullptr; }
    CudaHandle &operator=(CudaHandle &&o) noexcept {
        if (this != &o) { reset(); h = o.h; o.h = nullptr; }
        return *this;
    }
    ~CudaHandle() { reset(); }
    void reset() {
        if (h) Destroy(h);
        h = nullptr;
    }
    operator H() const { return h; }
};
using Stream = CudaHandle<cudaStream_t, cudaStreamDestroy>;
using Event = CudaHandle<cudaEvent_t, cudaEventDestroy>;

#endif
