// common.cuh -- shared device helpers and host-side plumbing for libsdr_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <atomic>
#include <cstddef>
#include <memory>
#include <new>

#include "../../include/sdr_b200.h"

namespace sdr {

// ---- host-side error plumbing -----------------------------------------------------------
inline int cuda_status(cudaError_t e) { return e == cudaSuccess ? SDR_OK : SDR_ERR_CUDA_BASE + (int)e; }
#define SDR_CUDA_TRY(expr)                                  \
    do {                                                    \
        cudaError_t _e = (expr);                            \
        if (_e != cudaSuccess) return sdr::cuda_status(_e); \
    } while (0)

extern std::atomic<uint64_t> g_launches;
inline void count_launch(uint64_t n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
inline int launch_status() { return cuda_status(cudaGetLastError()); }

// RAII device selection that restores the caller's current device (handles must not depend on
// thread-local CUDA state: SURVEY 8b "Threading").
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) {
            err = cudaSetDevice(dev);
            ok = (err == cudaSuccess);
        }
    }
    // every int-returning entry point checks this: a failed cudaSetDevice must not let the call run on the
    // caller's current device
    int status() const { return ok ? SDR_OK : SDR_ERR_CUDA_BASE + (int)err; }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

// SM count of the CURRENT device (launchers run under a DeviceGuard).  Cached per device ordinal; the cache entries
// are atomics, so concurrent first calls from handles on different threads / devices are benign.
inline int current_sm_count() {
    static std::atomic<int> cache[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    if (dev >= 0 && dev < 64) {
        const int c = cache[dev].load(std::memory_order_relaxed);
        if (c > 0) return c;
    }
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return 1;
    if (dev >= 0 && dev < 64) cache[dev].store(sms, std::memory_order_relaxed);
    return sms;
}

// SDR_OK, SDR_ERR_NO_DEVICE when the runtime sees no device, SDR_ERR_INVALID_ARG for an ordinal out of range
inline int check_device(int dev) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return SDR_ERR_NO_DEVICE;
    }
    if (dev < 0 || dev >= n) return SDR_ERR_INVALID_ARG;
    return SDR_OK;
}

// the caller's stream, or one the handle creates and destroys
struct StreamRef {
    cudaStream_t s = nullptr;
    bool owned = false;
    StreamRef() = default;
    StreamRef(const StreamRef &) = delete;
    StreamRef &operator=(const StreamRef &) = delete;
    ~StreamRef() {
        if (owned) cudaStreamDestroy(s);
    }
    int init(void *user) {
        if (user) {
            s = (cudaStream_t)user;
            owned = false;
            return SDR_OK;
        }
        cudaError_t e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        owned = (e == cudaSuccess);
        return cuda_status(e);
    }
};

// one device allocation, freed with its owner (on the device current at that point: a DeviceGuard outlives it)
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    // grow-only scratch: at least `bytes`, with slack so that slowly growing calls rarely reallocate
    int reserve(size_t bytes) {
        if (bytes <= cap) return SDR_OK;
        return alloc(bytes + bytes / 8 + 256);
    }
    // exactly `bytes` (tables and state whose size is fixed); the old contents are dropped
    int alloc(size_t bytes) {
        release();
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            p = nullptr;
            return cuda_status(e);
        }
        cap = bytes;
        return SDR_OK;
    }
    // exactly `bytes`, filled from the host in stream order
    int upload(const void *host, size_t bytes, cudaStream_t st) {
        int rc = alloc(bytes);
        if (rc) return rc;
        return cuda_status(cudaMemcpyAsync(p, host, bytes, cudaMemcpyHostToDevice, st));
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// an owned sub-handle, released with the ABI's own destroy function
template <auto Destroy>
struct AbiDeleter {
    template <class T>
    void operator()(T *h) const { Destroy(h); }
};
template <class T, auto Destroy>
using Owned = std::unique_ptr<T, AbiDeleter<Destroy>>;

// ---- handle lifecycle -------------------------------------------------------------------
// A handle H derives from a copyable host-state struct (configuration, geometry, host tables, stream position) that
// holds `int dev`, and adds its device resources: `StreamRef stream` first (destroyed last), then sub-handles, DevBufs.
// It supplies
//     int alloc(void *user_stream, const H *src)   stream, tables and buffers for the host state; src: clone source
//     int copy_device(const H &src)                 the source's carried device state (clone only)
// and the templates below do the rest.

// *err = code (err may be null); returns the null handle
inline std::nullptr_t fail(int *err, int code) {
    if (err) *err = code;
    return nullptr;
}

template <class H>
void destroy_handle(H *h) {
    if (!h) return;
    DeviceGuard g(h->dev);
    delete h;
}

// after the handle's own argument checks: device check, host state (init(H &) -> error code), then alloc
template <class H, class Init>
H *create_handle(int *err, int dev, void *user_stream, Init &&init) {
    int dummy;
    if (!err) err = &dummy;
    if ((*err = check_device(dev)) != SDR_OK) return nullptr;
    H *h = new (std::nothrow) H;
    if (!h) return fail(err, SDR_ERR_MALLOC_FAILED);
    h->dev = dev;
    DeviceGuard g(dev);
    *err = init(*h);
    if (!*err) *err = g.ok ? h->alloc(user_stream, nullptr) : g.status();
    if (!*err) return h;
    delete h;
    return nullptr;
}

// a handle with the source's host state and a copy of its device state; it allocates on the source's stream when the
// caller owns that stream, else on a stream of its own
template <class State, class H>
H *clone_handle(const H *src, int *err) {
    int dummy;
    if (!err) err = &dummy;
    if (!src) return fail(err, SDR_ERR_NULL_HANDLE);
    H *h = new (std::nothrow) H;
    if (!h) return fail(err, SDR_ERR_MALLOC_FAILED);
    static_cast<State &>(*h) = static_cast<const State &>(*src);
    DeviceGuard g(h->dev);
    *err = g.status();
    // the source's pending work is part of the state it hands over (and alloc may read its device tables)
    if (!*err) *err = cuda_status(cudaStreamSynchronize(src->stream.s));
    if (!*err) *err = h->alloc(src->stream.owned ? nullptr : (void *)src->stream.s, src);
    if (!*err) *err = h->copy_device(*src);
    if (!*err) return h;
    delete h;
    return nullptr;
}

// ---- device helpers ---------------------------------------------------------------------
#ifdef __CUDACC__

// (b as f32 - 128.0) / 128.0, exactly (src/rtltcp.rs:160-163).  byte `idx` of `word`.
// 0x4B000000 | b is the float 8388608 + b; (8388608 + b)/128 = 65536 + b/128 is exact in f32 and
// so is the subtraction of 65537, hence one PRMT + one FFMA give the reference's value bit for bit.
__device__ __forceinline__ float unpack_byte(uint32_t word, int idx) {
    const uint32_t m = __byte_perm(word, 0x4B000000u, 0x7540u | (uint32_t)idx);
    return __fmaf_rn(__uint_as_float(m), 0.0078125f, -65537.0f);
}
__device__ __forceinline__ float2 unpack_iq16(uint32_t word, int pair) {  // pair 0: bytes 0,1 ; pair 1: bytes 2,3
    return make_float2(unpack_byte(word, 2 * pair), unpack_byte(word, 2 * pair + 1));
}
__device__ __forceinline__ float2 unpack_iq_u16(uint16_t h) {
    return make_float2(unpack_byte((uint32_t)h, 0), unpack_byte((uint32_t)h, 1));
}

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
// sm_100 packed FP32: one FADD2 per complex add / subtract.  Same flops per cycle as two FADDs (FADD2 issues at half
// rate, profiles/r01_f32x2_rate_probe.txt) but half the issue slots -- a gain for the issue-bound FFT kernels, a loss
// for some others (measured per kernel, see fft.cu), hence a template switch rather than a global one.
__device__ __forceinline__ float2 cadd_p(float2 a, float2 b) {
    unsigned long long r;
    asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&r);
}
__device__ __forceinline__ float2 csub_p(float2 a, float2 b) {
    unsigned long long r;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(*reinterpret_cast<unsigned long long *>(&a)), "l"(*reinterpret_cast<unsigned long long *>(&b)));
    return *reinterpret_cast<float2 *>(&r);
}
template <bool PK> __device__ __forceinline__ float2 cadd_t(float2 a, float2 b) { return PK ? cadd_p(a, b) : cadd(a, b); }
template <bool PK> __device__ __forceinline__ float2 csub_t(float2 a, float2 b) { return PK ? csub_p(a, b) : csub(a, b); }

#endif  // __CUDACC__

}  // namespace sdr
