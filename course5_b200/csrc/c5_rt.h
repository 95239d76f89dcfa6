// c5_rt.h — thin runtime layer under the library: device memory, copies, launches, sorts.
//
// Product build (default): CUDA runtime + CUB on the context's device.
// -DC5_HOSTSIM: the same translation units compiled so that "device" memory is host memory
// and every kernel body runs as a serial host loop. That build exists ONLY so the device
// functions' logic can be exercised by `-m "not gpu"` tests in a container without a GPU
// (tests/hostsim/); it is never loaded by course5_b200 and is not a fallback.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include <cuda_runtime.h>

#define C5_HD __host__ __device__ __forceinline__

#ifdef C5_HOSTSIM
constexpr bool kHostSim = true;
#else
constexpr bool kHostSim = false;
#endif

namespace c5 {

struct Error {
    int code;
    std::string text;
};

// Thrown inside the library, caught at the C ABI (no exception crosses it).
[[noreturn]] void fail(int code, const std::string& text);

#define C5_CUDA(expr)                                                                              \
    do {                                                                                           \
        cudaError_t _e = (expr);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            ::c5::fail(-2, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" + __FILE__ +  \
                               ":" + std::to_string(__LINE__) + ")");                              \
        }                                                                                          \
    } while (0)

// ---- memory ---------------------------------------------------------------------------------
void* dev_alloc(size_t bytes);
void dev_free(void* p);
void dev_zero(void* p, size_t bytes, cudaStream_t s);
void h2d(void* dst, const void* src, size_t bytes, cudaStream_t s);
void d2h(void* dst, const void* src, size_t bytes, cudaStream_t s);
void d2d(void* dst, const void* src, size_t bytes, cudaStream_t s);
// rows of `width` bytes, `height` of them, from src (pitch spitch) to dst (pitch dpitch), device to device
void d2d_2d(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height, cudaStream_t s);
void stream_sync(cudaStream_t s);
// `waiter` waits for the work enqueued on `producer` so far, through `ev` (recorded on `producer`).
void wait_for(cudaStream_t waiter, cudaStream_t producer, cudaEvent_t ev);
void* host_pinned_alloc(size_t bytes); // page-locked host memory (results the stream copies back while the host runs on)
void host_pinned_free(void* p);
size_t dev_bytes_in_use();

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    bool owner = true; // false: a view of memory another DevBuf owns (sibling contexts share the mesh)
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n), owner(o.owner) {
        o.p = nullptr;
        o.n = 0;
        o.owner = true;
    }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) {
            release();
            p = o.p;
            n = o.n;
            owner = o.owner;
            o.p = nullptr;
            o.n = 0;
            o.owner = true;
        }
        return *this;
    }
    void alias(const DevBuf& o) { // the owner must outlive this view
        release();
        p = o.p;
        n = o.n;
        owner = false;
    }
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        if (count) p = static_cast<T*>(dev_alloc(count * sizeof(T)));
        n = count;
    }
    void ensure(size_t count) {
        if (count > n) alloc(count);
    }
    void release() {
        if (p && owner) dev_free(p);
        p = nullptr;
        n = 0;
        owner = true;
    }
    size_t bytes() const { return n * sizeof(T); }
};

// ---- sorts / compaction (CUB on the device; std:: in hostsim) --------------------------------
// Stable LSD radix sorts of (key, value) pairs, in place.
void sort_pairs_u64(uint64_t* keys, uint32_t* vals, size_t n, int end_bit, cudaStream_t s);
void sort_pairs_u32(uint32_t* keys, uint32_t* vals, size_t n, int end_bit, cudaStream_t s);
// out[k] = i for the k-th i with flags[i] != 0; returns the count (synchronises s).
size_t select_flagged(const uint8_t* flags, uint32_t* out, size_t n, cudaStream_t s);

// ---- launches --------------------------------------------------------------------------------
extern thread_local uint64_t* g_launch_counter; // bumped once per kernel launch (or host loop)

inline void count_launch() {
    if (g_launch_counter) ++*g_launch_counter;
}

// The pixel kernel and the kernels that run beside it on an SM (a view's prologue and grazing-ray kernel) ask for one
// L1 / shared-memory split, so that a block of one can take the place a block of the other leaves without the SM
// draining first to change its split. Once per kernel and device.
void prefer_side_carveout(const void* kernel, int device);
template <class... A>
void prefer_side_carveout(void (*kernel)(A...), int device) {
    prefer_side_carveout(reinterpret_cast<const void*>(kernel), device);
}

#ifdef __CUDACC__
template <class F>
__global__ void k_for_each(int64_t n, F f) {
    const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
    if (i < n) f(i);
}

// f must be a trivially copyable functor with a C5_HD operator()(int64_t) const.
template <class F>
void for_each(cudaStream_t s, int64_t n, const F& f) {
    if (n <= 0) return;
    count_launch();
    if (kHostSim) {
        for (int64_t i = 0; i < n; i++) f(i);
    } else {
        const int block = 256;
        k_for_each<<<static_cast<unsigned>((n + block - 1) / block), block, 0, s>>>(n, f);
        C5_CUDA(cudaGetLastError());
    }
}
#endif

} // namespace c5
