// c5_rt.cu — runtime layer: device memory, copies, CUB sorts (host equivalents under C5_HOSTSIM).
#include "c5_rt.h"

#include <algorithm>
#include <atomic>
#include <mutex>
#include <unordered_map>
#include <numeric>
#include <vector>

#ifndef C5_HOSTSIM
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>
#endif

namespace c5 {

thread_local uint64_t* g_launch_counter = nullptr;
static std::atomic<size_t> g_bytes{0};

[[noreturn]] void fail(int code, const std::string& text) {
    throw Error{code, text};
}

// Allocation sizes are tracked on the host so c5_mesh_info.device_bytes is exact.
static std::mutex g_alloc_mu;
static std::unordered_map<void*, size_t> g_allocs;

void* dev_alloc(size_t bytes) {
    void* p = nullptr;
    if (kHostSim) {
        p = std::aligned_alloc(256, ((bytes + 255) / 256) * 256);
        if (!p) fail(-3, "host allocation failed (hostsim)");
    } else {
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            fail(e == cudaErrorMemoryAllocation ? -3 : -2,
                 std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
        }
    }
    {
        std::lock_guard<std::mutex> lock(g_alloc_mu);
        g_allocs[p] = bytes;
    }
    g_bytes += bytes;
    return p;
}

void dev_free(void* p) {
    if (!p) return;
    size_t bytes = 0;
    {
        std::lock_guard<std::mutex> lock(g_alloc_mu);
        auto it = g_allocs.find(p);
        if (it != g_allocs.end()) {
            bytes = it->second;
            g_allocs.erase(it);
        }
    }
    if (kHostSim) {
        std::free(p);
    } else {
        cudaFree(p);
    }
    g_bytes -= bytes;
}

size_t dev_bytes_in_use() {
    return g_bytes.load();
}

void dev_zero(void* p, size_t bytes, cudaStream_t s) {
    if (!bytes) return;
    if (kHostSim) {
        std::memset(p, 0, bytes);
    } else {
        C5_CUDA(cudaMemsetAsync(p, 0, bytes, s));
    }
}

void h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (!bytes) return;
    if (kHostSim) {
        std::memcpy(dst, src, bytes);
    } else {
        C5_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
    }
}

void d2h(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (!bytes) return;
    if (kHostSim) {
        std::memcpy(dst, src, bytes);
    } else {
        C5_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
    }
}

void d2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
    if (!bytes) return;
    if (kHostSim) {
        std::memmove(dst, src, bytes);
    } else {
        C5_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
    }
}

void d2d_2d(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height, cudaStream_t s) {
    if (!width || !height) return;
    if (kHostSim) {
        for (size_t r = 0; r < height; r++) {
            std::memcpy(static_cast<char*>(dst) + r * dpitch, static_cast<const char*>(src) + r * spitch, width);
        }
    } else {
        C5_CUDA(cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, cudaMemcpyDeviceToDevice, s));
    }
}

void* host_pinned_alloc(size_t bytes) {
    void* p = nullptr;
    if (kHostSim) {
        p = std::malloc(bytes ? bytes : 1);
        if (!p) fail(-3, "host allocation failed");
    } else {
        C5_CUDA(cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable));
    }
    return p;
}

void host_pinned_free(void* p) {
    if (!p) return;
    if (kHostSim) std::free(p);
    else cudaFreeHost(p);
}

void stream_sync(cudaStream_t s) {
    if (!kHostSim) C5_CUDA(cudaStreamSynchronize(s));
}

// 100 KB of shared memory per SM. Beside seven blocks of the pixel kernel (1 KB each, reserved by the hardware) that
// holds four blocks of the solid mask (22 KB each) or seven of the grazing-ray kernel (11 KB each); alone, the
// grazing-ray kernel gets eight blocks per SM (C3 on one B200: 0.52 ms, 0.47 with the twelve of its grid). The pixel
// kernel alone pays 1 % for the L1 this takes (3.49 -> 3.53 ms); 64 KB cost the grazing-ray kernel alone 40 % and
// the pipelined views half the gain (profiles/r15_arms_c3_one_b200.jsonl).
constexpr int64_t kSideSmemBytes = 100 * 1024;

void prefer_side_carveout(const void* kernel, int device) {
    if (kHostSim) return;
    static std::mutex mu;
    static std::vector<std::pair<const void*, int>> done;
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<const void*, int> key{kernel, device};
    if (std::find(done.begin(), done.end(), key) != done.end()) return;
    int per_sm = 0;
    C5_CUDA(cudaDeviceGetAttribute(&per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, device));
    // a percentage of the most an SM can hold, rounded down here and up by the driver to a split the SM has
    const int percent = static_cast<int>(std::min<int64_t>(100, kSideSmemBytes * 100 / per_sm));
    C5_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, percent));
    done.push_back(key);
}

void wait_for(cudaStream_t waiter, cudaStream_t producer, cudaEvent_t ev) {
    if (!kHostSim) {
        C5_CUDA(cudaEventRecord(ev, producer));
        C5_CUDA(cudaStreamWaitEvent(waiter, ev, 0));
    }
}

#ifdef C5_HOSTSIM

template <class K>
static void host_sort_pairs(K* keys, uint32_t* vals, size_t n) {
    std::vector<size_t> idx(n);
    std::iota(idx.begin(), idx.end(), size_t{0});
    std::stable_sort(idx.begin(), idx.end(), [&](size_t a, size_t b) { return keys[a] < keys[b]; });
    std::vector<K> k2(n);
    std::vector<uint32_t> v2(n);
    for (size_t i = 0; i < n; i++) {
        k2[i] = keys[idx[i]];
        v2[i] = vals[idx[i]];
    }
    std::copy(k2.begin(), k2.end(), keys);
    std::copy(v2.begin(), v2.end(), vals);
}

void sort_pairs_u64(uint64_t* keys, uint32_t* vals, size_t n, int, cudaStream_t) {
    count_launch();
    host_sort_pairs(keys, vals, n);
}
void sort_pairs_u32(uint32_t* keys, uint32_t* vals, size_t n, int, cudaStream_t) {
    count_launch();
    host_sort_pairs(keys, vals, n);
}
size_t select_flagged(const uint8_t* flags, uint32_t* out, size_t n, cudaStream_t) {
    count_launch();
    size_t k = 0;
    for (size_t i = 0; i < n; i++) {
        if (flags[i]) out[k++] = static_cast<uint32_t>(i);
    }
    return k;
}

#else

template <class K>
static void cub_sort_pairs(K* keys, uint32_t* vals, size_t n, int end_bit, cudaStream_t s) {
    if (n < 2) return;
    if (n > 0x7FFFFFFFull) fail(-1, "sort: more than 2^31 items");
    count_launch();
    DevBuf<K> k2;
    DevBuf<uint32_t> v2;
    k2.alloc(n);
    v2.alloc(n);
    size_t temp_bytes = 0;
    C5_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, k2.p, vals, v2.p, static_cast<int>(n), 0,
                                            end_bit, s));
    DevBuf<uint8_t> temp;
    temp.alloc(temp_bytes ? temp_bytes : 1);
    C5_CUDA(cub::DeviceRadixSort::SortPairs(temp.p, temp_bytes, keys, k2.p, vals, v2.p, static_cast<int>(n), 0,
                                            end_bit, s));
    d2d(keys, k2.p, n * sizeof(K), s);
    d2d(vals, v2.p, n * sizeof(uint32_t), s);
    stream_sync(s);
}

void sort_pairs_u64(uint64_t* keys, uint32_t* vals, size_t n, int end_bit, cudaStream_t s) {
    cub_sort_pairs(keys, vals, n, end_bit, s);
}
void sort_pairs_u32(uint32_t* keys, uint32_t* vals, size_t n, int end_bit, cudaStream_t s) {
    cub_sort_pairs(keys, vals, n, end_bit, s);
}

size_t select_flagged(const uint8_t* flags, uint32_t* out, size_t n, cudaStream_t s) {
    if (n == 0) return 0;
    if (n > 0x7FFFFFFFull) fail(-1, "select: more than 2^31 items");
    count_launch();
    DevBuf<int> d_count;
    d_count.alloc(1);
    cub::CountingInputIterator<uint32_t> iota(0);
    size_t temp_bytes = 0;
    C5_CUDA(cub::DeviceSelect::Flagged(nullptr, temp_bytes, iota, flags, out, d_count.p, static_cast<int>(n), s));
    DevBuf<uint8_t> temp;
    temp.alloc(temp_bytes ? temp_bytes : 1);
    C5_CUDA(cub::DeviceSelect::Flagged(temp.p, temp_bytes, iota, flags, out, d_count.p, static_cast<int>(n), s));
    int count = 0;
    d2h(&count, d_count.p, sizeof(int), s);
    stream_sync(s);
    return static_cast<size_t>(count);
}

#endif

} // namespace c5
