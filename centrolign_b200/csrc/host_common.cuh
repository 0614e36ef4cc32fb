// host_common.cuh -- what the host files of the library share: the error string behind clb_last_error(), the cache of
// pinned-host and device blocks, staged buffers drawn from it, the checks of a graph batch and of the device index, the
// worker pool over windows and the CLB_COUNT_CALLS counters.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "centrolign_b200.h"

namespace clb {

// Sets this thread's clb_last_error() message and returns `code`.
int fail(int code, const std::string& msg);
// A failed CUDA call: CLB_ENOMEM for an allocation failure, CLB_ECUDA otherwise, message "<expr>: <CUDA's error string>".
int cuda_fail(cudaError_t e, const char* expr);

}  // namespace clb

// Returns the code of a failed CUDA call, or (CUDA_TRY_CLEANUP) stores it in `rc` and jumps to `cleanup`.
#define CUDA_TRY(expr)                                                    \
    do {                                                                  \
        const cudaError_t e_ = (expr);                                    \
        if (e_ != cudaSuccess) return clb::cuda_fail(e_, #expr);          \
    } while (0)
#define CUDA_TRY_CLEANUP(expr)                                            \
    do {                                                                  \
        const cudaError_t e_ = (expr);                                    \
        if (e_ != cudaSuccess) {                                          \
            rc = clb::cuda_fail(e_, #expr);                               \
            goto cleanup;                                                 \
        }                                                                 \
    } while (0)

namespace clb {

// Process-wide cache of pinned-host and device blocks.  cudaHostAlloc / cudaFreeHost of the
// multi-GB staging buffers cost seconds per call; a Stitcher calls the batch entry point once per
// guide-tree node, so blocks are kept and reused (best fit) until clb_release_cached_memory().
class MemCache {
public:
    void* host_alloc(size_t bytes, size_t* cap) {
        bytes = round_up(bytes);
        {
            std::lock_guard<std::mutex> lk(mu_);
            auto it = host_.lower_bound(bytes);
            if (it != host_.end() && it->first <= 2 * bytes + (size_t(1) << 20)) {
                void* p = it->second;
                *cap = it->first;
                host_.erase(it);
                return p;
            }
        }
        void* p = nullptr;
        if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            trim();
            if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        }
        *cap = bytes;
        return p;
    }
    void host_release(void* p, size_t cap) {
        std::lock_guard<std::mutex> lk(mu_);
        host_.emplace(cap, p);
    }
    void* dev_alloc(int device, size_t bytes, size_t* cap, bool any_larger) {
        bytes = round_up(bytes);
        {
            std::lock_guard<std::mutex> lk(mu_);
            auto& m = dev_[device];
            auto it = m.lower_bound(bytes);
            if (it != m.end() && (any_larger || it->first <= 2 * bytes + (size_t(1) << 20))) {
                void* p = it->second;
                *cap = it->first;
                m.erase(it);
                return p;
            }
        }
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) {
            cudaGetLastError();
            trim();
            if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        }
        *cap = bytes;
        return p;
    }
    void dev_release(int device, void* p, size_t cap) {
        std::lock_guard<std::mutex> lk(mu_);
        dev_[device].emplace(cap, p);
    }
    size_t dev_cached(int device) {
        std::lock_guard<std::mutex> lk(mu_);
        size_t t = 0;
        for (auto& kv : dev_[device]) t += kv.first;
        return t;
    }
    void trim() {
        std::lock_guard<std::mutex> lk(mu_);
        for (auto& kv : host_) cudaFreeHost(kv.second);
        host_.clear();
        int cur = 0;
        cudaGetDevice(&cur);
        for (auto& d : dev_) {
            cudaSetDevice(d.first);
            for (auto& kv : d.second) cudaFree(kv.second);
            d.second.clear();
        }
        cudaSetDevice(cur);
    }

private:
    static size_t round_up(size_t b) { return (std::max<size_t>(b, 1) + 4095) & ~size_t(4095); }
    std::mutex mu_;
    std::multimap<size_t, void*> host_;
    std::map<int, std::multimap<size_t, void*>> dev_;
};
extern MemCache g_cache;

// n elements in an optional pinned host block and a device twin, both drawn from g_cache and given back to it on
// destruction.  The alloc functions return CLB_OK or CLB_ENOMEM.
template <class T>
struct Staged {
    T* h = nullptr;
    T* d = nullptr;
    size_t n = 0, cap_h = 0, cap_d = 0;
    int dev = 0;
    Staged() = default;
    Staged(const Staged&) = delete;
    Staged& operator=(const Staged&) = delete;
    ~Staged() { release(); }
    int alloc_host(size_t count) {
        n = count;
        h = (T*)g_cache.host_alloc(n * sizeof(T), &cap_h);
        return h ? CLB_OK : CLB_ENOMEM;
    }
    // any_larger: any cached block of at least n elements will do (otherwise only one of at most about twice that size)
    int alloc_dev(int device, bool any_larger = false) {
        dev = device;
        d = (T*)g_cache.dev_alloc(device, n * sizeof(T), &cap_d, any_larger);
        return d ? CLB_OK : CLB_ENOMEM;
    }
    int alloc(int device, size_t count, bool host, bool any_larger = false) {
        n = count;
        if (host && alloc_host(count) != CLB_OK) return CLB_ENOMEM;
        return alloc_dev(device, any_larger);
    }
    size_t bytes() const { return n * sizeof(T); }
    void release() {
        if (h) g_cache.host_release(h, cap_h);
        if (d) g_cache.dev_release(dev, d, cap_d);
        h = d = nullptr;
    }
};

// CLB_EINVAL if `g` or one of its offset arrays is null, or, for n_windows > 0, a payload array that is not empty.
int check_graph_batch(const clb_graph_batch* g, int64_t n_windows = -1);

// Window w of a graph batch.  `off` / `ids` are the predecessor lists of a clb_graph_batch or the successor lists of a
// clb_succ_graph_batch.
struct GraphWindow {
    uint32_t n, n_edge, n_src, n_snk;
    const uint32_t* off;  // [n + 1]
    const uint32_t* ids;  // [n_edge]
    const uint32_t* src;  // [n_src]
    const uint32_t* snk;  // [n_snk]
    const uint8_t* label; // [n]
};
// Slices window w out of g: CLB_EINVAL unless the offsets rise from 0 to n_edge and every id, source and sink is a node
// of the window.
int graph_window(const clb_graph_batch& g, int64_t w, GraphWindow& out);

// CLB_ECUDA without a CUDA device (there is no CPU fallback), CLB_EINVAL for a device index out of range.
int require_device(int device);

// Frees the arenas the chaining calls keep per device (chain_host.cu; clb_release_cached_memory).
void chain_release_cache();

// Host threads of a pool over n windows: one below serial_below windows, else up to 32.
inline unsigned pool_threads(int64_t n, int64_t serial_below) {
    return n < serial_below ? 1u : std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
}

// fn(thread, w) -> CLB code for every window w of [0, n), on pool_threads(n, serial_below) threads (the calling thread is
// thread 0) that take `grain` windows at a time.  Stops at the first failure: returns its code and the window in *bad.
template <class Fn>
int for_each_window(int64_t n, int64_t grain, int64_t serial_below, const Fn& fn, int64_t* bad = nullptr) {
    std::atomic<int64_t> next(0), bad_w(-1);
    std::atomic<int> status(CLB_OK);
    auto worker = [&](unsigned t) {
        for (;;) {
            const int64_t w0 = next.fetch_add(grain);
            if (w0 >= n || status.load() != CLB_OK) return;
            for (int64_t w = w0; w < std::min(n, w0 + grain); ++w) {
                const int r = fn(t, w);
                if (r != CLB_OK) {
                    int ok = CLB_OK;
                    if (status.compare_exchange_strong(ok, r)) bad_w.store(w);
                    return;
                }
            }
        }
    };
    const unsigned nthreads = pool_threads(n, serial_below);
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nthreads; ++t) pool.emplace_back(worker, t);
    worker(0);
    for (auto& t : pool) t.join();
    if (bad) *bad = bad_w.load();
    return status.load();
}

// CLB_EINVAL unless devices[] lists n_devices >= 1 ordinals, none twice.  `who` starts the message.
int check_devices(int n_devices, const int* devices, const char* who);

// The scaffolding of the _multi entry points.  Deals n_items independent items to the devices with clb_balanced_partition
// on cost[] (the part index per item goes to part_out if it is not null), then runs run(k, sel) -> CLB code on one host
// thread per device that got items, where sel lists the items of devices[k] in ascending order.  Returns the first failure
// in device order, its message prefixed with "device <ordinal>: ".
template <class Fn>
int deal_to_devices(int n_devices, const int* devices, int32_t n_items, const int64_t* cost, int32_t* part_out, const Fn& run) {
    std::vector<int32_t> part(n_items);
    const int rc = clb_balanced_partition(n_items, cost, n_devices, part.data());
    if (rc != CLB_OK) return rc;
    if (part_out) std::copy(part.begin(), part.end(), part_out);
    std::vector<std::vector<int32_t>> sel(n_devices);
    for (int32_t w = 0; w < n_items; ++w) sel[part[w]].push_back(w);
    // each thread has its own CUDA context binding and error string; the error strings are handed to the caller's thread
    std::vector<int> rcs(n_devices, CLB_OK);
    std::vector<std::string> errs(n_devices);
    std::vector<std::thread> pool;
    for (int k = 0; k < n_devices; ++k)
        if (!sel[k].empty())
            pool.emplace_back([&, k] {
                rcs[k] = run(k, sel[k]);
                if (rcs[k] != CLB_OK) errs[k] = clb_last_error();
            });
    for (auto& t : pool) t.join();
    for (int k = 0; k < n_devices; ++k)
        if (rcs[k] != CLB_OK) return fail(rcs[k], "device " + std::to_string(devices[k]) + ": " + errs[k]);
    return CLB_OK;
}

// CLB_COUNT_CALLS: evidence for integration tests that the GPU path really ran.  Counts the calls of an entry point and
// their windows, and prints "<kPrefix>calls C windows W" at exit.
template <const char* kPrefix>
void count_call(int64_t n_windows) {
    if (!getenv("CLB_COUNT_CALLS")) return;
    static std::atomic<int64_t> calls(0), windows(0);
    static std::once_flag once;
    std::call_once(once, [] {
        atexit([] { fprintf(stderr, "%scalls %lld windows %lld\n", kPrefix, (long long)calls.load(), (long long)windows.load()); });
    });
    calls += 1;
    windows += n_windows;
}

}  // namespace clb
