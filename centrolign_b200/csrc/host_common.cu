// host_common.cu -- the host plumbing every entry family of the C ABI uses (host_common.cuh), and the library-wide
// entry points: clb_last_error, clb_device_count, clb_warm_up, clb_release_cached_memory.
#include <new>

#include "host_common.cuh"

namespace {
thread_local std::string g_err;
}  // namespace

namespace clb {

MemCache g_cache;

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

int cuda_fail(cudaError_t e, const char* expr) {
    return fail(e == cudaErrorMemoryAllocation ? CLB_ENOMEM : CLB_ECUDA, std::string(expr) + ": " + cudaGetErrorString(e));
}

int check_graph_batch(const clb_graph_batch* g, int64_t n_windows) {
    if (!g || !g->node_off || !g->edge_off || !g->pred_off || !g->src_off || !g->snk_off) return CLB_EINVAL;
    if (n_windows > 0) {  // the payload arrays may only be null when they are empty
        if (g->node_off[n_windows] > 0 && !g->label) return CLB_EINVAL;
        if (g->edge_off[n_windows] > 0 && !g->pred) return CLB_EINVAL;
        if (g->src_off[n_windows] > 0 && !g->src) return CLB_EINVAL;
        if (g->snk_off[n_windows] > 0 && !g->snk) return CLB_EINVAL;
    }
    return CLB_OK;
}

int graph_window(const clb_graph_batch& g, int64_t w, GraphWindow& out) {
    const int64_t n0 = g.node_off[w];
    const uint32_t n = (uint32_t)(g.node_off[w + 1] - n0);
    out.n = n;
    out.n_edge = (uint32_t)(g.edge_off[w + 1] - g.edge_off[w]);
    out.n_src = (uint32_t)(g.src_off[w + 1] - g.src_off[w]);
    out.n_snk = (uint32_t)(g.snk_off[w + 1] - g.snk_off[w]);
    out.off = g.pred_off + n0 + w;
    out.ids = g.pred + g.edge_off[w];
    out.src = g.src + g.src_off[w];
    out.snk = g.snk + g.snk_off[w];
    out.label = g.label + n0;
    if (out.off[0] != 0 || out.off[n] != out.n_edge) return CLB_EINVAL;
    for (uint32_t v = 0; v < n; ++v)
        if (out.off[v + 1] < out.off[v]) return CLB_EINVAL;
    for (uint32_t k = 0; k < out.n_edge; ++k)
        if (out.ids[k] >= n) return CLB_EINVAL;
    for (uint32_t k = 0; k < out.n_src; ++k)
        if (out.src[k] >= n) return CLB_EINVAL;
    for (uint32_t k = 0; k < out.n_snk; ++k)
        if (out.snk[k] >= n) return CLB_EINVAL;
    return CLB_OK;
}

int require_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return fail(CLB_ECUDA, "no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(CLB_EINVAL, "device index out of range");
    return CLB_OK;
}

}  // namespace clb

// Context creation off the critical path: a process that knows it will use `device` calls this first thing; the CUDA
// runtime serialises initialisation itself, so later calls of the library simply find the context there (or wait for it).
namespace {
std::mutex g_warm_mu;
std::thread* g_warm_thread = nullptr;
void join_warm_up() {
    std::thread* t = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_warm_mu);
        t = g_warm_thread;
        g_warm_thread = nullptr;
    }
    if (t) {
        t->join();
        delete t;
    }
}
}  // namespace

extern "C" {

const char* clb_last_error(void) { return g_err.c_str(); }

int clb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

void clb_warm_up(int device) {
    std::lock_guard<std::mutex> lk(g_warm_mu);
    static bool started = false;
    if (started) return;
    started = true;
    g_warm_thread = new (std::nothrow) std::thread([device] {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
            cudaGetLastError();
            return;  // no device: the first real call reports it
        }
        if (cudaSetDevice(device) == cudaSuccess) cudaFree(nullptr);
        cudaGetLastError();
    });
    if (g_warm_thread) atexit(join_warm_up);
}

void clb_release_cached_memory(void) {
    clb::g_cache.trim();
    clb::chain_release_cache();
}

}  // extern "C"
