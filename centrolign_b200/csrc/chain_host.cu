// chain_host.cu -- host side of clb_chain_dp (include/centrolign_b200.h): lays out the reference's search
// structures for the device (shapes only -- see chain_device.cuh; large problems are laid out by the device itself,
// chain_layout_kernels.cu), runs the DP kernel, and performs the reference's traceback (Anchorer::traceback_sparse_dp, include/centrolign/anchorer.hpp:2473-2547).
//
// Shapes reproduced here:
//   * MaxSearchTree: implicit binary heap 0..n-1 filled with the sorted keys by an in-order walk
//     (max_search_tree.hpp:108-150); one per (p1, p2, shift) for the gap-free trees, keys (offset, match)
//     (anchorer.hpp:2143-2215);
//   * OrthogonalMaxSearchTree: the same heap over keys ((shift, match), offset), and for every node outside
//     the two outer spines a cross structure over the node's subtree ordered by offset, ties in the outer
//     key order (stable sort on key 2 only, orthogonal_max_search_tree.hpp:175-239, max_search_tree.hpp:100-106).
// There is no CPU fallback: without a CUDA device the call fails.
#include <chrono>
#include <cstring>
#include <limits>
#include <numeric>

#include "chain_device.cuh"
#include "host_common.cuh"

namespace clb {
cudaError_t launch_chain(ChainArgs args, int grid, int* cluster, int prepare_grid, cudaStream_t stream, cudaEvent_t after_prepare);
cudaError_t launch_chain_small_batch(const ChainArgs* d_args, int n, int smem_bytes, bool any_global, cudaStream_t stream);
int chain_max_grid(int device);
cudaError_t chain_layout_scratch_bytes(const ChainLayoutDims& d, size_t* bytes);
cudaError_t chain_layout_sort(const ChainLayoutIn& in, const ChainLayoutDims& d, char* scratch, cudaStream_t st, int64_t* n_groups, int64_t* h2d_bytes);
cudaError_t chain_layout_build(const ChainLayoutDims& d, int64_t G, char* scratch, const ChainLayoutOut& o, cudaStream_t st, int64_t* n_inner);
}  // namespace clb

using clb::fail;

namespace {

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// heap index of every in-order position of an n-node implicit heap (max_search_tree.hpp:119-150); the device layout
// places its entries with the same function
void inorder_layout(uint32_t n, std::vector<uint32_t>& heap_of_pos) {
    heap_of_pos.resize(n);
    for (uint32_t k = 0; k < n; ++k) heap_of_pos[k] = clb::heap_of_inorder(k, n);
}

// Σ over x < n of the bit length of x
int64_t bitlen_prefix(int64_t n) {
    int64_t s = 0;
    for (int b = 1; b <= 33 && (int64_t(1) << (b - 1)) < n; ++b) s += n - (int64_t(1) << (b - 1));
    return s;
}
// inner-list slots of an n-node orthogonal tree, Σ heap_nanc over its nodes, level by level in closed form: on level d,
// position t has heap_nanc = min(bit length of t, bit length of 2^d - 1 - t)
int64_t inner_slots(int64_t n) {
    int64_t s = 0;
    for (int d = 2; n >= 2 && d <= clb::heap_depth((uint32_t)(n - 1)); ++d) {
        const int64_t full = int64_t(1) << d, half = full / 2;
        const int64_t c = std::min(full, n - (full - 1));  // nodes on level d
        s += bitlen_prefix(std::min(c, half));
        if (c > half) s += bitlen_prefix(half) - bitlen_prefix(full - c);
    }
    return s;
}

// All device data of one call lives in one arena: [copied segments][zero-filled segments].  The arena, its pinned
// staging twin, the stream and the events are kept per device across calls (the Anchorer's fill-in pass makes
// thousands of small chaining calls per alignment), up to kArenaKeep bytes.
struct DeviceArena {
    char* d = nullptr;
    size_t cap = 0;
    char* h = nullptr;  // pinned
    size_t hcap = 0;
    char* ls = nullptr;  // scratch of the device layout, kept and released with the arena
    size_t ls_cap = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evp = nullptr;
};
constexpr size_t kArenaKeep = size_t(1) << 30;
constexpr size_t kDirectCopyBytes = size_t(32) << 20;  // copy regions above this size go to the device without a pinned staging twin
constexpr size_t kChainBatchArena = size_t(4) << 20;  // a problem up to this arena size joins a batched launch (one CTA per problem)
constexpr int kChainClusterMax = 16;  // CTAs of the cluster a mid-sized problem runs in (non-portable size; launch_chain halves it if refused)

// State kept per device ordinal, each behind its own mutex: calls on one device are serialised, calls on different devices
// are not.  A slot is made on first use and never erased, so a reference to it stays valid while others are added.
template <class T>
class PerDevice {
public:
    struct Slot {
        std::mutex mu;
        T state;
    };
    Slot& at(int device) {
        std::lock_guard<std::mutex> lk(mu_);
        return slots_[device];
    }
    // fn(device, state) for every slot, each under its own lock
    template <class Fn>
    void for_each(const Fn& fn) {
        std::lock_guard<std::mutex> lk(mu_);
        for (auto& kv : slots_) {
            std::lock_guard<std::mutex> ls(kv.second.mu);
            fn(kv.first, kv.second.state);
        }
    }

private:
    std::mutex mu_;
    std::map<int, Slot> slots_;
};
PerDevice<DeviceArena> g_arenas;

cudaError_t ensure_stream(DeviceArena& ar) {  // on the current device
    if (ar.stream) return cudaSuccess;
    cudaError_t e = cudaStreamCreateWithFlags(&ar.stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&ar.ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&ar.ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&ar.evp);
    return e;
}

// Which side lays out a problem that runs on its own.  Auto: the device from kDeviceLayoutMinEntries tree entries on, if its
// scratch fits in free device memory.  CLB_CHAIN_LAYOUT=host|device forces a side (A/B runs, tests); check builds both and
// compares the copy regions byte for byte.  Problems the batched launch takes always keep the host layout.
enum class LayoutSide { Auto, Host, Device, Check };
LayoutSide layout_side_knob() {
    const char* v = getenv("CLB_CHAIN_LAYOUT");
    if (!v) return LayoutSide::Auto;
    if (!strcmp(v, "host")) return LayoutSide::Host;
    if (!strcmp(v, "device")) return LayoutSide::Device;
    if (!strcmp(v, "check")) return LayoutSide::Check;
    return LayoutSide::Auto;
}
// tools/chain_layout_bench.py on a B200 (profiles/r03_chain_layout.json, DESIGN.md section 10): the device layout is the faster
// one at every size measured, 10^4 tree entries up; below that a call is dominated by its launches either way
constexpr int64_t kDeviceLayoutMinEntries = 10000;

// fn(begin, end) over [0, n) on up to 16 host threads (the layout of a million-match problem is tens of millions of
// small steps; the Anchorer calls us from one thread)
template <class Fn>
void parallel_for(int64_t n, int64_t min_per_thread, const Fn& fn) {
    const int64_t hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    const int64_t nt = std::max<int64_t>(1, std::min<int64_t>(hw, n / std::max<int64_t>(1, min_per_thread)));
    if (nt <= 1) {
        fn((int64_t)0, n);
        return;
    }
    std::vector<std::thread> th;
    for (int64_t t = 1; t < nt; ++t) th.emplace_back([&, t] { fn(n * t / nt, n * (t + 1) / nt); });
    fn((int64_t)0, n / nt);
    for (auto& x : th) x.join();
}

struct SortKey {
    uint64_t hi, lo;
    uint32_t e;
    bool operator<(const SortKey& o) const { return hi != o.hi ? hi < o.hi : lo < o.lo; }
};
// sorts `keys` on the host threads: sorted chunks, then pairwise merges
void parallel_sort(std::vector<SortKey>& keys) {
    const int64_t n = (int64_t)keys.size();
    const int64_t hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    int64_t nt = 1;
    while (nt * 2 <= hw && n / (nt * 2) >= 65536) nt *= 2;
    if (nt == 1) {
        std::sort(keys.begin(), keys.end());
        return;
    }
    parallel_for(nt, 1, [&](int64_t a, int64_t b) {
        for (int64_t t = a; t < b; ++t) std::sort(keys.begin() + n * t / nt, keys.begin() + n * (t + 1) / nt);
    });
    std::vector<SortKey> tmp(keys.size());
    for (int64_t w = 1; w < nt; w *= 2) {
        parallel_for(nt / (2 * w), 1, [&](int64_t a, int64_t b) {
            for (int64_t g = a; g < b; ++g) {
                const int64_t lo = n * (g * 2 * w) / nt, mid = n * (g * 2 * w + w) / nt, hi = n * (g * 2 * w + 2 * w) / nt;
                std::merge(keys.begin() + lo, keys.begin() + mid, keys.begin() + mid, keys.begin() + hi, tmp.begin() + lo);
            }
        });
        keys.swap(tmp);
    }
}

struct ArenaPlan {
    struct Seg {
        size_t off, bytes;
        const void* src;
    };
    std::vector<Seg> segs;
    size_t copy_bytes = 0, zero_bytes = 0;
    static size_t align(size_t x) { return (x + 255) & ~size_t(255); }
    template <class T>
    size_t copy(const std::vector<T>& v) { return copy(v.data(), v.size() * sizeof(T)); }
    size_t copy(const void* src, size_t bytes) {
        const size_t off = copy_bytes;
        segs.push_back(Seg{off, bytes, src});
        copy_bytes = align(copy_bytes + std::max<size_t>(bytes, 1));
        return off;
    }
    size_t zero(size_t bytes) {  // offset relative to the start of the zero region
        const size_t off = zero_bytes;
        zero_bytes = align(zero_bytes + std::max<size_t>(bytes, 1));
        return off;
    }
};

// The arrays of the copy region, in arena order.  The raw ones are the caller's arrays as they are; the others are laid
// out by the host (chain_host.cu) or by the device (chain_layout_kernels.cu).
enum CopySeg {
    kSegDp, kSegBp, kSegSins, kSegIns, kSegQoff, kSegQm, kSegW, kSegQc1, kSegQa1, kSegQa2, kSegQo, kSegPg, kSegGs, kSegGb, kSegGn, kSegPb,
    kSegGk, kSegGm, kSegOs, kSegOo, kSegOm, kSegIb, kSegIn, kSegIo, kSegEr, kSegs
};
constexpr const char* kSegName[kSegs] = {"dp_init", "bp0", "sins_live", "ins", "qry_live", "qry_match", "weight", "qry_chain1", "qa1",
                                         "qa2", "qoff", "pair_grp_off", "grp_shift", "grp_base", "grp_n", "pair_base", "gf_key", "gf_match",
                                         "or_shift", "or_off", "or_match", "in_base", "in_n", "in_off", "ent_rank"};
constexpr size_t kSegElem[kSegs] = {4, 4, 8, sizeof(clb::InsRec), 8, 4, 4, 4, 4, 4, 4, 8, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4, 4};
bool seg_is_raw(int k) { return k == kSegDp || (k >= kSegQm && k <= kSegQo); }

// The sizes a layout needs, known before any table exists
struct LayoutCounts {
    int64_t M = 0, n_qry = 0, S_live = 0, n_ins = 0, npair = 0, G = 0, E = 0, n_inner = 0, max_q = 0;
    int C1 = 0, C2 = 0, P = 0;
    uint32_t max_n = 0;  // largest orthogonal tree (largest pair), 0 without entries
    int64_t pairs_used = 0;  // pairs with entries: the fewest gap-free trees there can be
    int64_t seg_count(int k) const {
        const int64_t Eo = P > 0 ? E : 0;
        switch (k) {
            case kSegDp: case kSegBp: case kSegW: return M;
            case kSegSins: case kSegQoff: return S_live + 1;
            case kSegIns: return n_ins;
            case kSegQm: case kSegQc1: return n_qry;
            case kSegQa1: return M * C1;
            case kSegQa2: case kSegQo: return M * C2;
            case kSegPg: case kSegPb: return npair + 1;
            case kSegGs: case kSegGb: case kSegGn: return G;
            case kSegGk: case kSegGm: return E;
            case kSegIo: case kSegEr: return n_inner;
            default: return Eo;  // or_*, in_base, in_n
        }
    }
};

// A laid-out problem: the scalar kernel arguments, and where its arrays sit in the copy region (o) and in the zero
// region (z_*) of its arena.
struct ChainLayout {
    clb::ChainArgs scalars{};  // every pointer null: bind() sets them
    size_t copy_bytes = 0, zero_bytes = 0;
    size_t arena_bytes() const { return copy_bytes + zero_bytes; }
    size_t o[kSegs];
    size_t z_qrec, z_gford, z_gfbest, z_orord, z_bit, z_cbest, z_cbp, z_cnt, z_ranks;
};

// the copy region (sources: src[k], null where the device builds the array) and the zero region of a problem of size c
void plan_layout(const LayoutCounts& c, const void* const* src, ChainLayout& L, ArenaPlan& plan) {
    for (int k = 0; k < kSegs; ++k) L.o[k] = plan.copy(src ? src[k] : nullptr, (size_t)c.seg_count(k) * kSegElem[k]);
    const int64_t T = 2 * c.P, E = c.E;
    L.z_qrec = plan.zero((size_t)c.n_qry * c.C2 * sizeof(clb::QueryRec));
    L.z_gford = plan.zero((size_t)E * 4); L.z_gfbest = plan.zero((size_t)E * 8);
    L.z_orord = plan.zero((size_t)T * E * 4); L.z_bit = plan.zero((size_t)T * c.n_inner * 8);
    L.z_cbest = plan.zero((size_t)c.M * 16); L.z_cbp = plan.zero((size_t)(c.max_q * c.C2 * (T + 1)) * 4 * 2); L.z_cnt = plan.zero(8);
}

// The kernel arguments of a laid-out problem whose copy region is at device address c and zero region at z.  The only
// code that knows which array lives in which region.  arena_bytes covers both regions, copy_bytes the copy region.
clb::ChainArgs bind(const ChainLayout& L, char* c, char* z) {
    clb::ChainArgs a = L.scalars;
    const size_t* o = L.o;
    a.dp = (float*)(c + o[kSegDp]); a.backptr = (uint32_t*)(c + o[kSegBp]);
    a.sins_off = (const int64_t*)(c + o[kSegSins]); a.ins = (const clb::InsRec*)(c + o[kSegIns]);
    a.qry_off = (const int64_t*)(c + o[kSegQoff]); a.qry_match = (const uint32_t*)(c + o[kSegQm]);
    a.weight = (const float*)(c + o[kSegW]); a.qry_chain1 = (const uint32_t*)(c + o[kSegQc1]);
    a.qa1 = (const int32_t*)(c + o[kSegQa1]); a.qa2 = (const int32_t*)(c + o[kSegQa2]); a.qoff = (const uint32_t*)(c + o[kSegQo]);
    a.pair_grp_off = (const int64_t*)(c + o[kSegPg]); a.grp_shift = (const int32_t*)(c + o[kSegGs]);
    a.grp_base = (const uint32_t*)(c + o[kSegGb]); a.grp_n = (const uint32_t*)(c + o[kSegGn]); a.pair_base = (const uint32_t*)(c + o[kSegPb]);
    a.gf_key = (const uint32_t*)(c + o[kSegGk]); a.gf_match = (const uint32_t*)(c + o[kSegGm]);
    a.or_shift = (const int32_t*)(c + o[kSegOs]); a.or_off = (const uint32_t*)(c + o[kSegOo]); a.or_match = (const uint32_t*)(c + o[kSegOm]);
    a.in_base = (const uint32_t*)(c + o[kSegIb]); a.in_n = (const uint32_t*)(c + o[kSegIn]); a.in_off = (const uint32_t*)(c + o[kSegIo]);
    a.ent_rank = (const uint32_t*)(c + o[kSegEr]);
    a.qrec = (clb::QueryRec*)(z + L.z_qrec);
    a.gf_ord = (uint32_t*)(z + L.z_gford); a.gf_best = (unsigned long long*)(z + L.z_gfbest);
    a.or_ord = (uint32_t*)(z + L.z_orord); a.bit = (unsigned long long*)(z + L.z_bit);
    a.rank_pool = a.rank_stride ? (uint32_t*)(z + L.z_ranks) : nullptr;
    a.cand_best = (unsigned long long*)(z + L.z_cbest); a.cand_bp = (uint32_t*)(z + L.z_cbp); a.counters = (unsigned long long*)(z + L.z_cnt);
    a.arena_base = c;
    a.arena_bytes = (int64_t)L.arena_bytes();
    a.copy_bytes = (int64_t)L.copy_bytes;
    return a;
}

// A batch of small problems being collected by clb_chain_dp_batch: every problem whose arena fits shared memory is
// laid out as usual, its copy segments are appended to ONE staging buffer, and its layout is recorded; flush() then needs
// one H2D copy, one launch (a CTA per problem) and one D2H copy for all.
std::atomic<int64_t> g_batch_flushes(0), g_batch_problems(0);  // CLB_COUNT_CALLS: launches of the batched kernel / problems in them
struct DeferredProblem {
    ChainLayout layout;
    size_t arena_off = 0;       // of the problem's copy region in the combined buffer
    size_t res_off = 0;         // of its results (match-count floats / words) in the compact result buffers
    int64_t n_match = 0;
    const clb_chain_problem* p = nullptr;
    float* dp_out = nullptr;
    int64_t* backptr_out = nullptr;
    int64_t* chain_out = nullptr;
    int64_t* chain_len = nullptr;
    float* opt_score = nullptr;
};
struct BatchCtx {
    std::vector<char> staging;  // concatenated copy regions (256-byte aligned)
    std::vector<DeferredProblem> items;
    size_t res_total = 0;
    int max_smem = 0;
};

}  // namespace

// the reference's traceback on the final DP values and back-pointers (anchorer.hpp:2483-2534)
static int chain_traceback(const clb_chain_problem* p, const float* h_dp, const uint32_t* h_bp, float* dp_out, int64_t* backptr_out,
                           int64_t* chain_out, int64_t* chain_len, float* opt_score) {
    const float kLowest = std::numeric_limits<float>::lowest();
    const int64_t M = p->n_match;
    float opt_value = kLowest;
    int64_t opt = -1;
    for (int64_t m = 0; m < M; ++m) {
        float dp_val = h_dp[m];
        const float fin = p->final_term[m];
        if (fin == kLowest) dp_val = fin;
        else dp_val += fin;
        if (dp_val > opt_value && dp_val > p->min_score) {
            opt_value = dp_val;
            opt = m;
        }
    }
    int64_t len = 0;
    for (int64_t here = opt; here >= 0; here = h_bp[here] == 0xffffffffu ? -1 : (int64_t)h_bp[here]) {
        if (len >= M) return fail(CLB_ECUDA, "internal: back-pointer cycle");
        chain_out[len++] = here;
    }
    std::reverse(chain_out, chain_out + len);
    *chain_len = len;
    if (opt_score) *opt_score = opt_value;
    if (dp_out) memcpy(dp_out, h_dp, M * sizeof(float));
    if (backptr_out)
        for (int64_t m = 0; m < M; ++m) backptr_out[m] = h_bp[m] == 0xffffffffu ? -1 : (int64_t)h_bp[m];
    return CLB_OK;
}

// The host layout: every table of the copy region built on up to 16 host threads.  The batched path and every problem
// below the device-layout threshold use it; CLB_CHAIN_LAYOUT=check compares the device layout with it.
struct HostLayout {
    LayoutCounts c;
    std::vector<uint32_t> bp0;
    std::vector<int64_t> sins_live, qry_live, pair_grp_off;
    std::vector<clb::InsRec> ins;
    std::vector<int32_t> grp_shift, or_shift;
    std::vector<uint32_t> grp_base32, grp_n, pair_base32, gf_key, gf_match, or_off, or_match, in_base32, in_n, in_off, ent_rank;
    const void* src[kSegs] = {};
};

static int host_layout(const clb_chain_problem* p, HostLayout& H) {
    const int64_t M = p->n_match, S = p->n_step, E = p->ins_off[M], n_qry = p->qry_off[S];
    const int C1 = p->n_chain1, C2 = p->n_chain2, P = p->num_pw, T = 2 * P;
    const int64_t npair = (int64_t)C1 * C2;
    auto& grp_n = H.grp_n;
    auto& gf_key = H.gf_key;
    auto& gf_match = H.gf_match;
    auto& pair_grp_off = H.pair_grp_off;
    auto& grp_shift = H.grp_shift;
    auto& or_shift = H.or_shift;
    auto& or_off = H.or_off;
    auto& or_match = H.or_match;
    auto& in_n = H.in_n;
    auto& in_off = H.in_off;
    auto& ent_rank = H.ent_rank;
    auto& ins = H.ins;
    std::vector<uint32_t> ent_match(E), ent_pair(E);
    for (int64_t m = 0; m < M; ++m)
        for (int64_t e = p->ins_off[m]; e < p->ins_off[m + 1]; ++e) {
            ent_match[e] = (uint32_t)m;
            ent_pair[e] = p->ins_p1[e] * (uint32_t)C2 + p->ins_p2[e];
        }
    // step -> entries, in the reference's order (anchorer.hpp:2301-2310); positions double as sequence numbers
    std::vector<int64_t> sins_off(S + 1, 0);
    std::vector<uint32_t> sins_entry;
    sins_entry.reserve(E);
    int64_t max_q = 0;
    for (int64_t s = 0; s < S; ++s) {
        for (int64_t k = p->end_off[s]; k < p->end_off[s + 1]; ++k) {
            const uint32_t m = p->end_match[k];
            for (int64_t e = p->ins_off[m]; e < p->ins_off[m + 1]; ++e)
                if (!p->ins_active || p->ins_active[e]) sins_entry.push_back((uint32_t)e);
        }
        sins_off[s + 1] = (int64_t)sins_entry.size();
        max_q = std::max(max_q, p->qry_off[s + 1] - p->qry_off[s]);
    }
    if ((int64_t)sins_entry.size() >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "more than 2^32 insertions");
    if (max_q * C2 * (T + 1) >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "too many queries in one step");

    std::vector<uint32_t> order(E);
    std::iota(order.begin(), order.end(), 0u);
    std::vector<uint32_t> heap_of_pos;

    // gap-free trees: one per (pair, shift), keys (offset, match)
    std::vector<int64_t> grp_base;
    pair_grp_off.assign(npair + 1, 0);
    gf_key.resize(E);
    gf_match.resize(E);
    std::vector<uint32_t> ent_gf_grp(E), ent_gf_node(E);
    std::vector<SortKey> keys(E);
    parallel_for(E, 1 << 16, [&](int64_t a, int64_t b) {  // (pair, shift, offset, match)
        for (int64_t e = a; e < b; ++e)
            keys[e] = SortKey{((uint64_t)ent_pair[e] << 32) | ((uint32_t)p->ins_shift[e] ^ 0x80000000u),
                              ((uint64_t)p->ins_offset[e] << 32) | ent_match[e], (uint32_t)e};
    });
    parallel_sort(keys);
    for (int64_t i = 0; i < E; ++i) order[i] = keys[i].e;
    for (int64_t i = 0; i < E;) {
        int64_t j = i;
        while (j < E && ent_pair[order[j]] == ent_pair[order[i]] && p->ins_shift[order[j]] == p->ins_shift[order[i]]) ++j;
        const uint32_t g = (uint32_t)grp_base.size(), n = (uint32_t)(j - i);
        grp_base.push_back(i);
        grp_shift.push_back(p->ins_shift[order[i]]);
        grp_n.push_back(n);
        pair_grp_off[ent_pair[order[i]] + 1] += 1;
        inorder_layout(n, heap_of_pos);
        for (uint32_t k = 0; k < n; ++k) {
            const uint32_t e = order[i + k], h = heap_of_pos[k];
            gf_key[i + h] = p->ins_offset[e];
            gf_match[i + h] = ent_match[e];
            ent_gf_grp[e] = g;
            ent_gf_node[e] = h;
        }
        i = j;
    }
    for (int64_t pr = 0; pr < npair; ++pr) pair_grp_off[pr + 1] += pair_grp_off[pr];

    // orthogonal trees: one shape per pair, keys ((shift, match), offset)
    std::vector<int64_t> pair_base(npair + 1, 0), in_base, ent_rank_off;
    std::vector<uint32_t> ent_or_node;
    int64_t n_inner = 0;
    if (P > 0) {
        or_shift.resize(E); or_off.resize(E); or_match.resize(E); in_n.assign(E, 0); in_base.assign(E, -1);
        ent_or_node.resize(E); ent_rank_off.assign(E + 1, 0);
        parallel_for(E, 1 << 16, [&](int64_t a, int64_t b) {  // (pair, shift, match)
            for (int64_t e = a; e < b; ++e)
                keys[e] = SortKey{((uint64_t)ent_pair[e] << 32) | ((uint32_t)p->ins_shift[e] ^ 0x80000000u), (uint64_t)ent_match[e], (uint32_t)e};
        });
        parallel_sort(keys);
        for (int64_t i = 0; i < E; ++i) order[i] = keys[i].e;
        for (int64_t e = 0; e < E; ++e) pair_base[ent_pair[e] + 1] += 1;
        for (int64_t pr = 0; pr < npair; ++pr) pair_base[pr + 1] += pair_base[pr];
        std::vector<uint32_t> pos_of_heap, sub_lo, sub_n, nanc;
        std::vector<uint8_t> spine;
        // pass 1: shapes, inner-list sizes and bases
        for (int64_t pr = 0; pr < npair; ++pr) {
            const int64_t ob = pair_base[pr];
            const uint32_t n = (uint32_t)(pair_base[pr + 1] - ob);
            if (!n) continue;
            inorder_layout(n, heap_of_pos);
            for (uint32_t k = 0; k < n; ++k) {
                const uint32_t e = order[ob + k], h = heap_of_pos[k];
                or_shift[ob + h] = p->ins_shift[e];
                or_off[ob + h] = p->ins_offset[e];
                or_match[ob + h] = ent_match[e];
                ent_or_node[e] = h;
            }
            spine.assign(n, 0);  // orthogonal_max_search_tree.hpp:175-182: the two outer spines carry no cross tree
            for (uint64_t c = 0; c < n; c = 2 * c + 1) spine[c] = 1;
            for (uint64_t c = 2; c < n; c = 2 * c + 2) spine[c] = 1;
            sub_n.assign(n, 1);
            for (uint32_t h = n; h-- > 1;) sub_n[(h - 1) / 2] += sub_n[h];
            nanc.assign(n, 0);
            for (uint32_t h = 0; h < n; ++h) {
                nanc[h] = (h ? nanc[(h - 1) / 2] : 0) + (spine[h] ? 0 : 1);
                if (!spine[h]) {
                    in_base[ob + h] = n_inner;
                    in_n[ob + h] = sub_n[h];
                    n_inner += sub_n[h];
                }
            }
            for (uint32_t k = 0; k < n; ++k) ent_rank_off[order[ob + k] + 1] = nanc[heap_of_pos[k]];
        }
        for (int64_t e = 0; e < E; ++e) ent_rank_off[e + 1] += ent_rank_off[e];
        if (ent_rank_off[E] != n_inner) return fail(CLB_ECUDA, "internal: inner list accounting mismatch");
        in_off.resize(n_inner);
        ent_rank.resize(n_inner);
        // pass 2: inner lists by merging children lists, one tree level at a time from the leaves up (the nodes of a
        // level are independent); a list holds outer key-order positions and is stored where the device will read it
        std::vector<uint32_t> in_pos(n_inner);
        for (int64_t pr = 0; pr < npair; ++pr) {
            const int64_t ob = pair_base[pr];
            const uint32_t n = (uint32_t)(pair_base[pr + 1] - ob);
            if (!n) continue;
            inorder_layout(n, heap_of_pos);
            pos_of_heap.resize(n);
            for (uint32_t k = 0; k < n; ++k) pos_of_heap[heap_of_pos[k]] = k;
            auto depth_of = [](uint32_t h) { return 31 - __builtin_clz(h + 1); };  // heap index -> depth
            for (int d = depth_of(n - 1); d >= 0; --d) {
                const int64_t first = (int64_t(1) << d) - 1, last = std::min<int64_t>(n, (int64_t(2) << d) - 1);
                parallel_for(last - first, std::max<int64_t>(1, 65536 / std::max<int64_t>(1, n >> d)), [&](int64_t a0, int64_t b0) {
                    for (int64_t hh = first + a0; hh < first + b0; ++hh) {
                        const uint32_t h = (uint32_t)hh;
                        if (in_base[ob + h] < 0) continue;  // spine: never queried, never built
                        const uint32_t l = 2 * h + 1, r = 2 * h + 2;
                        uint32_t* out = in_pos.data() + in_base[ob + h];
                        const uint32_t* L = l < n ? in_pos.data() + in_base[ob + l] : nullptr;
                        const uint32_t* R = r < n ? in_pos.data() + in_base[ob + r] : nullptr;
                        const uint32_t nl = l < n ? in_n[ob + l] : 0, nr = r < n ? in_n[ob + r] : 0;
                        const uint32_t self = pos_of_heap[h];
                        auto off_of = [&](uint32_t pos) { return or_off[ob + heap_of_pos[pos]]; };
                        // positions of the left subtree < self < positions of the right subtree: ties in offset resolve by side
                        const uint32_t so = off_of(self);
                        uint32_t a = 0, b = 0, k = 0;
                        bool self_done = false;
                        while (a < nl || b < nr || !self_done) {
                            // candidates in position order: L[a] < self < R[b]; pick the smallest (offset, position)
                            int pick = -1;
                            uint32_t bo = 0;
                            if (a < nl) { pick = 0; bo = off_of(L[a]); }
                            if (!self_done && (pick < 0 || so < bo)) { pick = 1; bo = so; }
                            if (b < nr) {
                                const uint32_t ro = off_of(R[b]);
                                if (pick < 0 || ro < bo) pick = 2;
                            }
                            out[k++] = pick == 0 ? L[a++] : (pick == 1 ? self : R[b++]);
                            if (pick == 1) self_done = true;
                        }
                        // offsets of the list entries and the rank of every element in this list
                        const int64_t ib = in_base[ob + h];
                        for (uint32_t kk = 0; kk < k; ++kk) {
                            const uint32_t pos = out[kk], eh = heap_of_pos[pos];
                            in_off[ib + kk] = or_off[ob + eh];
                            ent_rank[ent_rank_off[order[ob + pos]] + (depth_of(eh) - d)] = kk;  // climbing order: the element's own node first
                        }
                    }
                });
            }
        }
    }
    // insertion records in the reference's order, and the remaining per-entry tables in 32-bit form
    if (n_inner >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "search structures exceed 2^32 inner slots");
    if ((int64_t)sins_entry.size() >= (int64_t(1) << 31)) return fail(CLB_EINVAL, "more than 2^31 insertions");
    ins.resize(sins_entry.size());
    for (size_t i = 0; i < sins_entry.size(); ++i) {
        const uint32_t e = sins_entry[i];
        clb::InsRec& r = ins[i];
        r.match = ent_match[e];
        r.gf_base = (uint32_t)grp_base[ent_gf_grp[e]];
        r.gf_node = ent_gf_node[e];
        r.or_base = P > 0 ? (uint32_t)pair_base[ent_pair[e]] : 0;
        r.or_node = P > 0 ? ent_or_node[e] : 0;
        r.shift = p->ins_shift[e];
        r.rank_off = P > 0 ? (uint32_t)ent_rank_off[e] : 0;
        r.n_rank = P > 0 ? (uint32_t)(ent_rank_off[e + 1] - ent_rank_off[e]) : 0;
    }
    H.grp_base32.assign(grp_base.begin(), grp_base.end());
    H.pair_base32.assign(pair_base.begin(), pair_base.end());
    H.in_base32.resize(in_base.size());
    for (size_t k = 0; k < in_base.size(); ++k) H.in_base32[k] = in_base[k] < 0 ? clb::kChainNone : (uint32_t)in_base[k];
    // the device walks only the steps in which something happens (a caller may list every node of graph 1 as a step; the
    // builders of hostcpp/chain_b200.hpp list the nodes with events): the offsets are cumulative, so dropping an empty step
    // drops one equal entry of either list
    H.sins_live.reserve(S + 1); H.qry_live.reserve(S + 1);
    H.sins_live.push_back(sins_off[0]); H.qry_live.push_back(p->qry_off[0]);
    for (int64_t s = 0; s < S; ++s)
        if (sins_off[s + 1] != sins_off[s] || p->qry_off[s + 1] != p->qry_off[s]) {
            H.sins_live.push_back(sins_off[s + 1]);
            H.qry_live.push_back(p->qry_off[s + 1]);
        }
    H.bp0.assign(M, clb::kChainNone);
    LayoutCounts& c = H.c;
    c.M = M; c.n_qry = n_qry; c.S_live = (int64_t)H.sins_live.size() - 1; c.n_ins = (int64_t)ins.size(); c.npair = npair;
    c.G = (int64_t)grp_n.size(); c.E = E; c.n_inner = n_inner; c.max_q = max_q; c.C1 = C1; c.C2 = C2; c.P = P;
    for (int64_t pr = 0; pr < npair; ++pr) c.max_n = std::max<uint32_t>(c.max_n, H.pair_base32[pr + 1] - H.pair_base32[pr]);
    const void* src[kSegs] = {p->dp_init, H.bp0.data(), H.sins_live.data(), ins.data(), H.qry_live.data(), p->qry_match, p->weight,
                              p->qry_chain1, p->qa1, p->qa2, p->qoff, pair_grp_off.data(), grp_shift.data(), H.grp_base32.data(),
                              grp_n.data(), H.pair_base32.data(), gf_key.data(), gf_match.data(), or_shift.data(), or_off.data(),
                              or_match.data(), H.in_base32.data(), in_n.data(), in_off.data(), ent_rank.data()};
    std::copy(src, src + kSegs, H.src);
    (void)T;
    return CLB_OK;
}

// The sizes of the device layout from linear passes over the caller's arrays, with the host layout's checks of them in
// the host layout's order.  No table is built.
static int count_layout(const clb_chain_problem* p, LayoutCounts& c) {
    const int64_t M = p->n_match, S = p->n_step, E = p->ins_off[M];
    const int C1 = p->n_chain1, C2 = p->n_chain2, P = p->num_pw, T = 2 * P;
    const int64_t npair = (int64_t)C1 * C2;
    std::vector<uint32_t> act(M);
    for (int64_t m = 0; m < M; ++m) {
        uint32_t n = 0;
        for (int64_t e = p->ins_off[m]; e < p->ins_off[m + 1]; ++e) n += !p->ins_active || p->ins_active[e];
        act[m] = n;
    }
    int64_t n_ins = 0, S_live = 0, max_q = 0;
    for (int64_t s = 0; s < S; ++s) {
        int64_t here = 0;
        for (int64_t k = p->end_off[s]; k < p->end_off[s + 1]; ++k) here += act[p->end_match[k]];
        n_ins += here;
        S_live += here > 0 || p->qry_off[s + 1] != p->qry_off[s];
        max_q = std::max(max_q, p->qry_off[s + 1] - p->qry_off[s]);
    }
    if (n_ins >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "more than 2^32 insertions");
    if (max_q * C2 * (T + 1) >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "too many queries in one step");
    std::vector<int64_t> hist(npair, 0);
    for (int64_t e = 0; e < E; ++e) hist[p->ins_p1[e] * (int64_t)C2 + p->ins_p2[e]] += 1;
    c = LayoutCounts{};
    for (int64_t pr = 0; pr < npair; ++pr) {
        c.max_n = std::max<uint32_t>(c.max_n, (uint32_t)hist[pr]);
        c.pairs_used += hist[pr] > 0;
        if (P > 0) c.n_inner += inner_slots(hist[pr]);
    }
    if (P == 0) c.max_n = 0;  // as the host layout's: no orthogonal trees
    if (c.n_inner >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "search structures exceed 2^32 inner slots");
    if (n_ins >= (int64_t(1) << 31)) return fail(CLB_EINVAL, "more than 2^31 insertions");
    c.M = M; c.n_qry = p->qry_off[S]; c.S_live = S_live; c.n_ins = n_ins; c.npair = npair; c.E = E; c.max_q = max_q;
    c.C1 = C1; c.C2 = C2; c.P = P;
    return CLB_OK;
}

// whether the device layout's scratch and the problem's arena fit in the device's free memory
static bool device_layout_fits(int device, const LayoutCounts& c, size_t arena_bytes, bool has_active, int64_t n_end, int64_t S) {
    const clb::ChainLayoutDims dims{c.M, S, c.E, n_end, c.npair, c.C2, c.P, 0, has_active};
    size_t scratch = 0, free_b = 0, total_b = 0;
    if (cudaSetDevice(device) != cudaSuccess || clb::chain_layout_scratch_bytes(dims, &scratch) != cudaSuccess) return false;
    return cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && scratch + arena_bytes < free_b;
}

static int chain_dp_impl(int device, const clb_chain_problem* p, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                         int64_t* chain_len, float* opt_score, clb_chain_stats* stats, BatchCtx* ctx);

extern "C" int clb_chain_dp(int device, const clb_chain_problem* p, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                            int64_t* chain_len, float* opt_score, clb_chain_stats* stats) {
    return chain_dp_impl(device, p, dp_out, backptr_out, chain_out, chain_len, opt_score, stats, nullptr);
}

static int chain_dp_impl(int device, const clb_chain_problem* p, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                         int64_t* chain_len, float* opt_score, clb_chain_stats* stats, BatchCtx* ctx) {
    const double t_start = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    struct CallTimer {  // evidence for integration tests that the GPU path really ran, and what it cost
        static std::atomic<int64_t>& us() { static std::atomic<int64_t> v(0); return v; }
        static std::atomic<int64_t>* phase() { static std::atomic<int64_t> v[4]; return v; }  // layout, staging, gpu, traceback
        double t0;
        bool on;
        ~CallTimer() { if (on) us() += (int64_t)((now_ms() - t0) * 1e3); }
    } call_timer{t_start, getenv("CLB_COUNT_CALLS") != nullptr};
    if (call_timer.on && p) {
        static std::atomic<int64_t> calls(0), matches(0);
        static std::once_flag once;
        std::call_once(once, [] {
            atexit([] {
                fprintf(stderr, "[clb] chain calls %lld matches %lld seconds %.3f (layout %.3f, staging %.3f, gpu %.3f, traceback %.3f); "
                                "%lld of them in %lld batched launches\n",
                        (long long)calls.load(), (long long)matches.load(), CallTimer::us().load() * 1e-6,
                        CallTimer::phase()[0].load() * 1e-6, CallTimer::phase()[1].load() * 1e-6, CallTimer::phase()[2].load() * 1e-6,
                        CallTimer::phase()[3].load() * 1e-6, (long long)g_batch_problems.load(), (long long)g_batch_flushes.load());
            });
        });
        calls += 1;
        matches += p->n_match;
    }
    if (!p || !chain_out || !chain_len) return fail(CLB_EINVAL, "null problem or output");
    if (p->num_pw < 0 || p->num_pw > CLB_MAX_PW) return fail(CLB_EINVAL, "num_pw outside 0..3");
    if (p->n_match < 0 || p->n_step < 0 || p->n_chain1 < 0 || p->n_chain2 < 0) return fail(CLB_EINVAL, "negative sizes");
    if (p->n_match > 0 && (p->n_chain1 < 1 || p->n_chain2 < 1)) return fail(CLB_EINVAL, "matches but no chains");
    if (p->n_match >= (int64_t(1) << 31)) return fail(CLB_EINVAL, "more than 2^31 matches");
    if (const char* dump_dir = getenv("CLB_DUMP_DIR")) {  // debugging aid: every problem a caller sends, in the format of oracle/chain_shim.cpp
        static std::atomic<int> seq(0);
        if (p->n_match > 0 && p->ins_off && p->end_off && p->qry_off) {
            const std::string path = std::string(dump_dir) + "/chain_" + std::to_string(seq++) + ".bin";
            if (FILE* f = fopen(path.c_str(), "wb")) {
                const std::string kind = p->num_pw == 0 ? "gapfree" : "affine";
                auto put = [&](const std::string& name, uint32_t code, const void* data, uint64_t n, size_t elem) {
                    const std::string full = kind + "." + name;
                    const uint32_t len = (uint32_t)full.size();
                    fwrite(&len, 4, 1, f); fwrite(full.data(), 1, len, f); fwrite(&code, 4, 1, f); fwrite(&n, 8, 1, f);
                    if (n && data) fwrite(data, elem, n, f);
                };
                const int64_t M_ = p->n_match, S_ = p->n_step, E_ = p->ins_off[M_], NE = p->end_off[S_], NQ = p->qry_off[S_];
                const double prm[11] = {(double)p->num_pw, p->gap_open[0], p->gap_open[1], p->gap_open[2], p->gap_extend[0], p->gap_extend[1],
                                        p->gap_extend[2], p->scale, (double)p->n_chain1, (double)p->n_chain2, 0.0};
                put("params", 4, prm, 11, 8);
                put("min_score", 0, &p->min_score, 1, 4);
                put("expect_chain", 3, nullptr, 0, 8);
                put("weight", 0, p->weight, M_, 4); put("dp_init", 0, p->dp_init, M_, 4); put("final_term", 0, p->final_term, M_, 4);
                put("end_off", 3, p->end_off, S_ + 1, 8); put("end_match", 2, p->end_match, NE, 4);
                put("qry_off", 3, p->qry_off, S_ + 1, 8); put("qry_match", 2, p->qry_match, NQ, 4); put("qry_chain1", 2, p->qry_chain1, NQ, 4);
                put("ins_off", 3, p->ins_off, M_ + 1, 8); put("ins_p1", 2, p->ins_p1, E_, 4); put("ins_p2", 2, p->ins_p2, E_, 4);
                put("ins_shift", 1, p->ins_shift, E_, 4); put("ins_offset", 2, p->ins_offset, E_, 4);
                std::vector<uint32_t> act(E_, 1u);
                if (p->ins_active) for (int64_t e = 0; e < E_; ++e) act[e] = p->ins_active[e];
                put("ins_active", 2, act.data(), E_, 4);
                put("qa1", 1, p->qa1, (uint64_t)M_ * p->n_chain1, 4); put("qa2", 1, p->qa2, (uint64_t)M_ * p->n_chain2, 4);
                put("qoff", 2, p->qoff, (uint64_t)M_ * p->n_chain2, 4);
                fclose(f);
            }
        }
    }
    const bool layout_only = getenv("CLB_CHAIN_LAYOUT_ONLY") != nullptr;  // host-layout timing without a device (no results)
    if (!layout_only)
        if (const int rc = clb::require_device(device)) return rc;
    *chain_len = 0;
    const float kLowest = std::numeric_limits<float>::lowest();
    if (opt_score) *opt_score = kLowest;
    const int64_t M = p->n_match, S = p->n_step;
    if (M == 0) return CLB_OK;
    if (!p->weight || !p->dp_init || !p->final_term || !p->end_off || !p->qry_off || !p->ins_off || !p->qa1 || !p->qa2 || !p->qoff)
        return fail(CLB_EINVAL, "null problem arrays");
    const int C1 = p->n_chain1, C2 = p->n_chain2, P = p->num_pw, T = 2 * P;
    const int64_t npair = (int64_t)C1 * C2;
    const int64_t E = p->ins_off[M];  // tree entries
    if (E < 0 || E >= (int64_t(1) << 32) - 1) return fail(CLB_EINVAL, "entry count out of range");
    const int64_t n_end = p->end_off[S], n_qry = p->qry_off[S];
    for (int64_t k = 0; k < n_end; ++k)
        if (p->end_match[k] >= (uint64_t)M) return fail(CLB_EINVAL, "end_match out of range");
    for (int64_t k = 0; k < n_qry; ++k)
        if (p->qry_match[k] >= (uint64_t)M || p->qry_chain1[k] >= (uint32_t)C1) return fail(CLB_EINVAL, "query out of range");
    for (int64_t e = 0; e < E; ++e)
        if (p->ins_p1[e] >= (uint32_t)C1 || p->ins_p2[e] >= (uint32_t)C2) return fail(CLB_EINVAL, "insert path out of range");

    // ------------------------------------------------------------------ layout ------------------------------------------------------------------
    // The host layout, or, for a problem that runs on its own and has at least kDeviceLayoutMinEntries tree entries, the
    // device layout straight into the arena (chain_layout_kernels.cu).  CLB_CHAIN_LAYOUT=host|device|check overrides the choice.
    const LayoutSide knob = layout_only ? LayoutSide::Host : layout_side_knob();
    LayoutCounts cnt;
    bool on_device = false;
    if (knob != LayoutSide::Host && (knob != LayoutSide::Auto || E >= kDeviceLayoutMinEntries)) {
        if (const int rc = count_layout(p, cnt)) return rc;
        // a problem the batched launch takes keeps the host layout: its copy region is staged with the others'
        ChainLayout L0{};
        ArenaPlan plan0;
        LayoutCounts lower = cnt;  // the arena with the fewest gap-free trees the problem can have
        lower.G = cnt.pairs_used;
        plan_layout(lower, nullptr, L0, plan0);
        const size_t lower_total = plan0.copy_bytes + plan0.zero_bytes;
        on_device = !(ctx && !getenv("CLB_CHAIN_NO_SMALL")) || lower_total > kChainBatchArena;
        if (on_device && knob == LayoutSide::Auto) on_device = device_layout_fits(device, cnt, lower_total, p->ins_active != nullptr, p->end_off[S], S);
    }
    const bool on_host = !on_device || knob == LayoutSide::Check;
    HostLayout H;
    if (on_host) {
        if (const int rc = host_layout(p, H)) return rc;
        if (on_device) {  // check: the linear counts of the device path against the host layout's
            const char* what = cnt.n_ins != H.c.n_ins ? "insertion count" : cnt.S_live != H.c.S_live ? "live step count"
                             : cnt.n_inner != H.c.n_inner ? "inner slot count" : nullptr;
            if (what) return fail(CLB_ECUDA, std::string("CLB_CHAIN_LAYOUT=check: the device layout's ") + what + " differs from the host layout's");
        }
        cnt = H.c;
    }
    double t_built = now_ms();
    if (layout_only) {
        fprintf(stderr, "[clb] chain layout only: %lld matches, %lld entries, %lld inner slots, %.1f ms\n", (long long)M, (long long)E,
                (long long)cnt.n_inner, t_built - t_start);
        return fail(CLB_ECUDA, "CLB_CHAIN_LAYOUT_ONLY: layout timed, nothing computed");
    }
    const char* layout_name = on_device ? (on_host ? "check" : "device") : "host";

    // ------------------------------------------------------------------ device ------------------------------------------------------------------
    int rc = CLB_OK;
    clb::ChainArgs a{};
    std::vector<float> h_dp(M);
    std::vector<uint32_t> h_bp(M);
    int grid = 1;
    auto& arena_slot = g_arenas.at(device);
    std::lock_guard<std::mutex> arena_lock(arena_slot.mu);
    DeviceArena& ar = arena_slot.state;
    bool keep = true;
    {
        ArenaPlan plan;
        ChainLayout L{};
        const int64_t n_inner = cnt.n_inner, max_q = cnt.max_q;
        int64_t h2d = 0;
        double t_staged = 0;
        clb::ChainLayoutDims dims{M, S, E, p->end_off[S], npair, C2, P, cnt.max_n ? clb::heap_depth(cnt.max_n - 1) : 0, p->ins_active != nullptr};
        if (on_device) {  // phase 1: per-entry tables and sorts on the device; its read-back is the number of gap-free trees
            CUDA_TRY_CLEANUP(cudaSetDevice(device));
            CUDA_TRY_CLEANUP(ensure_stream(ar));
            size_t scratch = 0;
            CUDA_TRY_CLEANUP(clb::chain_layout_scratch_bytes(dims, &scratch));
            if (ar.ls_cap < scratch) {
                if (ar.ls) cudaFree(ar.ls);
                ar.ls = nullptr;
                ar.ls_cap = 0;
                CUDA_TRY_CLEANUP(cudaMalloc((void**)&ar.ls, scratch));
                ar.ls_cap = scratch;
            }
            const clb::ChainLayoutIn in{p->ins_off, p->ins_p1, p->ins_p2, p->ins_shift, p->ins_offset, p->ins_active, p->end_off, p->end_match, p->qry_off};
            int64_t G = 0;
            CUDA_TRY_CLEANUP(clb::chain_layout_sort(in, dims, ar.ls, ar.stream, &G, &h2d));
            if (on_host && G != cnt.G) {
                rc = fail(CLB_ECUDA, "CLB_CHAIN_LAYOUT=check: the device layout's gap-free tree count differs from the host layout's");
                goto cleanup;
            }
            cnt.G = G;
        }
        {
            const void* raw[kSegs] = {};  // the device layout copies only the caller's arrays
            raw[kSegDp] = p->dp_init; raw[kSegQm] = p->qry_match; raw[kSegW] = p->weight; raw[kSegQc1] = p->qry_chain1;
            raw[kSegQa1] = p->qa1; raw[kSegQa2] = p->qa2; raw[kSegQo] = p->qoff;
            plan_layout(cnt, on_device ? raw : H.src, L, plan);
        }
        // subtree-block ranks of every orthogonal walk (2 * (depth + 1) blocks at most), if memory allows
        int rank_stride = 0;
        if (P > 0 && n_qry > 0 && !getenv("CLB_CHAIN_NO_RANKS")) {
            const uint32_t max_n = std::max<uint32_t>(1, cnt.max_n);
            rank_stride = 2 * (32 - __builtin_clz(max_n));
            const size_t bytes = (size_t)n_qry * C2 * 2 * rank_stride * 4;
            bool fits = bytes <= (size_t(64) << 20);  // small pools always fit; cudaMemGetInfo costs more than a small problem
            if (!fits) {
                size_t free_b = 0, total_b = 0;
                cudaSetDevice(device);
                fits = cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && bytes < free_b / 4 + (ar.cap > 0 ? ar.cap / 4 : 0);
            }
            if (fits) L.z_ranks = plan.zero(bytes);
            else rank_stride = 0;
        }
        L.copy_bytes = plan.copy_bytes;
        L.zero_bytes = plan.zero_bytes;
        clb::ChainArgs& b = L.scalars;
        b.num_pw = P; b.n_chain1 = C1; b.n_chain2 = C2; b.scale = p->scale;
        for (int k = 0; k < 3; ++k) {
            b.gap_open[k] = p->gap_open[k];
            b.gap_extend[k] = p->gap_extend[k];
            b.scale_ext[k] = p->scale * p->gap_extend[k];  // anchorer.hpp:2330: local_scale * gap_extend[pw / 2] (* shift on the device)
        }
        b.n_match = M; b.n_step = cnt.S_live; b.n_entry = E; b.n_inner = n_inner; b.n_qry = n_qry; b.n_ins = cnt.n_ins;
        b.cand_bp_stride = max_q * C2 * (T + 1);
        b.rank_stride = rank_stride;
        const size_t total = plan.copy_bytes + plan.zero_bytes;
        if (!on_device && ctx && total <= kChainBatchArena && !getenv("CLB_CHAIN_NO_SMALL")) {
            // batched small problem: stage the copy region and keep the layout; flush() binds it to the staged arena
            DeferredProblem d;
            d.arena_off = ctx->staging.size();
            ctx->staging.resize(d.arena_off + plan.copy_bytes);
            for (const auto& sg : plan.segs)
                if (sg.bytes) memcpy(ctx->staging.data() + d.arena_off + sg.off, sg.src, sg.bytes);
            d.layout = L;
            d.res_off = ctx->res_total;
            ctx->res_total += (size_t)M;
            if (total <= (size_t)clb::kChainSmallArena) ctx->max_smem = std::max(ctx->max_smem, (int)((total + 15) / 16 * 16));
            d.n_match = M; d.p = p; d.dp_out = dp_out; d.backptr_out = backptr_out; d.chain_out = chain_out; d.chain_len = chain_len;
            d.opt_score = opt_score;
            ctx->items.push_back(d);
            if (stats) {
                stats->build_ms = t_built - t_start;
                stats->steps = S;
                stats->inserts = cnt.n_ins;
                stats->queries = n_qry * C2;
                stats->tree_bytes = (int64_t)total;
                stats->h2d_bytes = (int64_t)plan.copy_bytes;
                stats->d2h_bytes = M * 8;
            }
            return CLB_OK;
        }
        keep = total <= kArenaKeep;
        CUDA_TRY_CLEANUP(cudaSetDevice(device));
        CUDA_TRY_CLEANUP(ensure_stream(ar));
        if (ar.cap < total) {
            if (ar.d) cudaFree(ar.d);
            ar.d = nullptr;
            ar.cap = 0;
            const size_t want = keep ? std::max(total, std::min(kArenaKeep, 2 * total)) : total;
            CUDA_TRY_CLEANUP(cudaMalloc((void**)&ar.d, want));
            ar.cap = want;
        }
        char* zr = ar.d + plan.copy_bytes;
        if (on_device) {
            // phase 2: the caller's raw arrays go up as they are, every other table is written by the layout kernels
            for (int k = 0; k < kSegs; ++k)
                if (seg_is_raw(k) && plan.segs[k].bytes) {
                    CUDA_TRY_CLEANUP(cudaMemcpyAsync(ar.d + plan.segs[k].off, plan.segs[k].src, plan.segs[k].bytes, cudaMemcpyHostToDevice, ar.stream));
                    h2d += (int64_t)plan.segs[k].bytes;
                }
            CUDA_TRY_CLEANUP(cudaMemsetAsync(ar.d + L.o[kSegBp], 0xff, (size_t)M * 4, ar.stream));  // bp0: kChainNone
            char* c = ar.d;
            const clb::ChainLayoutOut out{(int64_t*)(c + L.o[kSegSins]), (clb::InsRec*)(c + L.o[kSegIns]), (int64_t*)(c + L.o[kSegQoff]),
                                          (int64_t*)(c + L.o[kSegPg]), (int32_t*)(c + L.o[kSegGs]), (uint32_t*)(c + L.o[kSegGb]),
                                          (uint32_t*)(c + L.o[kSegGn]), (uint32_t*)(c + L.o[kSegPb]), (uint32_t*)(c + L.o[kSegGk]),
                                          (uint32_t*)(c + L.o[kSegGm]), (int32_t*)(c + L.o[kSegOs]), (uint32_t*)(c + L.o[kSegOo]),
                                          (uint32_t*)(c + L.o[kSegOm]), (uint32_t*)(c + L.o[kSegIb]), (uint32_t*)(c + L.o[kSegIn]),
                                          (uint32_t*)(c + L.o[kSegIo]), (uint32_t*)(c + L.o[kSegEr])};
            int64_t dev_inner = 0;
            CUDA_TRY_CLEANUP(clb::chain_layout_build(dims, cnt.G, ar.ls, out, ar.stream, &dev_inner));
            if (P > 0 && E > 0 && dev_inner != n_inner) {
                rc = fail(CLB_ECUDA, "internal: inner list accounting mismatch");
                goto cleanup;
            }
            if (on_host) {  // check: the copy region byte for byte against the host layout's
                std::vector<char> got;
                for (int k = 0; k < kSegs && rc == CLB_OK; ++k) {
                    const size_t bytes = plan.segs[k].bytes;
                    if (!bytes) continue;
                    got.resize(bytes);
                    CUDA_TRY_CLEANUP(cudaMemcpy(got.data(), ar.d + plan.segs[k].off, bytes, cudaMemcpyDeviceToHost));
                    const char* want = (const char*)H.src[k];
                    if (memcmp(got.data(), want, bytes) == 0) continue;
                    size_t i = 0;
                    while (got[i] == want[i]) ++i;
                    rc = fail(CLB_ECUDA, std::string("CLB_CHAIN_LAYOUT=check: the device layout differs from the host layout in ") + kSegName[k] + "[" +
                                             std::to_string(i / kSegElem[k]) + "]");
                }
                if (rc != CLB_OK) goto cleanup;
            }
            t_built = t_staged = now_ms();
        } else {
            // A large problem is copied segment by segment straight from the caller's arrays: pinning a staging twin of tens to
            // hundreds of MB costs more (≈ 1 ms per MB) than the driver's own staging of a pageable copy, and a problem of that size
            // comes a few times per alignment.  Small problems -- thousands per alignment -- share one pinned twin that stays.
            const bool direct = plan.copy_bytes > kDirectCopyBytes && ar.hcap < plan.copy_bytes;
            if (!direct && ar.hcap < plan.copy_bytes) {
                if (ar.h) cudaFreeHost(ar.h);
                ar.h = nullptr;
                ar.hcap = 0;
                const size_t want = std::max(plan.copy_bytes, std::min(kDirectCopyBytes, 2 * plan.copy_bytes));
                CUDA_TRY_CLEANUP(cudaHostAlloc((void**)&ar.h, want, cudaHostAllocDefault));
                ar.hcap = want;
            }
            if (!direct)
                for (const auto& sg : plan.segs)
                    if (sg.bytes) memcpy(ar.h + sg.off, sg.src, sg.bytes);
            t_staged = now_ms();
            if (direct) {
                for (const auto& sg : plan.segs)
                    if (sg.bytes) CUDA_TRY_CLEANUP(cudaMemcpyAsync(ar.d + sg.off, sg.src, sg.bytes, cudaMemcpyHostToDevice, ar.stream));
            } else {
                CUDA_TRY_CLEANUP(cudaMemcpyAsync(ar.d, ar.h, plan.copy_bytes, cudaMemcpyHostToDevice, ar.stream));
            }
            h2d = (int64_t)plan.copy_bytes;
        }
        CUDA_TRY_CLEANUP(cudaMemsetAsync(zr, 0, plan.zero_bytes, ar.stream));
        a = bind(L, ar.d, zr);
        a.copy_bytes = (int64_t)total;  // the single-problem path copies the zeroed region too
        // How the phases of a step are separated.  A step has `warps_per_step` independent warp-sized work items on average:
        // a handful run in one CTA (__syncthreads), up to as many as the largest cluster has warps in ONE thread-block cluster
        // (hardware cluster barrier, the items of a step spread over its SMs), more in a cooperative grid over all SMs (grid.sync).
        const int64_t S_live = cnt.S_live;
        const double warps_per_step = S_live ? ((double)cnt.n_ins + (double)n_qry * C2) * (T + 1) / (double)S_live : 0.0;
        const int max_grid = clb::chain_max_grid(device);
        const int warps_per_cta = P == 0 ? 28 : 16;  // chain_kernels.cu: the gap-free kernel runs with 896 threads
        int cluster = 1;
        if (getenv("CLB_CHAIN_GRID")) {
            grid = std::max(1, std::min(max_grid, atoi(getenv("CLB_CHAIN_GRID"))));
        } else if (getenv("CLB_CHAIN_CLUSTER")) {
            cluster = std::max(1, std::min(16, atoi(getenv("CLB_CHAIN_CLUSTER"))));
        } else if (warps_per_step > (double)kChainClusterMax * warps_per_cta) {
            grid = max_grid;  // more items than the largest cluster has warps: measured 335 ms (cluster of 16) -> 232 ms (148 CTAs) at 441 items
        } else if (warps_per_step > 1.5 * warps_per_cta) {
            while (cluster < kChainClusterMax && cluster * warps_per_cta < warps_per_step) cluster *= 2;
        }
        if (total <= (size_t)clb::kChainSmallArena && !getenv("CLB_CHAIN_NO_SMALL") && !getenv("CLB_CHAIN_GRID")) grid = 0;
        const int prepare_grid = (int)std::max<int64_t>(1, std::min<int64_t>((n_qry * C2 + 7) / 8, 8 * (int64_t)max_grid));
        CUDA_TRY_CLEANUP(cudaEventRecord(ar.ev0, ar.stream));
        CUDA_TRY_CLEANUP(clb::launch_chain(a, grid, &cluster, prepare_grid, ar.stream, ar.evp));
        CUDA_TRY_CLEANUP(cudaEventRecord(ar.ev1, ar.stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(h_dp.data(), a.dp, M * sizeof(float), cudaMemcpyDeviceToHost, ar.stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(h_bp.data(), a.backptr, M * sizeof(uint32_t), cudaMemcpyDeviceToHost, ar.stream));
        CUDA_TRY_CLEANUP(cudaStreamSynchronize(ar.stream));
        if (call_timer.on) {
            CallTimer::phase()[0] += (int64_t)((t_built - t_start) * 1e3);
            CallTimer::phase()[1] += (int64_t)((t_staged - t_built) * 1e3);
            CallTimer::phase()[2] += (int64_t)((now_ms() - t_staged) * 1e3);
        }
        float ms = 0.f;
        CUDA_TRY_CLEANUP(cudaEventElapsedTime(&ms, ar.ev0, ar.ev1));
        if (getenv("CLB_TIMING")) {
            float pms = 0.f;
            cudaEventElapsedTime(&pms, ar.ev0, ar.evp);
            fprintf(stderr, "[clb] chain: build %.1f ms (%s layout), alloc+stage %.1f ms (%.0f MB arena, %.0f MB copied), prepare kernel %.2f ms, "
                            "DP kernel %.2f ms, enqueue..sync %.1f ms (grid %d, cluster %d, %lld of %lld steps with events, %.0f warp items per step, "
                            "rank pool %s)\n",
                    t_built - t_start, layout_name, t_staged - t_built, total / 1e6, h2d / 1e6, pms, ms - pms, now_ms() - t_staged, grid, cluster,
                    (long long)S_live, (long long)S, warps_per_step, rank_stride ? "on" : "off");
        }
        if (stats) {
            stats->build_ms = t_built - t_start;
            stats->kernel_ms = ms;
            stats->steps = S;
            stats->inserts = cnt.n_ins;
            stats->queries = n_qry * C2;
            stats->tree_bytes = (int64_t)total;
            stats->h2d_bytes = h2d;
            stats->d2h_bytes = M * 8;
            stats->kernel_launches = (grid == 0 || n_qry == 0) ? 1 : 2;
        }
    }
    rc = chain_traceback(p, h_dp.data(), h_bp.data(), dp_out, backptr_out, chain_out, chain_len, opt_score);
    if (rc != CLB_OK) goto cleanup;
    if (stats) stats->total_ms = now_ms() - t_start;
cleanup:
    if (!keep || rc != CLB_OK) {  // large arenas are not kept: other calls of the library size themselves by free memory
        if (ar.d) cudaFree(ar.d);
        if (ar.h) cudaFreeHost(ar.h);
        ar.d = ar.h = nullptr;
        ar.cap = ar.hcap = 0;
    }
    if ((!keep || rc != CLB_OK || ar.ls_cap > kArenaKeep) && ar.ls) {  // the layout scratch: the same rule, and never kept above kArenaKeep
        cudaFree(ar.ls);
        ar.ls = nullptr;
        ar.ls_cap = 0;
    }
    return rc;
}

// Device and pinned buffers of the batched path, per device, grown on demand and kept (the flushes of one device are
// serialised: a flush is one copy in, one launch, one copy out).
namespace {
struct BatchArena {
    char* d_arena = nullptr; size_t arena_cap = 0;
    clb::ChainArgs* d_args = nullptr; size_t args_cap = 0;
    float* d_dp = nullptr; uint32_t* d_bp = nullptr; size_t res_cap = 0;
    char* d_zero = nullptr; size_t zero_cap = 0;     // zero regions of the problems that run from global memory
    char* h_stage = nullptr; size_t stage_cap = 0;   // pinned: copy regions, then the kernel arguments
    char* h_res = nullptr; size_t hres_cap = 0;      // pinned: dp values, then back-pointers
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};
PerDevice<BatchArena> g_batch_arenas;

template <class T>
cudaError_t grow_device(T*& ptr, size_t& cap, size_t want) {
    if (want <= cap) return cudaSuccess;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    const size_t bytes = std::max<size_t>(want + want / 2, 1 << 20);
    cudaError_t e = cudaMalloc((void**)&ptr, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
}
cudaError_t grow_pinned(char*& ptr, size_t& cap, size_t want) {
    if (want <= cap) return cudaSuccess;
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
    const size_t bytes = std::max<size_t>(want + want / 2, 1 << 20);
    cudaError_t e = cudaHostAlloc((void**)&ptr, bytes, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = bytes;
    return e;
}

// One H2D copy, ONE launch (a CTA per problem), one D2H copy and the tracebacks for every deferred problem of `ctxs`.
int flush_contexts(int device, BatchCtx* const* ctxs, int64_t n_ctx, clb_chain_stats* stats) {
    size_t stage_bytes = 0, res_total = 0;
    int64_t nb = 0;
    int max_smem = 0;
    for (int64_t c = 0; c < n_ctx; ++c) {
        stage_bytes += ArenaPlan::align(ctxs[c]->staging.size());
        res_total += ctxs[c]->res_total;
        nb += (int64_t)ctxs[c]->items.size();
        max_smem = std::max(max_smem, ctxs[c]->max_smem);
    }
    if (nb == 0) return CLB_OK;
    int rc = CLB_OK;
    auto& batch_slot = g_batch_arenas.at(device);
    std::lock_guard<std::mutex> lk(batch_slot.mu);
    BatchArena& ba = batch_slot.state;
    const double t_start = now_ms();
    CUDA_TRY(cudaSetDevice(device));
    if (!ba.stream) {
        CUDA_TRY(cudaStreamCreateWithFlags(&ba.stream, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreate(&ba.e0));
        CUDA_TRY(cudaEventCreate(&ba.e1));
    }
    const size_t args_bytes = (size_t)nb * sizeof(clb::ChainArgs);
    CUDA_TRY(grow_device(ba.d_arena, ba.arena_cap, stage_bytes));
    CUDA_TRY(grow_device(ba.d_args, ba.args_cap, args_bytes));
    if (res_total * 4 > ba.res_cap) {
        size_t cap_dp = ba.res_cap, cap_bp = ba.res_cap;
        CUDA_TRY(grow_device(ba.d_dp, cap_dp, res_total * 4));
        CUDA_TRY(grow_device(ba.d_bp, cap_bp, res_total * 4));
        ba.res_cap = std::min(cap_dp, cap_bp);
    }
    CUDA_TRY(grow_pinned(ba.h_stage, ba.stage_cap, stage_bytes + args_bytes));
    CUDA_TRY(grow_pinned(ba.h_res, ba.hres_cap, res_total * 8));
    clb::ChainArgs* h_args = reinterpret_cast<clb::ChainArgs*>(ba.h_stage + stage_bytes);
    float* h_dp = reinterpret_cast<float*>(ba.h_res);
    uint32_t* h_bp = reinterpret_cast<uint32_t*>(ba.h_res + res_total * 4);
    size_t zero_total = 0;  // problems too large for shared memory keep their zero-initialised region in global memory
    for (int64_t c = 0; c < n_ctx; ++c)
        for (const DeferredProblem& d : ctxs[c]->items)
            if (d.layout.arena_bytes() > (size_t)clb::kChainSmallArena) zero_total += ArenaPlan::align(d.layout.zero_bytes);
    CUDA_TRY(grow_device(ba.d_zero, ba.zero_cap, zero_total));
    {
        size_t seg = 0, res_base = 0, zero_off = 0;
        int64_t k = 0;
        for (int64_t c = 0; c < n_ctx; ++c) {
            const BatchCtx& ctx = *ctxs[c];
            if (!ctx.staging.empty()) memcpy(ba.h_stage + seg, ctx.staging.data(), ctx.staging.size());
            for (const DeferredProblem& d : ctx.items) {
                // the copy region is the staged copy; the zero region follows it (shared memory: the kernel lays both out
                // behind each other) or is this problem's part of the cleared buffer
                char* const copy = ba.d_arena + seg + d.arena_off;
                const bool in_smem = d.layout.arena_bytes() <= (size_t)clb::kChainSmallArena;
                clb::ChainArgs a = bind(d.layout, copy, in_smem ? copy + d.layout.copy_bytes : ba.d_zero + zero_off);
                if (!in_smem) zero_off += ArenaPlan::align(d.layout.zero_bytes);
                a.out_dp = ba.d_dp + res_base + d.res_off;
                a.out_backptr = ba.d_bp + res_base + d.res_off;
                h_args[k++] = a;
            }
            seg += ArenaPlan::align(ctx.staging.size());
            res_base += ctx.res_total;
        }
    }
    const double t_staged = now_ms();
    CUDA_TRY(cudaMemcpyAsync(ba.d_arena, ba.h_stage, stage_bytes, cudaMemcpyHostToDevice, ba.stream));
    CUDA_TRY(cudaMemcpyAsync(ba.d_args, h_args, args_bytes, cudaMemcpyHostToDevice, ba.stream));
    if (zero_total) CUDA_TRY(cudaMemsetAsync(ba.d_zero, 0, zero_total, ba.stream));
    CUDA_TRY(cudaEventRecord(ba.e0, ba.stream));
    CUDA_TRY(clb::launch_chain_small_batch(ba.d_args, (int)nb, max_smem, zero_total > 0, ba.stream));
    CUDA_TRY(cudaEventRecord(ba.e1, ba.stream));
    CUDA_TRY(cudaMemcpyAsync(h_dp, ba.d_dp, res_total * 4, cudaMemcpyDeviceToHost, ba.stream));
    CUDA_TRY(cudaMemcpyAsync(h_bp, ba.d_bp, res_total * 4, cudaMemcpyDeviceToHost, ba.stream));
    CUDA_TRY(cudaStreamSynchronize(ba.stream));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, ba.e0, ba.e1));
    if (stats) {
        stats->kernel_ms += ms;
        stats->kernel_launches += 1;
    }
    const double t_done = now_ms();
    {
        size_t res_base = 0;
        for (int64_t c = 0; c < n_ctx && rc == CLB_OK; ++c) {
            for (const DeferredProblem& d : ctxs[c]->items) {
                rc = chain_traceback(d.p, h_dp + res_base + d.res_off, h_bp + res_base + d.res_off, d.dp_out, d.backptr_out, d.chain_out, d.chain_len,
                                     d.opt_score);
                if (rc != CLB_OK) break;
            }
            res_base += ctxs[c]->res_total;
        }
    }
    if (getenv("CLB_TIMING"))
        fprintf(stderr, "[clb] chain batch: %lld problems in one launch, %.2f MB staged in %.2f ms, kernel %.2f ms, copies+sync %.2f ms, tracebacks %.2f ms\n",
                (long long)nb, stage_bytes / 1e6, t_staged - t_start, ms, t_done - t_staged - ms, now_ms() - t_done);
    g_batch_flushes += 1;
    g_batch_problems += nb;
    return rc;
}
}  // namespace

// Many independent chaining problems in one call.  The Anchorer's fill-in pass (anchorer.hpp:619-699) chains the
// matches inside every gap of the main chain separately -- thousands of problems of a few dozen matches each; one at a
// time each pays a layout, a staging copy, a launch on ONE SM and a read-back.  Here every problem that fits shared
// memory is laid out on the host, all of them are staged in one buffer and solved by ONE launch with a CTA per problem
// (chain_small_batch_kernel), and the results come back in one copy; larger problems run through clb_chain_dp.
extern "C" int clb_chain_dp_batch(int device, int64_t n_problems, const clb_chain_problem* const* problems, float* const* dp_out,
                                  int64_t* const* backptr_out, int64_t* const* chain_out, int64_t* chain_len, float* opt_score,
                                  clb_chain_stats* stats) {
    const double t_start = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_problems < 0 || (n_problems > 0 && (!problems || !chain_out || !chain_len))) return fail(CLB_EINVAL, "clb_chain_dp_batch: null arguments");
    BatchCtx ctx;
    clb_chain_stats one{};
    for (int64_t k = 0; k < n_problems; ++k) {
        if (!problems[k] || !chain_out[k]) return fail(CLB_EINVAL, "clb_chain_dp_batch: null problem or output");
        const int rc = chain_dp_impl(device, problems[k], dp_out ? dp_out[k] : nullptr, backptr_out ? backptr_out[k] : nullptr, chain_out[k],
                                     &chain_len[k], opt_score ? &opt_score[k] : nullptr, stats ? &one : nullptr, &ctx);
        if (rc != CLB_OK) return rc;
        if (stats) {
            stats->build_ms += one.build_ms; stats->kernel_ms += one.kernel_ms; stats->steps += one.steps; stats->inserts += one.inserts;
            stats->queries += one.queries; stats->tree_bytes += one.tree_bytes; stats->h2d_bytes += one.h2d_bytes;
            stats->d2h_bytes += one.d2h_bytes; stats->kernel_launches += one.kernel_launches;
        }
    }
    BatchCtx* const one_ctx[1] = {&ctx};
    const int rc = flush_contexts(device, one_ctx, 1, stats);
    if (rc != CLB_OK) return rc;
    if (stats) stats->total_ms = now_ms() - t_start;
    return CLB_OK;
}

// The batched call over several devices: the problems are dealt by a work estimate and every device runs
// clb_chain_dp_batch on its share, from its own host thread.
extern "C" int clb_chain_dp_batch_multi(int n_devices, const int* devices, int64_t n_problems, const clb_chain_problem* const* problems,
                                        float* const* dp_out, int64_t* const* backptr_out, int64_t* const* chain_out, int64_t* chain_len,
                                        float* opt_score, int32_t* part_out, clb_chain_stats* stats) {
    const double t_start = now_ms();
    if (stats) memset(stats, 0, sizeof(*stats));
    if (const int rc = clb::check_devices(n_devices, devices, "clb_chain_dp_batch_multi")) return rc;
    if (n_problems < 0 || n_problems >= (int64_t(1) << 31) || (n_problems > 0 && (!problems || !chain_out || !chain_len)))
        return fail(CLB_EINVAL, "clb_chain_dp_batch_multi: null arguments or too many problems");
    for (int k = 0; k < n_devices; ++k)
        if (const int rc = clb::require_device(devices[k])) return rc;
    // the DP costs about a step's latency times the steps (DESIGN.md section 10), and the layout grows with the events
    std::vector<int64_t> cost((size_t)n_problems);
    for (int64_t k = 0; k < n_problems; ++k) {
        const clb_chain_problem* p = problems[k];
        if (!p || !chain_out[k]) return fail(CLB_EINVAL, "clb_chain_dp_batch_multi: null problem or output");
        cost[k] = std::max<int64_t>(0, p->n_step) + (p->ins_off && p->n_match > 0 ? p->ins_off[p->n_match] : 0) +
                  (p->qry_off && p->n_step > 0 ? p->qry_off[p->n_step] : 0);
    }
    std::vector<clb_chain_stats> dev_stats(n_devices);
    const int rc = clb::deal_to_devices(n_devices, devices, (int32_t)n_problems, cost.data(), part_out, [&](int d, const std::vector<int32_t>& sel) -> int {
        // the share's pointers in share order; chain lengths and optima come back through local arrays
        const size_t n = sel.size();
        std::vector<const clb_chain_problem*> ps(n);
        std::vector<float*> dps(n, nullptr);
        std::vector<int64_t*> bps(n, nullptr), chains(n);
        std::vector<int64_t> lens(n, 0);
        std::vector<float> opts(n, 0.f);
        for (size_t i = 0; i < n; ++i) {
            ps[i] = problems[sel[i]];
            if (dp_out) dps[i] = dp_out[sel[i]];
            if (backptr_out) bps[i] = backptr_out[sel[i]];
            chains[i] = chain_out[sel[i]];
        }
        const int r = clb_chain_dp_batch(devices[d], (int64_t)n, ps.data(), dps.data(), bps.data(), chains.data(), lens.data(), opts.data(),
                                         stats ? &dev_stats[d] : nullptr);
        if (r != CLB_OK) return r;
        for (size_t i = 0; i < n; ++i) {
            chain_len[sel[i]] = lens[i];
            if (opt_score) opt_score[sel[i]] = opts[i];
        }
        return CLB_OK;
    });
    if (rc != CLB_OK) return rc;
    if (stats) {
        for (const clb_chain_stats& one : dev_stats) {
            stats->build_ms += one.build_ms; stats->kernel_ms += one.kernel_ms; stats->steps += one.steps; stats->inserts += one.inserts;
            stats->queries += one.queries; stats->tree_bytes += one.tree_bytes; stats->h2d_bytes += one.h2d_bytes;
            stats->d2h_bytes += one.d2h_bytes; stats->kernel_launches += one.kernel_launches;
        }
        stats->total_ms = now_ms() - t_start;
    }
    return CLB_OK;
}

// The same in two halves, for callers that prepare problems on several host threads (the drop-in Anchorer runs the
// fill-in subproblems of anchorer.hpp:657-693 on a thread pool): clb_chain_job_create lays one problem out in the CALLING
// thread -- no device work, thread-safe -- and clb_chain_jobs_run solves the jobs of any number of threads in one launch.
struct clb_chain_job {
    BatchCtx ctx;
    int device = 0;
};

extern "C" int clb_chain_job_create(int device, const clb_chain_problem* problem, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                                    int64_t* chain_len, float* opt_score, clb_chain_job** job) {
    if (!job) return fail(CLB_EINVAL, "clb_chain_job_create: null job pointer");
    *job = nullptr;
    if (!problem || !chain_out || !chain_len) return fail(CLB_EINVAL, "clb_chain_job_create: null arguments");
    clb_chain_job* j = new (std::nothrow) clb_chain_job();
    if (!j) return fail(CLB_ENOMEM, "clb_chain_job_create: out of host memory");
    j->device = device;
    // a problem too large for one SM's shared memory is solved here and now (ctx stays empty)
    const int rc = chain_dp_impl(device, problem, dp_out, backptr_out, chain_out, chain_len, opt_score, nullptr, &j->ctx);
    if (rc != CLB_OK) {
        delete j;
        return rc;
    }
    if (j->ctx.items.empty()) {  // solved already (or nothing to solve): no job
        delete j;
        return CLB_OK;
    }
    *job = j;
    return CLB_OK;
}

extern "C" int clb_chain_jobs_run(int device, int64_t n_jobs, clb_chain_job* const* jobs) {
    if (n_jobs < 0 || (n_jobs > 0 && !jobs)) return fail(CLB_EINVAL, "clb_chain_jobs_run: null arguments");
    std::vector<BatchCtx*> ctxs;
    ctxs.reserve((size_t)n_jobs);
    for (int64_t k = 0; k < n_jobs; ++k) {
        if (!jobs[k]) return fail(CLB_EINVAL, "clb_chain_jobs_run: null job");
        if (jobs[k]->device != device) return fail(CLB_EINVAL, "clb_chain_jobs_run: job was created for another device");
        if (!jobs[k]->ctx.items.empty()) ctxs.push_back(&jobs[k]->ctx);
    }
    const int rc = flush_contexts(device, ctxs.data(), (int64_t)ctxs.size(), nullptr);
    if (rc == CLB_OK)
        for (BatchCtx* c : ctxs) {  // a job runs once
            c->items.clear();
            c->staging.clear();
            c->res_total = 0;
        }
    return rc;
}

extern "C" void clb_chain_job_destroy(clb_chain_job* job) { delete job; }

namespace clb {
void chain_release_cache() {
    g_arenas.for_each([](int device, DeviceArena& a) {
        cudaSetDevice(device);
        if (a.d) cudaFree(a.d);
        if (a.h) cudaFreeHost(a.h);
        if (a.ls) cudaFree(a.ls);
        if (a.ev0) cudaEventDestroy(a.ev0);
        if (a.ev1) cudaEventDestroy(a.ev1);
        if (a.evp) cudaEventDestroy(a.evp);
        if (a.stream) cudaStreamDestroy(a.stream);
        a = DeviceArena{};
    });
    g_batch_arenas.for_each([](int device, BatchArena& b) {
        cudaSetDevice(device);
        if (b.d_arena) cudaFree(b.d_arena);
        if (b.d_args) cudaFree(b.d_args);
        if (b.d_dp) cudaFree(b.d_dp);
        if (b.d_bp) cudaFree(b.d_bp);
        if (b.d_zero) cudaFree(b.d_zero);
        if (b.h_stage) cudaFreeHost(b.h_stage);
        if (b.h_res) cudaFreeHost(b.h_res);
        if (b.e0) cudaEventDestroy(b.e0);
        if (b.e1) cudaEventDestroy(b.e1);
        if (b.stream) cudaStreamDestroy(b.stream);
        b = BatchArena{};
    });
}
}  // namespace clb
