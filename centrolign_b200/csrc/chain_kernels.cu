// chain_kernels.cu -- sm_100a kernel of the sparse anchor-chaining DP (clb_chain_dp).
//
// Reference: Anchorer::sparse_affine_chain_dp main loop (include/centrolign/anchorer.hpp:2290-2417) and
// Anchorer::sparse_chain_dp main loop (:1640-1728); search structures max_search_tree.hpp:312-444 and
// orthogonal_max_search_tree.hpp:293-470.  Data layout and the equivalence argument: chain_device.cuh.
//
// A preparation kernel first computes, for all (query, path of graph 2) pairs at once, everything that does not
// depend on DP values: the gap-free tree of the query's diagonal and the shape of its three tree walks.
// Then one persistent kernel walks the graph-1 nodes ("steps") in topological order.  Per step:
//   A  every match ending here enters its DP value into the gap-free tree of its diagonal and into the
//      2*NumPW orthogonal value sets, for every path pair of its end point.  A work item is (entry, gap-free tree) or
//      (entry, one orthogonal value set): one warp, lanes over the ancestors of the entry's node (atomicMax on packed
//      words, Fenwick updates);
//   B  a work item is (match starting behind a forward edge, path of graph 2, gap-free tree) or (..., piece, parity):
//      one warp answers the query by the reference's own tree walk -- lane j owns the j-th node of either walk and the
//      subtree hanging off it (closed form, walk_step) -- keeps the first strictly greater candidate in the
//      reference's order (gap-free, then pieces 0..2P-1) and posts it with atomicMax keyed by (value, earlier first);
//      beside the queries, other threads apply the winners of the PREVIOUS step if they beat the match's current value
//      (update_dp, match_bank.hpp:171-184): queries never read DP values, insertions take max(stored, pending winner).
// The phases are separated by __syncthreads() (one CTA), by the hardware barrier of ONE thread-block cluster of up to 16
// CTAs (barrier.cluster.arrive.release / wait.acquire), or by a cooperative grid.sync(); the host picks by the number of
// work items per step (chain_host.cu).  Records that do not depend on DP values are loaded one phase ahead.
// Scores are float, gap terms double, every operation with an explicit rounding intrinsic so that no FMA
// contraction can change a bit relative to the reference's scalar code.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "chain_device.cuh"

namespace cg = cooperative_groups;

namespace clb {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kThreads = 512;
constexpr int kWarps = kThreads / 32;

__device__ __forceinline__ float mininf() { return -3.402823466e+38f; }  // numeric_limits<float>::lowest()

__device__ __forceinline__ uint32_t ford(float f) {  // order-preserving map float -> uint32 (-0 folded into +0)
    const uint32_t b = __float_as_uint(__fadd_rn(f, 0.0f));
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float funord(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
__device__ __forceinline__ unsigned long long pack(float v, uint32_t low) {
    return ((unsigned long long)ford(v) << 32) | low;
}
constexpr uint32_t kOrdLowest = 0x00800000u;  // ford(lowest()); 0 = never entered; both fail "ord > kOrdLowest"

// Loads.  SM = the whole problem was copied into shared memory (small problems: the Anchorer's fill-in pass makes
// thousands of chaining calls with a few dozen matches each, where a step is nothing but memory latency).
template <bool SM, class T>
__device__ __forceinline__ T ld_const(const T* p) {  // never written while a kernel runs
    if (SM) return *p;
    return __ldg(p);
}
template <bool SM, class T>
__device__ __forceinline__ T ld_live(const T* p) {  // written by other warps between barriers
    if (SM) return *reinterpret_cast<const volatile T*>(p);
    return __ldcg(p);
}
template <bool SM>
__device__ __forceinline__ uint4 ld_const4(const uint4* p) {
    if (SM) return *p;
    return __ldg(p);
}

// The walk shared by MaxSearchTree::range_max (max_search_tree.hpp:361-444) and the outer level of
// OrthogonalMaxSearchTree::range_max (orthogonal_max_search_tree.hpp:340-470), for one-sided key ranges:
//   prefix: in_range(x) <=> key[x] <  bound  (nothing lies below the range: its left walk takes every node)
//   suffix: in_range(x) <=> key[x] >  bound  (nothing lies above the range: its right walk takes every node)
// walk_shape finds the split node S and the in-range decisions along the conditional side (LSB first).  The walk
// is uniform over the warp; to avoid one memory round trip per tree level, the range flags of a node and of its
// descendants four levels down (31 nodes) are fetched by the 31 lanes at once and the next moves are resolved
// from the resulting bit mask.
template <class InRange>
__device__ void walk_shape(uint32_t n, bool prefix, const InRange& in_range, int lane, uint32_t& S_out, uint32_t& bits_out) {
    uint32_t wbase = kChainNone;
    unsigned wbits = 0;
    auto flag = [&](uint32_t y) -> bool {
        const uint32_t rel = y + 1;
        int d = -1;
        if (wbase != kChainNone) {
            const uint32_t b = wbase + 1;
            d = (31 - __clz(rel)) - (31 - __clz(b));
            if (d < 0 || d > 4 || (rel >> d) != b) d = -1;
        }
        if (d < 0) {  // fetch the window rooted at y
            wbase = y;
            bool f = false;
            if (lane < 31) {
                uint32_t idx = y;
                if (lane < 30) {
                    const int dj = 31 - __clz(lane + 2);
                    idx = (rel << dj) - 1 + (uint32_t)(lane + 2 - (1 << dj));
                    if ((rel << dj) < rel) idx = kChainNone;  // overflow: no such node
                }
                if (idx < n) f = in_range(idx);
            }
            wbits = __ballot_sync(kFull, f);
            d = 0;
        }
        if (d == 0) return (wbits >> 30) & 1u;
        const uint32_t k = rel - ((wbase + 1) << d);
        return (wbits >> ((1u << d) - 2 + k)) & 1u;
    };
    uint32_t cursor = 0;
    while (cursor < n && !flag(cursor)) cursor = prefix ? 2 * cursor + 1 : 2 * cursor + 2;
    S_out = cursor < n ? cursor : kChainNone;
    uint32_t bits = 0;
    if (cursor < n) {
        int nbit = 0;
        uint32_t c = prefix ? 2 * cursor + 2 : 2 * cursor + 1;  // the conditional side: right walk of a prefix, left walk of a suffix
        while (c < n) {
            const bool f = flag(c);
            bits |= (uint32_t)f << nbit;
            ++nbit;
            c = (f == prefix) ? 2 * c + 2 : 2 * c + 1;  // prefix: in range -> right, else left; suffix: in range -> left, else right
        }
    }
    bits_out = bits;
}

// Expands a stored walk into the blocks the reference tests.  Its order is: S, then the left walk, then the right walk,
// every taken node followed by the subtree hanging off the walk on the inner side.  The j-th node of either walk has a
// closed form (heap indices + 1 are the bit strings of the root paths), so lane j of a warp finds its two nodes and two
// subtrees without walking:
//   unconditional side (left walk of a prefix range, right walk of a suffix range): always outward;
//   conditional side: decision bit i says whether node i is in range (taken, continue outward) or not (continue inward).
struct WalkStep {
    uint32_t node, sub;  // heap indices of the walk node and of the subtree root hanging inside the range
    bool node_ok, sub_ok;
};
__device__ __forceinline__ WalkStep walk_step(uint32_t n, bool prefix, uint32_t S, uint32_t bits, int side, int j) {
    const bool cond = (side == 1) == prefix;
    const unsigned long long x0 = 2ull * ((unsigned long long)S + 1ull) + (unsigned)side;  // heap index + 1 of the walk's first node
    unsigned long long x;
    bool taken = true;
    if (!cond) {
        x = side == 0 ? (x0 << j) : (((x0 + 1ull) << j) - 1ull);
    } else {
        const uint32_t path = side == 0 ? ~bits : bits;  // child bit per step: left walk taken -> 0, right walk taken -> 1
        x = (x0 << j) | (unsigned long long)(j ? (__brev(path) >> (32 - j)) : 0u);
        taken = (bits >> j) & 1u;
    }
    WalkStep w;
    const bool exists = j < 31 && x <= (unsigned long long)n;
    const unsigned long long xs = side == 0 ? 2ull * x + 1ull : 2ull * x;  // left walk: right child; right walk: left child
    w.node_ok = exists && taken;
    w.sub_ok = w.node_ok && xs <= (unsigned long long)n;
    w.node = (uint32_t)(x - 1ull);
    w.sub = (uint32_t)(xs - 1ull);
    return w;
}
// position of a block in the reference's test order (only the order matters): S = 0, left walk, right walk
__device__ __forceinline__ uint32_t walk_key(int side, int j, int kind) { return 1u + 64u * (unsigned)side + 2u * (unsigned)j + (unsigned)kind; }

// first index in [lo, hi) whose value is >= q, by 32-ary search over the warp (uniform result)
template <bool SM>
__device__ int64_t warp_lower_bound(const int32_t* arr, int64_t lo, int64_t hi, int q, int lane) {
    while (hi - lo > 32) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t at = lo + (int64_t)lane * step;
        const bool less = at < hi && ld_const<SM>(&arr[at]) < q;
        const int cnt = __popc(__ballot_sync(kFull, less));  // pivots below q form a prefix
        if (cnt == 0) return lo;
        const int64_t nlo = lo + (int64_t)(cnt - 1) * step + 1;
        hi = min(hi, lo + (int64_t)cnt * step);
        lo = nlo;
    }
    const bool less = lo + lane < hi && ld_const<SM>(&arr[lo + lane]) < q;
    return lo + __popc(__ballot_sync(kFull, less));
}

// number of entries of the ascending list `a[0, n)` that are < key, 8-ary search with independent probes
template <bool SM>
__device__ __forceinline__ uint32_t count_less(const uint32_t* a, uint32_t n, uint32_t key) {
    uint32_t lo = 0, hi = n;  // answer in [lo, hi]
    while (hi - lo > 7) {
        const uint32_t step = (hi - lo) >> 3;
        uint32_t v[7];
#pragma unroll
        for (int i = 0; i < 7; ++i) v[i] = ld_const<SM>(&a[lo + (i + 1) * step - 1]);
        int c = 0;
#pragma unroll
        for (int i = 0; i < 7; ++i) c += v[i] < key;
        const uint32_t nlo = lo + c * step;
        hi = c == 7 ? hi : lo + (c + 1) * step - 1;
        lo = nlo;
    }
    uint32_t v[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) v[i] = lo + i < hi ? ld_const<SM>(&a[lo + i]) : kChainNone;
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < 7; ++i) c += (lo + i < hi) && v[i] < key;
    return lo + c;
}

}  // namespace

// Everything about a (query, path of graph 2) pair that does not depend on DP values (anchorer.hpp:2374-2381).
template <bool SM>
__device__ void prepare_queries(const ChainArgs& A, int lane, int64_t gwarp, int64_t nwarp) {
    const int C1 = A.n_chain1, C2 = A.n_chain2;
    for (int64_t qc = gwarp; qc < A.n_qry * C2; qc += nwarp) {
        const int64_t k = qc / C2;
        const int c2 = (int)(qc - k * C2);
        const uint32_t m = A.qry_match[k], c1 = A.qry_chain1[k];
        QueryRec r;
        r.match = m;
        r.weight = A.weight[m];
        r.offset = A.qoff[(int64_t)m * C2 + c2];
        r.q = (int)((uint32_t)A.qa1[(int64_t)m * C1 + c1] - (uint32_t)A.qa2[(int64_t)m * C2 + c2]);
        r.gf_base = r.gf_n = r.or_base = r.or_n = 0;
        r.gf_S = r.ev_S = r.od_S = kChainNone;
        r.gf_bits = r.ev_bits = r.od_bits = 0;
        if (r.offset != 0) {
            const int64_t pair = (int64_t)c1 * C2 + c2;
            const int64_t g1 = A.pair_grp_off[pair + 1];
            const int64_t g = warp_lower_bound<SM>(A.grp_shift, A.pair_grp_off[pair], g1, r.q, lane);
            if (g < g1 && ld_const<SM>(&A.grp_shift[g]) == r.q) {  // the diagonal exists (anchorer.hpp:2379-2382)
                r.gf_base = A.grp_base[g];
                r.gf_n = A.grp_n[g];
                const uint32_t* key = A.gf_key + r.gf_base;
                const uint32_t offset = r.offset;
                walk_shape(r.gf_n, true, [&](uint32_t x) { return ld_const<SM>(&key[x]) < offset; }, lane, r.gf_S, r.gf_bits);
            }
            if (A.num_pw > 0) {
                r.or_base = A.pair_base[pair];
                r.or_n = A.pair_base[pair + 1] - r.or_base;
                const int32_t* shift = A.or_shift + r.or_base;
                const int q = r.q;
                if (r.or_n) {
                    walk_shape(r.or_n, false, [&](uint32_t x) { return ld_const<SM>(&shift[x]) > q; }, lane, r.ev_S, r.ev_bits);
                    walk_shape(r.or_n, true, [&](uint32_t x) { return ld_const<SM>(&shift[x]) < q; }, lane, r.od_S, r.od_bits);
                    if (A.rank_pool) {  // how many elements of every subtree block lie below the query offset
                        for (int par = 0; par < 2; ++par) {
                            const uint32_t S = par ? r.od_S : r.ev_S;
                            if (S == kChainNone) continue;
                            const uint32_t bits = par ? r.od_bits : r.ev_bits;
                            uint32_t* pool = A.rank_pool + ((int64_t)qc * 2 + par) * A.rank_stride;
                            const WalkStep wl = walk_step(r.or_n, par == 1, S, bits, 0, lane), wr = walk_step(r.or_n, par == 1, S, bits, 1, lane);
                            const unsigned lm = __ballot_sync(kFull, wl.sub_ok), rm = __ballot_sync(kFull, wr.sub_ok);
                            const unsigned below = (1u << lane) - 1u;
                            for (int side = 0; side < 2; ++side) {  // subtree blocks in walk order: the left walk's, then the right walk's
                                const WalkStep& w = side ? wr : wl;
                                const int j = side ? __popc(lm) + __popc(rm & below) : __popc(lm & below);
                                if (w.sub_ok && j < A.rank_stride)
                                    pool[j] = count_less<SM>(A.in_off + ld_const<SM>(&A.in_base[r.or_base + w.sub]), ld_const<SM>(&A.in_n[r.or_base + w.sub]), r.offset);
                            }
                        }
                    }
                }
            }
        }
        r.or_base2 = r.or_base;
        r.or_n2 = r.or_n;
        if (lane == 0) A.qrec[qc] = r;
    }
}

__global__ void __launch_bounds__(256) chain_prepare_kernel(const ChainArgs A) {
    prepare_queries<false>(A, threadIdx.x & 31, ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, ((int64_t)gridDim.x * blockDim.x) >> 5);
}

// 16-byte loads of DP-independent records that are issued one phase before they are needed (the next step's first work
// item of this warp): volatile so that the compiler keeps them where they are written.
__device__ __forceinline__ uint4 ld_early(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ int64_t ld_early(const int64_t* p) {
    int64_t v;
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ld_early(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// warp-wide maximum of (hi, lo) pairs in lexicographic order, hi == 0 means "nothing"; returns the lane that holds it
// (kFull lanes must call), or -1
__device__ __forceinline__ int warp_argmax(uint32_t hi, uint32_t lo, uint32_t& hi_out) {
    const uint32_t mh = __reduce_max_sync(kFull, hi);
    hi_out = mh;
    if (mh == 0) return -1;
    const uint32_t ml = __reduce_max_sync(kFull, hi == mh ? lo : 0u);
    return __ffs(__ballot_sync(kFull, hi == mh && lo == ml)) - 1;
}

// NK: work items per insertion / per (query, chain2) pair known at compile time (1 = gap-free chaining, 7 = three gap
// pieces), 0 = 2 * num_pw + 1 read from the arguments.
template <bool SM, int NK>
__device__ __forceinline__ void chain_steps(const ChainArgs& A) {
    cg::grid_group grid = cg::this_grid();
    const int mode = SM ? 0 : A.sync_mode;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    // the shared-memory flavour is one CTA per problem whatever the grid is (a batch launch has one CTA per problem);
    // with several CTAs, consecutive work items of a step go to different CTAs (a step has a few dozen items)
    const uint32_t nctas = mode == 0 ? 1u : gridDim.x, cta = mode == 0 ? 0u : blockIdx.x;
    const uint32_t gwarp = (uint32_t)wib * nctas + cta, nwarp = nctas * (blockDim.x >> 5);
    const uint32_t gthread = cta * blockDim.x + threadIdx.x, nthread = nctas * blockDim.x;
    const int C2 = A.n_chain2, T = 2 * A.num_pw;
    // work items: an insertion has one item for the gap-free tree of its diagonal and one per orthogonal value set; a
    // (query, chain2) pair has one item for the gap-free tree and one per (piece, parity), in the reference's candidate order
    const uint32_t n_kind = NK ? (uint32_t)NK : (uint32_t)(T + 1);
    const uint32_t slots = n_kind;
    unsigned long long n_tree_queries = 0;
    constexpr bool kEarly = !SM;  // records of the next step are fetched one phase ahead (global memory only)

    auto barrier = [&]() {
        if (mode == 0) __syncthreads();
        else if (mode == 1) asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        else grid.sync();
    };
    // update_dp of the winners of the previous step (match_bank.hpp:171-184).  Runs beside the queries of the current step,
    // which never read DP values; an insertion of the current step took the maximum of the stored value and the pending
    // winner (effective_dp).  The candidate words are double-buffered by step parity; the thread that applies a winner
    // also clears its word, a full step before that buffer is posted to again.
    auto apply_winners = [&](int64_t q0, int64_t q1, unsigned long long* cand, const uint32_t* cand_bp) {
        for (uint32_t qi = gthread; qi < (uint32_t)(q1 - q0); qi += nthread) {
            const uint32_t m = ld_const<SM>(&A.qry_match[q0 + qi]);
            const unsigned long long pk = ld_live<SM>(&cand[m]);
            if (!pk) continue;
            const uint32_t order = ~(uint32_t)pk;
            if (order / ((uint32_t)C2 * slots) != qi) continue;  // the winner was posted by another query of this match
            const float v = funord((uint32_t)(pk >> 32));
            if (v > ld_live<SM>(&A.dp[m])) {
                A.dp[m] = v;
                A.backptr[m] = ld_live<SM>(&cand_bp[order]);
            }
            cand[m] = 0;
        }
    };
    auto effective_dp = [&](uint32_t m, const unsigned long long* cand) -> float {
        const unsigned long long pk = ld_live<SM>(&cand[m]);
        float dpv = ld_live<SM>(&A.dp[m]);
        if (pk) {
            const float v = funord((uint32_t)(pk >> 32));
            if (v > dpv) dpv = v;
        }
        return dpv;
    };
    // the two records of this warp's first work items of a step
    struct InsEarly { uint4 a, b; uint32_t ib, cn, rank; };
    struct QryEarly { uint4 r0, rs; };
    auto ins_item = [&](uint32_t it, int64_t i0, int64_t& i, uint32_t& u) {
        const uint32_t ii = it / n_kind;
        u = it - ii * n_kind;
        i = i0 + ii;
    };
    auto fetch_ins = [&](int64_t i0, InsEarly& e) {
        int64_t i; uint32_t u;
        ins_item(gwarp, i0, i, u);
        if (i < A.n_ins) {
            e.a = ld_early(reinterpret_cast<const uint4*>(&A.ins[i]));
            e.b = ld_early(reinterpret_cast<const uint4*>(&A.ins[i]) + 1);
        }
    };
    auto fetch_levels = [&](int64_t i0, InsEarly& e) {  // needs e.a, e.b
        int64_t i; uint32_t u;
        ins_item(gwarp, i0, i, u);
        if (i < A.n_ins && u > 0 && lane < (int)e.b.w) {
            const uint32_t a = ((e.b.x + 1) >> lane) - 1;
            e.ib = ld_early(&A.in_base[e.a.w + a]);
            e.cn = ld_early(&A.in_n[e.a.w + a]);
            e.rank = ld_early(&A.ent_rank[e.b.z + lane]);
        }
    };
    auto qry_second = [&](uint32_t type) -> int { return type == 0 ? 1 : 2 + (int)((type - 1) & 1u); };
    auto fetch_qry = [&](int64_t q0, QryEarly& e) {
        const uint32_t qc = gwarp / n_kind, type = gwarp - qc * n_kind;
        const int64_t idx = q0 * C2 + qc;
        if (idx < A.n_qry * C2) {
            const uint4* rp = reinterpret_cast<const uint4*>(&A.qrec[idx]);
            e.r0 = ld_early(rp);
            e.rs = ld_early(rp + qry_second(type));
        }
    };

    const int64_t S = A.n_step;
    if (S <= 0) return;
    int64_t i0 = A.sins_off[0], i1 = A.sins_off[1], q0 = A.qry_off[0], q1 = A.qry_off[1];
    int64_t pq0 = 0, pq1 = 0;  // queries of the previous step, whose winners are still to be applied
    InsEarly ie = {}, ie_next = {};
    QryEarly qe = {}, qe_next = {};
    if (kEarly) {
        fetch_ins(i0, ie);
        fetch_levels(i0, ie);
        fetch_qry(q0, qe);
    }
    for (int64_t s = 0; s < S; ++s) {
        unsigned long long* cand_prev = A.cand_best + ((s + 1) & 1) * A.n_match;  // posted in step s-1
        unsigned long long* cand_cur = A.cand_best + (s & 1) * A.n_match;         // posted in this step
        uint32_t* bp_prev = A.cand_bp + ((s + 1) & 1) * A.cand_bp_stride;
        uint32_t* bp_cur = A.cand_bp + (s & 1) * A.cand_bp_stride;
        const int64_t s2 = s + 2 <= S ? s + 2 : S;
        int64_t i2, q2;  // used by the next step
        if (kEarly) {
            i2 = ld_early(&A.sins_off[s2]);
            q2 = ld_early(&A.qry_off[s2]);
        } else {
            i2 = A.sins_off[s2];
            q2 = A.qry_off[s2];
        }
        if (kEarly) {
            fetch_ins(i1, ie_next);
            fetch_qry(q1, qe_next);
        }
        // -------------------------------- A: inserts (anchorer.hpp:2301-2345) --------------------------------
        const uint32_t n_ins_items = (uint32_t)(i1 - i0) * n_kind;
        for (uint32_t it = gwarp; it < n_ins_items; it += nwarp) {
            int64_t i; uint32_t u;
            ins_item(it, i0, i, u);
            const bool early = kEarly && it == gwarp;
            const uint4 ra = early ? ie.a : ld_const4<SM>(reinterpret_cast<const uint4*>(&A.ins[i]));
            const uint4 rb = early ? ie.b : ld_const4<SM>(reinterpret_cast<const uint4*>(&A.ins[i]) + 1);
            const uint32_t m = ra.x, gf_base = ra.y, gf_node = ra.z, or_base = ra.w, or_node = rb.x, rank_off = rb.z;
            const int shift = (int)rb.y, nr = (int)rb.w;
            uint32_t ib = 0, cn = 0, rank = 0;
            if (u > 0 && lane < nr) {  // lane = level: the node itself and its ancestors below the outer spines
                if (early) {
                    ib = ie.ib; cn = ie.cn; rank = ie.rank;
                } else {
                    const uint32_t a = ((or_node + 1) >> lane) - 1;
                    ib = ld_const<SM>(&A.in_base[or_base + a]);
                    cn = ld_const<SM>(&A.in_n[or_base + a]);
                    rank = ld_const<SM>(&A.ent_rank[rank_off + lane]);
                }
            }
            const float dpv = effective_dp(m, cand_prev);
            if (!(dpv > mininf())) continue;  // entering lowest() changes nothing in the reference's trees
            if (u == 0) {  // gap-free tree of the entry's diagonal: lanes = the node and its ancestors
                if (lane == 0) A.gf_ord[gf_base + gf_node] = ford(dpv);
                const uint32_t anc = (gf_node + 1) >> lane;
                if (anc) atomicMax(&A.gf_best[gf_base + anc - 1], pack(dpv, ~(uint32_t)i));
            } else if constexpr (NK != 1) {
                // anchorer.hpp:2328-2335: odd pieces add, even pieces subtract local_scale * gap_extend * shift
                const int t = (int)u - 1;
                const double gap = __dmul_rn(A.scale_ext[t >> 1], (double)shift);
                const float v = __double2float_rn((t & 1) ? __dadd_rn((double)dpv, gap) : __dsub_rn((double)dpv, gap));
                if (!(v > mininf())) continue;  // anchorer.hpp:2338
                if (lane == 0) A.or_ord[(int64_t)t * A.n_entry + or_base + or_node] = ford(v);
                if (lane < nr) {
                    const unsigned long long pk = pack(v, or_node);
                    unsigned long long* bit = A.bit + (int64_t)t * A.n_inner + ib;
                    for (uint32_t k = rank; k < cn; k |= k + 1) atomicMax(&bit[k], pk);
                }
            }
        }
        if (i0 != i1) barrier();
        if (kEarly) fetch_levels(i1, ie_next);

        // ---------------- update_dp of the previous step + B: queries (anchorer.hpp:2352-2416) ----------------
        if (pq0 != pq1) apply_winners(pq0, pq1, cand_prev, bp_prev);
        auto post = [&](uint32_t m, uint32_t qc, uint32_t slot, float cand, uint32_t bp) {  // one lane
            const uint32_t order = qc * slots + slot;
            bp_cur[order] = bp;
            atomicMax(&cand_cur[m], pack(cand, ~order));
        };
        const uint32_t n_items = (uint32_t)(q1 - q0) * (uint32_t)C2 * n_kind;
        for (uint32_t item = gwarp; item < n_items; item += nwarp) {
            const uint32_t qc = item / n_kind, type = item - qc * n_kind;  // (query, chain2) pair inside the step
            const bool early = kEarly && item == gwarp;
            const uint4* rp = reinterpret_cast<const uint4*>(&A.qrec[q0 * C2 + qc]);
            const uint4 r0 = early ? qe.r0 : ld_const4<SM>(rp);  // match, weight, offset, q
            const uint32_t offset = r0.z;
            if (offset == 0) continue;  // nothing on this path reaches the match: every range [0, 0) is empty
            const uint4 rs = early ? qe.rs : ld_const4<SM>(rp + qry_second(type));  // tree base, size, S, decision bits of the walk
            const uint32_t m = r0.x, base = rs.x, n = rs.y, S0 = rs.z, bits = rs.w;
            const float w = __uint_as_float(r0.y);
            const int q = (int)r0.w;
            if (n == 0 || S0 == kChainNone) continue;
            ++n_tree_queries;
            const bool prefix = type == 0 || ((type - 1) & 1u);
            const WalkStep wl = walk_step(n, prefix, S0, bits, 0, lane), wr = walk_step(n, prefix, S0, bits, 1, lane);
            // this lane's blocks: S (lane 0), its node and hanging subtree on either walk
            uint32_t best_hi = 0, best_lo = 0, best_sel = 0;  // (ord, ~key) and what identifies the match
            auto consider = [&](uint32_t ord, uint32_t key, uint32_t sel) {
                if (ord > kOrdLowest && (ord > best_hi || (ord == best_hi && ~key > best_lo))) {
                    best_hi = ord;
                    best_lo = ~key;
                    best_sel = sel;
                }
            };
            if (NK == 1 || type == 0) {
                // same diagonal (anchorer.hpp:2379-2389): MaxSearchTree::range_max((0, min), (offset, min))
                const uint32_t vS = lane == 0 ? ld_live<SM>(&A.gf_ord[base + S0]) : 0u;
                const uint32_t vl = wl.node_ok ? ld_live<SM>(&A.gf_ord[base + wl.node]) : 0u;
                const uint32_t vr = wr.node_ok ? ld_live<SM>(&A.gf_ord[base + wr.node]) : 0u;
                const unsigned long long sl = wl.sub_ok ? ld_live<SM>(&A.gf_best[base + wl.sub]) : 0ull;
                const unsigned long long sr = wr.sub_ok ? ld_live<SM>(&A.gf_best[base + wr.sub]) : 0ull;
                consider(vS, 0, S0);
                consider(vl, walk_key(0, lane, 0), wl.node);
                consider((uint32_t)(sl >> 32), walk_key(0, lane, 1), 0x80000000u | (~(uint32_t)sl & 0x7fffffffu));  // the insertion sequence number (< 2^31)
                consider(vr, walk_key(1, lane, 0), wr.node);
                consider((uint32_t)(sr >> 32), walk_key(1, lane, 1), 0x80000000u | (~(uint32_t)sr & 0x7fffffffu));
                uint32_t top;
                const int src = warp_argmax(best_hi, best_lo, top);
                if (src < 0) continue;
                if (lane == src) {
                    const uint32_t bm = (best_sel & 0x80000000u) ? ld_const<SM>(&A.ins[best_sel & 0x7fffffffu].match) : ld_const<SM>(&A.gf_match[base + best_sel]);
                    post(m, qc, 0, __fadd_rn(funord(top), w), bm);
                }
                continue;
            }
            if constexpr (NK != 1) {
            // one orthogonal value set (anchorer.hpp:2390-2413): piece k; parity 0 = even (shift > q), 1 = odd (shift < q)
            const int t = (int)type - 1, k = t >> 1, par = t & 1;
            const uint32_t* ord_t = A.or_ord + (int64_t)t * A.n_entry + base;
            const unsigned long long* bit_t = A.bit + (int64_t)t * A.n_inner;
            const unsigned lm = __ballot_sync(kFull, wl.sub_ok), rm = __ballot_sync(kFull, wr.sub_ok);
            const unsigned below = (1u << lane) - 1u;
            // nodes on the walks: the node's own element counts if its offset lies below the query's
            {
                const uint32_t oS = lane == 0 ? ld_const<SM>(&A.or_off[base + S0]) : 0xffffffffu;
                const uint32_t ol = wl.node_ok ? ld_const<SM>(&A.or_off[base + wl.node]) : 0xffffffffu;
                const uint32_t orr = wr.node_ok ? ld_const<SM>(&A.or_off[base + wr.node]) : 0xffffffffu;
                const uint32_t vS = lane == 0 ? ld_live<SM>(&ord_t[S0]) : 0u;
                const uint32_t vl = wl.node_ok ? ld_live<SM>(&ord_t[wl.node]) : 0u;
                const uint32_t vr = wr.node_ok ? ld_live<SM>(&ord_t[wr.node]) : 0u;
                if (oS < offset) consider(vS, 0, S0);
                if (ol < offset) consider(vl, walk_key(0, lane, 0), wl.node);
                if (orr < offset) consider(vr, walk_key(1, lane, 0), wr.node);
            }
            // hanging subtrees: Fenwick prefix maximum over the elements with offset below the query's
            const uint32_t* ranks = A.rank_pool ? A.rank_pool + (((q0 * C2 + qc) * 2 + par) * A.rank_stride) : nullptr;
            uint32_t ib2[2] = {0, 0}, cnt2[2] = {0, 0};
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                const WalkStep& ws = side ? wr : wl;
                if (ws.sub_ok) {
                    const int j = side ? __popc(lm) + __popc(rm & below) : __popc(lm & below);
                    ib2[side] = ld_const<SM>(&A.in_base[base + ws.sub]);
                    cnt2[side] = (ranks && j < A.rank_stride) ? ld_const<SM>(&ranks[j])
                                                               : count_less<SM>(A.in_off + ib2[side], ld_const<SM>(&A.in_n[base + ws.sub]), offset);
                }
            }
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                uint32_t c = cnt2[side];
                unsigned long long r = 0;
                while (c) {  // the probe addresses only depend on the count: eight probes in flight
                    unsigned long long x[8];
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) {
                        x[jj] = c ? ld_live<SM>(&bit_t[ib2[side] + c - 1]) : 0ull;
                        c &= c - 1;  // 0 stays 0
                    }
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) r = x[jj] > r ? x[jj] : r;
                }
                if (r) consider((uint32_t)(r >> 32), walk_key(side, lane, 1), (uint32_t)r);
            }
            uint32_t top;
            const int src = warp_argmax(best_hi, best_lo, top);  // first block, in walk order, that attains the maximum value
            if (src < 0) continue;
            if (lane == src) {
                const double eq = __dmul_rn(A.gap_extend[k], (double)q);
                const double pen = __dmul_rn(A.scale, par ? __dadd_rn(A.gap_open[k], eq) : __dsub_rn(A.gap_open[k], eq));
                const float cand = __double2float_rn(__dsub_rn((double)__fadd_rn(funord(top), w), pen));
                post(m, qc, (uint32_t)(1 + t), cand, ld_const<SM>(&A.or_match[base + best_sel]));
            }
            }  // NK != 1
        }
        if (q0 != q1 || pq0 != pq1) barrier();
        pq0 = q0; pq1 = q1;
        i0 = i1; i1 = i2; q0 = q1; q1 = q2;
        ie = ie_next; qe = qe_next;
    }
    if (pq0 != pq1)  // the last step's winners
        apply_winners(pq0, pq1, A.cand_best + ((S + 1) & 1) * A.n_match, A.cand_bp + ((S + 1) & 1) * A.cand_bp_stride);
    if (lane == 0 && n_tree_queries) atomicAdd(A.counters, n_tree_queries);
}

// The gap-free kernel needs fewer registers and runs with 28 warps: a step of a pairwise problem has about twenty work items.
constexpr int kThreadsGapFree = 896;
template <int NK>
__global__ void __launch_bounds__(NK == 1 ? kThreadsGapFree : kThreads, 1) chain_kernel(const __grid_constant__ ChainArgs A) {
    chain_steps<false, NK>(A);
}
typedef void (*ChainKernel)(const ChainArgs);
static ChainKernel chain_kernel_for(int num_pw) {
    return num_pw == 0 ? (ChainKernel)chain_kernel<1> : num_pw == 3 ? (ChainKernel)chain_kernel<7> : (ChainKernel)chain_kernel<0>;
}

// Small problems: one CTA copies the whole arena into shared memory, rebases the pointers, prepares the queries,
// runs the same step loop on shared memory and copies the DP values and back-pointers out again.
__device__ __forceinline__ void chain_small_body(const ChainArgs& G, uint4* arena_smem) {
    const char* gbase = G.arena_base;
    const int64_t ncopy = (G.copy_bytes + 15) / 16, nall = (G.arena_bytes + 15) / 16;
    for (int64_t i = threadIdx.x; i < ncopy; i += kThreads)
        arena_smem[i] = __ldg(reinterpret_cast<const uint4*>(gbase) + i);
    for (int64_t i = ncopy + threadIdx.x; i < nall; i += kThreads) arena_smem[i] = make_uint4(0u, 0u, 0u, 0u);
    ChainArgs A = G;
    char* sbase = reinterpret_cast<char*>(arena_smem);
#define CLB_REBASE(f) A.f = reinterpret_cast<decltype(A.f)>(sbase + (reinterpret_cast<const char*>(G.f) - gbase))
    CLB_REBASE(dp); CLB_REBASE(backptr); CLB_REBASE(sins_off); CLB_REBASE(ins); CLB_REBASE(qry_off); CLB_REBASE(qry_match);
    CLB_REBASE(qrec); CLB_REBASE(weight); CLB_REBASE(qry_chain1); CLB_REBASE(qa1); CLB_REBASE(qa2); CLB_REBASE(qoff);
    CLB_REBASE(pair_grp_off); CLB_REBASE(grp_shift); CLB_REBASE(grp_base); CLB_REBASE(grp_n); CLB_REBASE(pair_base);
    CLB_REBASE(gf_key); CLB_REBASE(gf_match); CLB_REBASE(gf_ord); CLB_REBASE(gf_best); CLB_REBASE(or_shift); CLB_REBASE(or_off);
    CLB_REBASE(or_match); CLB_REBASE(or_ord); CLB_REBASE(in_base); CLB_REBASE(in_n); CLB_REBASE(in_off); CLB_REBASE(bit);
    CLB_REBASE(ent_rank); CLB_REBASE(cand_best); CLB_REBASE(cand_bp); CLB_REBASE(counters);
    if (G.rank_pool) CLB_REBASE(rank_pool);
#undef CLB_REBASE
    __syncthreads();
    prepare_queries<true>(A, threadIdx.x & 31, threadIdx.x >> 5, kWarps);
    __syncthreads();
    chain_steps<true, 0>(A);
    __syncthreads();
    float* const odp = G.out_dp ? G.out_dp : G.dp;
    uint32_t* const obp = G.out_backptr ? G.out_backptr : G.backptr;
    for (int64_t m = threadIdx.x; m < G.n_match; m += kThreads) {
        odp[m] = A.dp[m];
        obp[m] = A.backptr[m];
    }
}

// Small problems: one CTA copies the whole arena into shared memory, rebases the pointers, prepares the queries,
// runs the same step loop on shared memory and copies the DP values and back-pointers out again.
__global__ void __launch_bounds__(kThreads, 1) chain_small_kernel(const ChainArgs G) {
    extern __shared__ uint4 arena_smem[];
    chain_small_body(G, arena_smem);
}

// The same for a batch of independent problems: CTA b solves problem b (clb_chain_dp_batch, clb_chain_jobs_run).  A problem
// whose arena fits shared memory runs there; a larger one runs on its arena in global memory (copy region as staged, zero
// region cleared by the host's memset), its queries prepared by chain_batch_prepare_kernel beforehand.
__global__ void __launch_bounds__(256) chain_batch_prepare_kernel(const ChainArgs* __restrict__ problems) {
    __shared__ ChainArgs G;
    if (threadIdx.x == 0) G = problems[blockIdx.x];
    __syncthreads();
    if (G.arena_bytes <= (int64_t)kChainSmallArena || G.n_qry == 0) return;
    prepare_queries<false>(G, threadIdx.x & 31, threadIdx.x >> 5, blockDim.x >> 5);
}

__global__ void __launch_bounds__(kThreads, 1) chain_small_batch_kernel(const ChainArgs* __restrict__ problems) {
    extern __shared__ uint4 arena_smem[];
    __shared__ ChainArgs G;
    if (threadIdx.x == 0) G = problems[blockIdx.x];
    __syncthreads();
    if (G.arena_bytes <= (int64_t)kChainSmallArena) {
        chain_small_body(G, arena_smem);
        return;
    }
    chain_steps<false, 0>(G);
    __syncthreads();
    for (int64_t m = threadIdx.x; m < G.n_match; m += kThreads) {
        G.out_dp[m] = G.dp[m];
        G.out_backptr[m] = G.backptr[m];
    }
}

// Function attributes belong to the current device, so they are set at every launch (a process may chain on several
// devices); setting one costs a few microseconds of host time.
cudaError_t launch_chain_small_batch(const ChainArgs* d_args, int n, int smem_bytes, bool any_global, cudaStream_t stream) {
    const cudaError_t e0 = cudaFuncSetAttribute(chain_small_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kChainSmallArena);
    if (e0 != cudaSuccess) return e0;
    if (any_global) chain_batch_prepare_kernel<<<n, 256, 0, stream>>>(d_args);
    chain_small_batch_kernel<<<n, kThreads, (size_t)smem_bytes, stream>>>(d_args);
    return cudaGetLastError();
}

// grid == 0: the whole problem fits into shared memory (one CTA).  Otherwise one CTA, or `*cluster` > 1 CTAs of ONE
// thread-block cluster (hardware barrier between the phases of a step), or a cooperative grid of `grid` > 1 CTAs.
// On return *cluster is the cluster size the kernel was launched with (1 without a cluster).
cudaError_t launch_chain(ChainArgs args, int grid, int* cluster_io, int prepare_grid, cudaStream_t stream, cudaEvent_t after_prepare) {
    int cluster = *cluster_io;
    *cluster_io = 1;
    if (grid == 0) {
        const cudaError_t e0 = cudaFuncSetAttribute(chain_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kChainSmallArena);
        if (e0 != cudaSuccess) return e0;
        if (after_prepare) cudaEventRecord(after_prepare, stream);
        chain_small_kernel<<<1, kThreads, (size_t)((args.arena_bytes + 15) / 16 * 16), stream>>>(args);
        return cudaGetLastError();
    }
    if (args.n_qry > 0) chain_prepare_kernel<<<prepare_grid, 256, 0, stream>>>(args);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    if (after_prepare) cudaEventRecord(after_prepare, stream);
    const ChainKernel kern = chain_kernel_for(args.num_pw);
    const int threads = args.num_pw == 0 ? kThreadsGapFree : kThreads;
    if (cluster > 1) {
        // clusters of 16 on the current device; a refusal shows at launch
        cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        cudaGetLastError();
        args.sync_mode = 1;
        for (; cluster > 1; cluster /= 2) {  // a cluster size the device cannot place falls back to the next smaller one
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(cluster);
            cfg.blockDim = dim3(threads);
            cfg.stream = stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = cluster;
            at[0].val.clusterDim.y = 1;
            at[0].val.clusterDim.z = 1;
            cfg.attrs = at;
            cfg.numAttrs = 1;
            e = cudaLaunchKernelEx(&cfg, kern, args);
            if (e == cudaSuccess) {
                *cluster_io = cluster;
                return e;
            }
            cudaGetLastError();
        }
    }
    if (grid > 1) {
        args.sync_mode = 2;
        void* params[] = {(void*)&args};
        return cudaLaunchCooperativeKernel((const void*)kern, dim3(grid), dim3(threads), params, 0, stream);
    }
    args.sync_mode = 0;
    kern<<<1, threads, 0, stream>>>(args);
    return cudaGetLastError();
}

int chain_max_grid(int device) {
    int per_sm = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, chain_kernel<0>, kThreads, 0) != cudaSuccess) return 1;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) return 1;
    return per_sm > 0 ? sms : 1;
}

}  // namespace clb
