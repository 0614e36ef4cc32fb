// chain_layout_kernels.cu -- the search structures of one chaining problem laid out on the device (see the device-layout
// section of chain_device.cuh).  The tables are exactly those of the host layout in chain_host.cu, array for array and
// byte for byte: CLB_CHAIN_LAYOUT=check builds both and compares them.
//
//   * per-entry tables: entry -> match and entry -> path pair, and the active entries of every match;
//   * the insertion list: for every step the active entries of the matches ending there, in end_match order (prefix sums
//     over the end slots give the positions), and the steps in which something happens;
//   * two stable radix sorts: gap-free order (pair, shift, offset, match) and orthogonal order (pair, shift, match).
//     Entries are numbered in match order, so a stable sort that starts from entry order breaks the remaining ties by
//     match exactly as the host's 128-bit keys do;
//   * gap-free trees: group heads, sizes and the heap index of every entry (heap_of_inorder);
//   * orthogonal trees: heap placement, inner-list sizes and bases (a prefix sum in pair, heap order), rank offsets
//     (a prefix sum in entry order) and the inner lists themselves, one launch per tree level from the deepest up.
//     The list of node x is its subtree's elements ordered by (offset, in-order position), which is the host merge's
//     tie rule (left subtree < x < right subtree).  An element's slot in x's list is its slot in its child's list, plus
//     the elements of the sibling list and x itself that precede it, counted by binary search in the sibling list.
// CUB (the toolkit's CCCL) supplies the generic sorts and scans; the tree kernels are ours.
#include <cub/cub.cuh>

#include <algorithm>

#include "chain_device.cuh"

namespace clb {
namespace {

constexpr int kThreads = 256;

#define LAYOUT_LOOP(i, n) for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < (n); i += (int64_t)gridDim.x * blockDim.x)

template <class K, class... A>
cudaError_t run(int64_t n, cudaStream_t st, K kernel, A... args) {
    if (n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((n + kThreads - 1) / kThreads, 148 * 16);
    kernel<<<grid, kThreads, 0, st>>>(n, args...);
    return cudaGetLastError();
}

#define TRY(x)                                   \
    do {                                         \
        const cudaError_t e_ = (x);              \
        if (e_ != cudaSuccess) return e_;        \
    } while (0)

// scratch buffer carve-up; with base == 0 it only measures
struct Scratch {
    int64_t *ins_off, *end_off, *qry_off, *end_cnt, *end_pos;
    uint32_t *p1, *p2, *offset, *end_match, *ent_match, *ent_pair, *act_cnt, *step_flag, *step_pos;
    int32_t* shift;
    uint8_t* active;
    uint32_t *key32_in, *key32_out, *iota, *vals_tmp, *gf_ord, *or_ord, *flag, *gid, *grp_pair;
    uint32_t *ent_gf_grp, *ent_gf_node, *ent_or_node, *nd_e;
    uint64_t *hi, *hi_perm, *hi_sorted, *or_keys, *in_n64, *in_base64, *nanc64, *rank_off64;
    void* cub;
    size_t cub_bytes, total;
};

int hi_bits(const ChainLayoutDims& d) {
    int b = 0;
    while (b < 31 && (int64_t(1) << b) < d.npair) ++b;
    return 32 + b;
}

cudaError_t cub_bytes_needed(const ChainLayoutDims& d, size_t* out) {
    size_t m = 0, b = 0;
    const int64_t n = std::max<int64_t>(d.E, 1);
    TRY(cub::DeviceRadixSort::SortPairs(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr, n));
    m = std::max(m, b);
    TRY(cub::DeviceRadixSort::SortPairs(nullptr, b, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr, (uint32_t*)nullptr, n));
    m = std::max(m, b);
    TRY(cub::DeviceScan::InclusiveSum(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, n));
    m = std::max(m, b);
    const int64_t ns = std::max<int64_t>({n, d.n_end + 1, d.S + 1});
    TRY(cub::DeviceScan::ExclusiveSum(nullptr, b, (const uint64_t*)nullptr, (uint64_t*)nullptr, ns));
    m = std::max(m, b);
    TRY(cub::DeviceScan::ExclusiveSum(nullptr, b, (const int64_t*)nullptr, (int64_t*)nullptr, ns));
    m = std::max(m, b);
    TRY(cub::DeviceScan::ExclusiveSum(nullptr, b, (const uint32_t*)nullptr, (uint32_t*)nullptr, ns));
    m = std::max(m, b);
    *out = m;
    return cudaSuccess;
}

Scratch carve(const ChainLayoutDims& d, char* base, size_t cub_bytes) {
    Scratch s{};
    size_t off = 0;
    auto take = [&](auto*& ptr, int64_t n) {
        using T = std::remove_reference_t<decltype(*ptr)>;
        ptr = reinterpret_cast<T*>(base + off);
        off = (off + (size_t)std::max<int64_t>(n, 1) * sizeof(T) + 255) & ~size_t(255);
    };
    const int64_t E = d.E, Eo = d.P > 0 ? d.E : 0;
    take(s.ins_off, d.M + 1); take(s.end_off, d.S + 1); take(s.qry_off, d.S + 1);
    take(s.end_cnt, d.n_end + 1); take(s.end_pos, d.n_end + 1);
    take(s.p1, E); take(s.p2, E); take(s.offset, E); take(s.shift, E); take(s.active, d.has_active ? E : 0);
    take(s.end_match, d.n_end); take(s.ent_match, E); take(s.ent_pair, E); take(s.act_cnt, d.M);
    take(s.step_flag, d.S + 1); take(s.step_pos, d.S + 1);
    take(s.key32_in, E); take(s.key32_out, E); take(s.iota, E); take(s.vals_tmp, E); take(s.gf_ord, E);
    take(s.flag, E); take(s.gid, E); take(s.grp_pair, E); take(s.ent_gf_grp, E); take(s.ent_gf_node, E);
    take(s.hi, E); take(s.hi_perm, E); take(s.hi_sorted, E);
    take(s.or_ord, Eo); take(s.or_keys, Eo); take(s.ent_or_node, Eo); take(s.nd_e, Eo);
    take(s.in_n64, Eo); take(s.in_base64, Eo); take(s.nanc64, Eo); take(s.rank_off64, Eo);
    char* c = nullptr;
    take(c, (int64_t)cub_bytes);
    s.cub = c;
    s.cub_bytes = cub_bytes;
    s.total = off;
    return s;
}

// ------------------------------------------------------------- kernels -------------------------------------------------------------

// entry -> match, entry -> pair, active entries per match
__global__ void k_match_entries(int64_t M, const int64_t* ins_off, const uint32_t* p1, const uint32_t* p2, const uint8_t* active, int C2,
                                uint32_t* ent_match, uint32_t* ent_pair, uint32_t* act_cnt) {
    LAYOUT_LOOP(m, M) {
        uint32_t cnt = 0;
        for (int64_t e = ins_off[m]; e < ins_off[m + 1]; ++e) {
            ent_match[e] = (uint32_t)m;
            ent_pair[e] = p1[e] * (uint32_t)C2 + p2[e];
            cnt += active ? (active[e] != 0) : 1u;
        }
        act_cnt[m] = cnt;
    }
}

__global__ void k_entry_keys(int64_t E, const uint32_t* offset, const int32_t* shift, const uint32_t* ent_pair, uint32_t* key32, uint32_t* iota,
                             uint64_t* hi) {
    LAYOUT_LOOP(e, E) {
        key32[e] = offset[e];
        iota[e] = (uint32_t)e;
        hi[e] = ((uint64_t)ent_pair[e] << 32) | ((uint32_t)shift[e] ^ 0x80000000u);
    }
}

__global__ void k_gather_hi(int64_t E, const uint32_t* perm, const uint64_t* hi, uint64_t* out) {
    LAYOUT_LOOP(i, E) out[i] = hi[perm[i]];
}

__global__ void k_group_flags(int64_t E, const uint64_t* sorted, uint32_t* flag) {
    LAYOUT_LOOP(i, E) flag[i] = i == 0 || sorted[i] != sorted[i - 1];
}

// active insertions of every end slot (slots before end_off[0] belong to no step)
__global__ void k_end_counts(int64_t n, int64_t n_end, const int64_t* end_off, const uint32_t* end_match, const uint32_t* act_cnt, int64_t* cnt) {
    LAYOUT_LOOP(k, n) cnt[k] = (k < n_end && k >= end_off[0]) ? (int64_t)act_cnt[end_match[k]] : 0;
}

// steps in which something happens (chain_host.cu: the device walks only those)
__global__ void k_step_flags(int64_t n, int64_t S, const int64_t* end_off, const int64_t* end_pos, const int64_t* qry_off, uint32_t* flag) {
    LAYOUT_LOOP(s, n) flag[s] = s < S && (end_pos[end_off[s + 1]] != end_pos[end_off[s]] || qry_off[s + 1] != qry_off[s]);
}

__global__ void k_step_live(int64_t n, int64_t S, const int64_t* end_off, const int64_t* end_pos, const int64_t* qry_off, const uint32_t* flag,
                            const uint32_t* pos, int64_t* sins_live, int64_t* qry_live) {
    LAYOUT_LOOP(s, n) {
        if (s == 0) {
            sins_live[0] = 0;
            qry_live[0] = qry_off[0];
        }
        if (s < S && flag[s]) {
            const uint32_t j = pos[s] + 1;
            sins_live[j] = end_pos[end_off[s + 1]];
            qry_live[j] = qry_off[s + 1];
        }
    }
}

// insertion records in the reference's order
__global__ void k_ins(int64_t n_end, const int64_t* end_off, const uint32_t* end_match, const int64_t* end_pos, const int64_t* ins_off,
                      const uint8_t* active, const int32_t* shift, const uint32_t* ent_pair, const uint32_t* ent_gf_grp, const uint32_t* ent_gf_node,
                      const uint32_t* grp_base, const uint32_t* pair_base, const uint32_t* ent_or_node, const uint64_t* rank_off64,
                      const uint64_t* nanc64, int P, InsRec* ins) {
    LAYOUT_LOOP(k, n_end) {
        if (k < end_off[0]) continue;
        const uint32_t m = end_match[k];
        int64_t pos = end_pos[k];
        for (int64_t e = ins_off[m]; e < ins_off[m + 1]; ++e) {
            if (active && !active[e]) continue;
            InsRec r;
            r.match = m;
            r.gf_base = grp_base[ent_gf_grp[e]];
            r.gf_node = ent_gf_node[e];
            r.or_base = P > 0 ? pair_base[ent_pair[e]] : 0;
            r.or_node = P > 0 ? ent_or_node[e] : 0;
            r.shift = shift[e];
            r.rank_off = P > 0 ? (uint32_t)rank_off64[e] : 0;
            r.n_rank = P > 0 ? (uint32_t)nanc64[e] : 0;
            ins[pos++] = r;
        }
    }
}

__global__ void k_group_heads(int64_t E, const uint32_t* flag, const uint32_t* gid, const uint32_t* gf_ord, const uint64_t* hi_sorted,
                              const int32_t* shift, uint32_t* grp_base, int32_t* grp_shift, uint32_t* grp_pair) {
    LAYOUT_LOOP(i, E) {
        if (!flag[i]) continue;
        const uint32_t g = gid[i] - 1;
        grp_base[g] = (uint32_t)i;
        grp_shift[g] = shift[gf_ord[i]];
        grp_pair[g] = (uint32_t)(hi_sorted[i] >> 32);
    }
}

__global__ void k_group_n(int64_t G, int64_t E, const uint32_t* grp_base, uint32_t* grp_n) {
    LAYOUT_LOOP(g, G) grp_n[g] = (uint32_t)((g + 1 < G ? (int64_t)grp_base[g + 1] : E) - grp_base[g]);
}

// first group / first outer node of every pair (pair npair: the totals)
__global__ void k_pair_offsets(int64_t n, int64_t G, const uint32_t* grp_pair, int64_t E, const uint64_t* or_keys, int64_t* pair_grp_off,
                               uint32_t* pair_base) {
    LAYOUT_LOOP(pr, n) {
        int64_t lo = 0, hi = G;
        while (lo < hi) {
            const int64_t mid = (lo + hi) / 2;
            if (grp_pair[mid] < (uint64_t)pr) lo = mid + 1;
            else hi = mid;
        }
        pair_grp_off[pr] = lo;
        if (pair_base) {
            lo = 0, hi = E;
            while (lo < hi) {
                const int64_t mid = (lo + hi) / 2;
                if ((or_keys[mid] >> 32) < (uint64_t)pr) lo = mid + 1;
                else hi = mid;
            }
            pair_base[pr] = (uint32_t)lo;
        }
    }
}

__global__ void k_gf_place(int64_t E, const uint32_t* gf_ord, const uint32_t* gid, const uint32_t* grp_base, const uint32_t* grp_n,
                           const uint32_t* offset, const uint32_t* ent_match, uint32_t* gf_key, uint32_t* gf_match, uint32_t* ent_gf_grp,
                           uint32_t* ent_gf_node) {
    LAYOUT_LOOP(i, E) {
        const uint32_t e = gf_ord[i], g = gid[i] - 1, b = grp_base[g];
        const uint32_t h = heap_of_inorder((uint32_t)(i - b), grp_n[g]);
        gf_key[b + h] = offset[e];
        gf_match[b + h] = ent_match[e];
        ent_gf_grp[e] = g;
        ent_gf_node[e] = h;
    }
}

__global__ void k_or_place(int64_t E, const uint32_t* or_ord, const uint64_t* or_keys, const uint32_t* pair_base, const int32_t* shift,
                           const uint32_t* offset, const uint32_t* ent_match, int32_t* or_shift, uint32_t* or_off, uint32_t* or_match,
                           uint32_t* in_n, uint32_t* ent_or_node, uint32_t* nd_e, uint64_t* in_n64, uint64_t* nanc64) {
    LAYOUT_LOOP(i, E) {
        const uint32_t e = or_ord[i], pr = (uint32_t)(or_keys[i] >> 32), ob = pair_base[pr], n = pair_base[pr + 1] - ob;
        const uint32_t h = heap_of_inorder((uint32_t)(i - ob), n), j = ob + h;
        or_shift[j] = shift[e];
        or_off[j] = offset[e];
        or_match[j] = ent_match[e];
        const uint32_t sz = heap_on_spine(h) ? 0 : heap_subtree_size(h, n);
        in_n[j] = sz;
        in_n64[j] = sz;
        ent_or_node[e] = h;
        nd_e[j] = e;
        nanc64[e] = heap_nanc(h);
    }
}

__global__ void k_in_base(int64_t E, const uint32_t* in_n, const uint64_t* in_base64, uint32_t* in_base) {
    LAYOUT_LOOP(j, E) in_base[j] = in_n[j] ? (uint32_t)in_base64[j] : kChainNone;
}

// elements of a sorted list below v (or_equal: at most v)
__device__ inline uint32_t count_below(const uint32_t* a, uint32_t n, uint32_t v, bool or_equal) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) / 2;
        const uint32_t x = a[mid];
        if (x < v || (or_equal && x == v)) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// the inner lists of the non-spine nodes of depth d: every element of their subtrees finds its slot
__global__ void k_inner_level(int64_t E, int d, const uint32_t* nd_e, const uint32_t* ent_pair, const uint32_t* pair_base, const uint32_t* or_off,
                              const uint32_t* in_base, const uint32_t* in_n, const uint64_t* rank_off64, uint32_t* in_off, uint32_t* ent_rank) {
    LAYOUT_LOOP(j, E) {
        const uint32_t e = nd_e[j], pr = ent_pair[e], ob = pair_base[pr], n = pair_base[pr + 1] - ob, h = (uint32_t)j - ob;
        const int dy = heap_depth(h);
        if (dy < d) continue;
        const uint32_t x = (uint32_t)((((uint64_t)h + 1) >> (dy - d)) - 1);
        const uint32_t xb = in_base[ob + x];
        if (xb == kChainNone) continue;  // spine: no list
        const uint32_t oy = or_off[j];
        auto below = [&](uint64_t c, bool or_equal) -> uint32_t {  // elements of child c's list before oy
            if (c >= n) return 0;
            return count_below(in_off + in_base[ob + c], in_n[ob + c], oy, or_equal);
        };
        const uint64_t l = 2 * (uint64_t)x + 1, r = l + 1;
        const uint64_t ro = rank_off64[e];
        uint32_t slot;
        if (dy == d) {
            slot = below(l, true) + below(r, false);  // left subtree < x < right subtree on equal offsets
        } else {
            const uint64_t c = (((uint64_t)h + 1) >> (dy - d - 1)) - 1;
            const uint32_t rank_in_child = ent_rank[ro + (dy - d - 1)];
            const uint32_t ox = or_off[ob + x];
            if (c == l) slot = rank_in_child + below(r, false) + (ox < oy ? 1u : 0u);
            else slot = rank_in_child + below(l, true) + (ox <= oy ? 1u : 0u);
        }
        in_off[xb + slot] = oy;
        ent_rank[ro + (dy - d)] = slot;
    }
}

template <class T>
cudaError_t up(T* dst, const T* src, int64_t n, cudaStream_t st, int64_t* h2d) {
    if (n <= 0) return cudaSuccess;
    *h2d += n * (int64_t)sizeof(T);
    return cudaMemcpyAsync(dst, src, (size_t)n * sizeof(T), cudaMemcpyHostToDevice, st);
}

}  // namespace

cudaError_t chain_layout_scratch_bytes(const ChainLayoutDims& d, size_t* bytes) {
    size_t cb = 0;
    TRY(cub_bytes_needed(d, &cb));
    *bytes = carve(d, nullptr, cb).total;
    return cudaSuccess;
}

// Phase 1: upload, per-entry tables, both sorts, gap-free group ids.  Synchronises the stream: *n_groups is read back.
cudaError_t chain_layout_sort(const ChainLayoutIn& in, const ChainLayoutDims& d, char* scratch, cudaStream_t st, int64_t* n_groups,
                              int64_t* h2d_bytes) {
    size_t cb = 0;
    TRY(cub_bytes_needed(d, &cb));
    const Scratch s = carve(d, scratch, cb);
    const int64_t E = d.E;
    TRY(up(s.ins_off, in.ins_off, d.M + 1, st, h2d_bytes));
    TRY(up(s.end_off, in.end_off, d.S + 1, st, h2d_bytes));
    TRY(up(s.qry_off, in.qry_off, d.S + 1, st, h2d_bytes));
    TRY(up(s.end_match, in.end_match, d.n_end, st, h2d_bytes));
    TRY(up(s.p1, in.ins_p1, E, st, h2d_bytes));
    TRY(up(s.p2, in.ins_p2, E, st, h2d_bytes));
    TRY(up(s.shift, in.ins_shift, E, st, h2d_bytes));
    TRY(up(s.offset, in.ins_offset, E, st, h2d_bytes));
    if (d.has_active) TRY(up(s.active, in.ins_active, E, st, h2d_bytes));
    TRY(run(d.M, st, k_match_entries, (const int64_t*)s.ins_off, (const uint32_t*)s.p1, (const uint32_t*)s.p2,
            (const uint8_t*)(d.has_active ? s.active : nullptr), d.C2, s.ent_match, s.ent_pair, s.act_cnt));
    *n_groups = 0;
    if (E == 0) return cudaStreamSynchronize(st);
    TRY(run(E, st, k_entry_keys, (const uint32_t*)s.offset, (const int32_t*)s.shift, (const uint32_t*)s.ent_pair, s.key32_in, s.iota, s.hi));
    const int hb = hi_bits(d);
    size_t tb = s.cub_bytes;
    // gap-free order: by offset, then stably by (pair, shift)
    TRY(cub::DeviceRadixSort::SortPairs(s.cub, tb, (const uint32_t*)s.key32_in, s.key32_out, (const uint32_t*)s.iota, s.vals_tmp, E, 0, 32, st));
    TRY(run(E, st, k_gather_hi, (const uint32_t*)s.vals_tmp, (const uint64_t*)s.hi, s.hi_perm));
    tb = s.cub_bytes;
    TRY(cub::DeviceRadixSort::SortPairs(s.cub, tb, (const uint64_t*)s.hi_perm, s.hi_sorted, (const uint32_t*)s.vals_tmp, s.gf_ord, E, 0, hb, st));
    if (d.P > 0) {  // orthogonal order: stably by (pair, shift) from entry order
        tb = s.cub_bytes;
        TRY(cub::DeviceRadixSort::SortPairs(s.cub, tb, (const uint64_t*)s.hi, s.or_keys, (const uint32_t*)s.iota, s.or_ord, E, 0, hb, st));
    }
    TRY(run(E, st, k_group_flags, (const uint64_t*)s.hi_sorted, s.flag));
    tb = s.cub_bytes;
    TRY(cub::DeviceScan::InclusiveSum(s.cub, tb, (const uint32_t*)s.flag, s.gid, E, st));
    uint32_t g = 0;
    TRY(cudaMemcpyAsync(&g, s.gid + (E - 1), sizeof(g), cudaMemcpyDeviceToHost, st));
    TRY(cudaStreamSynchronize(st));
    *n_groups = g;
    return cudaSuccess;
}

// Phase 2: every laid-out table, into the arena.  Synchronises the stream; *n_inner is the inner-slot total the device
// counted (the caller compares it with its own).
cudaError_t chain_layout_build(const ChainLayoutDims& d, int64_t G, char* scratch, const ChainLayoutOut& o, cudaStream_t st, int64_t* n_inner) {
    size_t cb = 0;
    TRY(cub_bytes_needed(d, &cb));
    const Scratch s = carve(d, scratch, cb);
    const int64_t E = d.E, S = d.S;
    size_t tb;
    // steps and insertion positions
    TRY(run(d.n_end + 1, st, k_end_counts, d.n_end, (const int64_t*)s.end_off, (const uint32_t*)s.end_match, (const uint32_t*)s.act_cnt, s.end_cnt));
    tb = s.cub_bytes;
    TRY(cub::DeviceScan::ExclusiveSum(s.cub, tb, (const int64_t*)s.end_cnt, s.end_pos, d.n_end + 1, st));
    TRY(run(S + 1, st, k_step_flags, S, (const int64_t*)s.end_off, (const int64_t*)s.end_pos, (const int64_t*)s.qry_off, s.step_flag));
    tb = s.cub_bytes;
    TRY(cub::DeviceScan::ExclusiveSum(s.cub, tb, (const uint32_t*)s.step_flag, s.step_pos, S + 1, st));
    TRY(run(S + 1, st, k_step_live, S, (const int64_t*)s.end_off, (const int64_t*)s.end_pos, (const int64_t*)s.qry_off, (const uint32_t*)s.step_flag,
            (const uint32_t*)s.step_pos, o.sins_live, o.qry_live));
    // gap-free trees
    TRY(run(E, st, k_group_heads, (const uint32_t*)s.flag, (const uint32_t*)s.gid, (const uint32_t*)s.gf_ord, (const uint64_t*)s.hi_sorted,
            (const int32_t*)s.shift, o.grp_base, o.grp_shift, s.grp_pair));
    TRY(run(G, st, k_group_n, E, (const uint32_t*)o.grp_base, o.grp_n));
    if (d.P == 0) TRY(cudaMemsetAsync(o.pair_base, 0, (size_t)(d.npair + 1) * sizeof(uint32_t), st));
    TRY(run(d.npair + 1, st, k_pair_offsets, G, (const uint32_t*)s.grp_pair, E, (const uint64_t*)s.or_keys, o.pair_grp_off,
            d.P > 0 ? o.pair_base : (uint32_t*)nullptr));
    TRY(run(E, st, k_gf_place, (const uint32_t*)s.gf_ord, (const uint32_t*)s.gid, (const uint32_t*)o.grp_base, (const uint32_t*)o.grp_n,
            (const uint32_t*)s.offset, (const uint32_t*)s.ent_match, o.gf_key, o.gf_match, s.ent_gf_grp, s.ent_gf_node));
    // orthogonal trees
    *n_inner = 0;
    uint64_t tail[4] = {0, 0, 0, 0};
    if (d.P > 0 && E > 0) {
        TRY(run(E, st, k_or_place, (const uint32_t*)s.or_ord, (const uint64_t*)s.or_keys, (const uint32_t*)o.pair_base, (const int32_t*)s.shift,
                (const uint32_t*)s.offset, (const uint32_t*)s.ent_match, o.or_shift, o.or_off, o.or_match, o.in_n, s.ent_or_node, s.nd_e, s.in_n64,
                s.nanc64));
        tb = s.cub_bytes;
        TRY(cub::DeviceScan::ExclusiveSum(s.cub, tb, (const uint64_t*)s.in_n64, s.in_base64, E, st));
        tb = s.cub_bytes;
        TRY(cub::DeviceScan::ExclusiveSum(s.cub, tb, (const uint64_t*)s.nanc64, s.rank_off64, E, st));
        TRY(run(E, st, k_in_base, (const uint32_t*)o.in_n, (const uint64_t*)s.in_base64, o.in_base));
        for (int lev = d.max_depth; lev >= 2; --lev)  // depths 0 and 1 are spine only
            TRY(run(E, st, k_inner_level, lev, (const uint32_t*)s.nd_e, (const uint32_t*)s.ent_pair, (const uint32_t*)o.pair_base,
                    (const uint32_t*)o.or_off, (const uint32_t*)o.in_base, (const uint32_t*)o.in_n, (const uint64_t*)s.rank_off64, o.in_off,
                    o.ent_rank));
        TRY(cudaMemcpyAsync(&tail[0], s.in_base64 + (E - 1), 8, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(&tail[1], s.in_n64 + (E - 1), 8, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(&tail[2], s.rank_off64 + (E - 1), 8, cudaMemcpyDeviceToHost, st));
        TRY(cudaMemcpyAsync(&tail[3], s.nanc64 + (E - 1), 8, cudaMemcpyDeviceToHost, st));
    }
    TRY(run(d.n_end, st, k_ins, (const int64_t*)s.end_off, (const uint32_t*)s.end_match, (const int64_t*)s.end_pos, (const int64_t*)s.ins_off,
            (const uint8_t*)(d.has_active ? s.active : nullptr), (const int32_t*)s.shift, (const uint32_t*)s.ent_pair, (const uint32_t*)s.ent_gf_grp,
            (const uint32_t*)s.ent_gf_node, (const uint32_t*)o.grp_base, (const uint32_t*)o.pair_base, (const uint32_t*)s.ent_or_node,
            (const uint64_t*)s.rank_off64, (const uint64_t*)s.nanc64, d.P, o.ins));
    TRY(cudaStreamSynchronize(st));
    if (d.P > 0 && E > 0) *n_inner = tail[0] + tail[1] == tail[2] + tail[3] ? (int64_t)(tail[0] + tail[1]) : -1;
    return cudaSuccess;
}

}  // namespace clb
