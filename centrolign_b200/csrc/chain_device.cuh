// chain_device.cuh -- device-side layout of the sparse anchor-chaining DP (clb_chain_dp).
//
// The reference keeps, per pair of paths (p1, p2) of the two graphs,
//   * one MaxSearchTree per diagonal ("gap-free" trees, keyed (offset on p2, match));
//     reference: include/centrolign/anchorer.hpp:2136-2241, include/centrolign/max_search_tree.hpp
//   * 2*NumPW OrthogonalMaxSearchTrees keyed ((shift, match), offset on p2), all with the same keys;
//     reference: anchorer.hpp:2084-2111, include/centrolign/orthogonal_max_search_tree.hpp
// Both are static in SHAPE (implicit heap layout, filled in key order, max_search_tree.hpp:108-150) and only
// their values move.  Here the same shapes are laid out once, by the host (chain_host.cu) or for large problems by the
// device (chain_layout_kernels.cu), and the value side
// is held in atomically-max-able words so that all updates of one DP step can run in parallel:
//   gap-free tree node x : best[x] = max over the subtree of x of pack(value, ~insertion sequence number)
//                          -- exactly the reference's subtree_max pointer, which moves only on a strictly
//                          greater value and therefore names the EARLIEST inserted maximum
//                          (max_search_tree.hpp:312-358);
//   orthogonal tree node r: a Fenwick tree over the elements of r's subtree sorted by offset, holding
//                          pack(value, outer node index): the reference's cross tree compares
//                          (value, outer index) pairs (orthogonal_max_search_tree.hpp:74), so its range
//                          maxima are unique, and its queries are always prefixes [0, offset)
//                          (anchorer.hpp:2396-2407), which a Fenwick tree over max answers.
// The queries walk the outer trees exactly as the reference's range_max does and take the FIRST block, in
// that walk's order, that attains the maximum (strict '>' replaces, max_search_tree.hpp:361-444,
// orthogonal_max_search_tree.hpp:340-470).
//
// Values are stored as order-preserving 32-bit images of the reference's floats ("ord", 0 = never entered), so
// that zero-filled memory is the initial state and comparisons are integer comparisons.  Everything about a query
// that does not depend on DP values -- its diagonal's tree, the shape of its three tree walks -- is computed for
// all queries at once by a preparation kernel (QueryRec), so that a DP step only has to look at values.
#pragma once
#include <stdint.h>

namespace clb {

constexpr int kChainMaxTrees = 6;            // 2 * NumPW orthogonal value sets
constexpr uint32_t kChainNone = 0xffffffffu;
constexpr int kChainSmallArena = 216 * 1024;   // problems whose whole arena fits run from shared memory

// One tree insertion (a match end on one path pair), in the reference's insertion order; the index of the
// record is the insertion sequence number that breaks ties inside the gap-free trees.
struct InsRec {
    uint32_t match;
    uint32_t gf_base;   // first node of the gap-free tree of its diagonal
    uint32_t gf_node;   // its heap index in that tree
    uint32_t or_base;   // first outer node of the path pair's orthogonal trees
    uint32_t or_node;   // its outer heap index
    int32_t shift;
    uint32_t rank_off;  // ranks in the inner lists of its non-spine ancestors, self first
    uint32_t n_rank;
};

// One (query, path of graph 2) pair.  A tree walk is stored as its split node S and the in-range decisions along
// the one conditional side of the walk (the other side takes every node), LSB first.
struct QueryRec {
    uint32_t match;
    float weight;
    uint32_t offset;    // 0 = nothing on this path reaches the match: no candidates
    int32_t q;          // query shift
    uint32_t gf_base, gf_n;   // gap-free tree of diagonal q, gf_n == 0 if there is none
    uint32_t gf_S, gf_bits;   // prefix walk over keys < offset
    uint32_t or_base, or_n;
    uint32_t ev_S, ev_bits;   // even pieces: shift > q (suffix walk)
    uint32_t or_base2, or_n2; // or_base, or_n again: every kind of work item reads two 16-byte quarters of the record
    uint32_t od_S, od_bits;   // odd pieces:  shift < q (prefix walk)
};

struct ChainArgs {
    int num_pw;
    int n_chain1, n_chain2;
    double scale_ext[3];   // local_scale * gap_extend[k]
    double gap_open[3], gap_extend[3], scale;
    int64_t n_match;
    float* dp;             // [n_match] starts as dp_init
    uint32_t* backptr;     // [n_match] kChainNone = none
    int64_t n_step;
    const int64_t* sins_off;   // [n_step+1] insertions of the step
    const InsRec* ins;
    int64_t n_ins;
    const int64_t* qry_off;    // [n_step+1]
    const uint32_t* qry_match;
    QueryRec* qrec;            // [n_qry * n_chain2]
    int64_t n_qry;
    // raw query data, read by the preparation kernel only
    const float* weight;
    const uint32_t* qry_chain1;
    const int32_t* qa1;
    const int32_t* qa2;
    const uint32_t* qoff;
    const int64_t* pair_grp_off;  // [npair+1] diagonals of the pair, ascending shift
    const int32_t* grp_shift;
    const uint32_t* grp_base;
    const uint32_t* grp_n;
    const uint32_t* pair_base;    // [npair+1] first outer node of the pair
    // gap-free trees
    const uint32_t* gf_key;       // [n_entry] offset key, heap layout per tree
    const uint32_t* gf_match;     // [n_entry]
    uint32_t* gf_ord;             // [n_entry] value of the node
    unsigned long long* gf_best;  // [n_entry] subtree maximum
    // orthogonal trees
    const int32_t* or_shift;      // [n_entry] heap layout per pair
    const uint32_t* or_off;
    const uint32_t* or_match;
    uint32_t* or_ord;             // [2*num_pw][n_entry]
    const uint32_t* in_base;      // [n_entry] per outer node: first slot of its inner list, kChainNone on the outer spines
    const uint32_t* in_n;
    const uint32_t* in_off;       // [n_inner] offsets of the inner lists, ascending
    unsigned long long* bit;      // [2*num_pw][n_inner] Fenwick trees over max
    const uint32_t* ent_rank;     // [n_inner]
    int64_t n_inner;
    int64_t n_entry;
    // per-step candidate exchange
    unsigned long long* cand_best;  // [2][n_match] by step parity: pack(value, ~order), 0 = none
    uint32_t* cand_bp;              // [2][cand_bp_stride] by step parity, cand_bp_stride = max queries per step * n_chain2 * (2*num_pw+1)
    int64_t cand_bp_stride;
    unsigned long long* counters;   // [0] tree queries answered
    // ranks of the subtree blocks of every orthogonal walk, computed by the preparation kernel: per (query, chain2,
    // parity) rank_stride words, one per subtree block in walk order; nullptr = computed on the fly
    uint32_t* rank_pool;
    int rank_stride;
    const char* arena_base;  // the arena all pointers above point into, and its size
    int64_t arena_bytes;
    int64_t copy_bytes;      // shared-memory kernels: this many bytes are copied from arena_base, the rest of the arena starts as zero
    float* out_dp;           // batched launch: compact result arrays of the problem (nullptr: results go back into dp / backptr)
    uint32_t* out_backptr;
    int sync_mode;     // how the phases of a step are separated: 0 one CTA (__syncthreads), 1 one thread-block cluster
                       // (barrier.cluster), 2 cooperative grid (grid.sync)
};

// ---------------------------------------------------------------------------------------------------------------------
// Shapes of the implicit heaps, shared by the host layout (chain_host.cu) and the device layout (chain_layout_kernels.cu).
// An n-node heap is a complete binary tree: levels full except the last, which is filled from the left.  Every subtree
// of it is again such a tree.

#ifdef __CUDA_ARCH__
#define CLB_CLZ(x) __clz(x)
#else
#define CLB_CLZ(x) __builtin_clz(x)
#endif

// depth of heap node h (< 2^32 - 1)
__host__ __device__ inline int heap_depth(uint32_t h) { return 31 - CLB_CLZ(h + 1); }

// nodes of the left subtree of the root of an m-node heap
__host__ __device__ inline uint32_t heap_left_size(uint32_t m) {
    if (m <= 1) return 0;
    const int hgt = 31 - CLB_CLZ(m);  // the root's height: levels 0..hgt
    const uint32_t half = 1u << (hgt - 1);
    const uint32_t last = m - ((1u << hgt) - 1);  // nodes on the last level, 1 .. 2^hgt
    return half - 1 + (last < half ? last : half);
}

// the heap index of in-order position k of an n-node heap: the node the reference's in-order fill
// (max_search_tree.hpp:119-150) gives the k-th smallest key; a descent from the root over the subtree sizes
__host__ __device__ inline uint32_t heap_of_inorder(uint32_t k, uint32_t n) {
    uint32_t h = 0, m = n;
    for (;;) {
        const uint32_t ls = heap_left_size(m);
        if (k == ls) return h;
        if (k < ls) {
            h = 2 * h + 1;
            m = ls;
        } else {
            k -= ls + 1;
            h = 2 * h + 2;
            m -= ls + 1;
        }
    }
}

// the two outer spines of an orthogonal tree carry no inner list (orthogonal_max_search_tree.hpp:175-182)
__host__ __device__ inline bool heap_on_spine(uint32_t h) {
    const uint64_t a = (uint64_t)h + 1, b = (uint64_t)h + 2;
    return (a & (a - 1)) == 0 || (b & (b - 1)) == 0;
}

// nodes in the subtree of heap node h of an n-node heap (h < n)
__host__ __device__ inline uint32_t heap_subtree_size(uint32_t h, uint32_t n) {
    const int d = heap_depth(h), H = heap_depth(n - 1);
    const uint64_t w = uint64_t(1) << (H - d);               // width of the subtree's last level
    const uint64_t first = ((uint64_t)h + 1) * w - 1;        // its first heap index there
    const uint64_t present = n > first ? (n - first < w ? n - first : w) : 0;
    return (uint32_t)(w - 1 + present);
}

// non-spine nodes on the path from the root to h, h included: the inner lists h is an element of.  At depth d with
// level position t, the ancestor at depth j is on the left spine iff t >> (d - j) == 0 and on the right spine iff it is
// all ones, so the path leaves the spines min(bit length of t, bit length of its complement) levels above h.
__host__ __device__ inline uint32_t heap_nanc(uint32_t h) {
    const int d = heap_depth(h);
    if (d == 0) return 0;
    const uint32_t t = h + 1 - (1u << d), u = ((1u << d) - 1) ^ t;
    const uint32_t bt = t ? 32 - CLB_CLZ(t) : 0, bu = u ? 32 - CLB_CLZ(u) : 0;
    return bt < bu ? bt : bu;
}

// ---------------------------------------------------------------------------------------------------------------------
// Device layout (chain_layout_kernels.cu): the tables chain_host.cu's host layout builds, built by kernels straight into
// the copy region of the call's arena.  Phase 1 (chain_layout_sort) uploads the caller's raw entry and step arrays into
// a scratch buffer, builds the per-entry tables and sorts the entries; its one read-back is the number of gap-free trees,
// which the arena plan needs.  Phase 2 (chain_layout_build) writes every laid-out table.

struct ChainLayoutDims {
    int64_t M, S, E, n_end, npair;
    int C2, P;
    int max_depth;    // depth of the deepest orthogonal node: floor(log2(largest tree))
    bool has_active;  // the problem has an ins_active array
};

// destinations in the arena (device pointers); the orthogonal ones are unused when P == 0
struct ChainLayoutOut {
    int64_t* sins_live;
    InsRec* ins;
    int64_t* qry_live;
    int64_t* pair_grp_off;
    int32_t* grp_shift;
    uint32_t* grp_base;
    uint32_t* grp_n;
    uint32_t* pair_base;
    uint32_t* gf_key;
    uint32_t* gf_match;
    int32_t* or_shift;
    uint32_t* or_off;
    uint32_t* or_match;
    uint32_t* in_base;
    uint32_t* in_n;
    uint32_t* in_off;
    uint32_t* ent_rank;
};

// the caller's raw arrays the layout reads (host pointers)
struct ChainLayoutIn {
    const int64_t* ins_off;
    const uint32_t *ins_p1, *ins_p2;
    const int32_t* ins_shift;
    const uint32_t* ins_offset;
    const uint8_t* ins_active;  // may be null: every entry active
    const int64_t* end_off;
    const uint32_t* end_match;
    const int64_t* qry_off;
};

}  // namespace clb
