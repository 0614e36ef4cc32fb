// integration/shadow/centrolign/anchorer.hpp -- zero-edit drop-in of the B200 chaining DP into the reference.
//
// With `integration/shadow` BEFORE the reference's include directory, every `#include "centrolign/anchorer.hpp"`
// lands here.  The untouched reference header is read first (#include_next); then the two member templates that
// hold the chaining DP are given EXPLICIT SPECIALIZATIONS for exactly the production instantiation that
// Anchorer::anchor_chain selects (reference: include/centrolign/anchorer.hpp:1271-1278 and :1286-1291, with
// BGraph = BaseGraph, XMerge = PathMerge<uint32_t, uint8_t> as chosen by Core, include/centrolign/core.hpp:336-338,
// and NumPW = 3).  Name lookup in the reference's own `_gen_sparse_affine` / `_gen_sparse` calls then picks the
// specializations: same signature, same call sites, no reference line edited.  The bit-packed instantiation that
// restrain_memory selects (:1263-1264) is specialized the same way; the 64-bit variants keep the reference's generic code.
//
// The specializations build what the reference builds before its main loop (MatchBank, forward edges,
// post-switch distances, topological order -- the reference's own classes), hand the flat problem to
// clb_chain_dp through centrolign_b200/hostcpp/chain_b200.hpp, and turn the returned match ranks into anchor_t
// records exactly as Anchorer::traceback_sparse_dp (:2506-2536) and the annotation loop (:2443-2468) do.
#ifndef CENTROLIGN_B200_SHADOW_ANCHORER_HPP
#define CENTROLIGN_B200_SHADOW_ANCHORER_HPP

#include_next "centrolign/anchorer.hpp"

#include "centrolign/chain_merge.hpp"
#include "centrolign/forward_edges.hpp"
#include "centrolign/match_bank.hpp"
#include "centrolign/packed_forward_edges.hpp"
#include "centrolign/packed_match_bank.hpp"
#include "centrolign/packed_vector.hpp"
#include "centrolign/vector_support.hpp"
#include "centrolign/path_merge.hpp"
#include "centrolign/post_switch_distances.hpp"
#include "centrolign/topological_order.hpp"

#include "chain_b200.hpp"

#include <chrono>
#include <cstdio>
#include <cstdlib>

namespace centrolign {
namespace b200_chain {

inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

typedef PathMerge<uint32_t, uint8_t> XMerge;
typedef MatchBank<uint32_t, uint16_t, float> Bank;
typedef ForwardEdges<XMerge::node_id_t, XMerge::chain_id_t> FwdEdges;
typedef std::vector<std::pair<int32_t, Bank::match_id_t>> ShiftMatchVector;
typedef std::vector<std::pair<uint32_t, Bank::match_id_t>> DistMatchVector;
// the bit-packed containers of restrain_memory (anchorer.hpp:1236-1248)
typedef PackedMatchBank<uint32_t, float> PackedBank;
typedef VectorPair<SignedPackedVector, PackedVector, int32_t, PackedBank::match_id_t> PackedShiftMatchVector;
typedef VectorPair<PackedVector, PackedVector, uint32_t, PackedBank::match_id_t> PackedDistMatchVector;

// The flat problem holds, per match, one query shift per path of graph 1 and two words per path of graph 2 (qa1 / qa2 /
// qoff), and indexes tree entries with 32 bits.  A merge of hundreds of paths with millions of matches would need tens of
// GB for them on the host, in pinned staging and on the device; such a problem stays on the reference's CPU code
// (CLB_CHAIN_MAX_TABLE_GB, default 16).
inline bool flat_problem_too_large(const std::vector<match_set_t>& match_sets, size_t num_match_sets, size_t chains1, size_t chains2) {
    static const double budget_gb = getenv("CLB_CHAIN_MAX_TABLE_GB") ? atof(getenv("CLB_CHAIN_MAX_TABLE_GB")) : 16.0;
    double matches = 0.0;
    for (size_t s = 0; s < num_match_sets && s < match_sets.size(); ++s)
        matches += (double)match_sets[s].walks1.size() * (double)match_sets[s].walks2.size();
    const double table_bytes = matches * 4.0 * ((double)chains1 + 2.0 * (double)chains2);
    return table_bytes > budget_gb * 1e9 || matches >= 2147483648.0;  // (the library indexes matches with 31 bits)
}

// anchors of a chain of match ranks: the loop body of traceback_sparse_dp (anchorer.hpp:2510-2527), forward order
inline std::vector<anchor_t> anchors_of(const std::vector<int64_t>& chain, const centrolign_b200::ChainProblem& P,
                                        const std::vector<match_set_t>& match_sets) {
    std::vector<anchor_t> anchors;
    anchors.reserve(chain.size());
    for (int64_t rank : chain) {
        const auto& idx = P.ids[(size_t)rank];
        anchors.emplace_back();
        auto& anchor = anchors.back();
        auto& match_set = match_sets[std::get<0>(idx)];
        anchor.walk1 = match_set.walks1[std::get<1>(idx)];
        anchor.count1 = match_set.count1;
        anchor.walk2 = match_set.walks2[std::get<2>(idx)];
        anchor.count2 = match_set.count2;
        anchor.full_length = match_set.full_length;
        anchor.match_set = std::get<0>(idx);
        anchor.idx1 = std::get<1>(idx);
        anchor.idx2 = std::get<2>(idx);
    }
    return anchors;
}

}  // namespace b200_chain

// ---- sparse_affine_chain_dp: the 32-bit instantiations Anchorer::anchor_chain selects (anchorer.hpp:1258-1278) ----
//   * production:        std::vector-backed containers (:1276-1277);
//   * restrain_memory:   bit-packed MatchBank / forward edges / distance vectors (:1263-1264) -- what Core switches to for
//                        merges of many paths (core.hpp:194), i.e. the largest chaining calls of a progressive alignment.
// Both build the same flat problem: packed and unpacked containers answer every query identically and iterate in the
// same order (packed_match_bank.hpp:146-163, packed_forward_edges.hpp:86-101).  The 64-bit instantiations (:1267-1268,
// :1281-1282: >= 2^32 anchors or a diagonal difference >= 2^31) keep the reference's generic code: the flat problem and the
// device search structures index matches with 32 bits, and a problem of that size does not fit one GPU's HBM anyway.
#define CLB_AFFINE_CHAIN_SPECIALIZATION(SHIFT_MATCH_VEC, DIST_MATCH_VEC, DIST_VEC, ANCHOR_VEC, MBANK, FWD)                         \
    template <>                                                                                                                    \
    inline std::vector<anchor_t>                                                                                                   \
    Anchorer::sparse_affine_chain_dp<uint32_t, uint16_t, uint32_t, int32_t, uint32_t, float, SHIFT_MATCH_VEC, DIST_MATCH_VEC,      \
                                     DIST_VEC, ANCHOR_VEC, MBANK, FWD, BaseGraph, b200_chain::XMerge, 3>(                          \
        const std::vector<match_set_t>& match_sets, const BaseGraph& graph1, const BaseGraph& graph2,                              \
        const b200_chain::XMerge& xmerge1, const b200_chain::XMerge& xmerge2, const std::array<double, 3>& gap_open,               \
        const std::array<double, 3>& gap_extend, double local_scale, size_t num_match_sets, bool suppress_verbose_logging,         \
        const std::vector<uint64_t>* sources1, const std::vector<uint64_t>* sources2, const std::vector<uint64_t>* sinks1,         \
        const std::vector<uint64_t>* sinks2, const std::unordered_set<std::tuple<size_t, size_t, size_t>>* masked_matches) const { \
        using namespace b200_chain;                                                                                                \
        if (flat_problem_too_large(match_sets, num_match_sets, xmerge1.chain_size(), xmerge2.chain_size()))                        \
            /* the per-match x per-path tables of the flat problem would not fit: the reference's own generic code, through its   \
               64-bit instantiation (anchorer.hpp:1281-1282), which this header does not specialize */                            \
            return sparse_affine_chain_dp<uint64_t, uint32_t, uint64_t, int64_t, uint64_t, float,                                  \
                                          std::vector<std::pair<int64_t, MatchBank<uint64_t, uint32_t, float>::match_id_t>>,       \
                                          std::vector<std::pair<uint64_t, MatchBank<uint64_t, uint32_t, float>::match_id_t>>,      \
                                          std::vector<uint64_t>, std::vector<uint64_t>, MatchBank<uint64_t, uint32_t, float>,     \
                                          b200_chain::FwdEdges, BaseGraph, b200_chain::XMerge, 3>(                                 \
                match_sets, graph1, graph2, xmerge1, xmerge2, gap_open, gap_extend, local_scale, num_match_sets,                  \
                suppress_verbose_logging, sources1, sources2, sinks1, sinks2, masked_matches);                                    \
        const double t0 = now_s();                                                                                                 \
        MBANK match_bank(graph1, match_sets, num_match_sets, true, masked_matches);                   /* anchorer.hpp:1861 */      \
        PostSwitchDistances<DIST_VEC> switch_dists1(graph1, xmerge1), switch_dists2(graph2, xmerge2); /* :1871-1872 */             \
        std::vector<bool> mask_to, mask_from;                                                                                      \
        std::tie(mask_to, mask_from) = generate_forward_edge_masks(graph1, match_sets, num_match_sets); /* :2267-2269 */           \
        FWD forward_edges(xmerge1, &mask_to, &mask_from);                                                                          \
        const auto order1 = topological_order(graph1); /* :2290 */                                                                 \
        auto weight_of = [&](const match_set_t& ms) -> float {                                                                     \
            return score_function->anchor_weight(ms.count1, ms.count2, ms.walks1.front().size(), ms.full_length);                  \
        };                                                                                                                         \
        const double t1 = now_s();                                                                                                 \
        auto P = centrolign_b200::build_affine_chain_problem<int32_t>(match_bank, forward_edges, switch_dists1, switch_dists2,     \
                                                                      graph1, order1, xmerge1, xmerge2, match_sets, num_match_sets, \
                                                                      gap_open, gap_extend, local_scale, sources1, sources2,       \
                                                                      sinks1, sinks2, weight_of);                                  \
        const double t2 = now_s();                                                                                                 \
        float opt_value = 0.0f;                                                                                                    \
        auto traceback = anchors_of(P.solve(centrolign_b200::chain_device(), &opt_value), P, match_sets);                                                        \
        if (getenv("CLB_TIMING") && P.n_match() > 10000)                                                                           \
            fprintf(stderr, "[clb] affine chaining of %zu matches (" #MBANK "): reference-side tables %.3f s, flat problem %.3f s, " \
                            "clb_chain_dp %.3f s\n", P.n_match(), t1 - t0, t2 - t1, now_s() - t2);                                 \
        annotate_scores(traceback); /* :2536 */                                                                                    \
        /* gap length and score between the anchors (:2443-2468) */                                                               \
        centrolign_b200::annotate_gaps<int32_t>(traceback, xmerge1, xmerge2, switch_dists1, switch_dists2, gap_open, gap_extend,   \
                                                local_scale, sources1, sources2, sinks1, sinks2);                                  \
        if (!suppress_verbose_logging) {                                                                                           \
            logging::log(logging::Debug, "Optimal chain consists of " + std::to_string(traceback.size()) + " matches with score " + \
                                             (opt_value == std::numeric_limits<float>::lowest() ? std::string("-inf")              \
                                                                                                : std::to_string(opt_value)));     \
        }                                                                                                                          \
        return traceback;                                                                                                          \
    }
CLB_AFFINE_CHAIN_SPECIALIZATION(b200_chain::ShiftMatchVector, b200_chain::DistMatchVector, std::vector<uint32_t>, std::vector<uint32_t>,
                                b200_chain::Bank, b200_chain::FwdEdges)
CLB_AFFINE_CHAIN_SPECIALIZATION(b200_chain::PackedShiftMatchVector, b200_chain::PackedDistMatchVector, PackedVector, PackedVector,
                                b200_chain::PackedBank, PackedForwardEdges)
#undef CLB_AFFINE_CHAIN_SPECIALIZATION

// ---- sparse_chain_dp, production instantiation (anchorer.hpp:1291), for the two reachability structures Core uses with
// it: PathMerge<uint32_t, uint8_t> in the alignment subproblems (core.hpp:336-338) and ChainMerge in the per-sequence
// scale calibration (src/core.cpp:150-157) ----
#define CLB_GAPFREE_CHAIN_SPECIALIZATION(XM)                                                                                       \
    template <>                                                                                                                    \
    inline std::vector<anchor_t>                                                                                                   \
    Anchorer::sparse_chain_dp<uint32_t, uint32_t, uint16_t, uint32_t, float, b200_chain::DistMatchVector, std::vector<uint32_t>,  \
                              b200_chain::Bank, ForwardEdges<XM::node_id_t, XM::chain_id_t>, BaseGraph, XM>(                      \
        const std::vector<match_set_t>& match_sets, const BaseGraph& graph1, const XM& chain_merge1, const XM& chain_merge2,       \
        size_t num_match_sets, bool suppress_verbose_logging, const std::vector<uint64_t>* sources1,                               \
        const std::vector<uint64_t>* sources2, const std::vector<uint64_t>* sinks1, const std::vector<uint64_t>* sinks2,           \
        const std::unordered_set<std::tuple<size_t, size_t, size_t>>* masked_matches) const {                                      \
        using namespace b200_chain;                                                                                                \
        Bank match_bank(graph1, match_sets, num_match_sets, true, masked_matches); /* anchorer.hpp:1531 */                         \
        std::vector<bool> mask_to, mask_from;                                                                                      \
        std::tie(mask_to, mask_from) = generate_forward_edge_masks(graph1, match_sets, num_match_sets); /* :1620-1622 */           \
        ForwardEdges<XM::node_id_t, XM::chain_id_t> forward_edges(chain_merge1, &mask_to, &mask_from);                             \
        const auto order1 = topological_order(graph1); /* :1640 */                                                                 \
        auto weight_of = [&](const match_set_t& ms) -> float {                                                                     \
            return score_function->anchor_weight(ms.count1, ms.count2, ms.walks1.front().size(), ms.full_length);                  \
        };                                                                                                                         \
        auto P = centrolign_b200::build_gapfree_chain_problem(match_bank, forward_edges, graph1, order1, chain_merge1,             \
                                                              chain_merge2, match_sets, num_match_sets, sources1, sources2,        \
                                                              sinks1, sinks2, weight_of);                                          \
        auto traceback = anchors_of(P.solve(centrolign_b200::chain_device()), P, match_sets);                                                                    \
        annotate_scores(traceback); /* :2536 */                                                                                    \
        (void)suppress_verbose_logging;                                                                                            \
        return traceback;                                                                                                          \
    }
CLB_GAPFREE_CHAIN_SPECIALIZATION(b200_chain::XMerge)
CLB_GAPFREE_CHAIN_SPECIALIZATION(ChainMerge)
#undef CLB_GAPFREE_CHAIN_SPECIALIZATION

// ---- fill_in_anchor_chain (anchorer.hpp:619-699) for the production types: the subproblems between the anchors of the
// main chain are independent -- each has its own subgraphs, matches, budget and result slot -- so they run on a pool of
// host threads whose chaining calls share kernel launches (centrolign_b200/hostcpp/chain_batcher.hpp).  Extraction, the
// division of matches and budgets, and the merge of the results are the reference's own functions, called in its order.
#define CLB_FILL_IN_SPECIALIZATION(XM)                                                                                                      \
template <>                                                                                                                                 \
inline void Anchorer::fill_in_anchor_chain<BaseGraph, XM>(                                                                                  \
    std::vector<anchor_t>& anchors, std::vector<match_set_t>& matches, const BaseGraph& graph1, const BaseGraph& graph2,                    \
    const SentinelTableau& tableau1, const SentinelTableau& tableau2, const XM& xmerge1, const XM& xmerge2,                                 \
    bool restrain_memory, ChainAlgorithm local_chaining_algorithm, double anchor_scale,                                                     \
    const std::unordered_set<std::tuple<size_t, size_t, size_t>>* masked_matches) const {                                                   \
    if (anchors.empty()) {                                                                                                                  \
        logging::log(logging::Debug, "Skipping fill-in anchoring on an empty chain");                                                       \
        return;                                                                                                                             \
    }                                                                                                                                       \
    auto gaps = extract_graphs_between(anchors, graph1, graph2, tableau1, tableau2, xmerge1, xmerge2);                                      \
    project_paths(graph1, graph2, gaps);                                                                                                    \
    std::vector<std::vector<std::pair<size_t, std::pair<std::vector<size_t>, std::vector<size_t>>>>> origin;                                \
    auto gap_matches = divvy_matches(matches, graph1, graph2, gaps, origin);                                                                \
    const auto budgets = assign_reanchor_budget(gaps);                                                                                      \
    std::vector<std::vector<anchor_t>> gap_chains(gaps.size());                                                                             \
    centrolign_b200::batched_parallel_for(gaps.size(), centrolign_b200::default_devices(), [&](size_t g) {                                  \
        auto& sub1 = gaps[g].first;                                                                                                         \
        auto& sub2 = gaps[g].second;                                                                                                        \
        XM gap_merge1(sub1.subgraph), gap_merge2(sub2.subgraph);                                                                            \
        /* masked (set, walk1, walk2) triples in the numbering of this gap's match sets (:662-679) */                                       \
        std::unordered_set<std::tuple<size_t, size_t, size_t>> masked_here;                                                                 \
        if (masked_matches && !masked_matches->empty()) {                                                                                   \
            for (size_t set = 0; set < origin[g].size(); ++set) {                                                                           \
                const size_t parent_set = origin[g][set].first;                                                                             \
                const std::vector<size_t>& from1 = origin[g][set].second.first;                                                             \
                const std::vector<size_t>& from2 = origin[g][set].second.second;                                                            \
                for (size_t a = 0; a < from1.size(); ++a)                                                                                   \
                    for (size_t b = 0; b < from2.size(); ++b)                                                                               \
                        if (masked_matches->count(std::make_tuple(parent_set, from1[a], from2[b]))) masked_here.emplace(set, a, b);         \
            }                                                                                                                               \
        }                                                                                                                                   \
        gap_chains[g] = anchor_chain(gap_matches[g], sub1.subgraph, sub2.subgraph, gap_merge1, gap_merge2, restrain_memory, &sub1.sources,  \
                                     &sub2.sources, &sub1.sinks, &sub2.sinks, budgets[g], true, local_chaining_algorithm, anchor_scale,     \
                                     &masked_here);                                                                                         \
    });                                                                                                                                     \
    merge_fill_in_chains(anchors, gap_chains, gaps, origin);                                                                                \
    logging::log(logging::Debug, "Filled-in anchor chain consists of " + std::to_string(anchors.size()) + " anchors");                      \
}
CLB_FILL_IN_SPECIALIZATION(b200_chain::XMerge)  // alignment subproblems (core.hpp:336-338)
CLB_FILL_IN_SPECIALIZATION(ChainMerge)          // per-sequence scale calibration (src/core.cpp:150-157, :222)
#undef CLB_FILL_IN_SPECIALIZATION

}  // namespace centrolign

#endif
