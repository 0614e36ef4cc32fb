// chain_b200.hpp -- C++ host layer of the sparse anchor-chaining DP (clb_chain_dp, include/centrolign_b200.h).
//
// The reference runs its chaining DP inside two member templates of Anchorer,
//
//     sparse_affine_chain_dp<UIntSet, UIntMatch, UIntDist, IntShift, UIntAnchor, ScoreFloat, ..., MBank, FwdEdges>
//         (match_sets, graph1, graph2, xmerge1, xmerge2, gap_open, gap_extend, local_scale, num_match_sets,
//          suppress_verbose_logging, sources1, sources2, sinks1, sinks2, masked_matches)
//                                                    reference: include/centrolign/anchorer.hpp:1812-2471
//     sparse_chain_dp<UIntDist, UIntSet, UIntMatch, UIntAnchor, ScoreFloat, ..., MBank, FwdEdges>
//         (match_sets, graph1, chain_merge1, chain_merge2, num_match_sets, ...)
//                                                    reference: include/centrolign/anchorer.hpp:1511-1750
//
// both called from Anchorer::anchor_chain (anchorer.hpp:1213-1307).  The functions below take the objects
// those templates build before their main loop -- the MatchBank, the ForwardEdges, the two
// PostSwitchDistances, the XMerge reachability structures, the topological order of graph 1 -- read them
// through their public interfaces, and write the flat clb_chain_problem the CUDA library consumes: per
// match the tree keys of its end point for every path pair and the query shifts / offsets of its start
// point for every path, and per graph-1 node the matches that end there and the (match, chain) queries of
// its forward edges, all in the reference's own iteration order.  The gap-measuring lambdas of the
// reference (anchorer.hpp:1875-2000) are restated here because the lead / final gap terms and the anchor
// annotations need them.  No DP happens on the host; errors surface as std::runtime_error.
#ifndef CENTROLIGN_B200_CHAIN_HPP
#define CENTROLIGN_B200_CHAIN_HPP

#include <array>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <limits>
#include <stdexcept>
#include <string>
#include <tuple>
#include <type_traits>
#include <vector>

#include "centrolign_b200.h"
#include "chain_batcher.hpp"

namespace centrolign_b200 {

// Owns the arrays a clb_chain_problem points into.
struct ChainProblem {
    int num_pw = 0;
    double gap_open[CLB_MAX_PW] = {0, 0, 0}, gap_extend[CLB_MAX_PW] = {0, 0, 0}, scale = 1.0;
    int32_t n_chain1 = 0, n_chain2 = 0;
    float min_score = 0.0f;
    std::vector<float> weight, dp_init, final_term;
    std::vector<int64_t> end_off{0}, qry_off{0}, ins_off{0};
    std::vector<uint32_t> end_match, qry_match, qry_chain1, ins_p1, ins_p2, ins_offset, qoff;
    std::vector<int32_t> ins_shift, qa1, qa2;
    std::vector<uint8_t> ins_active;  // empty = all active
    std::vector<std::tuple<size_t, size_t, size_t>> ids;  // rank -> (match set, walk1 index, walk2 index)

    size_t n_match() const { return weight.size(); }

    clb_chain_problem view() const {
        clb_chain_problem p;
        p.num_pw = num_pw;
        for (int k = 0; k < CLB_MAX_PW; ++k) {
            p.gap_open[k] = gap_open[k];
            p.gap_extend[k] = gap_extend[k];
        }
        p.scale = scale;
        p.n_chain1 = n_chain1;
        p.n_chain2 = n_chain2;
        p.n_match = (int64_t)weight.size();
        p.weight = weight.data();
        p.dp_init = dp_init.data();
        p.final_term = final_term.data();
        p.min_score = min_score;
        p.n_step = (int64_t)end_off.size() - 1;
        p.end_off = end_off.data();
        p.end_match = end_match.data();
        p.qry_off = qry_off.data();
        p.qry_match = qry_match.data();
        p.qry_chain1 = qry_chain1.data();
        p.ins_off = ins_off.data();
        p.ins_p1 = ins_p1.data();
        p.ins_p2 = ins_p2.data();
        p.ins_shift = ins_shift.data();
        p.ins_offset = ins_offset.data();
        p.ins_active = ins_active.empty() ? nullptr : ins_active.data();
        p.qa1 = qa1.data();
        p.qa2 = qa2.data();
        p.qoff = qoff.data();
        return p;
    }

    // Runs the DP + traceback on the GPU; returns the chain as match ranks in forward order.  Inside a fill-in pool
    // (batched_parallel_for) the problem runs on the device of the calling worker's batcher, not on `device`.
    std::vector<int64_t> solve(int device = 0, float* opt_score = nullptr, clb_chain_stats* stats = nullptr,
                               std::vector<float>* dp_out = nullptr, std::vector<int64_t>* backptr_out = nullptr) const {
        const clb_chain_problem p = view();
        std::vector<int64_t> chain(weight.size() + 1);
        int64_t len = 0;
        if (dp_out) dp_out->assign(weight.size(), 0.0f);
        if (backptr_out) backptr_out->assign(weight.size(), -1);
        if (ChainBatcher* batcher = stats ? nullptr : ChainBatcher::current()) {
            // a worker of a fill-in pool: lay the problem out here, share the launch with the other workers (chain_batcher.hpp)
            clb_chain_job* job = nullptr;
            const int rc = clb_chain_job_create(batcher->device(), &p, dp_out ? dp_out->data() : nullptr, backptr_out ? backptr_out->data() : nullptr,
                                                chain.data(), &len, opt_score, &job);
            if (rc != CLB_OK) throw std::runtime_error(std::string("centrolign_b200: ") + clb_last_error());
            if (job) {
                struct Guard {
                    clb_chain_job* j;
                    ~Guard() { clb_chain_job_destroy(j); }
                } guard{job};
                batcher->solve(job);
            }
            chain.resize((size_t)len);
            return chain;
        }
        const int rc = clb_chain_dp(device, &p, dp_out ? dp_out->data() : nullptr, backptr_out ? backptr_out->data() : nullptr,
                                    chain.data(), &len, opt_score, stats);
        if (rc != CLB_OK) throw std::runtime_error(std::string("centrolign_b200: ") + clb_last_error());
        chain.resize((size_t)len);
        return chain;
    }
};

namespace detail {

// rank of every (set, i1, i2) in MatchBank iteration order (match_bank.hpp:188-267), UINT32_MAX if masked
template <class MBank, class MatchSets>
struct RankTable {
    std::vector<size_t> base;     // per set
    std::vector<uint32_t> rank;   // base[set] + i1 * walks2.size() + i2
    const MatchSets* sets;
    RankTable(const MBank& bank, const MatchSets& match_sets, size_t num_match_sets, ChainProblem& P) : sets(&match_sets) {
        base.assign(num_match_sets + 1, 0);
        for (size_t s = 0; s < num_match_sets; ++s)
            base[s + 1] = base[s] + match_sets[s].walks1.size() * match_sets[s].walks2.size();
        rank.assign(base[num_match_sets], 0xffffffffu);
        uint32_t r = 0;
        for (auto it = bank.begin(), end = bank.end(); it != end; ++it) {
            const auto idx = bank.get_match_indexes(*it);
            rank[at(std::get<0>(idx), std::get<1>(idx), std::get<2>(idx))] = r++;
            P.ids.emplace_back(std::get<0>(idx), std::get<1>(idx), std::get<2>(idx));
        }
    }
    size_t at(size_t s, size_t i1, size_t i2) const { return base[s] + i1 * (*sets)[s].walks2.size() + i2; }
    template <class MatchId>
    uint32_t operator()(const MBank& bank, const MatchId& id) const {
        const auto idx = bank.get_match_indexes(id);
        return rank[at(std::get<0>(idx), std::get<1>(idx), std::get<2>(idx))];
    }
};

// events of the main loop, in the reference's order (anchorer.hpp:2290-2416 / :1640-1727)
template <class MBank, class FwdEdges, class BGraph, class Ranks, class TopoOrder>
void collect_events(ChainProblem& P, const MBank& bank, const FwdEdges& forward_edges, const BGraph&, const Ranks& ranks,
                    const TopoOrder& order) {
    for (uint64_t node_id : order) {
        const size_t e0 = P.end_match.size(), q0 = P.qry_match.size();
        for (const auto& match_id : bank.ends_on(node_id)) P.end_match.push_back(ranks(bank, match_id));
        for (auto edge : forward_edges.edges(node_id)) {
            const uint64_t fwd_id = edge.first;
            const uint64_t chain1 = edge.second;
            for (const auto& match_id : bank.starts_on(fwd_id)) {
                P.qry_match.push_back(ranks(bank, match_id));
                P.qry_chain1.push_back((uint32_t)chain1);
            }
        }
        if (P.end_match.size() != e0 || P.qry_match.size() != q0) {
            P.end_off.push_back((int64_t)P.end_match.size());
            P.qry_off.push_back((int64_t)P.qry_match.size());
        }
    }
}

}  // namespace detail

// Gap geometry of sparse_affine_chain_dp.  The reference measures the indel between an END point (a node pair a chain
// element stops on, or a source pair) and a START point (the node pair the next element begins on, or a sink pair) as a
// difference of diagonals on a pair of paths (p1, p2) through the end point (anchorer.hpp:1875-1892):
//     end diagonal    d_end(p1,p2)   = index_on(e1,p1) - index_on(e2,p2)
//     reach diagonal  d_reach(p1,p2) = (predecessor_index(s1,p1) + D1(s1,p1)) - (predecessor_index(s2,p2) + D2(s2,p2))
// (the same two quantities the flat problem carries per match as ins_shift and qa1 - qa2), keeps the difference of smallest
// absolute value over the path pairs, and, for SETS of end / start points, folds over their product.  Here that is ONE
// routine, `closest`, over (pointer, count) views; the four shapes of the reference (:1937-2000 node->node, sources->node,
// node->sinks, sources->sinks) are its calls with one-element views.  Two details decide results and are kept: the
// product is walked starts-outer / ends-inner (:1985-1988; the one-sided shapes are that order with a trivial loop), and a
// candidate replaces the running value only if its ABSOLUTE value is below the running SIGNED value (:1954, :1971,
// :1991), so a negative running value is final.
template <typename IntShift, typename ScoreFloat, class XMerge, class SwitchDists, size_t NumPW>
struct GapGeometry {
    struct Nodes {  // a view of node ids
        const uint64_t* ptr;
        size_t n;
        Nodes(const uint64_t& one) : ptr(&one), n(1) {}
        Nodes(const std::vector<uint64_t>& v) : ptr(v.data()), n(v.size()) {}
    };
    const XMerge& xmerge1;
    const XMerge& xmerge2;
    const SwitchDists& switch_dists1;
    const SwitchDists& switch_dists2;
    const std::array<double, NumPW>& gap_open;
    const std::array<double, NumPW>& gap_extend;
    double local_scale;

    static IntShift unreachable() { return std::numeric_limits<IntShift>::max(); }

    IntShift end_diagonal(uint64_t e1, uint64_t e2, uint64_t p1, uint64_t p2) const {
        return xmerge1.index_on(e1, p1) - xmerge2.index_on(e2, p2);
    }
    IntShift reach_diagonal(uint64_t s1, uint64_t s2, uint64_t p1, uint64_t p2) const {
        return (xmerge1.predecessor_index(s1, p1) - xmerge2.predecessor_index(s2, p2) + switch_dists1.distance(s1, p1) -
                switch_dists2.distance(s2, p2));
    }
    // one end point to one start point: the diagonal difference of smallest absolute value over the path pairs through
    // the end point (first such pair in chains_on order), `unreachable()` if either graph has no walk between them
    IntShift between(uint64_t e1, uint64_t e2, uint64_t s1, uint64_t s2) const {
        IntShift best = unreachable();
        const bool walk1 = e1 == s1 || xmerge1.reachable(e1, s1), walk2 = e2 == s2 || xmerge2.reachable(e2, s2);
        if (walk1 && walk2)
            for (auto p1 : xmerge1.chains_on(e1))
                for (auto p2 : xmerge2.chains_on(e2)) {
                    const IntShift d = end_diagonal(e1, e2, p1, p2) - reach_diagonal(s1, s2, p1, p2);
                    if (std::abs(d) < std::abs(best)) best = d;
                }
        return best;
    }
    // sets of end points to sets of start points
    IntShift closest(Nodes ends1, Nodes ends2, Nodes starts1, Nodes starts2) const {
        IntShift running = unreachable();
        for (size_t a = 0; a < starts1.n; ++a)
            for (size_t b = 0; b < starts2.n; ++b)
                for (size_t c = 0; c < ends1.n; ++c)
                    for (size_t d = 0; d < ends2.n; ++d) {
                        const IntShift g = between(ends1.ptr[c], ends2.ptr[d], starts1.ptr[a], starts2.ptr[b]);
                        if (std::abs(g) < running) running = g;
                    }
        return running;
    }
    // score of an indel of `gap` diagonals: the best gap piece, 0 for no gap, lowest() if unreachable (:1906-1918)
    ScoreFloat score(IntShift gap) const {
        if (gap == 0) return ScoreFloat(0.0);
        ScoreFloat best = std::numeric_limits<ScoreFloat>::lowest();
        if (gap != unreachable())
            for (size_t pw = 0; pw < NumPW; ++pw)
                best = std::max<ScoreFloat>(best, -local_scale * (gap_open[pw] + gap_extend[pw] * std::abs(gap)));
        return best;
    }
    std::pair<IntShift, ScoreFloat> measured(Nodes ends1, Nodes ends2, Nodes starts1, Nodes starts2) const {
        const IntShift g = closest(ends1, ends2, starts1, starts2);
        return std::make_pair(g, score(g));
    }
};

// Gap lengths and scores between the elements of a finished chain (what anchorer.hpp:2443-2468 records in the anchors):
// one measurement per junction -- sources to the first anchor, anchor to anchor, last anchor to the sinks -- written to
// the records on both sides of the junction.
template <typename IntShift, class Anchors, class XMerge, class SwitchDists, size_t NumPW>
void annotate_gaps(Anchors& chain, const XMerge& xmerge1, const XMerge& xmerge2, const SwitchDists& switch_dists1,
                   const SwitchDists& switch_dists2, const std::array<double, NumPW>& gap_open,
                   const std::array<double, NumPW>& gap_extend, double local_scale, const std::vector<uint64_t>* sources1,
                   const std::vector<uint64_t>* sources2, const std::vector<uint64_t>* sinks1, const std::vector<uint64_t>* sinks2) {
    if (chain.empty()) return;
    GapGeometry<IntShift, float, XMerge, SwitchDists, NumPW> geo{xmerge1, xmerge2, switch_dists1, switch_dists2, gap_open, gap_extend, local_scale};
    if (sources1) {
        const auto lead = geo.measured(*sources1, *sources2, chain.front().walk1.front(), chain.front().walk2.front());
        chain.front().gap_before = lead.first;
        chain.front().gap_score_before = lead.second;
    }
    for (size_t i = 0; i + 1 < chain.size(); ++i) {
        const auto mid = geo.measured(chain[i].walk1.back(), chain[i].walk2.back(), chain[i + 1].walk1.front(), chain[i + 1].walk2.front());
        chain[i].gap_after = chain[i + 1].gap_before = mid.first;
        chain[i].gap_score_after = chain[i + 1].gap_score_before = mid.second;
    }
    if (sinks1) {
        const auto trail = geo.measured(chain.back().walk1.back(), chain.back().walk2.back(), *sinks1, *sinks2);
        chain.back().gap_after = trail.first;
        chain.back().gap_score_after = trail.second;
    }
}

// Flat problem of sparse_affine_chain_dp.  `weight_of(match_set)` is the reference's
// score_function->anchor_weight(count1, count2, walks1.front().size(), full_length) (anchorer.hpp:2023-2024).
template <typename IntShift, class MBank, class FwdEdges, class SwitchDists, class BGraph, class XMerge, class MatchSets,
          class TopoOrder, class WeightFn, size_t NumPW>
ChainProblem build_affine_chain_problem(const MBank& bank, const FwdEdges& forward_edges, const SwitchDists& switch_dists1,
                                        const SwitchDists& switch_dists2, const BGraph& graph1, const TopoOrder& order1,
                                        const XMerge& xmerge1, const XMerge& xmerge2, const MatchSets& match_sets,
                                        size_t num_match_sets, const std::array<double, NumPW>& gap_open,
                                        const std::array<double, NumPW>& gap_extend, double local_scale,
                                        const std::vector<uint64_t>* sources1, const std::vector<uint64_t>* sources2,
                                        const std::vector<uint64_t>* sinks1, const std::vector<uint64_t>* sinks2,
                                        const WeightFn& weight_of) {
    static_assert(NumPW >= 1 && NumPW <= CLB_MAX_PW, "1..3 gap pieces");
    typedef float ScoreFloat;  // the reference instantiates ScoreFloat = float (anchorer.hpp:1217)
    const ScoreFloat mininf = std::numeric_limits<ScoreFloat>::lowest();
    GapGeometry<IntShift, ScoreFloat, XMerge, SwitchDists, NumPW> geo{xmerge1, xmerge2, switch_dists1, switch_dists2,
                                                                      gap_open, gap_extend, local_scale};
    ChainProblem P;
    P.num_pw = (int)NumPW;
    for (size_t k = 0; k < NumPW; ++k) {
        P.gap_open[k] = gap_open[k];
        P.gap_extend[k] = gap_extend[k];
    }
    P.scale = local_scale;
    P.n_chain1 = (int32_t)xmerge1.chain_size();
    P.n_chain2 = (int32_t)xmerge2.chain_size();
    detail::RankTable<MBank, MatchSets> ranks(bank, match_sets, num_match_sets, P);
    const size_t C1 = xmerge1.chain_size(), C2 = xmerge2.chain_size();

    for (auto it = bank.begin(), end = bank.end(); it != end; ++it) {
        const auto& match_set = bank.match_set(*it);
        const uint64_t start1 = bank.walk1(*it).front(), start2 = bank.walk2(*it).front();
        const uint64_t end1 = bank.walk1(*it).back(), end2 = bank.walk2(*it).back();
        ScoreFloat weight = weight_of(match_set);
        P.weight.push_back(weight);
        if (sources1) {  // anchorer.hpp:2026-2039
            ScoreFloat lead_indel_score = geo.measured(*sources1, *sources2, start1, start2).second;
            if (lead_indel_score == mininf) weight = mininf;
            else weight += lead_indel_score;
        }
        P.dp_init.push_back(weight);
        P.final_term.push_back(sinks1 ? geo.measured(end1, end2, *sinks1, *sinks2).second : ScoreFloat(0.0));  // :2431-2438
        for (auto p1 : xmerge1.chains_on(end1))  // anchorer.hpp:2043-2048, 2309-2318
            for (auto p2 : xmerge2.chains_on(end2)) {
                P.ins_p1.push_back((uint32_t)p1);
                P.ins_p2.push_back((uint32_t)p2);
                P.ins_shift.push_back((int32_t)geo.end_diagonal(end1, end2, p1, p2));
                P.ins_offset.push_back((uint32_t)xmerge2.index_on(end2, p2));
            }
        P.ins_off.push_back((int64_t)P.ins_p1.size());
        // query shift (anchorer.hpp:1886-1892) is separable in wrapping arithmetic: (pred1 + D1) - (pred2 + D2)
        for (size_t c1 = 0; c1 < C1; ++c1)
            P.qa1.push_back((int32_t)(uint32_t)(uint64_t)((uint64_t)xmerge1.predecessor_index(start1, c1) +
                                                          (uint64_t)switch_dists1.distance(start1, c1)));
        for (size_t c2 = 0; c2 < C2; ++c2) {
            P.qa2.push_back((int32_t)(uint32_t)(uint64_t)((uint64_t)xmerge2.predecessor_index(start2, c2) +
                                                          (uint64_t)switch_dists2.distance(start2, c2)));
            // "we rely on -1's overflowing to 0" (anchorer.hpp:1898-1901); the sentinel has the XMerge's own integer width
            auto pred = xmerge2.predecessor_index(start2, c2);
            P.qoff.push_back((uint32_t)(decltype(pred))(pred + 1));
        }
    }
    P.min_score = 0.0f;
    if (sources1 && sinks1) P.min_score = geo.measured(*sources1, *sources2, *sinks1, *sinks2).second;  // :2419-2424
    detail::collect_events(P, bank, forward_edges, graph1, ranks, order1);
    return P;
}

// Flat problem of the gap-free sparse_chain_dp (anchorer.hpp:1511-1750): one search tree per (chain1, chain2)
// keyed (index on chain2, match) -- the same machinery with a single diagonal per chain pair and no gap pieces.
template <class MBank, class FwdEdges, class BGraph, class XMerge, class MatchSets, class TopoOrder, class WeightFn>
ChainProblem build_gapfree_chain_problem(const MBank& bank, const FwdEdges& forward_edges, const BGraph& graph1,
                                         const TopoOrder& order1, const XMerge& chain_merge1, const XMerge& chain_merge2,
                                         const MatchSets& match_sets, size_t num_match_sets,
                                         const std::vector<uint64_t>* sources1, const std::vector<uint64_t>* sources2,
                                         const std::vector<uint64_t>* sinks1, const std::vector<uint64_t>* sinks2,
                                         const WeightFn& weight_of) {
    typedef float ScoreFloat;
    const ScoreFloat mininf = std::numeric_limits<ScoreFloat>::lowest();
    ChainProblem P;
    P.num_pw = 0;
    P.n_chain1 = (int32_t)chain_merge1.chain_size();
    P.n_chain2 = (int32_t)chain_merge2.chain_size();
    detail::RankTable<MBank, MatchSets> ranks(bank, match_sets, num_match_sets, P);
    const size_t C1 = chain_merge1.chain_size(), C2 = chain_merge2.chain_size();
    for (auto it = bank.begin(), end = bank.end(); it != end; ++it) {
        const auto& match_set = bank.match_set(*it);
        const uint64_t start1 = bank.walk1(*it).front(), start2 = bank.walk2(*it).front();
        const uint64_t end1 = bank.walk1(*it).back(), end2 = bank.walk2(*it).back();
        ScoreFloat weight = weight_of(match_set);
        P.weight.push_back(weight);
        if (sources1) {  // anchorer.hpp:1559-1577
            bool found1 = false, found2 = false;
            for (auto src_id1 : *sources1)
                if (src_id1 == start1 || chain_merge1.reachable(src_id1, start1)) { found1 = true; break; }
            for (auto src_id2 : *sources2)
                if (src_id2 == start2 || chain_merge2.reachable(src_id2, start2)) { found2 = true; break; }
            if (!found1 || !found2) weight = mininf;
        }
        P.dp_init.push_back(weight);
        ScoreFloat fin = 0.0;  // anchorer.hpp:1730-1747
        if (sinks1) {
            fin = mininf;
            for (auto snk_id1 : *sinks1) {
                for (auto snk_id2 : *sinks2)
                    if ((snk_id1 == end1 || chain_merge1.reachable(end1, snk_id1)) &&
                        (snk_id2 == end2 || chain_merge2.reachable(end2, snk_id2))) { fin = 0.0; break; }
                if (fin == ScoreFloat(0.0)) break;
            }
        }
        P.final_term.push_back(fin);
        // every chain of graph 1 has a tree over all matches ending on a given chain of graph 2, key = index on that
        // chain (:1546-1552, 1595-1603); the match is entered only into the tree of its own graph-1 chain (:1657-1666)
        for (size_t c1 = 0; c1 < C1; ++c1) {
            P.ins_p1.push_back((uint32_t)c1);
            P.ins_p2.push_back((uint32_t)chain_merge2.chain(end2).first);
            P.ins_shift.push_back(0);
            P.ins_offset.push_back((uint32_t)chain_merge2.chain(end2).second);
            P.ins_active.push_back(c1 == chain_merge1.chain(end1).first ? 1 : 0);
        }
        P.ins_off.push_back((int64_t)P.ins_p1.size());
        for (size_t c1 = 0; c1 < C1; ++c1) P.qa1.push_back(0);
        for (size_t c2 = 0; c2 < C2; ++c2) {
            P.qa2.push_back(0);
            auto pred = chain_merge2.predecessor_index(start2, c2);  // :1699-1712: -1 = no reachable node, else [0, pred + 1)
            P.qoff.push_back((uint32_t)(decltype(pred))(pred + 1));
        }
    }
    P.min_score = 0.0f;  // traceback_sparse_dp(..., final_term, 0.0, ...), anchorer.hpp:1749
    detail::collect_events(P, bank, forward_edges, graph1, ranks, order1);
    return P;
}

}  // namespace centrolign_b200

#endif  // CENTROLIGN_B200_CHAIN_HPP
