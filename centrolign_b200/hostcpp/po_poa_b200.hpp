// po_poa_b200.hpp -- C++ host layer that keeps the reference's call signature.
//
// The reference's gap-fill entry point is the header template
//
//     template<int NumPW, class Graph>
//     Alignment po_poa(const Graph& graph1, const Graph& graph2,
//                      const std::vector<uint64_t>& sources1, const std::vector<uint64_t>& sources2,
//                      const std::vector<uint64_t>& sinks1,   const std::vector<uint64_t>& sinks2,
//                      const AlignmentParameters<NumPW>& params, int64_t* score_out = nullptr);
//                                  (reference: include/centrolign/alignment.hpp:78-85)
//
// centrolign_b200::po_poa below has the same argument list and the same meaning, and works on
// any type that models the reference's duck-typed Graph concept (node_size / label / previous,
// include/centrolign/graph.hpp:94-149) and any parameter struct with the reference's fields
// (match, mismatch, gap_open[], gap_extend[], alignment.hpp:56-65).  It flattens the graphs into
// the C-ABI batch layout and calls clb_popoa_batch (include/centrolign_b200.h); the CUDA library
// renumbers topologically and runs the sm_100a kernels.  Errors surface as std::runtime_error,
// the way the reference reports its own (src/stitcher.cpp:36); there is no CPU fallback.
//
// centrolign_b200::PoPoaBatch collects many windows and aligns them in one call -- that is what
// Stitcher::stitch should use (see INTEGRATION.md): its windows are independent and known up
// front (include/centrolign/stitcher.hpp:127-132).
#ifndef CENTROLIGN_B200_PO_POA_HPP
#define CENTROLIGN_B200_PO_POA_HPP

#include <cstdint>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <vector>

#include "centrolign_b200.h"
#include "devices.hpp"

namespace centrolign_b200 {

// Same shape as centrolign::AlignedPair (alignment.hpp:34-46); used when the caller does not
// supply the reference's own Alignment type.
struct AlignedPair {
    static constexpr uint64_t gap = uint64_t(-1);
    uint64_t node_id1 = gap;
    uint64_t node_id2 = gap;
    AlignedPair() = default;
    AlignedPair(uint64_t a, uint64_t b) : node_id1(a), node_id2(b) {}
    bool operator==(const AlignedPair& o) const { return node_id1 == o.node_id1 && node_id2 == o.node_id2; }
};
typedef std::vector<AlignedPair> Alignment;

// Same shape as centrolign::AlignmentParameters<NumPW> (alignment.hpp:56-65).
template <int NumPW>
struct AlignmentParameters {
    uint32_t match;
    uint32_t mismatch;
    uint32_t gap_open[NumPW];
    uint32_t gap_extend[NumPW];
};

// Accumulates windows (graph pairs) in the flat layout of clb_graph_batch.
class PoPoaBatch {
public:
    explicit PoPoaBatch(int device = 0) : devices_(1, device) { init(); }
    // Several GPUs of one box: the windows are dealt to the devices in cell-balanced bins (clb_popoa_batch_multi; the
    // windows of a stitch are independent, stitcher.hpp:157-203) and the results come back in window order.
    // CLB_DEVICES="0,1,2,3" in the environment gives a default-constructed Stitcher recorder the same list.
    explicit PoPoaBatch(const std::vector<int>& devices) : devices_(devices.empty() ? std::vector<int>(1, 0) : devices) { init(); }

    size_t size() const { return node_off_[0].size() - 1; }
    const std::vector<int>& devices() const { return devices_; }

    // one window = the argument list of the reference's po_poa, minus the parameters
    template <class Graph>
    void add(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
             const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
             const std::vector<uint64_t>& sinks2) {
        add_side(0, graph1, sources1, sinks1);
        add_side(1, graph2, sources2, sinks2);
    }

    // Align every window; alignments[w] / scores[w] are what po_poa would have returned for window w.
    template <int NumPW, class Params, class AlignmentT = Alignment>
    void align(const Params& params, std::vector<AlignmentT>& alignments, std::vector<int64_t>* scores = nullptr) const {
        static_assert(NumPW >= 1 && NumPW <= CLB_MAX_PW, "1..3 gap pieces");
        clb_params p;
        p.num_pw = NumPW;
        p.match = params.match;
        p.mismatch = params.mismatch;
        for (int k = 0; k < CLB_MAX_PW; ++k) {
            p.gap_open[k] = k < NumPW ? params.gap_open[k] : 0;
            p.gap_extend[k] = k < NumPW ? params.gap_extend[k] : 0;
        }
        const size_t nw = size();
        clb_graph_batch g[2];
        for (int s = 0; s < 2; ++s) {
            g[s].node_off = node_off_[s].data(); g[s].label = label_[s].data(); g[s].edge_off = edge_off_[s].data();
            g[s].pred_off = pred_off_[s].data(); g[s].pred = pred_[s].data(); g[s].src_off = src_off_[s].data();
            g[s].src = src_[s].data(); g[s].snk_off = snk_off_[s].data(); g[s].snk = snk_[s].data();
        }
        std::vector<int64_t> aln_off(nw + 1, 0), score(nw, 0);
        for (size_t w = 0; w < nw; ++w)
            aln_off[w + 1] = aln_off[w] + (node_off_[0][w + 1] - node_off_[0][w]) + (node_off_[1][w + 1] - node_off_[1][w]);
        std::vector<int32_t> pairs(2 * (size_t)aln_off[nw] + 2);
        std::vector<uint32_t> len(nw, 0);
        const int rc = devices_.size() == 1
                           ? clb_popoa_batch(devices_[0], (int32_t)nw, &g[0], &g[1], &p, score.data(), aln_off.data(), pairs.data(), len.data())
                           : clb_popoa_batch_multi((int)devices_.size(), devices_.data(), (int32_t)nw, &g[0], &g[1], &p, score.data(),
                                                   aln_off.data(), pairs.data(), len.data(), nullptr);
        if (rc != CLB_OK) throw std::runtime_error(std::string("centrolign_b200: ") + clb_last_error());
        alignments.assign(nw, AlignmentT());
        for (size_t w = 0; w < nw; ++w) {
            AlignmentT& a = alignments[w];
            a.reserve(len[w]);
            const int32_t* pr = pairs.data() + 2 * aln_off[w];
            for (uint32_t k = 0; k < len[w]; ++k) {
                typedef typename AlignmentT::value_type Pair;
                a.push_back(Pair(pr[2 * k] < 0 ? uint64_t(-1) : (uint64_t)pr[2 * k],
                                 pr[2 * k + 1] < 0 ? uint64_t(-1) : (uint64_t)pr[2 * k + 1]));
            }
        }
        if (scores) *scores = score;
    }

private:
    void init() {
        for (int s = 0; s < 2; ++s) {
            node_off_[s].push_back(0); edge_off_[s].push_back(0); src_off_[s].push_back(0); snk_off_[s].push_back(0);
        }
    }
    template <class Graph>
    void add_side(int s, const Graph& graph, const std::vector<uint64_t>& sources, const std::vector<uint64_t>& sinks) {
        const uint64_t n = graph.node_size();
        uint32_t e = 0;
        pred_off_[s].push_back(0);
        for (uint64_t v = 0; v < n; ++v) {
            label_[s].push_back((uint8_t)graph.label(v));
            for (uint64_t u : graph.previous(v)) {  // previous() order fixes the traceback tie-breaks
                pred_[s].push_back((uint32_t)u);
                ++e;
            }
            pred_off_[s].push_back(e);
        }
        for (uint64_t v : sources) src_[s].push_back((uint32_t)v);
        for (uint64_t v : sinks) snk_[s].push_back((uint32_t)v);
        node_off_[s].push_back(node_off_[s].back() + (int64_t)n);
        edge_off_[s].push_back(edge_off_[s].back() + (int64_t)e);
        src_off_[s].push_back(src_off_[s].back() + (int64_t)sources.size());
        snk_off_[s].push_back(snk_off_[s].back() + (int64_t)sinks.size());
    }

    std::vector<int> devices_;
    std::vector<int64_t> node_off_[2], edge_off_[2], src_off_[2], snk_off_[2];
    std::vector<uint8_t> label_[2];
    std::vector<uint32_t> pred_off_[2], pred_[2], src_[2], snk_[2];
};

// Drop-in for the reference's po_poa: same arguments, same result.
template <int NumPW, class Graph, class Params, class AlignmentT = Alignment>
AlignmentT po_poa(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
                  const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
                  const std::vector<uint64_t>& sinks2, const Params& params, int64_t* score_out = nullptr) {
    PoPoaBatch batch;
    batch.add(graph1, graph2, sources1, sources2, sinks1, sinks2);
    std::vector<AlignmentT> alns;
    std::vector<int64_t> scores;
    batch.align<NumPW, Params, AlignmentT>(params, alns, &scores);
    if (score_out) *score_out = scores[0];
    return alns[0];
}

// ---------------------------------------------------------------------------------------------------
// Wavefront variant.  Reference entry point (include/centrolign/alignment.hpp:117-125, body :2299-2338):
//
//     template<int NumPW, class Graph, class BackingMap = HashBackedMap>
//     Alignment pwfa_po_poa(const Graph& graph1, const Graph& graph2,
//                           sources1, sources2, sinks1, sinks2,
//                           const AlignmentParameters<NumPW>& params, int64_t prune_limit, int64_t* score_out = nullptr);
//
// The search walks next() lists, so PwfaBatch flattens SUCCESSOR lists in next() order (they and the
// order of the source lists decide ties, alignment.hpp:1788-1826) and calls clb_pwfa_batch.
class PwfaBatch {
public:
    explicit PwfaBatch(int device = 0) : devices_(1, device) { init(); }
    // Several GPUs of one box: the windows are dealt to the devices by (n1+1)+(n2+1) (clb_pwfa_batch_multi) and the
    // results come back in window order.
    explicit PwfaBatch(const std::vector<int>& devices) : devices_(devices.empty() ? std::vector<int>(1, 0) : devices) { init(); }

    size_t size() const { return node_off_[0].size() - 1; }
    const std::vector<int>& devices() const { return devices_; }

    template <class Graph>
    void add(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
             const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
             const std::vector<uint64_t>& sinks2) {
        add_side(0, graph1, sources1, sinks1);
        add_side(1, graph2, sources2, sinks2);
    }

    template <int NumPW, class Params, class AlignmentT = Alignment>
    void align(const Params& params, int64_t prune_limit, std::vector<AlignmentT>& alignments,
               std::vector<int64_t>* scores = nullptr) const {
        static_assert(NumPW >= 1 && NumPW <= CLB_MAX_PW, "1..3 gap pieces");
        clb_params p;
        p.num_pw = NumPW;
        p.match = params.match;
        p.mismatch = params.mismatch;
        for (int k = 0; k < CLB_MAX_PW; ++k) {
            p.gap_open[k] = k < NumPW ? params.gap_open[k] : 0;
            p.gap_extend[k] = k < NumPW ? params.gap_extend[k] : 0;
        }
        const size_t nw = size();
        clb_succ_graph_batch g[2];
        for (int s = 0; s < 2; ++s) {
            g[s].node_off = node_off_[s].data(); g[s].label = label_[s].data(); g[s].edge_off = edge_off_[s].data();
            g[s].pred_off = next_off_[s].data(); g[s].pred = next_[s].data(); g[s].src_off = src_off_[s].data();
            g[s].src = src_[s].data(); g[s].snk_off = snk_off_[s].data(); g[s].snk = snk_[s].data();
        }
        std::vector<int64_t> aln_off(nw + 1, 0), score(nw, 0);
        for (size_t w = 0; w < nw; ++w)
            aln_off[w + 1] = aln_off[w] + (node_off_[0][w + 1] - node_off_[0][w]) + (node_off_[1][w + 1] - node_off_[1][w]);
        std::vector<int32_t> pairs(2 * (size_t)aln_off[nw] + 2);
        std::vector<uint32_t> len(nw, 0);
        const int rc = devices_.size() == 1
                           ? clb_pwfa_batch(devices_[0], (int32_t)nw, &g[0], &g[1], &p, prune_limit, score.data(), aln_off.data(),
                                            pairs.data(), len.data(), nullptr)
                           : clb_pwfa_batch_multi((int)devices_.size(), devices_.data(), (int32_t)nw, &g[0], &g[1], &p, prune_limit,
                                                  score.data(), aln_off.data(), pairs.data(), len.data(), nullptr, nullptr);
        if (rc != CLB_OK) throw std::runtime_error(std::string("centrolign_b200: ") + clb_last_error());
        alignments.assign(nw, AlignmentT());
        for (size_t w = 0; w < nw; ++w) {
            AlignmentT& a = alignments[w];
            a.reserve(len[w]);
            const int32_t* pr = pairs.data() + 2 * aln_off[w];
            for (uint32_t k = 0; k < len[w]; ++k) {
                typedef typename AlignmentT::value_type Pair;
                a.push_back(Pair(pr[2 * k] < 0 ? uint64_t(-1) : (uint64_t)pr[2 * k],
                                 pr[2 * k + 1] < 0 ? uint64_t(-1) : (uint64_t)pr[2 * k + 1]));
            }
        }
        if (scores) *scores = score;
    }

private:
    void init() {
        for (int s = 0; s < 2; ++s) {
            node_off_[s].push_back(0); edge_off_[s].push_back(0); src_off_[s].push_back(0); snk_off_[s].push_back(0);
        }
    }
    template <class Graph>
    void add_side(int s, const Graph& graph, const std::vector<uint64_t>& sources, const std::vector<uint64_t>& sinks) {
        const uint64_t n = graph.node_size();
        uint32_t e = 0;
        next_off_[s].push_back(0);
        for (uint64_t v = 0; v < n; ++v) {
            label_[s].push_back((uint8_t)graph.label(v));
            for (uint64_t u : graph.next(v)) {  // next() order fixes the enumeration order of the search
                next_[s].push_back((uint32_t)u);
                ++e;
            }
            next_off_[s].push_back(e);
        }
        for (uint64_t v : sources) src_[s].push_back((uint32_t)v);
        for (uint64_t v : sinks) snk_[s].push_back((uint32_t)v);
        node_off_[s].push_back(node_off_[s].back() + (int64_t)n);
        edge_off_[s].push_back(edge_off_[s].back() + (int64_t)e);
        src_off_[s].push_back(src_off_[s].back() + (int64_t)sources.size());
        snk_off_[s].push_back(snk_off_[s].back() + (int64_t)sinks.size());
    }

    std::vector<int> devices_;
    std::vector<int64_t> node_off_[2], edge_off_[2], src_off_[2], snk_off_[2];
    std::vector<uint8_t> label_[2];
    std::vector<uint32_t> next_off_[2], next_[2], src_[2], snk_[2];
};

// Drop-in for the reference's pwfa_po_poa: same arguments, same result.
template <int NumPW, class Graph, class Params, class AlignmentT = Alignment>
AlignmentT pwfa_po_poa(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
                       const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
                       const std::vector<uint64_t>& sinks2, const Params& params, int64_t prune_limit,
                       int64_t* score_out = nullptr) {
    PwfaBatch batch;
    batch.add(graph1, graph2, sources1, sources2, sinks1, sinks2);
    std::vector<AlignmentT> alns;
    std::vector<int64_t> scores;
    batch.align<NumPW, Params, AlignmentT>(params, prune_limit, alns, &scores);
    if (score_out) *score_out = scores[0];
    return alns[0];
}

}  // namespace centrolign_b200

#endif  // CENTROLIGN_B200_PO_POA_HPP
