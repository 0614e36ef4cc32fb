// stitch_recorder.hpp -- turns the reference's serial gap-fill loop into ONE batched GPU call.
//
// Stitcher::stitch (reference: include/centrolign/stitcher.hpp:104-206) calls po_poa once per
// inter-anchor window and never looks at the result again: subalign() translates it to parent node ids
// (src/stitcher.cpp:66) and appends it to the stitched alignment (:75-77).  So while the reference's
// loop runs unchanged, the redirected po_poa call only RECORDS the window and hands back a one-pair
// marker (gap, gap) -- a pair the reference never produces -- and the redirected translate() call notes
// the window's back-translation tables.  When the loop is done, all recorded windows go to the GPU in
// one clb_popoa_batch per NumPW, and every marker is replaced, in order, by the translated alignment of
// its window.  The wavefront route (pwfa_po_poa, stitcher.hpp:336-339) is recorded the same way and goes
// out as one clb_pwfa_batch per NumPW.  Both routes use the GPUs of CLB_DEVICES (the _multi calls when it lists more
// than one).  Routing, gap-piece truncation, anchor copies and every other
// route are the reference's own code, executed as is.
#ifndef CENTROLIGN_B200_STITCH_RECORDER_HPP
#define CENTROLIGN_B200_STITCH_RECORDER_HPP

#include <cstdint>
#include <utility>
#include <vector>

#include <stdexcept>
#include <string>

#include "po_poa_b200.hpp"

namespace centrolign_b200 {

template <class AlignmentT>
class StitchRecorder {
public:
    typedef typename AlignmentT::value_type Pair;

    static StitchRecorder& instance() {
        static thread_local StitchRecorder rec;
        return rec;
    }

    bool active() const { return active_; }

    // Scope guard for a recording: if the reference's stitch throws (src/stitcher.cpp:36 does, and the GPU wrappers do on
    // CLB errors) the recorder is switched off again, so that later po_poa calls on this thread are aligned, not recorded.
    struct Scope {
        StitchRecorder& rec;
        explicit Scope(StitchRecorder& r) : rec(r) { rec.begin(); }
        ~Scope() { rec.abandon(); }
    };
    void abandon() {
        active_ = false;
        windows_.clear();
        translations_.clear();
    }

    void begin() {
        active_ = true;
        for (int k = 0; k < CLB_MAX_PW; ++k) {
            batch_[k] = PoPoaBatch(default_devices());  // CLB_DEVICES: several GPUs of the box share every stitch
            wbatch_[k] = PwfaBatch(default_devices());
            have_params_[k] = false;
        }
        windows_.clear();
        translations_.clear();
    }

    // the redirected po_poa call: remember the window, return the marker
    template <int NumPW, class Graph, class Params>
    AlignmentT record(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
                      const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
                      const std::vector<uint64_t>& sinks2, const Params& params) {
        windows_.push_back(std::make_pair(NumPW, batch_[NumPW - 1].size()));
        batch_[NumPW - 1].add(graph1, graph2, sources1, sources2, sinks1, sinks2);
        keep_params<NumPW>(params);
        return marker();
    }

    // the redirected pwfa_po_poa call
    template <int NumPW, class Graph, class Params>
    AlignmentT record_pwfa(const Graph& graph1, const Graph& graph2, const std::vector<uint64_t>& sources1,
                           const std::vector<uint64_t>& sources2, const std::vector<uint64_t>& sinks1,
                           const std::vector<uint64_t>& sinks2, const Params& params, int64_t prune_limit) {
        windows_.push_back(std::make_pair(-NumPW, wbatch_[NumPW - 1].size()));  // negative = wavefront route
        wbatch_[NumPW - 1].add(graph1, graph2, sources1, sources2, sinks1, sinks2);
        prune_limit_ = prune_limit;  // one value per Stitcher (2 * wfa_pruning_dist, stitcher.hpp:339)
        keep_params<NumPW>(params);
        return marker();
    }

private:
    static AlignmentT marker() {
        AlignmentT m;
        m.push_back(Pair(uint64_t(-1), uint64_t(-1)));
        return m;
    }
    template <int NumPW, class Params>
    void keep_params(const Params& params) {
        if (!have_params_[NumPW - 1]) {
            have_params_[NumPW - 1] = true;
            params_[NumPW - 1].match = params.match;
            params_[NumPW - 1].mismatch = params.mismatch;
            for (int k = 0; k < NumPW; ++k) {
                params_[NumPW - 1].gap_open[k] = params.gap_open[k];
                params_[NumPW - 1].gap_extend[k] = params.gap_extend[k];
            }
        }
    }

public:

    // the redirected translate call: true if `aln` is the marker of the window recorded last
    bool note_translation(const AlignmentT& aln, const std::vector<uint64_t>& back_translation1,
                          const std::vector<uint64_t>& back_translation2) {
        if (!active_ || !is_marker(aln) || translations_.size() >= windows_.size()) return false;
        translations_.push_back(std::make_pair(back_translation1, back_translation2));
        return true;
    }

    // run the batches and splice the results over the markers
    AlignmentT finish(AlignmentT&& stitched) {
        active_ = false;
        if (windows_.empty()) return std::move(stitched);
        size_t n_markers = 0;
        for (const Pair& p : stitched) n_markers += (p.node_id1 == uint64_t(-1) && p.node_id2 == uint64_t(-1)) ? 1 : 0;
        if (n_markers != windows_.size() || translations_.size() != windows_.size())
            throw std::runtime_error("centrolign_b200: the stitched alignment holds " + std::to_string(n_markers) + " window markers for " +
                                     std::to_string(windows_.size()) + " recorded windows and " + std::to_string(translations_.size()) +
                                     " translations");
        std::vector<AlignmentT> out[CLB_MAX_PW], wout[CLB_MAX_PW];
        if (batch_[0].size()) batch_[0].template align<1, GenericParams, AlignmentT>(params_[0], out[0]);
        if (batch_[1].size()) batch_[1].template align<2, GenericParams, AlignmentT>(params_[1], out[1]);
        if (batch_[2].size()) batch_[2].template align<3, GenericParams, AlignmentT>(params_[2], out[2]);
        if (wbatch_[0].size()) wbatch_[0].template align<1, GenericParams, AlignmentT>(params_[0], prune_limit_, wout[0]);
        if (wbatch_[1].size()) wbatch_[1].template align<2, GenericParams, AlignmentT>(params_[1], prune_limit_, wout[1]);
        if (wbatch_[2].size()) wbatch_[2].template align<3, GenericParams, AlignmentT>(params_[2], prune_limit_, wout[2]);
        AlignmentT result;
        result.reserve(stitched.size());
        size_t w = 0;
        for (const Pair& p : stitched) {
            if (p.node_id1 == uint64_t(-1) && p.node_id2 == uint64_t(-1)) {
                const int pw = windows_[w].first;
                const AlignmentT& sub = pw > 0 ? out[pw - 1][windows_[w].second] : wout[-pw - 1][windows_[w].second];
                const std::vector<uint64_t>& bt1 = translations_[w].first;
                const std::vector<uint64_t>& bt2 = translations_[w].second;
                for (const Pair& q : sub)  // same mapping as translate(), src/alignment.cpp:26-39
                    result.push_back(Pair(q.node_id1 == uint64_t(-1) ? q.node_id1 : bt1[q.node_id1],
                                          q.node_id2 == uint64_t(-1) ? q.node_id2 : bt2[q.node_id2]));
                ++w;
            } else {
                result.push_back(p);
            }
        }
        return result;
    }

private:
    struct GenericParams {
        uint32_t match, mismatch, gap_open[CLB_MAX_PW], gap_extend[CLB_MAX_PW];
    };
    static bool is_marker(const AlignmentT& aln) {
        return aln.size() == 1 && aln[0].node_id1 == uint64_t(-1) && aln[0].node_id2 == uint64_t(-1);
    }

    bool active_ = false;
    PoPoaBatch batch_[CLB_MAX_PW];
    PwfaBatch wbatch_[CLB_MAX_PW];
    int64_t prune_limit_ = 0;
    GenericParams params_[CLB_MAX_PW];
    bool have_params_[CLB_MAX_PW] = {false, false, false};
    std::vector<std::pair<int, size_t>> windows_;  // (+NumPW po_poa / -NumPW pwfa, index in that batch), in call order
    std::vector<std::pair<std::vector<uint64_t>, std::vector<uint64_t>>> translations_;
};

}  // namespace centrolign_b200

#endif
