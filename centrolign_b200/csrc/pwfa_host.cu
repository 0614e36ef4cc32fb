// pwfa_host.cu -- host side of clb_pwfa_batch and clb_pwfa_batch_multi (include/centrolign_b200.h): the wavefront
// variant of the gap fill, pwfa_po_poa (reference: include/centrolign/alignment.hpp:2299-2338).  Both run the same code
// on a selection of the caller's windows: clb_pwfa_batch selects all of them, the _multi call one share per device.
//
// Per window and side the host computes what the reference computes before its search loop --
// minmax_distance from the sources (minmax_distance.hpp:15-73), target_reachability of the sinks
// (target_reachability.hpp:15-33) -- packs them with label / sink flag / out-degree into one 16-byte
// record per node, appends the sources as the successor list of the virtual start node
// (alignment.hpp:1992-1997), converts the parameters (to_wfa_params, alignment.hpp:1613-1654) and groups
// the transition penalties into classes of equal value (see pwfa_kernels.cu).  The search and the
// traceback run on the device; there is no CPU fallback.
#include <algorithm>
#include <cstring>
#include <numeric>

#include "host_common.cuh"
#include "pwfa_device.cuh"

namespace clb {
cudaError_t launch_pwfa(const PwfaArgs& args, int grid, cudaStream_t stream);
}  // namespace clb

using clb::fail;
using clb::Staged;

namespace {

constexpr char kPwfaCalls[] = "[clb] pwfa ";  // CLB_COUNT_CALLS line of clb_pwfa_batch

uint32_t gcd_u32(uint32_t a, uint32_t b) {
    while (b) {
        const uint32_t r = a % b;
        a = b;
        b = r;
    }
    return a;
}

int ceil_log2(uint64_t v) {
    int l = 0;
    while ((uint64_t(1) << l) < v) ++l;
    return l;
}

struct SideOut {
    Staged<int4> info;
    Staged<uint32_t> next;
    Staged<uint8_t> nlab;
};

struct Scratch {
    std::vector<uint32_t> indeg, order;
    std::vector<int32_t> mind, maxd;
    std::vector<uint8_t> reach, sink;
};

// one side of one window -> node records + successor array (sources appended for the virtual start)
int flatten_side(const clb_succ_graph_batch& g, int64_t w, int4* info, uint32_t* next_out, uint8_t* nlab, Scratch& sc) {
    clb::GraphWindow gw;
    if (clb::graph_window(g, w, gw) != CLB_OK) return CLB_EINVAL;
    const uint32_t n = gw.n, E = gw.n_edge, nsrc = gw.n_src, nsnk = gw.n_snk;
    const uint32_t *no = gw.off, *nx = gw.ids, *src = gw.src, *snk = gw.snk;  // successor lists (see clb_succ_graph_batch)
    const uint8_t* label = gw.label;
    // the node records keep out-degrees and the source count in the 22 bits above kPwfaDegShift
    for (uint32_t v = 0; v < n; ++v)
        if (no[v + 1] - no[v] >= (1u << 22)) return CLB_EINVAL;
    if (nsrc >= (1u << 22)) return CLB_EINVAL;

    sc.indeg.assign(n + 1, 0);
    sc.order.resize(n + 1);
    for (uint32_t k = 0; k < E; ++k) ++sc.indeg[nx[k]];
    uint32_t cnt = 0;
    for (uint32_t v = 0; v < n; ++v)
        if (!sc.indeg[v]) sc.order[cnt++] = v;
    for (uint32_t k = 0; k < cnt; ++k) {
        const uint32_t v = sc.order[k];
        for (uint32_t e = no[v]; e < no[v + 1]; ++e)
            if (--sc.indeg[nx[e]] == 0) sc.order[cnt++] = nx[e];
    }
    if (cnt != n) return CLB_ECYCLE;
    // minmax_distance.hpp:22-60 ("not reached" nodes are never enqueued, their values are never read)
    const int32_t kUnreached = 0x3fffffff;
    sc.mind.assign(n + 1, kUnreached);
    sc.maxd.assign(n + 1, -1);
    for (uint32_t k = 0; k < nsrc; ++k) {
        sc.mind[src[k]] = 0;
        sc.maxd[src[k]] = 0;
    }
    for (uint32_t k = 0; k < n; ++k) {
        const uint32_t v = sc.order[k];
        if (sc.mind[v] == kUnreached) continue;
        for (uint32_t e = no[v]; e < no[v + 1]; ++e) {
            const uint32_t u = nx[e];
            sc.mind[u] = std::min(sc.mind[u], sc.mind[v] + 1);
            sc.maxd[u] = std::max(sc.maxd[u], sc.maxd[v] + 1);
        }
    }
    // target_reachability.hpp:18-30
    sc.reach.assign(n + 1, 0);
    sc.sink.assign(n + 1, 0);
    for (uint32_t k = 0; k < nsnk; ++k) {
        sc.reach[snk[k]] = 1;
        sc.sink[snk[k]] = 1;
    }
    for (uint32_t k = n; k-- > 0;) {
        const uint32_t v = sc.order[k];
        for (uint32_t e = no[v]; e < no[v + 1]; ++e)
            if (sc.reach[nx[e]]) sc.reach[v] = 1;
    }
    for (uint32_t v = 0; v < n; ++v) {
        const uint32_t word = (uint32_t)label[v] | (sc.reach[v] ? clb::kPwfaReach : 0u) | (sc.sink[v] ? clb::kPwfaSink : 0u) |
                              ((no[v + 1] - no[v]) << clb::kPwfaDegShift);
        info[v] = make_int4(sc.mind[v], sc.maxd[v], (int)no[v], (int)word);
    }
    // virtual start: distances -1 (alignment.hpp:2322-2323,2330-2331), never pruned for reachability, successors = sources
    info[n] = make_int4(-1, -1, (int)E, (int)(clb::kPwfaReach | (nsrc << clb::kPwfaDegShift)));
    for (uint32_t k = 0; k < E; ++k) {
        next_out[k] = nx[k];
        nlab[k] = label[nx[k]];
    }
    for (uint32_t k = 0; k < nsrc; ++k) {
        next_out[E + k] = src[k];
        nlab[E + k] = label[src[k]];
    }
    return CLB_OK;
}

// to_wfa_params (alignment.hpp:1630-1651): the penalties divided by their gcd and grouped into classes of equal value
// (a zero gap_open makes the reference divide by zero in its gcd)
int wfa_params(const clb_params* params, int64_t prune_limit, clb::PwfaParams& prm) {
    const int P = params->num_pw;
    prm = clb::PwfaParams{};
    uint32_t w_mismatch = 2 * (params->match + params->mismatch), w_open[3] = {0, 0, 0}, w_ext[3] = {0, 0, 0};
    uint32_t factor = w_mismatch;
    for (int k = 0; k < P; ++k) {
        w_open[k] = 2 * params->gap_open[k];
        w_ext[k] = 2 * params->gap_extend[k] + params->match;
        if (w_open[k] == 0 || w_ext[k] == 0 || factor == 0)
            return fail(CLB_EINVAL, "pwfa needs non-zero gap_open and mismatch+match (the reference's gcd divides by them)");
        factor = gcd_u32(factor, w_open[k]);
        factor = gcd_u32(factor, w_ext[k]);
    }
    if (factor == 0) return fail(CLB_EINVAL, "degenerate scoring parameters");
    w_mismatch /= factor;
    for (int k = 0; k < P; ++k) {
        w_open[k] /= factor;
        w_ext[k] /= factor;
    }
    {
        std::vector<uint32_t> pens = {w_mismatch, 0};
        for (int k = 0; k < P; ++k) {
            pens.push_back(w_open[k] + w_ext[k]);
            pens.push_back(w_ext[k]);
        }
        std::sort(pens.begin(), pens.end(), std::greater<uint32_t>());
        pens.erase(std::unique(pens.begin(), pens.end()), pens.end());
        prm.num_pw = P;
        prm.n_class = (int)pens.size();
        for (size_t c = 0; c < pens.size(); ++c) prm.pen[c] = pens[c];
        auto cls = [&](uint32_t p) { return (int)(std::find(pens.begin(), pens.end(), p) - pens.begin()); };
        prm.cls_mismatch = cls(w_mismatch);
        for (int k = 0; k < P; ++k) {
            prm.cls_open[k] = cls(w_open[k] + w_ext[k]);
            prm.cls_ext[k] = cls(w_ext[k]);
        }
        prm.match = params->match;
        prm.factor = factor;
        prm.prune_limit = (int)std::min<int64_t>(prune_limit, int64_t(1) << 30);
    }
    return CLB_OK;
}

// Windows sel[0..n_sel) of the batch on `device`, in one search launch plus the re-runs of windows whose tables had to be
// enlarged.  Window w = sel[i] is flattened, checked and reported under its own index w, and its results land where
// clb_pwfa_batch puts them; the device arrays hold the selected windows only.
int run_windows(int device, const clb_succ_graph_batch* g1, const clb_succ_graph_batch* g2, const clb::PwfaParams& prm,
                const int32_t* sel, int64_t n_sel, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs,
                uint32_t* aln_len, clb_pwfa_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    const int64_t nw = n_sel;
    const uint64_t max_pen = prm.pen[0];

    // layout
    std::vector<clb::PwfaWindow> win(nw);
    int64_t tot_info[2] = {0, 0}, tot_next[2] = {0, 0}, tot_pairs = 0;
    std::vector<int64_t> out_off(nw + 1, 0);
    for (int64_t i = 0; i < nw; ++i) {
        const int64_t w = sel[i];
        const int64_t n1 = g1->node_off[w + 1] - g1->node_off[w], n2 = g2->node_off[w + 1] - g2->node_off[w];
        if (n1 < 0 || n2 < 0 || n1 >= (int64_t(1) << 30) || n2 >= (int64_t(1) << 28))
            return fail(CLB_EINVAL, "window size out of range");
        // WFA scores are kept in 29 bits: every step costs at most max_pen
        if ((uint64_t)(n1 + n2 + 2) * (max_pen + 1) >= (uint64_t(1) << 29))
            return fail(CLB_EINVAL, "window " + std::to_string(w) + ": WFA score range exceeds 29 bits");
        if (aln_off[w + 1] - aln_off[w] < n1 + n2)
            return fail(CLB_EINVAL, "alignment capacity of window " + std::to_string(w) + " is below n1+n2");
        clb::PwfaWindow& W = win[i];
        W.n1 = (uint32_t)n1;
        W.n2 = (uint32_t)n2;
        W.info1 = tot_info[0];
        W.info2 = tot_info[1];
        W.next1 = tot_next[0];
        W.next2 = tot_next[1];
        W.out = tot_pairs;
        out_off[i] = tot_pairs;
        tot_info[0] += n1 + 1;
        tot_info[1] += n2 + 1;
        tot_next[0] += (g1->edge_off[w + 1] - g1->edge_off[w]) + (g1->src_off[w + 1] - g1->src_off[w]);
        tot_next[1] += (g2->edge_off[w + 1] - g2->edge_off[w]) + (g2->src_off[w + 1] - g2->src_off[w]);
        tot_pairs += n1 + n2;
        const int env_h = getenv("CLB_PWFA_HASH_LOG2") ? atoi(getenv("CLB_PWFA_HASH_LOG2")) : 0;
        const int env_q = getenv("CLB_PWFA_FIFO_LOG2") ? atoi(getenv("CLB_PWFA_FIFO_LOG2")) : 0;
        W.hash_log2 = (uint32_t)(env_h ? env_h : std::max(10, ceil_log2(16 * (uint64_t)(n1 + n2 + 2))));
        W.fifo_log2 = (uint32_t)(env_q ? env_q : std::max(10, ceil_log2((uint64_t)(n1 + n2 + 2))));
    }
    out_off[nw] = tot_pairs;

    if (cudaSetDevice(device) != cudaSuccess) return fail(CLB_ECUDA, "cudaSetDevice failed");
    SideOut so[2];
    for (int sd = 0; sd < 2; ++sd)
        if (so[sd].info.alloc(device, tot_info[sd], true) || so[sd].next.alloc(device, tot_next[sd], true) ||
            so[sd].nlab.alloc(device, tot_next[sd], true))
            return fail(CLB_ENOMEM, "pwfa: staging allocation failed");
    {
        std::vector<Scratch> scratch(clb::pool_threads(nw, 8));
        int64_t bad = -1;
        const int r = clb::for_each_window(nw, 1, 8, [&](unsigned t, int64_t i) {
            const int r1 = flatten_side(*g1, sel[i], so[0].info.h + win[i].info1, so[0].next.h + win[i].next1,
                                        so[0].nlab.h + win[i].next1, scratch[t]);
            if (r1 != CLB_OK) return r1;
            return flatten_side(*g2, sel[i], so[1].info.h + win[i].info2, so[1].next.h + win[i].next2, so[1].nlab.h + win[i].next2,
                                scratch[t]);
        }, &bad);
        if (r != CLB_OK)
            return fail(r, "window " + std::to_string(sel[bad]) + (r == CLB_ECYCLE ? ": graph has a cycle" : ": malformed graph arrays"));
    }

    int rc = CLB_OK;
    Staged<clb::PwfaWindow> s_win;
    Staged<int32_t> s_order, s_queue, s_status, s_aln;
    Staged<int64_t> s_score, s_wstats;
    Staged<uint32_t> s_len;
    Staged<char> s_ws;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<int32_t> pending(nw);
    int64_t h2d = 0;
    cudaDeviceProp prop;

    CUDA_TRY_CLEANUP(cudaGetDeviceProperties(&prop, device));
    CUDA_TRY_CLEANUP(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CUDA_TRY_CLEANUP(cudaEventCreate(&ev0));
    CUDA_TRY_CLEANUP(cudaEventCreate(&ev1));
    for (int sd = 0; sd < 2; ++sd) {
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(so[sd].info.d, so[sd].info.h, (size_t)tot_info[sd] * sizeof(int4), cudaMemcpyHostToDevice, stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(so[sd].next.d, so[sd].next.h, (size_t)tot_next[sd] * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(so[sd].nlab.d, so[sd].nlab.h, (size_t)tot_next[sd], cudaMemcpyHostToDevice, stream));
        h2d += tot_info[sd] * (int64_t)sizeof(int4) + tot_next[sd] * 5;
    }
    if (s_win.alloc(device, nw, true) || s_order.alloc(device, nw, true) || s_queue.alloc(device, 1, false) ||
        s_status.alloc(device, nw, true) || s_score.alloc(device, nw, true) || s_wstats.alloc(device, 4 * nw, true) ||
        s_len.alloc(device, nw, true) || s_aln.alloc(device, 2 * tot_pairs, true)) {
        rc = fail(CLB_ENOMEM, "pwfa: result buffer allocation failed");
        goto cleanup;
    }
    h2d += nw * (sizeof(clb::PwfaWindow) + sizeof(int32_t));

    std::iota(pending.begin(), pending.end(), 0);
    for (int round = 0; !pending.empty(); ++round) {
        if (round > 10) {
            rc = fail(CLB_ENOMEM, "pwfa: a window still overflows its tables after 10 enlargements");
            goto cleanup;
        }
        std::stable_sort(pending.begin(), pending.end(), [&](int32_t a, int32_t c) {
            return (int64_t)win[a].n1 + win[a].n2 > (int64_t)win[c].n1 + win[c].n2;
        });
        int64_t slot_bytes = 0;
        for (int32_t w : pending)
            slot_bytes = std::max<int64_t>(slot_bytes, ((int64_t(1) << win[w].hash_log2) +
                                                        (int64_t)prm.n_class * (int64_t(1) << win[w].fifo_log2)) * 16);
        size_t free_b = 0, total_b = 0;
        CUDA_TRY_CLEANUP(cudaMemGetInfo(&free_b, &total_b));
        const int warps_per_sm = getenv("CLB_PWFA_WARPS_PER_SM") ? std::max(1, atoi(getenv("CLB_PWFA_WARPS_PER_SM"))) : 16;
        int grid = (int)std::min<int64_t>((int64_t)pending.size(), (int64_t)prop.multiProcessorCount * warps_per_sm);
        grid = (int)std::min<int64_t>(grid, (int64_t)(free_b * 0.9) / slot_bytes);
        if (grid < 1) {
            rc = fail(CLB_ENOMEM, "pwfa: the tables of one window (" + std::to_string(slot_bytes) + " B) do not fit in device memory");
            goto cleanup;
        }
        s_ws.release();
        if (s_ws.alloc(device, (size_t)grid * slot_bytes, false, true)) {
            rc = fail(CLB_ENOMEM, "pwfa: workspace allocation failed");
            goto cleanup;
        }
        memcpy(s_win.h, win.data(), nw * sizeof(clb::PwfaWindow));
        memcpy(s_order.h, pending.data(), pending.size() * sizeof(int32_t));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_win.d, s_win.h, nw * sizeof(clb::PwfaWindow), cudaMemcpyHostToDevice, stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_order.d, s_order.h, pending.size() * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
        CUDA_TRY_CLEANUP(cudaMemsetAsync(s_queue.d, 0, sizeof(int32_t), stream));
        clb::PwfaArgs a{};
        a.info1 = so[0].info.d; a.info2 = so[1].info.d;
        a.next1 = so[0].next.d; a.next2 = so[1].next.d;
        a.nlab1 = so[0].nlab.d; a.nlab2 = so[1].nlab.d;
        a.win = s_win.d; a.order = s_order.d; a.n_run = (int32_t)pending.size(); a.queue = s_queue.d;
        a.workspace = s_ws.d; a.slot_bytes = slot_bytes;
        a.score = s_score.d; a.status = s_status.d; a.aln_len = s_len.d; a.aln = s_aln.d; a.wstats = s_wstats.d;
        a.prm = prm;
        CUDA_TRY_CLEANUP(cudaEventRecord(ev0, stream));
        CUDA_TRY_CLEANUP(clb::launch_pwfa(a, grid, stream));
        CUDA_TRY_CLEANUP(cudaEventRecord(ev1, stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_status.h, s_status.d, nw * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_wstats.h, s_wstats.d, 4 * nw * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
        CUDA_TRY_CLEANUP(cudaStreamSynchronize(stream));
        float ms = 0.f;
        CUDA_TRY_CLEANUP(cudaEventElapsedTime(&ms, ev0, ev1));
        if (stats) {
            stats->kernel_ms += ms;
            stats->kernel_launches += 1;
            stats->workspace_bytes = std::max<int64_t>(stats->workspace_bytes, (int64_t)grid * slot_bytes);
            stats->retries = round;
        }
        std::vector<int32_t> again;
        for (int32_t i : pending) {
            const int s = s_status.h[i];
            if (s == clb::kPwfaOk) {
                if (stats) {
                    stats->states += s_wstats.h[4 * i];
                    stats->dequeued += s_wstats.h[4 * i + 1];
                    stats->steps += s_wstats.h[4 * i + 3];
                }
            } else if (s == clb::kPwfaHashFull || s == clb::kPwfaFifoFull) {
                // the two grow together (queue entries per settled state are bounded by the out-degrees)
                win[i].hash_log2 += 2;
                win[i].fifo_log2 += 2;
                again.push_back(i);
            } else if (s == clb::kPwfaQueueDry) {
                // the reference dereferences an empty deque here (alignment.hpp:1738): its precondition is violated
                rc = fail(CLB_EINVAL, "window " + std::to_string(sel[i]) + ": no source reaches a sink within the pruning rule");
                goto cleanup;
            } else {
                rc = fail(CLB_ECUDA, "window " + std::to_string(sel[i]) + ": internal pwfa kernel error " + std::to_string(s));
                goto cleanup;
            }
        }
        pending.swap(again);
    }
    CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_score.h, s_score.d, nw * sizeof(int64_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_len.h, s_len.d, nw * sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY_CLEANUP(cudaMemcpyAsync(s_aln.h, s_aln.d, 2 * tot_pairs * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CUDA_TRY_CLEANUP(cudaStreamSynchronize(stream));
    for (int64_t i = 0; i < nw; ++i) {
        const int32_t w = sel[i];
        const uint32_t len = s_len.h[i];
        const int64_t cap = out_off[i + 1] - out_off[i];
        memcpy(aln_pairs + 2 * aln_off[w], s_aln.h + 2 * (out_off[i] + cap - len), 2 * (size_t)len * sizeof(int32_t));
        aln_len[w] = len;
        score_out[w] = s_score.h[i];
    }
    if (stats) {
        stats->h2d_bytes = h2d;
        stats->d2h_bytes = nw * 12 + 2 * tot_pairs * 4;
    }

cleanup:
    if (rc != CLB_OK) cudaDeviceSynchronize();  // nothing may still run on buffers that go back to the cache
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
    return rc;
}

// The argument checks of both entry points, in the order of clb_pwfa_batch.
int check_pwfa_args(int32_t n_windows, const clb_succ_graph_batch* g1, const clb_succ_graph_batch* g2, const clb_params* params,
                    int64_t prune_limit, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs, uint32_t* aln_len) {
    if (n_windows < 0 || !params || params->num_pw < 1 || params->num_pw > CLB_MAX_PW)
        return fail(CLB_EINVAL, "bad window count or NumPW outside 1..3");
    if (prune_limit < 0) return fail(CLB_EINVAL, "prune_limit must be >= 0");
    if (n_windows > 0 && (clb::check_graph_batch(g1, n_windows) || clb::check_graph_batch(g2, n_windows)))
        return fail(CLB_EINVAL, "null graph arrays");
    if (n_windows > 0 && (!score_out || !aln_off || !aln_pairs || !aln_len)) return fail(CLB_EINVAL, "null output arrays");
    return CLB_OK;
}

}  // namespace

extern "C" int clb_pwfa_batch(int device, int32_t n_windows, const clb_succ_graph_batch* g1, const clb_succ_graph_batch* g2,
                              const clb_params* params, int64_t prune_limit, int64_t* score_out, const int64_t* aln_off,
                              int32_t* aln_pairs, uint32_t* aln_len, clb_pwfa_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (const int rc = check_pwfa_args(n_windows, g1, g2, params, prune_limit, score_out, aln_off, aln_pairs, aln_len)) return rc;
    if (const int rc = clb::require_device(device)) return rc;
    clb::count_call<kPwfaCalls>(n_windows);
    if (n_windows == 0) return CLB_OK;
    clb::PwfaParams prm;
    if (const int rc = wfa_params(params, prune_limit, prm)) return rc;
    std::vector<int32_t> all(n_windows);
    std::iota(all.begin(), all.end(), 0);
    return run_windows(device, g1, g2, prm, all.data(), n_windows, score_out, aln_off, aln_pairs, aln_len, stats);
}

// The windows dealt to the devices by (n1+1)+(n2+1): the search settles about (n1+n2)*band states (DESIGN.md section 9),
// so a window's work grows with its side lengths, not with its cell count.
extern "C" int clb_pwfa_batch_multi(int n_devices, const int* devices, int32_t n_windows, const clb_succ_graph_batch* g1,
                                    const clb_succ_graph_batch* g2, const clb_params* params, int64_t prune_limit, int64_t* score_out,
                                    const int64_t* aln_off, int32_t* aln_pairs, uint32_t* aln_len, int32_t* part_out,
                                    clb_pwfa_stats* stats) {
    if (stats) memset(stats, 0, sizeof(*stats));
    if (const int rc = clb::check_devices(n_devices, devices, "clb_pwfa_batch_multi")) return rc;
    if (const int rc = check_pwfa_args(n_windows, g1, g2, params, prune_limit, score_out, aln_off, aln_pairs, aln_len)) return rc;
    for (int k = 0; k < n_devices; ++k)
        if (const int rc = clb::require_device(devices[k])) return rc;
    clb::count_call<kPwfaCalls>(n_windows);
    if (n_windows == 0) return CLB_OK;
    clb::PwfaParams prm;
    if (const int rc = wfa_params(params, prune_limit, prm)) return rc;
    std::vector<int64_t> cost(n_windows);
    for (int32_t w = 0; w < n_windows; ++w)
        cost[w] = (g1->node_off[w + 1] - g1->node_off[w] + 1) + (g2->node_off[w + 1] - g2->node_off[w] + 1);
    std::vector<clb_pwfa_stats> dev_stats(n_devices);
    const int rc = clb::deal_to_devices(n_devices, devices, n_windows, cost.data(), part_out, [&](int k, const std::vector<int32_t>& sel) {
        return run_windows(devices[k], g1, g2, prm, sel.data(), (int64_t)sel.size(), score_out, aln_off, aln_pairs, aln_len,
                           stats ? &dev_stats[k] : nullptr);
    });
    if (stats)
        for (const clb_pwfa_stats& d : dev_stats) {  // the devices run side by side: the longest kernel time, summed counters
            stats->kernel_ms = std::max(stats->kernel_ms, d.kernel_ms);
            stats->kernel_launches += d.kernel_launches;
            stats->retries += d.retries;
            stats->states += d.states;
            stats->dequeued += d.dequeued;
            stats->steps += d.steps;
            stats->h2d_bytes += d.h2d_bytes;
            stats->d2h_bytes += d.d2h_bytes;
            stats->workspace_bytes += d.workspace_bytes;
        }
    return rc;
}
