// popoa_host.cu -- host side of the C ABI (include/centrolign_b200.h).
//
// "Flattening": every window's two graphs arrive in the caller's node order, exactly as the
// reference's po_poa receives them (include/centrolign/alignment.hpp:78-85).  Here each graph
// is renumbered by a Kahn topological order (the reference does the same inside po_poa,
// alignment.hpp:806-807 / topological_order.hpp:11-60; DP values do not depend on which
// topological order is used), predecessor lists are rewritten in previous() order with the
// boundary index 0 appended last for sources (alignment.hpp:1069-1084), and the rows / columns
// the kernels must keep ("persisted") are chosen.  Flattening is multi-threaded over windows.
#include <algorithm>
#include <chrono>
#include <cstring>

#include "host_common.cuh"
#include "popoa_device.cuh"

namespace clb {
cudaError_t launch_popoa(int num_pw, const LaunchArgs& args, int grid, cudaStream_t stream);
cudaError_t launch_popoa_small(int num_pw, const LaunchArgs& args, int first, int count, int grid, cudaStream_t stream);  // popoa_small_kernels.cu
int popoa_smem_bytes();
void popoa_wait_profile(bool reset);  // -DCLB_PROFILE builds: where the warps of popoa_kernel wait
double int32_probe(int use_dpx, int sm_count);
int popoa_nsmid();
}  // namespace clb

using clb::fail;
using clb::g_cache;
using clb::Staged;

namespace {
constexpr char kPopoaCalls[] = "[clb] ";  // CLB_COUNT_CALLS line of clb_popoa_batch / clb_popoa_batch_multi
struct SideStage {
    Staged<uint32_t> info, depth, poff, pidx, sinks;
    Staged<int32_t> slot;
    std::vector<uint32_t> orig;  // matrix index -> caller node id (host only)
};
}  // namespace

struct clb_batch {
    int device = 0;
    int32_t nw = 0;
    clb_params params{};
    SideStage s[2];
    Staged<clb::WindowMeta> meta;
    Staged<int32_t> order;
    Staged<int64_t> score;
    Staged<int32_t> aln;
    Staged<uint32_t> aln_len;
    int32_t* d_queue = nullptr;
    char* d_workspace = nullptr;
    size_t workspace_cap = 0;
    int64_t slot_bytes = 0;
    int grid = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool uploaded = false, ran = false;
    clb_batch_stats stats{};
    std::vector<int64_t> out_off;  // pair offset per window in the device output
    std::vector<int32_t> sel;      // caller window id of batch window k (empty = identity)
    bool shared_workspace = false; // workspace owned by the caller of the chunked one-shot path; slots by SM id
    int32_t n_big = 0;             // order[0 .. n_big) go to popoa_kernel, the rest (matrices of <= kSmallCells cells) to popoa_small_kernel
    int sm_count = 0;
    int64_t max_ws_bytes = 0;      // largest single-window workspace of this batch
};

namespace {
// panel configuration of the tiled fill (LaunchArgs::panel_rows, clb::panel_rows_for): read once.  CLB_PANEL_ROWS
// sets the height (a multiple of 64 rows), 0 switches tiling off, "auto" = about n1/8 per window; unset = 2048 rows
// (measured on configs[1]: 1024 / 2048 / 4096 / auto within 1.5 % of each other, 2048 best)
int panel_cfg() {
    static const int v = [] {
        const char* e = getenv("CLB_PANEL_ROWS");
        if (!e) return clb::kPanelRowsMax;
        if (!strcmp(e, "auto")) return -1;
        const int h = atoi(e);
        return h <= 0 ? 0 : std::max(128, h / clb::kRowBlock * clb::kRowBlock);  // tiny panels only add hand-overs
    }();
    return v;
}

struct FlattenScratch {
    std::vector<uint32_t> succ_off, succ, indeg, stack, tpos;
    std::vector<uint8_t> is_src;
};

// Topological numbering of one graph: successor lists + Kahn's algorithm with a stack (keeps chains contiguous).
// Fills sc.tpos[v] = 1-based rank, orig[rank] = v (and leaves the successor lists in sc); returns the number of
// nodes ranked (< n: the graph has a cycle).
uint32_t topological_ranks(uint32_t n, const uint32_t* po, const uint32_t* pr, uint32_t E, FlattenScratch& sc, uint32_t* orig) {
    sc.succ_off.assign(n + 2, 0);
    sc.succ.resize(E + 1);
    sc.indeg.resize(n + 1);
    sc.stack.clear();
    sc.tpos.assign(n + 1, 0);
    sc.is_src.assign(n + 1, 0);
    for (uint32_t k = 0; k < E; ++k) sc.succ_off[pr[k] + 2]++;
    for (uint32_t v = 0; v < n; ++v) sc.succ_off[v + 2] += sc.succ_off[v + 1];
    for (uint32_t v = 0; v < n; ++v)
        for (uint32_t k = po[v]; k < po[v + 1]; ++k) sc.succ[sc.succ_off[pr[k] + 1]++] = v;
    // succ_off[v] .. succ_off[v+1] now delimit v's successors
    for (uint32_t v = 0; v < n; ++v) {
        sc.indeg[v] = po[v + 1] - po[v];
        if (sc.indeg[v] == 0) sc.stack.push_back(v);
    }
    uint32_t cnt = 0;
    // Which of several nodes that become ready together goes first does not change any DP value (alignment.hpp:806-807:
    // any topological order) but it changes how far back predecessors lie.  Fewest successors first, then largest
    // in-degree: an alternative allele is numbered before the backbone node next to it and a merge node before a
    // sibling allele, which keeps both alleles of ADJACENT SNP bubbles within distance 2 of their predecessors
    // (plain LIFO order leaves one of them at distance 3: 35 % -> 12 % of the 128-column strips of configs[1] then
    // need the generic step of the fill kernel).  Ties keep the LIFO order.
    auto goes_later = [&](uint32_t a, uint32_t b) {  // true: a is popped after b, i.e. sits deeper in the stack
        const uint32_t sa = sc.succ_off[a + 1] - sc.succ_off[a], sb = sc.succ_off[b + 1] - sc.succ_off[b];
        if (sa != sb) return sa > sb;
        return po[a + 1] - po[a] < po[b + 1] - po[b];
    };
    while (!sc.stack.empty()) {
        const uint32_t v = sc.stack.back();
        sc.stack.pop_back();
        sc.tpos[v] = ++cnt;
        orig[cnt] = v;
        const size_t base = sc.stack.size();
        for (uint32_t k = sc.succ_off[v]; k < sc.succ_off[v + 1]; ++k)
            if (--sc.indeg[sc.succ[k]] == 0) sc.stack.push_back(sc.succ[k]);
        if (sc.stack.size() - base > 1) std::stable_sort(sc.stack.begin() + (ptrdiff_t)base, sc.stack.end(), goes_later);
    }
    return cnt;
}

// Flatten one side of one window.  Returns CLB_OK / CLB_EINVAL / CLB_ECYCLE.
int flatten_side(const clb_graph_batch& g, int64_t w, int side, SideStage& st, clb::WindowMeta& m, FlattenScratch& sc,
                 int64_t& int_ops_deg /* sum of in-degrees incl. boundary edges */) {
    clb::GraphWindow gw;
    if (clb::graph_window(g, w, gw) != CLB_OK) return CLB_EINVAL;
    const uint32_t n = gw.n, E = gw.n_edge, nsrc = gw.n_src, nsnk = gw.n_snk;
    const uint32_t *po = gw.off, *pr = gw.ids, *src = gw.src, *snk = gw.snk;

    const int64_t nb = (side == 0 ? m.node1 : m.node2);
    const int64_t pb = (side == 0 ? m.poff1 : m.poff2);
    const int64_t xb = (side == 0 ? m.pidx1 : m.pidx2);
    const int64_t kb = (side == 0 ? m.snk1 : m.snk2);
    uint32_t* info = st.info.h + nb;
    int32_t* slot = st.slot.h + nb;
    uint32_t* depth = st.depth.h + nb;
    uint32_t* poff = st.poff.h + pb;
    uint32_t* pidx = st.pidx.h + xb;
    uint32_t* orig = st.orig.data() + nb;
    const uint32_t cnt = topological_ranks(n, po, pr, E, sc, orig);
    if (cnt != n) return CLB_ECYCLE;
    for (uint32_t k = 0; k < nsrc; ++k) sc.is_src[src[k]] = 1;

    const uint32_t block = side == 0 ? (uint32_t)clb::kRowBlock : (uint32_t)clb::kStrip;
    info[0] = clb::kInfoPersist;
    depth[0] = 0;
    orig[0] = 0xffffffffu;
    poff[0] = 0;
    poff[1] = 0;  // the boundary index has no predecessors
    for (uint32_t i = 1; i <= n; ++i) info[i] = 0;
    uint32_t fill = 0;
    for (uint32_t i = 1; i <= n; ++i) {
        const uint32_t v = orig[i];
        uint32_t dmin = 0;
        const uint32_t first = fill;
        for (uint32_t k = po[v]; k < po[v + 1]; ++k) {
            const uint32_t p = sc.tpos[pr[k]];
            pidx[fill++] = p;
            if (depth[p] && (dmin == 0 || depth[p] + 1 < dmin)) dmin = depth[p] + 1;
            if (i - p > (uint32_t)clb::kNear || (i - 1) / block != (p - 1) / block) info[p] |= clb::kInfoPersist;
            if (i - p <= (uint32_t)clb::kNear) info[i] |= 1u << (clb::kInfoNearShift + (i - p - 1));
            else info[i] |= clb::kInfoFar;
        }
        if (sc.is_src[v]) {
            pidx[fill++] = 0;
            dmin = 1;
            info[i] |= clb::kInfoFar;
        }
        depth[i] = dmin;
        poff[i + 1] = fill;
        uint32_t word = (uint32_t)gw.label[v];
        if (fill - first == 1 && pidx[first] == i - 1) {  // regular: also for i == 1 with the boundary as its only predecessor
            word |= clb::kInfoRegular;
            info[i] &= ~(clb::kInfoFar | clb::kInfoNearMask);
            if (i > 1) info[i] |= 1u << clb::kInfoNearShift;
        }
        info[i] |= word;
        int_ops_deg += fill - first;
    }
    // tiled fill (popoa_kernels.cu): a panel takes rows R0-2 .. R0 over from the panel above through the workspace
    if (const uint32_t H = side == 0 ? (uint32_t)clb::panel_rows_for((int)n, panel_cfg()) : 0u)
        for (uint32_t r0 = H; r0 < n; r0 += H)
            for (uint32_t t = 0; t < 3; ++t) info[r0 - t] |= clb::kInfoPersist;
    uint32_t* sinks = st.sinks.h + kb;
    for (uint32_t k = 0; k < nsnk; ++k) {
        sinks[k] = sc.tpos[snk[k]];
        if (side == 0) info[sinks[k]] |= clb::kInfoPersist;  // M at (sink1, sink2) is read from the persisted row
    }
    uint32_t nslot = 0;
    for (uint32_t i = 0; i <= n; ++i) {
        if (info[i] & clb::kInfoPersist) {
            info[i] |= std::min<uint32_t>(nslot, clb::kInfoSlotEscape) << clb::kInfoSlotShift;
            slot[i] = (int32_t)nslot++;
        } else {
            slot[i] = -1;
        }
    }
    if (side == 0) { m.n1 = n; m.nsnk1 = nsnk; m.nrslot = nslot; }
    else { m.n2 = n; m.nsnk2 = nsnk; m.ncslot = nslot; }
    return CLB_OK;
}

}  // namespace

extern "C" {

void clb_batch_destroy(clb_batch* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->d_queue) g_cache.dev_release(b->device, b->d_queue, 4096);
    if (b->d_workspace && !b->shared_workspace) g_cache.dev_release(b->device, b->d_workspace, b->workspace_cap);
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

// Build a batch from all `n_windows` windows (sel == nullptr) or from the `n_sel` windows listed in `sel`.
static int create_internal(int device, int32_t n_windows, const clb_graph_batch* g1, const clb_graph_batch* g2,
                           const clb_params* params, const int32_t* sel, int32_t n_sel, clb_batch** out) {
    if (!out) return fail(CLB_EINVAL, "out is null");
    *out = nullptr;
    if (n_windows < 0 || !params || params->num_pw < 1 || params->num_pw > CLB_MAX_PW)
        return fail(CLB_EINVAL, "bad n_windows or num_pw (must be 1..3)");
    if (n_windows > 0 && (clb::check_graph_batch(g1, n_windows) || clb::check_graph_batch(g2, n_windows)))
        return fail(CLB_EINVAL, "null graph arrays");
    if (const int rc = clb::require_device(device)) return rc;
    CUDA_TRY(cudaSetDevice(device));

    clb_batch* b = new clb_batch();
    b->device = device;
    b->nw = sel ? n_sel : n_windows;
    b->params = *params;
    if (sel) b->sel.assign(sel, sel + n_sel);
    const int64_t nw = b->nw;
    auto src = [&](int64_t k) -> int64_t { return sel ? sel[k] : k; };
    const clb_graph_batch* gs[2] = {g1, g2};
    int rc = b->meta.alloc_host(nw) | b->order.alloc_host(nw) | b->score.alloc_host(nw) | b->aln_len.alloc_host(nw);
    int64_t tot_pairs = 0;
    b->out_off.assign(nw + 1, 0);
    for (int sd = 0; sd < 2 && rc == CLB_OK; ++sd) {
        int64_t N = 0, E = 0, S = 0, K = 0;
        for (int64_t k = 0; k < nw; ++k) {
            const int64_t w = src(k);
            if (w < 0 || w >= n_windows) { rc = CLB_EINVAL; break; }
            N += gs[sd]->node_off[w + 1] - gs[sd]->node_off[w];
            E += gs[sd]->edge_off[w + 1] - gs[sd]->edge_off[w];
            S += gs[sd]->src_off[w + 1] - gs[sd]->src_off[w];
            K += gs[sd]->snk_off[w + 1] - gs[sd]->snk_off[w];
        }
        if (N < 0 || E < 0 || S < 0 || K < 0) rc = CLB_EINVAL;
        SideStage& st = b->s[sd];
        rc |= st.info.alloc_host(N + nw + 2) | st.slot.alloc_host(N + nw) | st.depth.alloc_host(N + nw) |  // info: +2 pad, the fill reads up to two entries past a window
              st.poff.alloc_host(N + 2 * nw) | st.pidx.alloc_host(E + S) | st.sinks.alloc_host(K);
        st.orig.resize(N + nw);
    }
    if (rc != CLB_OK) {
        clb_batch_destroy(b);
        return fail(rc == CLB_EINVAL ? CLB_EINVAL : CLB_ENOMEM, "staging allocation failed");
    }
    {
        int64_t nb[2] = {0, 0}, eb[2] = {0, 0}, kb[2] = {0, 0};  // running node / pidx / sink bases per side
        for (int64_t k = 0; k < nw; ++k) {
            const int64_t w = src(k);
            clb::WindowMeta& m = b->meta.h[k];
            memset(&m, 0, sizeof(m));
            m.node1 = nb[0] + k; m.node2 = nb[1] + k;
            m.poff1 = nb[0] + 2 * k; m.poff2 = nb[1] + 2 * k;
            m.pidx1 = eb[0]; m.pidx2 = eb[1];
            m.snk1 = kb[0]; m.snk2 = kb[1];
            const int64_t n1 = g1->node_off[w + 1] - g1->node_off[w], n2 = g2->node_off[w + 1] - g2->node_off[w];
            if (n1 < 0 || n2 < 0 || n1 > 0x3fffffff || n2 > 0x3fffffff) {
                clb_batch_destroy(b);
                return fail(CLB_EINVAL, "window size out of range");
            }
            nb[0] += n1; nb[1] += n2;
            eb[0] += (g1->edge_off[w + 1] - g1->edge_off[w]) + (g1->src_off[w + 1] - g1->src_off[w]);
            eb[1] += (g2->edge_off[w + 1] - g2->edge_off[w]) + (g2->src_off[w + 1] - g2->src_off[w]);
            kb[0] += g1->snk_off[w + 1] - g1->snk_off[w];
            kb[1] += g2->snk_off[w + 1] - g2->snk_off[w];
            m.out = tot_pairs;
            b->out_off[k] = tot_pairs;
            tot_pairs += n1 + n2;
        }
        b->out_off[nw] = tot_pairs;
    }

    // multi-threaded flatten
    const double t_alloc_done = std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
    const unsigned nthreads = clb::pool_threads(nw, 64);
    std::vector<FlattenScratch> scratch(nthreads);
    std::vector<int64_t> ops_part(nthreads, 0);
    std::vector<double> cells_part(nthreads, 0.0);
    int64_t bad = -1;
    rc = clb::for_each_window(nw, 16, 64, [&](unsigned t, int64_t w) -> int {
        clb::WindowMeta& m = b->meta.h[w];
        int64_t deg1 = 0, deg2 = 0;
        int r = flatten_side(*g1, src(w), 0, b->s[0], m, scratch[t], deg1);
        if (r == CLB_OK) r = flatten_side(*g2, src(w), 1, b->s[1], m, scratch[t], deg2);
        if (r != CLB_OK) return r;
        // SURVEY 8(d): per cell a*b + 1 + 4P(a+b) + 2P add/max; summed over the window this factorises:
        //   sum_ij a_i*b_j = deg1*deg2,  sum_ij (a_i+b_j) = deg1*n2 + deg2*n1   (interior cells only)
        const int64_t P = b->params.num_pw;
        ops_part[t] += deg1 * deg2 + (int64_t)m.n1 * m.n2 * (1 + 2 * P) + 4 * P * (deg1 * (int64_t)m.n2 + deg2 * (int64_t)m.n1);
        cells_part[t] += ((double)m.n1 + 1.0) * ((double)m.n2 + 1.0);
        return CLB_OK;
    }, &bad);
    if (rc != CLB_OK) {
        clb_batch_destroy(b);
        return fail(rc, std::string(rc == CLB_ECYCLE ? "cyclic graph" : "malformed graph") + " in window " + std::to_string(src(bad)));
    }
    if (getenv("CLB_TIMING"))
        fprintf(stderr, "[clb] create: flatten %.3f s on %u threads\n",
                std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count() - t_alloc_done, nthreads);
    b->stats.cells = 0;
    b->stats.int_ops = 0;
    for (unsigned t = 0; t < nthreads; ++t) { b->stats.cells += cells_part[t]; b->stats.int_ops += ops_part[t]; }

    // work order: largest matrix first (longest-processing-time-first for the persistent CTAs)
    std::vector<int32_t> ord(nw);
    for (int64_t w = 0; w < nw; ++w) ord[w] = (int32_t)w;
    std::stable_sort(ord.begin(), ord.end(), [&](int32_t a, int32_t c) {
        const clb::WindowMeta &ma = b->meta.h[a], &mc = b->meta.h[c];
        return ((int64_t)ma.n1 + 1) * ((int64_t)ma.n2 + 1) > ((int64_t)mc.n1 + 1) * ((int64_t)mc.n2 + 1);
    });
    if (nw) memcpy(b->order.h, ord.data(), nw * sizeof(int32_t));
    // small windows (sorted to the end of the order) take the warp-per-window kernel and need no workspace
    b->n_big = (int32_t)nw;
    if (!getenv("CLB_NO_SMALL_WINDOWS"))
        while (b->n_big > 0) {
            const clb::WindowMeta& m = b->meta.h[ord[b->n_big - 1]];
            if (((int64_t)m.n1 + 1) * ((int64_t)m.n2 + 1) > clb::kSmallCells) break;
            --b->n_big;
        }
    b->slot_bytes = 16;
    b->stats.persist_bytes = 0;
    for (int64_t k = 0; k < b->n_big; ++k) {
        const int64_t w = ord[k];
        const clb::WindowMeta& m = b->meta.h[w];
        const int64_t ws = clb::workspace_bytes(m.n1, m.n2, m.nrslot, m.ncslot);
        if (clb::workspace_int4(m.n1, m.n2, m.nrslot, m.ncslot) >= (int64_t(1) << 31)) {
            clb_batch_destroy(b);
            return fail(CLB_ENOMEM, "window " + std::to_string(w) + " needs a workspace beyond the 32-bit offset range (32 GB)");
        }
        b->slot_bytes = std::max(b->slot_bytes, ws);
        b->stats.persist_bytes += ws;
    }
    b->max_ws_bytes = b->slot_bytes;
    b->slot_bytes = (b->slot_bytes + 255) & ~int64_t(255);
    if (b->aln.alloc_host(2 * tot_pairs) != CLB_OK) {
        clb_batch_destroy(b);
        return fail(CLB_ENOMEM, "pinned output allocation failed");
    }
    *out = b;
    return CLB_OK;
}

int clb_batch_create(int device, int32_t n_windows, const clb_graph_batch* g1, const clb_graph_batch* g2,
                     const clb_params* params, clb_batch** out) {
    return create_internal(device, n_windows, g1, g2, params, nullptr, 0, out);
}

static int upload_internal(clb_batch* b, char* shared_ws, int64_t shared_slot_bytes);

int clb_batch_upload(clb_batch* b) { return upload_internal(b, nullptr, 0); }

// shared_ws != nullptr: the workspace belongs to the caller (chunked one-shot path), slot pairs are picked by SM id
static int upload_internal(clb_batch* b, char* shared_ws, int64_t shared_slot_bytes) {
    if (!b) return fail(CLB_EINVAL, "null batch");
    if (b->uploaded) return fail(CLB_ESTATE, "batch already uploaded");
    CUDA_TRY(cudaSetDevice(b->device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, b->device));
    if (prop.major < 10) return fail(CLB_ECUDA, "device is not sm_100-class; this library ships sm_100a code only");
    b->sm_count = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&b->ev0));
    CUDA_TRY(cudaEventCreate(&b->ev1));
    int64_t h2d = 0;
#define UP(P_)                                                                                               \
    do {                                                                                                     \
        if ((P_).alloc_dev(b->device) != CLB_OK) return fail(CLB_ENOMEM, "device allocation failed (" #P_ ")");       \
        if ((P_).n) CUDA_TRY(cudaMemcpyAsync((P_).d, (P_).h, (P_).bytes(), cudaMemcpyHostToDevice, b->stream)); \
        h2d += (int64_t)(P_).bytes();                                                                        \
    } while (0)
    for (auto& s : b->s) {
        UP(s.info); UP(s.slot); UP(s.depth); UP(s.poff); UP(s.pidx); UP(s.sinks);
    }
    UP(b->meta);
    UP(b->order);
#undef UP
    if (b->score.alloc_dev(b->device) || b->aln.alloc_dev(b->device) || b->aln_len.alloc_dev(b->device))
        return fail(CLB_ENOMEM, "device allocation failed (outputs)");
    size_t qcap = 0;
    b->d_queue = (int32_t*)g_cache.dev_alloc(b->device, sizeof(int32_t), &qcap, false);
    if (!b->d_queue) return fail(CLB_ENOMEM, "device allocation failed (queue)");
    // A chunk whose largest window needs more than the shared slot (the slot was sized from the chunk with the most
    // cells; elongated or persist-heavy windows can need more with fewer cells) gets a workspace of its own below.
    if (shared_ws && b->max_ws_bytes > shared_slot_bytes) shared_ws = nullptr;
    if (shared_ws) {
        b->shared_workspace = true;
        b->d_workspace = shared_ws;
        b->slot_bytes = shared_slot_bytes;
        b->grid = std::max(1, std::min<int>(b->n_big, prop.multiProcessorCount));
        CUDA_TRY(cudaStreamSynchronize(b->stream));
        b->stats.h2d_bytes = h2d;
        b->stats.workspace_bytes = 0;
        b->uploaded = true;
        return CLB_OK;
    }
    // one workspace slot per persistent CTA; shrink the grid if memory is short
    size_t free_b = 0, total_b = 0;
    CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    free_b += g_cache.dev_cached(b->device);  // cached blocks are reusable (or trimmed on demand)
    int grid = std::max(1, std::min<int>(b->n_big, prop.multiProcessorCount));
    const int64_t budget = (int64_t)(free_b * 0.92);
    if (b->slot_bytes > budget) return fail(CLB_ENOMEM, "a single window's workspace exceeds device memory");
    // two workspace slots per CTA: one window being filled, the previous one being traced back
    if (2 * b->slot_bytes > budget) return fail(CLB_ENOMEM, "a single window's workspace exceeds device memory");
    grid = (int)std::min<int64_t>(grid, budget / (2 * b->slot_bytes));
    b->grid = std::max(1, grid);
    b->d_workspace = (char*)g_cache.dev_alloc(b->device, (size_t)b->grid * 2 * b->slot_bytes, &b->workspace_cap, true);
    if (!b->d_workspace) return fail(CLB_ENOMEM, "device allocation failed (workspace)");
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    b->stats.h2d_bytes = h2d;
    b->stats.workspace_bytes = (int64_t)b->grid * 2 * b->slot_bytes;
    b->uploaded = true;
    return CLB_OK;
}

static int launch_internal(clb_batch* b);
static int wait_internal(clb_batch* b);

int clb_batch_run(clb_batch* b) {
    const int rc = launch_internal(b);
    return rc == CLB_OK ? wait_internal(b) : rc;
}

static int launch_internal(clb_batch* b) {
    if (!b) return fail(CLB_EINVAL, "null batch");
    if (!b->uploaded) return fail(CLB_ESTATE, "upload the batch before running it");
    CUDA_TRY(cudaSetDevice(b->device));
    b->stats.kernel_launches = 0;
    CUDA_TRY(cudaEventRecord(b->ev0, b->stream));
    if (b->nw > 0) {
        CUDA_TRY(cudaMemsetAsync(b->d_queue, 0, sizeof(int32_t), b->stream));
        clb::LaunchArgs a;
        for (int sd = 0; sd < 2; ++sd) {
            clb::SideArrays& sa = sd == 0 ? a.s1 : a.s2;
            sa.info = b->s[sd].info.d; sa.slot = b->s[sd].slot.d; sa.depth = b->s[sd].depth.d;
            sa.poff = b->s[sd].poff.d; sa.pidx = b->s[sd].pidx.d; sa.sinks = b->s[sd].sinks.d;
        }
        a.meta = b->meta.d; a.order = b->order.d; a.n_windows = b->nw; a.queue = b->d_queue;
        a.workspace = b->d_workspace; a.slot_bytes = b->slot_bytes;
        a.score = b->score.d; a.aln = b->aln.d; a.aln_len = b->aln_len.d;
        a.prm.match = (int)b->params.match;
        a.prm.mismatch = (int)b->params.mismatch;
        for (int k = 0; k < 3; ++k) {
            a.prm.oe[k] = k < b->params.num_pw ? (int)(b->params.gap_open[k] + b->params.gap_extend[k]) : 0;
            a.prm.e[k] = k < b->params.num_pw ? (int)b->params.gap_extend[k] : 0;
        }
        // bit 1: force the generic fill step everywhere (results unchanged; tests use it to cover that path).
        // bit 0 (skip the traceback walk: results invalid, profiling the fill alone) exists only in -DCLB_PROFILE builds.
        a.debug_flags = getenv("CLB_DEBUG_FLAGS") ? atoi(getenv("CLB_DEBUG_FLAGS")) : 0;
#ifndef CLB_PROFILE
        a.debug_flags &= ~1;
#endif
        a.start_lag = getenv("CLB_START_LAG") ? atoi(getenv("CLB_START_LAG")) : 64;
        a.slot_by_smid = b->shared_workspace ? 1 : 0;
        a.panel_rows = panel_cfg();
        a.n_windows = b->n_big;  // the strip / tile kernel takes the windows above kSmallCells ...
        if (b->n_big > 0) {
            CUDA_TRY(clb::launch_popoa(b->params.num_pw, a, b->grid, b->stream));
            b->stats.kernel_launches += 1;
        }
        if (b->nw > b->n_big) {  // ... one warp per window takes the rest
            const int count = b->nw - b->n_big;
            const int sgrid = std::max(1, std::min(b->sm_count, (count + clb::kSmallWarps - 1) / clb::kSmallWarps));
            CUDA_TRY(clb::launch_popoa_small(b->params.num_pw, a, b->n_big, count, sgrid, b->stream));
            b->stats.kernel_launches += 1;
        }
    }
    CUDA_TRY(cudaEventRecord(b->ev1, b->stream));
    return CLB_OK;
}

static int wait_internal(clb_batch* b) {
    CUDA_TRY(cudaSetDevice(b->device));
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    if (getenv("CLB_WAIT_PROFILE")) clb::popoa_wait_profile(false);  // prints and clears the counters (no-op outside -DCLB_PROFILE builds)
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, b->ev0, b->ev1));
    b->stats.kernel_ms = ms;
    b->stats.fill_ms = 0.0;
    b->ran = true;
    return CLB_OK;
}

int clb_batch_download(clb_batch* b, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs, uint32_t* aln_len) {
    if (!b) return fail(CLB_EINVAL, "null batch");
    if (!b->ran) return fail(CLB_ESTATE, "run the batch before downloading results");
    if (b->nw > 0 && (!score_out || !aln_off || !aln_pairs || !aln_len)) return fail(CLB_EINVAL, "null output arrays");
    CUDA_TRY(cudaSetDevice(b->device));
    const int64_t nw = b->nw;
    auto dst_w = [&](int64_t k) -> int64_t { return b->sel.empty() ? k : b->sel[k]; };
    for (int64_t w = 0; w < nw; ++w)
        if (aln_off[dst_w(w) + 1] - aln_off[dst_w(w)] < b->out_off[w + 1] - b->out_off[w])
            return fail(CLB_EINVAL, "alignment capacity of window " + std::to_string(dst_w(w)) + " is below n1+n2");
    if (nw) {
        CUDA_TRY(cudaMemcpyAsync(b->score.h, b->score.d, b->score.bytes(), cudaMemcpyDeviceToHost, b->stream));
        CUDA_TRY(cudaMemcpyAsync(b->aln_len.h, b->aln_len.d, b->aln_len.bytes(), cudaMemcpyDeviceToHost, b->stream));
        if (b->aln.n) CUDA_TRY(cudaMemcpyAsync(b->aln.h, b->aln.d, b->aln.bytes(), cudaMemcpyDeviceToHost, b->stream));
        CUDA_TRY(cudaStreamSynchronize(b->stream));
    }
    b->stats.d2h_bytes = (int64_t)(b->score.bytes() + b->aln_len.bytes() + b->aln.bytes());
    // translate topological ranks back to the caller's node ids; pairs were written backwards
    // from the end of each window's region, so they are already in forward order
    clb::for_each_window(nw, 64, 64, [&](unsigned, int64_t w) -> int {
        const clb::WindowMeta& m = b->meta.h[w];
        const uint32_t len = b->aln_len.h[w];
        const int64_t cap = b->out_off[w + 1] - b->out_off[w];
        const int32_t* src = b->aln.h + 2 * (b->out_off[w] + cap - len);
        int32_t* dst = aln_pairs + 2 * aln_off[dst_w(w)];
        const uint32_t* o1 = b->s[0].orig.data() + m.node1;
        const uint32_t* o2 = b->s[1].orig.data() + m.node2;
        for (uint32_t k = 0; k < len; ++k) {
            const int32_t a = src[2 * k], c = src[2 * k + 1];
            dst[2 * k] = a < 0 ? CLB_GAP : (int32_t)o1[a + 1];
            dst[2 * k + 1] = c < 0 ? CLB_GAP : (int32_t)o2[c + 1];
        }
        aln_len[dst_w(w)] = len;
        score_out[dst_w(w)] = b->score.h[w];
        return CLB_OK;
    });
    return CLB_OK;
}

int clb_batch_get_stats(const clb_batch* b, clb_batch_stats* out) {
    if (!b || !out) return fail(CLB_EINVAL, "null argument");
    *out = b->stats;
    return CLB_OK;
}

int clb_popoa_batch(int device, int32_t n_windows, const clb_graph_batch* g1, const clb_graph_batch* g2,
                    const clb_params* params, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs,
                    uint32_t* aln_len) {
    const bool timing = getenv("CLB_TIMING") != nullptr;
    clb::count_call<kPopoaCalls>(n_windows);
    if (const char* dump_dir = getenv("CLB_DUMP_DIR")) {  // debugging aid: every batch a caller sends, for tools/check_dump.py
        static std::atomic<int> seq(0);
        if (n_windows > 0 && g1 && g2 && params) {
            const std::string path = std::string(dump_dir) + "/popoa_" + std::to_string(seq++) + ".bin";
            if (FILE* f = fopen(path.c_str(), "wb")) {
                const int64_t nw64 = n_windows;
                fwrite(&nw64, 8, 1, f);
                fwrite(params, sizeof(*params), 1, f);
                for (const clb_graph_batch* g : {g1, g2}) {
                    const int64_t N = g->node_off[n_windows], E = g->edge_off[n_windows], S = g->src_off[n_windows], K = g->snk_off[n_windows];
                    const int64_t hdr[4] = {N, E, S, K};
                    fwrite(hdr, 8, 4, f);
                    fwrite(g->node_off, 8, n_windows + 1, f); fwrite(g->label, 1, N, f); fwrite(g->edge_off, 8, n_windows + 1, f);
                    fwrite(g->pred_off, 4, N + n_windows, f); fwrite(g->pred, 4, E, f); fwrite(g->src_off, 8, n_windows + 1, f);
                    fwrite(g->src, 4, S, f); fwrite(g->snk_off, 8, n_windows + 1, f); fwrite(g->snk, 4, K, f);
                }
                fclose(f);
            }
        }
    }
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t0 = now(), t1 = t0, t2 = t0, t3 = t0, t4 = t0;
    // Large batches go through in chunks (largest windows first, geometrically growing host work), each with its
    // own stream: while the GPU works on chunk c the host flattens and uploads chunk c+1, and results of finished
    // chunks are copied back while later chunks still run.  All chunks share one workspace (slot pair = SM id).
    int64_t tot_nodes = 0;
    if (n_windows > 0 && g1 && g2 && g1->node_off && g2->node_off) tot_nodes = g1->node_off[n_windows] + g2->node_off[n_windows];
    // CLB_CHUNK_MIN_NODES lowers the node threshold (tests exercise the chunked path on small batches)
    const int64_t chunk_min_nodes = getenv("CLB_CHUNK_MIN_NODES") ? atoll(getenv("CLB_CHUNK_MIN_NODES")) : (int64_t(1) << 24);
    const bool chunked = n_windows >= 1024 && tot_nodes >= chunk_min_nodes && !getenv("CLB_NO_CHUNKS");
    auto one_batch = [&]() {
        clb_batch* b = nullptr;
        int rc = clb_batch_create(device, n_windows, g1, g2, params, &b);
        t1 = now();
        if (rc == CLB_OK) rc = clb_batch_upload(b);
        t2 = now();
        if (rc == CLB_OK) rc = clb_batch_run(b);
        t3 = now();
        if (rc == CLB_OK) rc = clb_batch_download(b, score_out, aln_off, aln_pairs, aln_len);
        t4 = now();
        clb_batch_destroy(b);
        if (timing)
            fprintf(stderr, "[clb] create %.3f s, upload %.3f s, run %.3f s, download %.3f s, destroy %.3f s\n", t1 - t0,
                    t2 - t1, t3 - t2, t4 - t3, now() - t4);
        return rc;
    };
    if (!chunked) return one_batch();
    if (clb::check_graph_batch(g1) || clb::check_graph_batch(g2) || !params) return fail(CLB_EINVAL, "null graph arrays");
    // windows by matrix size, largest first
    std::vector<int32_t> ord(n_windows);
    for (int32_t w = 0; w < n_windows; ++w) ord[w] = w;
    auto cells_of = [&](int32_t w) {
        return (g1->node_off[w + 1] - g1->node_off[w] + 1) * (g2->node_off[w + 1] - g2->node_off[w] + 1);
    };
    std::stable_sort(ord.begin(), ord.end(), [&](int32_t a, int32_t c) { return cells_of(a) > cells_of(c); });
    static const double kCut[] = {0.03, 0.09, 0.20, 0.40, 0.70, 1.0};
    std::vector<std::pair<int32_t, int32_t>> ranges;  // [begin, end) in ord
    {
        int64_t acc = 0;
        int32_t begin = 0;
        size_t cut = 0;
        for (int32_t i = 0; i < n_windows; ++i) {
            const int32_t w = ord[i];
            acc += (g1->node_off[w + 1] - g1->node_off[w]) + (g2->node_off[w + 1] - g2->node_off[w]);
            if (acc >= kCut[cut] * (double)tot_nodes || i == n_windows - 1) {
                ranges.emplace_back(begin, i + 1);
                begin = i + 1;
                while (cut + 1 < sizeof(kCut) / sizeof(kCut[0]) && acc >= kCut[cut] * (double)tot_nodes) ++cut;
            }
        }
    }
    std::vector<clb_batch*> chunks(ranges.size(), nullptr);
    char* shared_ws = nullptr;
    size_t shared_cap = 0;
    int64_t shared_slot = 0;
    int rc = CLB_OK;
    double t_create = 0, t_upload = 0;
    for (size_t c = 0; c < ranges.size() && rc == CLB_OK; ++c) {
        const double ta = now();
        rc = create_internal(device, n_windows, g1, g2, params, ord.data() + ranges[c].first,
                             ranges[c].second - ranges[c].first, &chunks[c]);
        const double tb = now();
        t_create += tb - ta;
        if (rc != CLB_OK) break;
        if (c == 0) {  // chunk 0 holds the largest windows: its slot size serves every chunk
            const int nsm = clb::popoa_nsmid();
            if (nsm <= 0) { rc = fail(CLB_ECUDA, "could not query the SM id space"); break; }
            shared_slot = (chunks[0]->max_ws_bytes + 255) & ~int64_t(255);
            shared_ws = (char*)g_cache.dev_alloc(device, (size_t)nsm * 2 * shared_slot, &shared_cap, true);
            if (!shared_ws) {  // one slot pair per SM does not fit: the single-batch path shrinks its grid to what does
                clb_batch_destroy(chunks[0]);
                return one_batch();
            }
        }
        rc = upload_internal(chunks[c], shared_ws, shared_slot);
        if (rc == CLB_OK) rc = launch_internal(chunks[c]);
        t_upload += now() - tb;
    }
    t2 = now();
    double t_down = 0, kernel_ms = 0;
    for (size_t c = 0; c < chunks.size() && rc == CLB_OK; ++c) {
        rc = wait_internal(chunks[c]);
        const double ta = now();
        if (rc == CLB_OK) rc = clb_batch_download(chunks[c], score_out, aln_off, aln_pairs, aln_len);
        t_down += now() - ta;
        kernel_ms += chunks[c]->stats.kernel_ms;
    }
    t3 = now();
    if (rc != CLB_OK) cudaDeviceSynchronize();  // no kernel may outlive the shared workspace
    for (clb_batch* b : chunks) clb_batch_destroy(b);
    if (shared_ws) g_cache.dev_release(device, shared_ws, shared_cap);
    if (timing)
        fprintf(stderr, "[clb] %zu chunks: create %.3f s, upload+launch %.3f s (issue phase %.3f s), wait+download %.3f s "
                        "(download %.3f s), sum of kernel times %.1f ms, total %.3f s\n",
                chunks.size(), t_create, t_upload, t2 - t0, t3 - t2, t_down, kernel_ms, now() - t0);
    (void)t1; (void)t4;
    return rc;
}

// Longest-processing-time-first assignment by cell count; ties go to the lowest part.  The same rule as
// centrolign_b200/sharding.py balanced_partition (tests compare the two).
int clb_balanced_partition(int32_t n_windows, const int64_t* cells, int n_parts, int32_t* part_out) {
    if (n_windows < 0 || n_parts < 1 || (n_windows > 0 && (!cells || !part_out))) return fail(CLB_EINVAL, "clb_balanced_partition: bad arguments");
    std::vector<int32_t> ord(n_windows);
    for (int32_t w = 0; w < n_windows; ++w) ord[w] = w;
    std::stable_sort(ord.begin(), ord.end(), [&](int32_t a, int32_t c) { return cells[a] > cells[c]; });
    std::vector<int64_t> load(n_parts, 0);
    for (int32_t w : ord) {
        int best = 0;
        for (int k = 1; k < n_parts; ++k)
            if (load[k] < load[best]) best = k;
        part_out[w] = best;
        load[best] += cells[w];
    }
    return CLB_OK;
}

int clb_popoa_batch_multi(int n_devices, const int* devices, int32_t n_windows, const clb_graph_batch* g1,
                          const clb_graph_batch* g2, const clb_params* params, int64_t* score_out, const int64_t* aln_off,
                          int32_t* aln_pairs, uint32_t* aln_len, int32_t* part_out) {
    if (const int rc = clb::check_devices(n_devices, devices, "clb_popoa_batch_multi")) return rc;
    if (n_devices == 1 || n_windows <= 1) {
        if (part_out) for (int32_t w = 0; w < n_windows; ++w) part_out[w] = 0;
        return clb_popoa_batch(devices[0], n_windows, g1, g2, params, score_out, aln_off, aln_pairs, aln_len);
    }
    if (n_windows < 0 || clb::check_graph_batch(g1) || clb::check_graph_batch(g2) || !params) return fail(CLB_EINVAL, "null graph arrays");
    clb::count_call<kPopoaCalls>(n_windows);
    std::vector<int64_t> cells(n_windows);
    for (int32_t w = 0; w < n_windows; ++w)
        cells[w] = (g1->node_off[w + 1] - g1->node_off[w] + 1) * (g2->node_off[w + 1] - g2->node_off[w] + 1);
    // one host thread (and CUDA context) per device; each writes only its own windows' entries of the output arrays
    return clb::deal_to_devices(n_devices, devices, n_windows, cells.data(), part_out, [&](int k, const std::vector<int32_t>& sel) {
        clb_batch* b = nullptr;
        int r = create_internal(devices[k], n_windows, g1, g2, params, sel.data(), (int32_t)sel.size(), &b);
        if (r == CLB_OK) r = clb_batch_upload(b);
        if (r == CLB_OK) r = clb_batch_run(b);
        if (r == CLB_OK) r = clb_batch_download(b, score_out, aln_off, aln_pairs, aln_len);
        clb_batch_destroy(b);
        return r;
    });
}

// Host-only diagnostic: the matrix index (1-based topological rank) flatten_side gives every node of one graph.
int clb_topological_ranks(uint32_t n_nodes, const uint32_t* pred_off, const uint32_t* pred, uint32_t* rank_out) {
    if (!pred_off || !rank_out || (n_nodes && pred_off[0] != 0)) return fail(CLB_EINVAL, "clb_topological_ranks: bad arguments");
    const uint32_t E = n_nodes ? pred_off[n_nodes] : 0;
    if (E && !pred) return fail(CLB_EINVAL, "clb_topological_ranks: bad arguments");
    for (uint32_t v = 0; v < n_nodes; ++v)
        if (pred_off[v + 1] < pred_off[v]) return fail(CLB_EINVAL, "clb_topological_ranks: predecessor offsets not monotone");
    for (uint32_t k = 0; k < E; ++k)
        if (pred[k] >= n_nodes) return fail(CLB_EINVAL, "clb_topological_ranks: predecessor id out of range");
    FlattenScratch sc;
    std::vector<uint32_t> orig((size_t)n_nodes + 1);
    if (topological_ranks(n_nodes, pred_off, pred, E, sc, orig.data()) != n_nodes) return fail(CLB_ECYCLE, "clb_topological_ranks: the graph has a cycle");
    for (uint32_t v = 0; v < n_nodes; ++v) rank_out[v] = sc.tpos[v];
    return CLB_OK;
}

double clb_int32_peak_tops(int device, int use_dpx) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return -1.0;
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -1.0;
    return clb::int32_probe(use_dpx, prop.multiProcessorCount);
}

}  // extern "C"
