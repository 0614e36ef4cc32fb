/*
 * centrolign_b200.h -- C ABI of the B200-native (sm_100a) gap-fill path.
 *
 * This is the drop-in boundary for the Stitcher's inter-anchor gap fill of
 * jeizenga/centrolign.  The reference has no FFI layer: its boundary is the C++ template
 *
 *     Alignment po_poa<NumPW, Graph>(graph1, graph2, sources1, sources2, sinks1, sinks2,
 *                                    const AlignmentParameters<NumPW>&, int64_t* score_out)
 *         -- reference: include/centrolign/alignment.hpp:78-85 (body :753-1163)
 *
 * called once per inter-anchor window from Stitcher::do_alignment
 * (reference: include/centrolign/stitcher.hpp:295-303) inside the serial loop of
 * Stitcher::stitch (stitcher.hpp:157-203).  The windows of one stitch() call are
 * independent, so this ABI takes a whole BATCH of windows; the C++ wrapper that keeps the
 * reference signature is centrolign_b200/hostcpp/po_poa_b200.hpp, and INTEGRATION.md
 * shows the lines a maintainer adds to stitcher.hpp.
 *
 * Conventions
 *   - plain pointers + sizes, caller-owned host memory, nothing retained after return;
 *   - node ids are window-relative and in the CALLER'S order (no topological order
 *     required; the library renumbers internally);
 *   - predecessor lists are in the graph's previous() order (graph.hpp:111) and source /
 *     sink lists in the caller's order: the reference's traceback tie-breaking
 *     (alignment.hpp:979-990, 1048-1137) depends on both and is reproduced exactly;
 *   - results: per window the optimal score (== *score_out of the reference) and the
 *     alignment as (node_id1, node_id2) int32 pairs, CLB_GAP (-1) = AlignedPair::gap
 *     (alignment.hpp:34-51), in forward order;
 *   - return value 0 = success, otherwise a CLB_E* code; clb_last_error() gives text.
 *     There is no CPU fallback: without a usable CUDA device every compute entry point
 *     fails with CLB_ECUDA.
 */
#ifndef CENTROLIGN_B200_H
#define CENTROLIGN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLB_GAP (-1)
#define CLB_MAX_PW 3

enum {
    CLB_OK = 0,
    CLB_EINVAL = 1,  /* malformed arguments (bad sizes, ids out of range, NumPW not in 1..3) */
    CLB_ECYCLE = 2,  /* a graph is not acyclic (the reference asserts, topological_order.hpp:56) */
    CLB_ECUDA = 3,   /* CUDA runtime / launch failure, or no device */
    CLB_ENOMEM = 4,  /* host or device allocation failed (a window's workspace does not fit) */
    CLB_ESTATE = 5   /* call sequence error on a clb_batch handle */
};

/* AlignmentParameters<NumPW> (alignment.hpp:56-65); penalties are stored positive. */
typedef struct clb_params {
    int32_t num_pw; /* 1..3 */
    uint32_t match;
    uint32_t mismatch;
    uint32_t gap_open[CLB_MAX_PW];
    uint32_t gap_extend[CLB_MAX_PW];
} clb_params;

/* One side (graph1 or graph2) of every window of a batch, concatenated. */
typedef struct clb_graph_batch {
    const int64_t* node_off;  /* [n_windows+1] first node of window w in label[] */
    const uint8_t* label;     /* [node_off[n_windows]] node labels (graph.label(id)), compared for equality */
    const int64_t* edge_off;  /* [n_windows+1] first edge of window w in pred[] */
    const uint32_t* pred_off; /* [node_off[n_windows]+n_windows]; window w owns n_w+1 window-relative
                                 CSR offsets starting at pred_off[node_off[w]+w] */
    const uint32_t* pred;     /* [edge_off[n_windows]] predecessor ids, previous() order */
    const int64_t* src_off;   /* [n_windows+1] */
    const uint32_t* src;      /* sources, caller order */
    const int64_t* snk_off;   /* [n_windows+1] */
    const uint32_t* snk;      /* sinks, caller order */
} clb_graph_batch;

/*
 * One-shot: align every window of the batch on `device`.
 *   score_out [n_windows]                          optimal scores
 *   aln_off   [n_windows+1]  (input)               window w's pairs go to aln_pairs[2*aln_off[w] ...];
 *                                                  capacity aln_off[w+1]-aln_off[w] must be >= n1_w+n2_w
 *   aln_pairs [2*aln_off[n_windows]]               (id1,id2) pairs, forward order
 *   aln_len   [n_windows]                          number of pairs written per window
 * Replaces n_windows calls of po_poa (alignment.hpp:78-85).
 */
int clb_popoa_batch(int device, int32_t n_windows, const clb_graph_batch* g1, const clb_graph_batch* g2,
                    const clb_params* params, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs,
                    uint32_t* aln_len);

/*
 * The same call over several GPUs of one box (BASELINE.json north_star: "work is sharded across the 8 GPUs of one box by
 * cell-balanced window bins ... results return through pinned host memory").  The windows of a stitch are independent
 * (include/centrolign/stitcher.hpp:157-203 reads only its own SubGraphInfo pair per window), so they are dealt to the
 * devices longest-first by DP cell count (n1+1)*(n2+1) (the measure of stitcher.hpp:241), one host thread and CUDA
 * context per device runs the single-device path on its share, and every window's result lands in the caller's arrays at
 * the same place as with clb_popoa_batch -- no device-to-device traffic, no collective.  devices[] lists distinct device
 * ordinals; n_devices == 1 is clb_popoa_batch.  If part_out is not NULL it receives, per window, the index into devices[]
 * the window ran on.
 */
int clb_popoa_batch_multi(int n_devices, const int* devices, int32_t n_windows, const clb_graph_batch* g1,
                          const clb_graph_batch* g2, const clb_params* params, int64_t* score_out, const int64_t* aln_off,
                          int32_t* aln_pairs, uint32_t* aln_len, int32_t* part_out);

/* Host-only: the cell-balanced assignment clb_popoa_batch_multi uses (longest-processing-time-first; ties to the lowest
 * part), part_out[w] in [0, n_parts). */
int clb_balanced_partition(int32_t n_windows, const int64_t* cells, int n_parts, int32_t* part_out);

/*
 * Staged form of the same call, for callers that keep a batch resident in HBM
 * (bench.py times clb_batch_run alone for the device-resident figure):
 *   create   : validate + renumber each graph topologically into pinned host staging
 *   upload   : host -> device copies, workspace allocation
 *   run      : all kernels (fill + traceback), synchronous; results stay on the device
 *   download : device -> host copy of scores / alignments, translated back to caller ids
 */
typedef struct clb_batch clb_batch;

int clb_batch_create(int device, int32_t n_windows, const clb_graph_batch* g1, const clb_graph_batch* g2,
                     const clb_params* params, clb_batch** out);
int clb_batch_upload(clb_batch* b);
int clb_batch_run(clb_batch* b);
int clb_batch_download(clb_batch* b, int64_t* score_out, const int64_t* aln_off, int32_t* aln_pairs,
                       uint32_t* aln_len);
void clb_batch_destroy(clb_batch* b);

/* Introspection for benchmarks (valid after clb_batch_run). */
typedef struct clb_batch_stats {
    double cells;            /* sum over windows of (n1+1)*(n2+1)  (stitcher.hpp:241) */
    double kernel_ms;        /* CUDA-event time of the last run on the batch's stream */
    double fill_ms;          /* of which: time inside the DP-fill kernel launches (0 if fused) */
    int64_t kernel_launches; /* kernels launched by the last run */
    int64_t h2d_bytes;       /* bytes clb_batch_upload copies */
    int64_t d2h_bytes;       /* bytes clb_batch_download copies */
    int64_t workspace_bytes; /* device workspace held by the batch */
    int64_t int_ops;         /* algorithmic INT32 add/max count of the fill (SURVEY.md 8d formula) */
    int64_t persist_bytes;   /* bytes of persisted rows/columns the fill writes to HBM (its algorithmic traffic) */
} clb_batch_stats;
int clb_batch_get_stats(const clb_batch* b, clb_batch_stats* out);

/*
 * Wavefront variant of the gap fill.  Replaces n_windows calls of
 *
 *     Alignment pwfa_po_poa<NumPW, Graph>(graph1, graph2, sources1, sources2, sinks1, sinks2,
 *                                         const AlignmentParameters<NumPW>&, int64_t prune_limit, int64_t* score_out)
 *         -- reference: include/centrolign/alignment.hpp:117-125 (body :2299-2338, search :1959-2033, :1712-1827),
 *            called from Stitcher::do_alignment (include/centrolign/stitcher.hpp:336-339) with
 *            prune_limit = 2 * wfa_pruning_dist.
 *
 * This algorithm walks the graphs FORWARD, so the two sides are given as SUCCESSOR lists: same struct
 * layout as clb_graph_batch, but pred_off / pred hold, per node, its successors in the graph's next()
 * order (include/centrolign/graph.hpp next()); that order and the caller's order of the source lists
 * decide ties (alignment.hpp:1788-1826) and are reproduced exactly: identical alignment, identical score.
 * Outputs as for clb_popoa_batch.  Preconditions are the reference's: acyclic graphs, some source reaches
 * some sink on both sides (else CLB_EINVAL where the reference would dereference an empty queue),
 * non-zero gap_open (the reference's gcd divides by it), prune_limit >= 0.
 */
typedef clb_graph_batch clb_succ_graph_batch;

typedef struct clb_pwfa_stats {
    double kernel_ms;        /* CUDA-event time of the search+traceback kernel(s) */
    int64_t kernel_launches; /* 1 + re-runs of windows whose tables had to be enlarged */
    int64_t retries;         /* enlargement rounds */
    int64_t states;          /* search states settled (first dequeues), all windows */
    int64_t dequeued;        /* queue entries dequeued */
    int64_t steps;           /* warp steps (each resolves up to 32 queue entries in order) */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t workspace_bytes; /* back-pointer tables + FIFOs held during the run */
} clb_pwfa_stats;

int clb_pwfa_batch(int device, int32_t n_windows, const clb_succ_graph_batch* g1, const clb_succ_graph_batch* g2,
                   const clb_params* params, int64_t prune_limit, int64_t* score_out, const int64_t* aln_off,
                   int32_t* aln_pairs, uint32_t* aln_len, clb_pwfa_stats* stats /* may be NULL */);

/*
 * The same call over several GPUs of one box, in the manner of clb_popoa_batch_multi: the windows are dealt to the
 * devices longest-first (clb_balanced_partition) by (n1+1)+(n2+1) -- the search settles about (n1+n2)*band states, so
 * a window's work follows its side lengths, not its cell count -- and one host thread per device runs the single-device
 * path on its share.  Every window's result lands in the caller's arrays at the same place as with clb_pwfa_batch, and
 * error messages name the caller's window index behind "device <ordinal>: ".  Windows whose tables must be enlarged are
 * re-run on their own device.  devices[] lists distinct ordinals (a repeat, or one out of range, is CLB_EINVAL).
 * part_out (may be NULL) receives, per window, the index into devices[] the window ran on.  stats (may be NULL): kernel_ms
 * is the largest over the devices (they run side by side); kernel_launches, retries, states, dequeued, steps, h2d_bytes,
 * d2h_bytes and workspace_bytes are sums over the devices.
 */
int clb_pwfa_batch_multi(int n_devices, const int* devices, int32_t n_windows, const clb_succ_graph_batch* g1,
                         const clb_succ_graph_batch* g2, const clb_params* params, int64_t prune_limit, int64_t* score_out,
                         const int64_t* aln_off, int32_t* aln_pairs, uint32_t* aln_len, int32_t* part_out /* may be NULL */,
                         clb_pwfa_stats* stats /* may be NULL */);

/*
 * Sparse anchor-chaining DP.  Replaces the main loops of
 *
 *     Anchorer::sparse_affine_chain_dp<...>   reference: include/centrolign/anchorer.hpp:1812-2471 (loop :2290-2417)
 *     Anchorer::sparse_chain_dp<...>          reference: include/centrolign/anchorer.hpp:1511-1750 (loop :1640-1728)
 *     Anchorer::traceback_sparse_dp           reference: include/centrolign/anchorer.hpp:2473-2547 (arg-max + back-pointer walk)
 *
 * called through the _gen_sparse_affine / _gen_sparse macros of Anchorer::anchor_chain (anchorer.hpp:1213-1307).
 * The C++ wrapper that keeps those signatures and produces this flat problem from the reference's own
 * MatchBank / ForwardEdges / PathMerge / PostSwitchDistances objects is centrolign_b200/hostcpp/chain_b200.hpp.
 *
 * A match is identified by its RANK in MatchBank iteration order (set, walk1 index, walk2 index ascending,
 * masked matches skipped; match_bank.hpp:251-267) -- order-isomorphic to the reference's match_id_t tuple, which
 * matters because match ids are the low-order part of every search-tree key.
 *
 * "Steps" are the nodes of graph 1 in the reference's topological order (only nodes with events need to be
 * listed).  At a step the reference first enters the DP value of every match ENDING on the node into its
 * search trees (anchorer.hpp:2301-2345), then, for every forward edge leaving the node and every match
 * STARTING on the edge's head, queries the trees and keeps the first strictly greater candidate
 * (:2352-2416).  The result depends on that order, on the order of equal keys inside the trees and on the
 * trees' own traversal order; all three are reproduced (see centrolign_b200/csrc/chain_host.cu).
 * Scores are IEEE float (the reference's ScoreFloat) with the gap terms evaluated in double, as there.
 */
typedef struct clb_chain_problem {
    int32_t num_pw;        /* 0: gap-free sparse_chain_dp; 1..3: sparse_affine_chain_dp with that many gap pieces */
    double gap_open[CLB_MAX_PW];
    double gap_extend[CLB_MAX_PW];
    double scale;          /* local_scale (anchorer.hpp:1821) */
    int32_t n_chain1;      /* xmerge1.chain_size() */
    int32_t n_chain2;      /* xmerge2.chain_size() */
    int64_t n_match;
    const float* weight;     /* [n_match] anchor_weight of the match's set, as ScoreFloat (anchorer.hpp:2367-2368) */
    const float* dp_init;    /* [n_match] single-anchor chain value incl. lead gap, or lowest() (anchorer.hpp:2023-2041) */
    const float* final_term; /* [n_match] final indel score, or lowest() = cannot reach a sink (anchorer.hpp:2431-2438) */
    float min_score;         /* the chain must beat the empty chain (anchorer.hpp:2419-2424) */
    int64_t n_step;
    const int64_t* end_off;     /* [n_step+1] into end_match */
    const uint32_t* end_match;  /* matches ending on the step's node, ends_on() order */
    const int64_t* qry_off;     /* [n_step+1] into qry_match / qry_chain1 */
    const uint32_t* qry_match;  /* matches starting on the head of a forward edge: edge order, then starts_on() order */
    const uint32_t* qry_chain1; /* the edge's chain on graph 1 */
    const int64_t* ins_off;     /* [n_match+1] into ins_*: one entry per (p1,p2) in chains_on(end1) x chains_on(end2), loop order */
    const uint32_t* ins_p1;
    const uint32_t* ins_p2;
    const int32_t* ins_shift;   /* index_on(end1,p1) - index_on(end2,p2)      (anchorer.hpp:1875-1880) */
    const uint32_t* ins_offset; /* index_on(end2,p2)                          (anchorer.hpp:1894-1896) */
    const uint8_t* ins_active;  /* NULL = all 1.  0 marks a key that shapes its search tree but is never entered: the gap-free
                                   sparse_chain_dp builds, for EVERY chain of graph 1, a tree over all matches ending on a chain
                                   of graph 2 (anchorer.hpp:1546-1552, 1595-1603) and enters a match only into the tree of its own
                                   graph-1 chain (:1661-1666); the idle keys still decide the tree's traversal order */
    const int32_t* qa1;  /* [n_match*n_chain1] predecessor_index(start1,c1) + D1(start1,c1), low 32 bits */
    const int32_t* qa2;  /* [n_match*n_chain2] predecessor_index(start2,c2) + D2(start2,c2), low 32 bits;
                            query shift = qa1 - qa2 in wrapping 32-bit arithmetic (anchorer.hpp:1886-1892) */
    const uint32_t* qoff; /* [n_match*n_chain2] predecessor_index(start2,c2) + 1, 0 = nothing reachable (anchorer.hpp:1898-1901) */
} clb_chain_problem;

typedef struct clb_chain_stats {
    double build_ms;   /* host: search-structure layout */
    double kernel_ms;  /* CUDA-event time of the DP kernel */
    double total_ms;   /* whole call */
    int64_t steps, inserts, queries; /* events processed; queries = (match, edge, chain2) triples */
    int64_t tree_bytes;              /* device bytes of the search structures */
    int64_t h2d_bytes, d2h_bytes;
    int64_t kernel_launches;
} clb_chain_stats;

/*
 * The chaining entry points below work on any device ordinal, and calls on different devices run side by side (each
 * device keeps its own buffers and lock); calls on one device are serialised where they use its buffers.
 *
 * Runs the DP on `device` and the reference's traceback.
 *   dp_out      [n_match] final DP values (may be NULL)
 *   backptr_out [n_match] back-pointer match rank, -1 = none (may be NULL)
 *   chain_out   [n_match] capacity; the optimal chain as match ranks in forward order
 *   chain_len   number of matches in the chain (0 = nothing beats min_score)
 *   opt_score   value of the optimum (lowest() if the chain is empty); may be NULL
 */
int clb_chain_dp(int device, const clb_chain_problem* problem, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                 int64_t* chain_len, float* opt_score, clb_chain_stats* stats /* may be NULL */);

/*
 * Many independent chaining problems in one call: the Anchorer's fill-in pass (include/centrolign/anchorer.hpp:619-699)
 * chains the matches inside every gap of the main chain separately, thousands of problems of a few dozen matches each.
 * Every problem whose search structures fit one SM's shared memory is staged into one buffer and solved by ONE kernel
 * launch with a CTA per problem; the others go through clb_chain_dp one by one.  Per problem k the outputs have the
 * meaning of clb_chain_dp: dp_out[k] / backptr_out[k] may be NULL (and the arrays themselves may be NULL), chain_out[k]
 * has capacity n_match of problem k, chain_len[k] and opt_score[k] (array may be NULL) receive the chain length and optimum.
 * stats (may be NULL) accumulates over the batch.
 */
int clb_chain_dp_batch(int device, int64_t n_problems, const clb_chain_problem* const* problems, float* const* dp_out,
                       int64_t* const* backptr_out, int64_t* const* chain_out, int64_t* chain_len, float* opt_score,
                       clb_chain_stats* stats /* may be NULL */);

/*
 * The batched call over several GPUs of one box.  The problems are dealt to the devices longest-first
 * (clb_balanced_partition) by a work estimate -- the DP costs about a step's latency times the steps, so n_step plus the
 * insert and query counts (ins_off[n_match] + qry_off[n_step]) -- and one host thread per device runs clb_chain_dp_batch
 * on its share.  Per problem the outputs are exactly those of clb_chain_dp.  devices[] lists distinct ordinals (a repeat,
 * or one out of range, is CLB_EINVAL); part_out (may be NULL) receives, per problem, the index into devices[] it ran on.
 * stats (may be NULL) accumulates over all problems as in clb_chain_dp_batch; total_ms is the wall time of the call.
 * One problem is never split over devices.
 */
int clb_chain_dp_batch_multi(int n_devices, const int* devices, int64_t n_problems, const clb_chain_problem* const* problems,
                             float* const* dp_out, int64_t* const* backptr_out, int64_t* const* chain_out, int64_t* chain_len,
                             float* opt_score, int32_t* part_out /* may be NULL */, clb_chain_stats* stats /* may be NULL */);

/*
 * The batched call in two halves, for a caller that prepares problems on several host threads (the drop-in Anchorer runs
 * the fill-in subproblems of include/centrolign/anchorer.hpp:657-693 on a thread pool, hostcpp/chain_batcher.hpp):
 *   clb_chain_job_create  lays ONE problem out for the device in the calling thread.  Thread-safe, no device work for a
 *                         problem that fits one SM's shared memory; a larger problem is solved by clb_chain_dp before the call
 *                         returns (its outputs are then final and *job is NULL).  The problem arrays and the output
 *                         pointers (meaning as in clb_chain_dp) must stay valid until the job has run.
 *   clb_chain_jobs_run    solves the jobs of any number of threads: one staging copy, ONE launch (a CTA per problem), one
 *                         read-back, then the tracebacks into every job's outputs.  A job runs once.
 *   clb_chain_job_destroy frees a job (NULL is allowed).
 */
typedef struct clb_chain_job clb_chain_job;
int clb_chain_job_create(int device, const clb_chain_problem* problem, float* dp_out, int64_t* backptr_out, int64_t* chain_out,
                         int64_t* chain_len, float* opt_score, clb_chain_job** job);
int clb_chain_jobs_run(int device, int64_t n_jobs, clb_chain_job* const* jobs);
void clb_chain_job_destroy(clb_chain_job* job);

/* Optional: starts creating the CUDA context of `device` on a background thread and returns at once, so that a process
 * which knows it will use the library overlaps the ~1 s of context creation with its own start-up work (the drop-in CLI
 * calls it from a static initializer; measured 8-10 s -> 7-9 s on the 2 x 100 kbp run).  Only the first call in a
 * process does anything; failures are silent here and surface in the first real call. */
void clb_warm_up(int device);

/* Measured INT32 issue-rate probe (a dependent-free add/max loop on every SM):
 * returns achieved 10^12 INT32 lane-ops per second on `device`, <0 on error. */
double clb_int32_peak_tops(int device, int use_dpx);

/* Host-only diagnostic (no device needed): the 1-based matrix index -- topological rank -- the flattening code gives
 * every node of one graph in predecessor-list form (the order replaces `topological_order`,
 * include/centrolign/topological_order.hpp:11-60; DP values do not depend on which topological order is used,
 * include/centrolign/alignment.hpp:806-807, but predecessor distances do -- DESIGN.md section 4).
 * Returns CLB_OK, CLB_EINVAL or CLB_ECYCLE. */
int clb_topological_ranks(uint32_t n_nodes, const uint32_t* pred_off /* [n_nodes+1] */, const uint32_t* pred,
                          uint32_t* rank_out /* [n_nodes] */);

/* Staging buffers (pinned host, device) are cached across calls; this frees the cache. */
void clb_release_cached_memory(void);

const char* clb_last_error(void);
int clb_device_count(void);

#ifdef __cplusplus
}
#endif
#endif /* CENTROLIGN_B200_H */
