"""Loader for tests/golden/popoa_golden.npz (written by tests/golden/make_golden.py)."""
import hashlib
import json
import os

import numpy as np

from centrolign_b200.batch import (AlignmentParameters, GraphSide, WindowBatch, batch_from_graph_pairs, graph_from_edges,
                                   successor_form, synth_windows)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "popoa_golden.npz")


PWFA_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pwfa_golden.npz")


def load_pwfa_golden():
    """tests/golden/pwfa_golden.npz (tests/golden/make_pwfa_golden.py): outputs of the unmodified reference's
    pwfa_po_poa.  Returns ([batch_v0, batch_v1] in successor form, params, cases[(variant, window, param, prune_limit)],
    scores, alignments)."""
    z = np.load(PWFA_GOLDEN)
    batches = []
    for v in ("v0", "v1"):
        sides = [GraphSide(*[z[f"{v}_{name}_{f}"] for f in
                             ("node_off", "label", "edge_off", "pred_off", "pred", "src_off", "src", "snk_off", "snk")])
                 for name in ("g1", "g2")]
        batches.append(WindowBatch(*sides))
    params = [AlignmentParameters(int(row[0]), int(row[1]), tuple(int(x) for x in row[2:2 + p]),
                                  tuple(int(x) for x in row[5:5 + p]))
              for row, p in zip(z["param_sets"], z["param_num_pw"])]
    alns = [z["aln"][z["aln_off"][k]:z["aln_off"][k + 1]] for k in range(len(z["score"]))]
    return batches, params, z["cases"], z["score"], alns


def load_golden():
    z = np.load(GOLDEN)
    sides = []
    for name in ("g1", "g2"):
        sides.append(GraphSide(*[z[f"{name}_{f}"] for f in
                                 ("node_off", "label", "edge_off", "pred_off", "pred", "src_off", "src", "snk_off", "snk")]))
    batch = WindowBatch(*sides)
    params = []
    for row, p in zip(z["param_sets"], z["param_num_pw"]):
        params.append(AlignmentParameters(int(row[0]), int(row[1]), tuple(int(x) for x in row[2:2 + p]),
                                          tuple(int(x) for x in row[5:5 + p])))
    alns = [z["aln"][z["aln_off"][w]:z["aln_off"][w + 1]] for w in range(batch.n_windows)]
    return batch, params, z["param_idx"], z["score"], alns


# Golden alignments of the reference's own unit test, src/test/test_alignment.cpp:684-773:
# two 7-node double-bubble graphs, AlignmentParameters<1>{match 1, mismatch 1, open 1, extend 1}.
_BUBBLE_EDGES = [(0, 1), (0, 2), (1, 3), (2, 3), (3, 4), (3, 5), (4, 6), (5, 6)]
G = -1
REFERENCE_UNIT_GOLDENS = [
    # (labels1, edges1, src1, snk1, labels2, edges2, src2, snk2, expected pairs)
    ("ACGTGCA", _BUBBLE_EDGES, [0], [6], "AGTTTGA", _BUBBLE_EDGES, [0], [6],
     [(0, 0), (2, 1), (3, 3), (4, 5), (6, 6)]),  # test_alignment.cpp:717-731
    ("ACGTGCAT", _BUBBLE_EDGES + [(7, 0)], [7], [6], "AGTTTGAT", _BUBBLE_EDGES + [(6, 7)], [0], [7],
     [(7, G), (0, 0), (2, 1), (3, 3), (4, 5), (6, 6), (G, 7)]),  # :733-753 lead / trail gaps
    ("AGTTTGAT", _BUBBLE_EDGES + [(6, 7)], [0], [7], "ACGTGCAT", _BUBBLE_EDGES + [(7, 0)], [7], [6],
     [(G, 7), (0, 0), (1, 2), (3, 3), (5, 4), (6, 6), (7, G)]),  # :755-771 flipped
]
# Tie-break probes measured on the built reference (SURVEY.md 8a "Empirical confirmation"):
TIEBREAK_PROBES = [
    # two equal diagonal predecessors on graph 1: the LAST prev1 in previous() order wins
    ("AAC", [(0, 2), (1, 2)], [0, 1], [2], "AC", [(0, 1)], [0], [1], (1, 1, (1,), (1,)), [(1, 0), (2, 1)]),
    ("AAC", [(1, 2), (0, 2)], [0, 1], [2], "AC", [(0, 1)], [0], [1], (1, 1, (1,), (1,)), [(0, 0), (2, 1)]),
    # two equal diagonal predecessors on graph 2: the FIRST prev2 wins
    ("AC", [(0, 1)], [0], [1], "AAC", [(0, 2), (1, 2)], [0, 1], [2], (1, 1, (1,), (1,)), [(0, 0), (1, 2)]),
    # mismatch vs insert+delete tie: gap close beats diagonal, I tested before D
    ("AG", [(0, 1)], [0], [1], "AC", [(0, 1)], [0], [1], (2, 2, (0,), (1,)), [(0, 0), (G, 1), (1, G)]),
]


CHAIN_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "chain_golden.npz")


def load_chain_golden():
    """tests/golden/chain_golden.npz (tests/golden/make_chain_golden.py): chaining problems in the flat
    clb_chain_problem layout with the chains the unmodified reference found.  Returns {case: {kind: ChainProblem}}."""
    from centrolign_b200.chain import problems_from_arrays

    z = np.load(CHAIN_GOLDEN)
    cases = sorted({k.split("/")[0] for k in z.files})
    return {c: problems_from_arrays(z, prefix=c + "/") for c in cases}


LIVE_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "live_golden.json")


def live_runs(name):
    """Inputs on which tests compare with the unmodified reference: [(batch, params, prune_limit)].  prune_limit is None
    for po_poa; for pwfa_po_poa the batch is in successor form."""
    prod = AlignmentParameters()
    if name == "po_poa_oracle":
        batch = synth_windows(24, first_index=100, seed=3, len_min=30, len_max=900, alt_len=41, alt_period=300)
        g = graph_from_edges("ACG", [(0, 1), (1, 2)], [0], [2])
        e = graph_from_edges("", [], [], [])
        return ([(batch, p, None) for p in (prod, prod.truncated(2), AlignmentParameters(1, 1, (1,), (1,)))]
                + [(batch_from_graph_pairs([(g, e), (e, g), (e, e)]), prod, None)])
    if name == "pwfa_oracle":
        batch = synth_windows(10, first_index=500, seed=5, len_min=200, len_max=3000, alt_len=41, alt_period=300)
        return [(sb, p, lim) for sb in (successor_form(batch), successor_form(batch, np.random.default_rng(1)))
                for p, lim in ((prod, 50), (prod.truncated(1), 8))]
    if name == "po_poa_gpu":
        return [(synth_windows(10, first_index=200, seed=9, len_min=100, len_max=1200, alt_len=61, alt_period=400), prod, None)]
    if name == "pwfa_gpu":
        sb = successor_form(synth_windows(8, first_index=1200, seed=2, len_min=500, len_max=7000))
        return [(sb, prod, 50), (sb, prod, 0)]
    raise KeyError(name)


def results_digest(scores, alns):
    """[(score, sha256 of the alignment as little-endian int32 pairs)] per window: the form live_golden.json keeps."""
    return [(int(s), hashlib.sha256(np.ascontiguousarray(a, "<i4").tobytes()).hexdigest()) for s, a in zip(scores, alns)]


def load_live_golden(name):
    """tests/golden/live_golden.json (tests/golden/make_live_golden.py): results_digest of every run of live_runs(name)."""
    with open(LIVE_GOLDEN) as f:
        return [[tuple(x) for x in run] for run in json.load(f)[name]]
