"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle
(oracle/po_poa_oracle.c), the committed reference fixtures, recorded results (tests/golden/live_golden.json)
and, where it is built, the unmodified reference itself (oracle/_ref/libclref.so).  Integer DP: bit-exact
scores and identical alignments are required."""
import numpy as np
import pytest

from centrolign_b200.batch import (AlignmentParameters, batch_from_graph_pairs, concat_batches,
                                   graph_from_edges, random_bubble_chain, random_dag, select_windows,
                                   sources_and_sinks, synth_windows)
from centrolign_b200.popoa import DeviceBatch, po_poa_batch
from checkers import CpuChecker  # test infrastructure: tests/checkers.py
from golden_io import REFERENCE_UNIT_GOLDENS, TIEBREAK_PROBES, live_runs, load_golden, load_live_golden, results_digest

pytestmark = pytest.mark.gpu

PROD = AlignmentParameters()


def _compare(batch, params, scores, alns, checker, tag):
    for w in range(batch.n_windows):
        s, a = checker.po_poa(batch, w, params)
        assert s == scores[w], f"{tag}: window {w} score {scores[w]} != {s} (n1={batch.g1.n(w)}, n2={batch.g2.n(w)})"
        assert np.array_equal(a, alns[w]), f"{tag}: window {w} alignment differs (n1={batch.g1.n(w)}, n2={batch.g2.n(w)})"


def _unit_batch(cases):
    return batch_from_graph_pairs([(graph_from_edges(c[0], c[1], c[2], c[3]), graph_from_edges(c[4], c[5], c[6], c[7]))
                                   for c in cases])


def test_reference_unit_goldens():
    batch = _unit_batch(REFERENCE_UNIT_GOLDENS)
    _, alns = po_poa_batch(batch, AlignmentParameters(1, 1, (1,), (1,)))
    for w, case in enumerate(REFERENCE_UNIT_GOLDENS):
        assert [tuple(x) for x in alns[w].tolist()] == case[8]


def test_tiebreak_probes():
    for w, case in enumerate(TIEBREAK_PROBES):
        batch = _unit_batch([case])
        _, alns = po_poa_batch(batch, AlignmentParameters(*case[8]))
        assert [tuple(x) for x in alns[0].tolist()] == case[9], f"probe {w}"


def test_golden_fixture():
    batch, params, pidx, scores, alns = load_golden()
    for k, p in enumerate(params):
        idx = np.nonzero(pidx == k)[0]
        sub = select_windows(batch, idx)
        got_s, got_a = po_poa_batch(sub, p)
        for n, w in enumerate(idx):
            assert got_s[n] == scores[w], f"golden window {w} (P={p.num_pw}): score {got_s[n]} != {scores[w]}"
            assert np.array_equal(got_a[n], alns[w]), f"golden window {w} (P={p.num_pw}): alignment differs"


def test_empty_and_degenerate_windows():
    oracle = CpuChecker("port")
    g = graph_from_edges("ACG", [(0, 1), (1, 2)], [0], [2])
    one = graph_from_edges("A", [], [0], [0])
    e = graph_from_edges("", [], [], [])
    nosink = graph_from_edges("AC", [(0, 1)], [0], [])
    batch = batch_from_graph_pairs([(g, e), (e, g), (e, e), (one, one), (one, g), (g, one), (g, nosink)])
    for p in (PROD, PROD.truncated(1), AlignmentParameters(1, 1, (1,), (1,))):
        scores, alns = po_poa_batch(batch, p)
        _compare(batch, p, scores, alns, oracle, "degenerate")
    scores, alns = po_poa_batch(batch_from_graph_pairs([]), PROD)
    assert len(scores) == 0 and alns == []


@pytest.mark.parametrize("num_pw", [1, 2, 3])
def test_random_small_graphs_vs_oracle(num_pw):
    oracle = CpuChecker("port")
    rng = np.random.default_rng(1000 + num_pw)
    pairs = []
    for t in range(400):
        sides = []
        for _ in range(2):
            if t % 2 == 0:
                n = int(rng.integers(2, 40))
                labels, edges = random_dag(rng, n, int(rng.integers(n, 3 * n)), alphabet="AC")
            else:
                labels, edges = random_bubble_chain(rng, int(rng.integers(2, 200)))
            src, snk = sources_and_sinks(len(labels), edges)
            sides.append(graph_from_edges(labels, edges, src, snk))
        pairs.append(tuple(sides))
    batch = batch_from_graph_pairs(pairs)
    for p in (PROD.truncated(num_pw), AlignmentParameters(3, 2, (1, 4, 9)[:num_pw], (3, 2, 1)[:num_pw])):
        scores, alns = po_poa_batch(batch, p)
        _compare(batch, p, scores, alns, oracle, f"random P={num_pw}")


def test_synthetic_hor_windows_vs_oracle():
    """Windows spanning several strips and row blocks, incl. long alternate-path bubbles."""
    oracle = CpuChecker("port")
    batch = concat_batches([
        synth_windows(24, first_index=0, seed=5, len_min=30, len_max=1500, alt_len=41, alt_period=300),
        synth_windows(6, first_index=50, seed=5, len_min=1500, len_max=3000),
    ])
    for p in (PROD, PROD.truncated(2)):
        scores, alns = po_poa_batch(batch, p)
        _compare(batch, p, scores, alns, oracle, f"synthetic P={p.num_pw}")


def test_skewed_shapes_vs_oracle():
    oracle = CpuChecker("port")
    rng = np.random.default_rng(7)
    pairs = []
    for n1, n2 in ((1, 300), (300, 1), (3, 700), (700, 3), (33, 65), (64, 32), (65, 33), (129, 31)):
        sides = []
        for n in (n1, n2):
            labels, edges = random_bubble_chain(rng, n, snp_rate=0.1, del_rate=0.03)
            src, snk = sources_and_sinks(len(labels), edges)
            sides.append(graph_from_edges(labels, edges, src, snk))
        pairs.append(tuple(sides))
    batch = batch_from_graph_pairs(pairs)
    scores, alns = po_poa_batch(batch, PROD)
    _compare(batch, PROD, scores, alns, oracle, "skewed")


def _irregular_chain(rng, length):
    """Backbone with SNP bubbles, short skip edges (distance 2..7: near, distance-3 and previous-lane far
    predecessors), long skip edges (far predecessors in earlier lanes / strips, several into one node) and
    extra source nodes joining the chain late (a boundary predecessor far from column 1)."""
    labels, edges = random_bubble_chain(rng, length, snp_rate=0.08, del_rate=0.04)
    labels = list(labels)
    edges = set(edges)
    for _ in range(max(2, length // 60)):  # short skips incl. distances 4..7
        p = int(rng.integers(0, length - 9))
        edges.add((p, p + 2 + int(rng.integers(0, 6))))
    for _ in range(max(2, length // 120)):  # long skips, sometimes two into the same node
        q = int(rng.integers(10, length))
        for _ in range(1 + int(rng.integers(0, 2))):
            p = int(rng.integers(max(0, q - 400), q - 8))
            edges.add((p, q))
    for _ in range(2):  # late sources
        a = len(labels)
        labels.append("ACGT"[int(rng.integers(0, 4))])
        edges.add((a, int(rng.integers(1, length))))
    edges = [(int(a), int(b)) for a, b in edges]
    rng.shuffle(edges)
    return "".join(labels), edges


@pytest.mark.parametrize("num_pw", [1, 3])
def test_wide_strips_irregular_graphs_vs_oracle(num_pw):
    """The 128-column strip path (windows of at least 384 columns) on graphs that are not the benchmark's:
    every predecessor shape the fill distinguishes (near 1..3, far through the fast and the generic path,
    persisted columns anywhere in a lane) on both sides, checked cell-exactly through score + alignment."""
    oracle = CpuChecker("port")
    rng = np.random.default_rng(4242 + num_pw)
    pairs = []
    for t in range(24):
        sides = []
        for _ in range(2):
            labels, edges = _irregular_chain(rng, int(rng.integers(400, 1300)))
            src, snk = sources_and_sinks(len(labels), edges)
            sides.append(graph_from_edges(labels, edges, src, snk))
        pairs.append(tuple(sides))
    batch = batch_from_graph_pairs(pairs)
    p = PROD.truncated(num_pw)
    scores, alns = po_poa_batch(batch, p)
    _compare(batch, p, scores, alns, oracle, f"wide irregular P={num_pw}")


_TILED_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
from centrolign_b200.batch import (AlignmentParameters, batch_from_graph_pairs, concat_batches, graph_from_edges,
                                   random_bubble_chain, sources_and_sinks, synth_windows)
from centrolign_b200.popoa import po_poa_batch
from checkers import CpuChecker
import test_popoa_gpu as t
oracle = CpuChecker("port")
rng = np.random.default_rng(77)
pairs = []
for k in range(40):
    sides = []
    for side in range(2):
        n = int(rng.integers(420, 1400))
        if k % 3 == 0: labels, edges = random_bubble_chain(rng, n, snp_rate=0.0, del_rate=0.0)   # low-entropy linear
        elif k % 3 == 1: labels, edges = random_bubble_chain(rng, n, snp_rate=0.1, del_rate=0.04)
        else: labels, edges = t._irregular_chain(rng, n)
        src, snk = sources_and_sinks(len(labels), edges)
        sides.append(graph_from_edges(labels, edges, src, snk))
    pairs.append(tuple(sides))
batch = concat_batches([batch_from_graph_pairs(pairs), synth_windows(6, first_index=50, seed=5, len_min=1500, len_max=3000)])
for p in (t.PROD, t.PROD.truncated(1)):
    scores, alns = po_poa_batch(batch, p)
    t._compare(batch, p, scores, alns, oracle, "tiled P=%d" % p.num_pw)
print("TILED-OK", batch.n_windows)
"""


def test_tiled_fill_small_panels():
    """The tiled fill (wide windows cut into row panels, tiles handed out from a queue; popoa_kernels.cu) with a
    panel height of 256 rows, so that windows of a few hundred rows already consist of several panels and every
    hand-over (rows R0-2..R0 through the workspace, the boundary column of strip 0) is exercised.  The panel height
    is read once per process (CLB_PANEL_ROWS), hence the child process."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CLB_PANEL_ROWS="256")
    code = _TILED_CHILD.format(root=root, tests=os.path.join(root, "tests"))
    res = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and "TILED-OK" in res.stdout, res.stdout[-3000:]


def test_live_against_unmodified_reference():
    """Equal to the results recorded in tests/golden/live_golden.json and, where oracle/_ref/libclref.so is built, to the
    unmodified reference's."""
    for (batch, p, _), want in zip(live_runs("po_poa_gpu"), load_live_golden("po_poa_gpu"), strict=True):
        scores, alns = po_poa_batch(batch, p)
        assert results_digest(scores, alns) == want, "differs from the recorded results"
        if CpuChecker.available("reference"):
            _compare(batch, p, scores, alns, CpuChecker("reference"), "reference")


def test_staged_api_is_repeatable_and_matches_one_shot():
    batch = synth_windows(12, first_index=300, seed=2, len_min=200, len_max=900)
    s1, a1 = po_poa_batch(batch, PROD)
    with DeviceBatch(batch, PROD) as db:
        db.upload()
        db.run()
        db.run()  # idempotent: a resident batch can be re-run (bench.py does)
        s2, a2 = db.download()
        st = db.stats()
        assert st.kernel_launches >= 1 and st.cells == float(batch.cells().sum()) and st.kernel_ms > 0
        assert np.array_equal(s1, s2)
        for x, y in zip(a1, a2):
            assert np.array_equal(x, y)


def test_size_independent_properties_large_windows():
    """Full-size windows (config 2 scale) are too slow for the oracle; check properties instead:
    the alignment is a valid source-to-sink walk pair, and re-scoring it with the affine
    pieces reproduces the reported optimum."""
    batch = synth_windows(3, first_index=1000, seed=4, len_min=6000, len_max=9000)
    scores, alns = po_poa_batch(batch, PROD)
    for w in range(batch.n_windows):
        assert_valid_and_rescore(batch, w, PROD, int(scores[w]), alns[w])


def test_30k_by_30k_window(monkeypatch):
    """One window of 30 000 x 30 000 nodes (9e8 cells, the largest single fill the workspace layout is meant for, VERDICT
    round 1 item 7): it runs, its alignment is a valid walk pair that re-scores to the reported optimum, and the generic
    fill step (a different code path through the same matrix) reports the same score and alignment."""
    batch = synth_windows(1, first_index=77, seed=5, len_min=30000, len_max=30000)
    scores, alns = po_poa_batch(batch, PROD)
    assert_valid_and_rescore(batch, 0, PROD, int(scores[0]), alns[0])
    monkeypatch.setenv("CLB_DEBUG_FLAGS", "2")
    scores2, alns2 = po_poa_batch(batch, PROD)
    assert int(scores2[0]) == int(scores[0]) and np.array_equal(alns2[0], alns[0])


def assert_valid_and_rescore(batch, w, p, score, aln):
    lab1, po1, pr1, src1, snk1 = batch.g1.window(w)
    lab2, po2, pr2, src2, snk2 = batch.g2.window(w)
    path1 = [int(a) for a, _ in aln if a >= 0]
    path2 = [int(b) for _, b in aln if b >= 0]
    for path, po, pr, src, snk in ((path1, po1, pr1, src1, snk1), (path2, po2, pr2, src2, snk2)):
        assert path[0] in set(src.tolist()) and path[-1] in set(snk.tolist())
        for u, v in zip(path[:-1], path[1:]):
            assert u in pr[po[v]:po[v + 1]].tolist()
    total, run, kind = 0, 0, 0

    def gap_cost(n):
        return min(o + e * n for o, e in zip(p.gap_open, p.gap_extend))

    for a, b in aln.tolist():
        k = 0 if (a >= 0 and b >= 0) else (1 if b < 0 else 2)
        if k != kind and run:
            total -= gap_cost(run)
            run = 0
        kind = k
        if k == 0:
            total += p.match if lab1[a] == lab2[b] else -p.mismatch
        else:
            run += 1
    if run:
        total -= gap_cost(run)
    assert total == score


def test_repeated_runs_are_identical_and_valid():
    """The fill warps of a CTA stream over windows and synchronise through progress words; any race
    would show up as run-to-run differences.  Re-run a mixed batch (narrow + wide strips, several
    windows per CTA) and demand identical bytes, plus the size-independent validity check."""
    batch = concat_batches([
        synth_windows(300, first_index=5000, seed=8, len_min=100, len_max=1200),
        synth_windows(40, first_index=6000, seed=8, len_min=1500, len_max=2500),
    ])
    ref_s, ref_a = po_poa_batch(batch, PROD)
    ref_s = ref_s.copy()
    for _ in range(2):
        s, a = po_poa_batch(batch, PROD)
        assert np.array_equal(s, ref_s)
        assert all(np.array_equal(x, y) for x, y in zip(a, ref_a))
    for w in range(0, batch.n_windows, 17):
        assert_valid_and_rescore(batch, w, PROD, int(ref_s[w]), ref_a[w])


def test_chunked_one_shot_matches_single_batch(monkeypatch):
    """Large one-shot calls are split into chunks that overlap host flattening, H2D, kernels and D2H
    (shared workspace, slot pair by SM id).  Same bytes as the single-batch path are required."""
    batch = concat_batches([
        synth_windows(1100, first_index=9000, seed=12, len_min=100, len_max=900),
        synth_windows(30, first_index=9500, seed=12, len_min=1500, len_max=2500),
    ])
    monkeypatch.setenv("CLB_NO_CHUNKS", "1")
    ref_s, ref_a = po_poa_batch(batch, PROD)
    ref_s = ref_s.copy()
    ref_a = [a.copy() for a in ref_a]
    monkeypatch.delenv("CLB_NO_CHUNKS")
    monkeypatch.setenv("CLB_CHUNK_MIN_NODES", "1")
    for _ in range(2):
        s, a = po_poa_batch(batch, PROD)
        assert np.array_equal(s, ref_s)
        assert all(np.array_equal(x, y) for x, y in zip(a, ref_a))
    for w in range(0, batch.n_windows, 97):
        assert_valid_and_rescore(batch, w, PROD, int(ref_s[w]), ref_a[w])


def test_chunked_one_shot_late_chunk_needs_larger_workspace(monkeypatch):
    """A window's workspace grows with its persisted rows / columns and its elongation, not only with its cell count: the
    chunked one-shot path sizes the shared slot from the chunk with the largest windows, so a persist-heavy or elongated
    window of a LATER chunk must get a workspace of its own (popoa_host.cu upload_internal) instead of overrunning its slot."""
    rng = np.random.default_rng(99)
    pairs = []
    for n1, n2 in ((260, 9), (9, 260), (300, 300)):  # elongated: few cells, long persisted columns / rows
        for _ in range(3):
            sides = []
            for n in (n1, n2):
                labels, edges = random_bubble_chain(rng, n, snp_rate=0.1, del_rate=0.03)
                if n >= 200:  # many far edges: nearly every row / column is persisted
                    edges = list(edges) + [(int(a), int(a) + 5 + int(rng.integers(0, 40))) for a in rng.integers(0, n - 50, size=n // 3)]
                src, snk = sources_and_sinks(len(labels), edges)
                sides.append(graph_from_edges(labels, edges, src, snk))
            pairs.append(tuple(sides))
    odd = batch_from_graph_pairs(pairs)
    batch = concat_batches([
        synth_windows(1100, first_index=9000, seed=13, len_min=100, len_max=400),
        synth_windows(8, first_index=9500, seed=13, len_min=420, len_max=450),  # chunk 0: most cells, few persisted rows
        odd,
    ])
    monkeypatch.setenv("CLB_NO_CHUNKS", "1")
    ref_s, ref_a = po_poa_batch(batch, PROD)
    ref_s = ref_s.copy()
    ref_a = [a.copy() for a in ref_a]
    monkeypatch.delenv("CLB_NO_CHUNKS")
    monkeypatch.setenv("CLB_CHUNK_MIN_NODES", "1")
    s, a = po_poa_batch(batch, PROD)
    assert np.array_equal(s, ref_s)
    assert all(np.array_equal(x, y) for x, y in zip(a, ref_a))
    oracle = CpuChecker("port")
    first_odd = batch.n_windows - odd.n_windows
    for w in range(first_odd, batch.n_windows):
        so, ao = oracle.po_poa(batch, w, PROD)
        assert so == s[w] and np.array_equal(ao, a[w]), f"window {w} differs from the oracle"


def test_multi_device_call_matches_single_device():
    """clb_popoa_batch_multi over every visible GPU (one on the test box: the threaded path with a single bin is still
    exercised through the two-window minimum) returns what clb_popoa_batch returns, in window order."""
    import torch

    from centrolign_b200.popoa import po_poa_batch_multi

    batch = synth_windows(40, first_index=700, seed=21, len_min=60, len_max=700)
    ref_s, ref_a = po_poa_batch(batch, PROD)
    devs = list(range(torch.cuda.device_count()))
    s, a, parts = po_poa_batch_multi(batch, PROD, devs, return_parts=True)
    assert np.array_equal(s, ref_s) and all(np.array_equal(x, y) for x, y in zip(a, ref_a))
    assert parts.min() >= 0 and parts.max() < len(devs)
    if len(devs) > 1:
        loads = np.bincount(parts, weights=batch.cells().astype(np.float64), minlength=len(devs))
        assert loads.min() > 0 and loads.max() - loads.min() <= batch.cells().max()
    with pytest.raises(Exception):
        po_poa_batch_multi(batch, PROD, [0, 0])


def test_small_and_strip_kernels_agree_on_every_fixture_window(monkeypatch):
    """Windows of at most 384 matrix cells take the warp-per-window kernel (popoa_small_kernels.cu), larger ones the strip
    kernel.  Both must reproduce the reference fixture; with CLB_NO_SMALL_WINDOWS every window is forced through the
    strip kernel, so each fixture window is checked on both paths."""
    batch, params, pidx, scores, alns = load_golden()
    cells = batch.cells()
    assert (cells <= 384).sum() > 50 and (cells > 384).sum() > 50  # the fixture exercises both routes
    for force_strip in (False, True):
        if force_strip:
            monkeypatch.setenv("CLB_NO_SMALL_WINDOWS", "1")
        for k, p in enumerate(params):
            idx = np.nonzero(pidx == k)[0]
            got_s, got_a = po_poa_batch(select_windows(batch, idx), p)
            for n, w in enumerate(idx):
                assert got_s[n] == scores[w], f"window {w} (force_strip={force_strip}): score {got_s[n]} != {scores[w]}"
                assert np.array_equal(got_a[n], alns[w]), f"window {w} (force_strip={force_strip}): alignment differs"


def test_small_window_kernel_random_dags_vs_oracle():
    """Thousands of tiny random DAG windows (the size the Stitcher really produces), all three parameter widths,
    through the warp-per-window kernel, each compared with the oracle."""
    oracle = CpuChecker("port")
    rng = np.random.default_rng(2024)
    pairs = []
    for t in range(1500):
        sides = []
        for _ in range(2):
            n = int(rng.integers(1, 19))
            labels, edges = random_dag(rng, n, int(rng.integers(0, 2 * n + 1)), alphabet="AC")
            src, snk = sources_and_sinks(len(labels), edges)
            sides.append(graph_from_edges(labels, edges, src, snk))
        pairs.append(tuple(sides))
    batch = batch_from_graph_pairs(pairs)
    assert (batch.cells() <= 384).all()
    for num_pw in (1, 2, 3):
        p = PROD.truncated(num_pw)
        scores, alns = po_poa_batch(batch, p)
        _compare(batch, p, scores, alns, oracle, f"small random DAGs, NumPW={num_pw}")
