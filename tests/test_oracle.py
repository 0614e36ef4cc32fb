"""CPU tests: pin the C oracle (oracle/po_poa_oracle.c) to the reference.

* the reference's own golden alignments (src/test/test_alignment.cpp:684-773),
* fixtures produced by the unmodified reference (tests/golden/popoa_golden.npz),
* recorded results on further windows (tests/golden/live_golden.json), and a live comparison with
  oracle/_ref/libclref.so on the same windows where it is built (oracle/Makefile, from the reference's sources).
"""
import numpy as np
import pytest

from centrolign_b200.batch import AlignmentParameters, batch_from_graph_pairs, graph_from_edges, successor_form
from checkers import CpuChecker  # test infrastructure: tests/checkers.py
from golden_io import (REFERENCE_UNIT_GOLDENS, TIEBREAK_PROBES, live_runs, load_chain_golden, load_golden, load_live_golden,
                       load_pwfa_golden, results_digest)


@pytest.fixture(scope="module")
def oracle():
    return CpuChecker("port")


def _unit_batch(cases):
    return batch_from_graph_pairs([(graph_from_edges(c[0], c[1], c[2], c[3]), graph_from_edges(c[4], c[5], c[6], c[7]))
                                   for c in cases])


def test_reference_unit_goldens(oracle):
    batch = _unit_batch(REFERENCE_UNIT_GOLDENS)
    p = AlignmentParameters(1, 1, (1,), (1,))
    for w, case in enumerate(REFERENCE_UNIT_GOLDENS):
        _, aln = oracle.po_poa(batch, w, p)
        assert [tuple(x) for x in aln.tolist()] == case[8]


def test_tiebreak_probes(oracle):
    batch = _unit_batch(TIEBREAK_PROBES)
    for w, case in enumerate(TIEBREAK_PROBES):
        _, aln = oracle.po_poa(batch, w, AlignmentParameters(*case[8]))
        assert [tuple(x) for x in aln.tolist()] == case[9], f"probe {w}"


def test_golden_fixture(oracle):
    batch, params, pidx, scores, alns = load_golden()
    assert batch.n_windows >= 300
    for w in range(batch.n_windows):
        s, a = oracle.po_poa(batch, w, params[pidx[w]])
        assert s == scores[w], f"window {w}: score"
        assert np.array_equal(a, alns[w]), f"window {w}: alignment"


def test_empty_sides(oracle):
    """po_poa with an empty graph falls back to the boundary row / column (alignment.hpp:991-1008)."""
    g = graph_from_edges("ACG", [(0, 1), (1, 2)], [0], [2])
    e = graph_from_edges("", [], [], [])
    batch = batch_from_graph_pairs([(g, e), (e, g), (e, e)])
    p = AlignmentParameters()
    s, a = oracle.po_poa(batch, 0, p)
    assert s == -(60 + 3 * 30) and a.tolist() == [[0, -1], [1, -1], [2, -1]]
    s, a = oracle.po_poa(batch, 1, p)
    assert s == -(60 + 3 * 30) and a.tolist() == [[-1, 0], [-1, 1], [-1, 2]]
    s, a = oracle.po_poa(batch, 2, p)
    assert s == 0 and len(a) == 0


def _check_live_runs(name, oracle):
    """The oracle on golden_io.live_runs(name): equal to the results recorded in tests/golden/live_golden.json and, where
    oracle/_ref/libclref.so is built, to the unmodified reference's."""
    ref = CpuChecker("reference") if CpuChecker.available("reference") else None
    for k, ((batch, p, lim), want) in enumerate(zip(live_runs(name), load_live_golden(name), strict=True)):
        scores, alns = oracle.run(batch, p, lim)
        assert results_digest(scores, alns) == want, f"{name} run {k}: differs from the recorded results"
        if ref is not None:
            rs, ra = ref.run(batch, p, lim)
            for w in range(batch.n_windows):
                assert scores[w] == rs[w] and np.array_equal(alns[w], ra[w]), f"{name} run {k} window {w} P={p.num_pw}"


def test_live_against_reference(oracle):
    """HOR-like windows up to 900 nodes with three parameter sets, and empty sides."""
    _check_live_runs("po_poa_oracle", oracle)


# ---- wavefront variant (oracle/pwfa_oracle.c) ------------------------------------------------------------
def test_pwfa_reference_unit_goldens(oracle):
    """src/test/test_alignment.cpp:717-771: pwfa_po_poa(..., prune_limit 4) gives the same golden pairs."""
    batch = successor_form(_unit_batch(REFERENCE_UNIT_GOLDENS))
    p = AlignmentParameters(1, 1, (1,), (1,))
    for w, case in enumerate(REFERENCE_UNIT_GOLDENS):
        _, aln = oracle.pwfa_po_poa(batch, w, p, 4)
        assert [tuple(x) for x in aln.tolist()] == case[8]


def test_pwfa_golden_fixture(oracle):
    batches, params, cases, scores, alns = load_pwfa_golden()
    assert len(cases) >= 1500
    for k, (variant, w, pi, lim) in enumerate(cases.tolist()):
        s, a = oracle.pwfa_po_poa(batches[variant], w, params[pi], lim)
        assert s == scores[k], f"case {k}: score"
        assert np.array_equal(a, alns[k]), f"case {k}: alignment"


def test_pwfa_live_against_reference(oracle):
    """Windows up to 3000 nodes in two successor orders, two parameter sets and prune limits."""
    _check_live_runs("pwfa_oracle", oracle)


# ---- sparse anchor-chaining DP (oracle/chain_oracle.c) ---------------------------------------------------
def test_chain_oracle_reproduces_reference_chains():
    """tests/golden/chain_golden.npz: flat problems + the chains Anchorer::sparse_chain_dp /
    sparse_affine_chain_dp of the unmodified reference returned (anchorer.hpp:1511-1750, 1812-2471)."""
    from checkers import chain_oracle

    gold = load_chain_golden()
    assert len(gold) >= 4
    for case in sorted(gold):
        for kind in ("gapfree", "affine", "local"):
            prob = gold[case][kind]
            chain, dp, bp, opt = chain_oracle(prob)
            assert np.array_equal(chain, prob.expect_chain), f"{case}/{kind}"
            assert len(chain) > 5
