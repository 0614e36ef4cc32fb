"""GPU parity tests of the wavefront variant: ``clb_pwfa_batch`` (hand-written sm_100a kernel) against the
CPU oracle (oracle/pwfa_oracle.c), the fixtures produced by the unmodified reference
(tests/golden/pwfa_golden.npz), recorded results (tests/golden/live_golden.json) and, where it is built,
the reference itself.  The algorithm's output is
defined by its dequeue order, so identical alignments and scores are required, not just equal scores."""
import numpy as np
import pytest

from centrolign_b200.batch import (AlignmentParameters, batch_from_graph_pairs, concat_batches,
                                   graph_from_edges, select_windows, successor_form, synth_windows)
from centrolign_b200.popoa import ClbError, PwfaStats, pwfa_po_poa_batch
from checkers import CpuChecker  # test infrastructure: tests/checkers.py
from golden_io import REFERENCE_UNIT_GOLDENS, live_runs, load_live_golden, load_pwfa_golden, results_digest

pytestmark = pytest.mark.gpu

PROD = AlignmentParameters()


def _unit_batch(cases):
    return batch_from_graph_pairs([(graph_from_edges(c[0], c[1], c[2], c[3]), graph_from_edges(c[4], c[5], c[6], c[7]))
                                   for c in cases])


def _compare(sb, params, lim, scores, alns, checker, tag):
    for w in range(sb.n_windows):
        s, a = checker.pwfa_po_poa(sb, w, params, lim)
        assert s == scores[w], f"{tag}: window {w} score {scores[w]} != {s}"
        assert np.array_equal(a, alns[w]), f"{tag}: window {w} alignment differs"


def test_reference_unit_goldens():
    sb = successor_form(_unit_batch(REFERENCE_UNIT_GOLDENS))
    _, alns = pwfa_po_poa_batch(sb, AlignmentParameters(1, 1, (1,), (1,)), 4)
    for a, case in zip(alns, REFERENCE_UNIT_GOLDENS):
        assert [tuple(x) for x in a.tolist()] == case[8]


def test_golden_fixture():
    batches, params, cases, scores, alns = load_pwfa_golden()
    groups = {}
    for k, (variant, w, pi, lim) in enumerate(cases.tolist()):
        groups.setdefault((variant, pi, lim), []).append((w, k))
    for (variant, pi, lim), items in groups.items():
        sub = select_windows(batches[variant], [w for w, _ in items])
        s, a = pwfa_po_poa_batch(sub, params[pi], lim)
        for n, (w, k) in enumerate(items):
            assert s[n] == scores[k], f"case {k} (window {w}, params {pi}, prune {lim}): score {s[n]} != {scores[k]}"
            assert np.array_equal(a[n], alns[k]), f"case {k} (window {w}, params {pi}, prune {lim}): alignment"


@pytest.mark.parametrize("num_pw", [1, 2, 3])
def test_hor_windows_vs_oracle(num_pw):
    port = CpuChecker("port")
    p = PROD.truncated(num_pw)
    batch = concat_batches([synth_windows(24, first_index=700, seed=6, len_min=100, len_max=2500, alt_len=61, alt_period=500),
                            synth_windows(4, first_index=900, seed=6, len_min=6000, len_max=8700)])
    for sb in (successor_form(batch), successor_form(batch, np.random.default_rng(num_pw))):
        st = PwfaStats()
        scores, alns = pwfa_po_poa_batch(sb, p, 50, stats=st)
        assert st.kernel_launches >= 1 and st.states > 0 and st.steps > 0
        _compare(sb, p, 50, scores, alns, port, f"P={num_pw}")


def test_live_against_unmodified_reference():
    """Equal to the results recorded in tests/golden/live_golden.json and, where oracle/_ref/libclref.so is built, to the
    unmodified reference's."""
    for (sb, p, lim), want in zip(live_runs("pwfa_gpu"), load_live_golden("pwfa_gpu"), strict=True):
        scores, alns = pwfa_po_poa_batch(sb, p, lim)
        assert results_digest(scores, alns) == want, f"prune={lim}: differs from the recorded results"
        if CpuChecker.available("reference"):
            _compare(sb, p, lim, scores, alns, CpuChecker("reference"), f"reference prune={lim}")


def test_table_enlargement_gives_the_same_result(monkeypatch):
    """Undersized back-pointer tables / FIFOs are detected on the device and the window is re-run larger."""
    batch = synth_windows(6, first_index=300, seed=9, len_min=800, len_max=2000)
    sb = successor_form(batch)
    ref_s, ref_a = pwfa_po_poa_batch(sb, PROD, 50)
    ref_s, ref_a = ref_s.copy(), [a.copy() for a in ref_a]
    monkeypatch.setenv("CLB_PWFA_HASH_LOG2", "9")
    monkeypatch.setenv("CLB_PWFA_FIFO_LOG2", "5")
    st = PwfaStats()
    s, a = pwfa_po_poa_batch(sb, PROD, 50, stats=st)
    assert st.retries >= 1
    assert np.array_equal(s, ref_s) and all(np.array_equal(x, y) for x, y in zip(a, ref_a))


def test_invalid_inputs_fail_loudly():
    g = graph_from_edges("ACG", [(0, 1), (1, 2)], [0], [2])
    sb = successor_form(batch_from_graph_pairs([(g, g)]))
    with pytest.raises(ClbError):
        pwfa_po_poa_batch(sb, PROD, -1)
    with pytest.raises(ClbError):
        pwfa_po_poa_batch(sb, AlignmentParameters(2, 2, (0,), (1,)), 4)  # zero gap_open: outside the reference's domain
    unreachable = graph_from_edges("ACG", [(0, 1)], [0], [2])  # the source cannot reach the sink
    with pytest.raises(ClbError):
        pwfa_po_poa_batch(successor_form(batch_from_graph_pairs([(unreachable, g)])), PROD, 50)
