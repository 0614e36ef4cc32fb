"""The chaining search structures laid out on the GPU (chain_layout_kernels.cu) against the host layout (chain_host.cu).

CLB_CHAIN_LAYOUT=check builds both layouts of a problem and compares their copy regions byte for byte: any difference
fails the call with CLB_ECUDA and names the first differing array.  CLB_CHAIN_LAYOUT=device and =host force one side;
the default picks the device from a size on."""
import numpy as np
import pytest

from centrolign_b200.chain import ChainProblem, ChainStats, chain_dp, chain_dp_batch_multi, synth_chain_problem
from checkers import chain_oracle  # test infrastructure: tests/checkers.py
from golden_io import load_chain_golden

pytestmark = pytest.mark.gpu

GOLD = load_chain_golden()
CASES = [(c, k) for c in sorted(GOLD) for k in sorted(GOLD[c])]


def _devices():
    from centrolign_b200.popoa import load_library

    return list(range(load_library().clb_device_count()))


def _run(prob, side, monkeypatch, device=0, stats=None):
    monkeypatch.setenv("CLB_CHAIN_LAYOUT", side)
    try:
        return chain_dp(prob, device=device, stats=stats)
    finally:
        monkeypatch.delenv("CLB_CHAIN_LAYOUT")


def _same(x, y):
    (c1, d1, b1, o1), (c2, d2, b2, o2) = x, y
    assert np.array_equal(c1, c2) and o1 == o2
    assert np.array_equal(d1.view(np.uint32), d2.view(np.uint32)) and np.array_equal(b1, b2)


@pytest.mark.parametrize("case,kind", CASES)
def test_fixture_layouts_agree(case, kind, monkeypatch):
    prob = GOLD[case][kind]
    _run(prob, "check", monkeypatch)
    host = _run(prob, "host", monkeypatch)
    dev = _run(prob, "device", monkeypatch)
    assert np.array_equal(dev[0], prob.expect_chain)
    _same(dev, host)


def _tiny(n, num_pw, same_shift=True):
    """n matches on one path pair: one orthogonal tree of n nodes (spines only for n <= 3)."""
    p = synth_chain_problem(max(n, 1), 1, 1, num_pw, seed=n, shifts=1 if same_shift else 4, offsets=3, inactive=0.0)
    if n == 0:
        p.arrays = {k: v[:0] if k not in ("end_off", "qry_off", "ins_off") else v[:1] for k, v in p.arrays.items()}
    return p


@pytest.mark.parametrize("num_pw", [0, 1, 3])
def test_small_trees_and_spines(num_pw, monkeypatch):
    for n in (1, 2, 3, 4, 5, 7):
        for same_shift in (True, False):
            prob = _tiny(n, num_pw, same_shift)
            got = _run(prob, "check", monkeypatch)
            _same(got, chain_oracle(prob))


@pytest.mark.parametrize("k", [6, 10])
@pytest.mark.parametrize("delta", [-1, 0, 1])
@pytest.mark.parametrize("num_pw", [0, 2])
def test_tree_sizes_around_powers_of_two(k, delta, num_pw, monkeypatch):
    """One pair with 2^k - 1, 2^k and 2^k + 1 entries: the last level empty but one, full, and with one node."""
    prob = synth_chain_problem((1 << k) + delta, 1, 1, num_pw, seed=k * 10 + delta + 1, shifts=2, offsets=8, inactive=0.0)
    got = _run(prob, "check", monkeypatch)
    _same(got, chain_oracle(prob))


@pytest.mark.parametrize("chains", [(2, 3), (3, 3)])
@pytest.mark.parametrize("num_pw", [0, 1, 3])
@pytest.mark.parametrize("empty_pair", [False, True])
def test_several_chains_ties_and_inactive_entries(chains, num_pw, empty_pair, monkeypatch):
    """Several entries per match, few distinct shifts and offsets (ties decided by match rank and by position in the inner
    lists), inactive entries, and a pair without entries."""
    prob = synth_chain_problem(3000, chains[0], chains[1], num_pw, seed=7 + num_pw, shifts=3, offsets=5, inactive=0.2,
                               empty_pair=empty_pair)
    got = _run(prob, "check", monkeypatch)
    _same(got, chain_oracle(prob))
    _same(_run(prob, "device", monkeypatch), got)


@pytest.mark.parametrize("num_pw", [0, 3])
def test_million_entries(num_pw, monkeypatch):
    prob = synth_chain_problem(120_000, 3, 3, num_pw, seed=1000 + num_pw, shifts=64, offsets=4096)
    assert prob.arrays["ins_off"][-1] >= 1_000_000
    got = _run(prob, "check", monkeypatch)
    _same(_run(prob, "host", monkeypatch), got)


def test_default_path_takes_the_device_layout_above_the_threshold(monkeypatch):
    prob = synth_chain_problem(40_000, 3, 3, 1, seed=5)  # 360 000 entries: above the automatic threshold
    st_auto, st_host = ChainStats(), ChainStats()
    monkeypatch.delenv("CLB_CHAIN_LAYOUT", raising=False)
    auto = chain_dp(prob, stats=st_auto)
    host = _run(prob, "host", monkeypatch, stats=st_host)
    _same(auto, host)
    # the device layout copies only the caller's arrays, the host layout the whole copy region
    assert st_auto.tree_bytes == st_host.tree_bytes and st_auto.h2d_bytes < st_host.h2d_bytes


def test_every_device(monkeypatch):
    prob = synth_chain_problem(2000, 3, 2, 2, seed=3, shifts=4, offsets=16)
    ref = chain_oracle(prob)
    for d in _devices():
        _same(_run(prob, "check", monkeypatch, device=d), ref)


def test_batch_multi_sends_large_problems_one_by_one():
    """A problem too large for the batched launch goes through the single-problem path, which lays it out on the device."""
    big = synth_chain_problem(40_000, 3, 3, 1, seed=11)
    small = synth_chain_problem(40, 1, 1, 1, seed=12)
    got = chain_dp_batch_multi([small, big, small], _devices())
    for prob, res in zip([small, big, small], got):
        _same(res, chain_dp(prob))


def test_check_reports_no_difference_on_a_problem_without_entries(monkeypatch):
    prob = _tiny(0, 1)
    chain, _, _, _ = _run(prob, "check", monkeypatch)
    assert len(chain) == 0
    # matches whose entries are all inactive: empty insertion list, trees still shaped
    p = synth_chain_problem(200, 2, 2, 1, seed=2, inactive=1.0)
    _same(_run(p, "check", monkeypatch), chain_oracle(p))
    assert isinstance(p, ChainProblem)
