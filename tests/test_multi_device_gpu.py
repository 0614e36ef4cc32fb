"""Several GPUs of one box for the wavefront gap fill (``clb_pwfa_batch_multi``) and the batched chaining DP
(``clb_chain_dp_batch_multi``), chaining on any device and on two devices at once, and the multi-device parts of the
C++ drop-in layer (the fill-in pool over a device list, CLB_DEVICES parsing).  The GPU tests use every visible device;
the ones that need two or more skip on a one-GPU box."""
import os
import re
import subprocess
import sys
import threading

import numpy as np
import pytest

from centrolign_b200.batch import (AlignmentParameters, batch_from_graph_pairs, concat_batches, graph_from_edges,
                                   select_windows, successor_form, synth_windows)
from checkers import CpuChecker, chain_oracle  # test infrastructure: tests/checkers.py
from golden_io import load_chain_golden, load_pwfa_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_DIR = os.path.join(ROOT, "centrolign_b200", "csrc")
PROD = AlignmentParameters()


def _devices():
    from centrolign_b200.popoa import load_library

    return list(range(load_library().clb_device_count()))


def _need_two():
    devs = _devices()
    if len(devs) < 2:
        pytest.skip("needs two or more GPUs; this box has %d" % len(devs))
    return devs


def _pwfa_costs(sb):
    n1 = np.diff(sb.g1.node_off)
    n2 = np.diff(sb.g2.node_off)
    return (n1 + 1) + (n2 + 1)


def _same(a, b):
    (sa, aa), (sb_, ab) = a, b
    return np.array_equal(sa, sb_) and len(aa) == len(ab) and all(np.array_equal(x, y) for x, y in zip(aa, ab))


# ------------------------------------------------------------------ C++ layer, no device ------------------------------------------------------------------

@pytest.fixture(scope="module")
def cpp_bin(tmp_path_factory):
    lib = os.path.join(LIB_DIR, "libcentrolign_b200.so")
    if not os.path.exists(lib):
        pytest.skip("libcentrolign_b200.so not built")
    out = str(tmp_path_factory.mktemp("multi_device") / "test_multi_device")
    subprocess.run(["g++", "-std=c++11", "-O1", "-pthread", "-I" + os.path.join(ROOT, "include"),
                    "-I" + os.path.join(ROOT, "centrolign_b200", "hostcpp"), os.path.join(ROOT, "tests", "cpp", "test_multi_device.cpp"),
                    "-L" + LIB_DIR, "-lcentrolign_b200", "-Wl,-rpath," + LIB_DIR, "-o", out], check=True)
    return out


def test_fill_in_pool_over_devices(cpp_bin):
    """hostcpp/chain_batcher.hpp over devices {0, 1} with a stand-in run function: every job runs exactly once, every
    launch carries jobs of one device, a worker's jobs go to its own device, {0} is the single-device pool, and an error
    in one device's launch comes back as an exception."""
    res = subprocess.run([cpp_bin, "--pool"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert res.returncode == 0 and "multi-device pool passed all tests!" in res.stdout, res.stdout


def test_solve_in_the_pool_creates_jobs_for_the_workers_device(cpp_bin):
    """ChainProblem::solve (hostcpp/chain_b200.hpp) called from the pool over devices {0, 1}: every job is created for the
    device of the calling worker's batcher -- not for the device argument of solve() -- and runs there.  The test program
    replaces clb_chain_job_create / clb_chain_job_destroy with stand-ins that record the device, so no GPU is needed."""
    res = subprocess.run([cpp_bin, "--solve"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert res.returncode == 0 and "solve passed all tests!" in res.stdout, res.stdout


@pytest.mark.parametrize("value,want", [("0,0,1", [0, 1]), ("1,0,1,0", [1, 0]), ("3", [3]), ("", [0])])
def test_device_list_parsing(cpp_bin, value, want):
    """CLB_DEVICES: a repeated ordinal counts once, first-seen order is kept, and chain_device() is the first entry."""
    env = dict(os.environ, CLB_DEVICES=value)
    out = subprocess.run([cpp_bin, "--devices"], stdout=subprocess.PIPE, text=True, env=env, check=True).stdout.split("\n")
    assert out[0].split()[1:] == [str(d) for d in want]
    assert out[1] == "chain_device %d" % want[0]


# ------------------------------------------------------------------ wavefront gap fill ------------------------------------------------------------------

@pytest.mark.gpu
def test_pwfa_golden_fixture_on_all_devices():
    from centrolign_b200.popoa import balanced_partition_c, pwfa_po_poa_batch_multi

    devs = _devices()
    batches, params, cases, scores, alns = load_pwfa_golden()
    groups = {}
    for k, (variant, w, pi, lim) in enumerate(cases.tolist()):
        groups.setdefault((variant, pi, lim), []).append((w, k))
    for (variant, pi, lim), items in groups.items():
        sub = select_windows(batches[variant], [w for w, _ in items])
        s, a, parts = pwfa_po_poa_batch_multi(sub, params[pi], lim, devs, return_parts=True)
        assert np.all((parts >= 0) & (parts < len(devs)))
        assert np.array_equal(parts, balanced_partition_c(_pwfa_costs(sub), len(devs)))
        for n, (w, k) in enumerate(items):
            assert s[n] == scores[k], f"case {k} (window {w}, params {pi}, prune {lim}): score {s[n]} != {scores[k]}"
            assert np.array_equal(a[n], alns[k]), f"case {k} (window {w}, params {pi}, prune {lim}): alignment"


@pytest.mark.gpu
@pytest.mark.parametrize("num_pw", [1, 2, 3])
def test_pwfa_hor_windows_vs_oracle_on_all_devices(num_pw):
    from centrolign_b200.popoa import PwfaStats, pwfa_po_poa_batch, pwfa_po_poa_batch_multi

    devs = _devices()
    port = CpuChecker("port")
    p = PROD.truncated(num_pw)
    batch = concat_batches([synth_windows(24, first_index=700, seed=6, len_min=100, len_max=2500, alt_len=61, alt_period=500),
                            synth_windows(4, first_index=900, seed=6, len_min=6000, len_max=8700)])
    for sb in (successor_form(batch), successor_form(batch, np.random.default_rng(num_pw))):
        st = PwfaStats()
        scores, alns = pwfa_po_poa_batch_multi(sb, p, 50, devs, stats=st)
        assert st.kernel_launches >= len(devs) and st.states > 0 and st.steps > 0 and st.kernel_ms > 0
        for w in range(sb.n_windows):
            s, a = port.pwfa_po_poa(sb, w, p, 50)
            assert s == scores[w], f"P={num_pw}: window {w} score {scores[w]} != {s}"
            assert np.array_equal(a, alns[w]), f"P={num_pw}: window {w} alignment differs"
        last = pwfa_po_poa_batch_multi(sb, p, 50, [devs[-1]])
        assert _same(last, pwfa_po_poa_batch(sb, p, 50, device=0))
        assert _same(last, (scores, alns))


@pytest.mark.gpu
def test_pwfa_table_enlargement_across_devices(monkeypatch):
    from centrolign_b200.popoa import PwfaStats, pwfa_po_poa_batch_multi

    devs = _devices()
    sb = successor_form(synth_windows(6 * len(devs), first_index=300, seed=9, len_min=800, len_max=2000))
    ref = pwfa_po_poa_batch_multi(sb, PROD, 50, devs)
    ref = (ref[0].copy(), [a.copy() for a in ref[1]])
    monkeypatch.setenv("CLB_PWFA_HASH_LOG2", "9")
    monkeypatch.setenv("CLB_PWFA_FIFO_LOG2", "5")
    st = PwfaStats()
    got = pwfa_po_poa_batch_multi(sb, PROD, 50, devs, stats=st)
    assert st.retries >= 1
    assert _same(got, ref)


@pytest.mark.gpu
def test_pwfa_multi_errors():
    from centrolign_b200.popoa import ClbError, pwfa_po_poa_batch_multi

    devs = _devices()
    g = graph_from_edges("ACGT", [(0, 1), (1, 2), (2, 3)], [0], [3])
    good = successor_form(batch_from_graph_pairs([(g, g)] * 4))
    for bad_devs in ([devs[0], devs[0]], [len(devs)], [devs[0], len(devs) + 3]):
        with pytest.raises(ClbError) as e:
            pwfa_po_poa_batch_multi(good, PROD, 50, bad_devs)
        assert e.value.code == 1, bad_devs
    unreachable = graph_from_edges("ACGT", [(0, 1), (2, 3)], [0], [3])  # the source cannot reach the sink
    n = max(4, 2 * len(devs))
    for k in (0, n - 1):
        pairs = [(g, g)] * n
        pairs[k] = (unreachable, g)
        with pytest.raises(ClbError) as e:
            pwfa_po_poa_batch_multi(successor_form(batch_from_graph_pairs(pairs)), PROD, 50, devs)
        assert f"window {k}:" in str(e.value), str(e.value)
    empty = select_windows(good, [])
    scores, alns = pwfa_po_poa_batch_multi(empty, PROD, 50, devs)
    assert len(scores) == 0 and alns == []


# ------------------------------------------------------------------ chaining ------------------------------------------------------------------

def _chain_problems():
    from centrolign_b200.chain import synth_fill_in_problems

    gold = load_chain_golden()
    probs = [gold[c][k] for c in sorted(gold) for k in sorted(gold[c])]
    return probs + synth_fill_in_problems(300, seed=11)


def _assert_equal_results(got, want):
    (chain, dp, bp, opt), (rchain, rdp, rbp, ropt) = got, want
    assert np.array_equal(chain, rchain) and opt == ropt
    assert np.array_equal(dp.view(np.uint32), rdp.view(np.uint32)) and np.array_equal(bp, rbp)


@pytest.mark.gpu
def test_chain_batch_on_all_devices_equals_one_by_one():
    """Per problem the chain, every DP value bit for bit and every back-pointer of clb_chain_dp, for the committed
    fixtures (every kind) and fill-in-sized problems."""
    from centrolign_b200.chain import ChainStats, chain_dp, chain_dp_batch_multi

    devs = _devices()
    probs = _chain_problems()
    st = ChainStats()
    got, parts = chain_dp_batch_multi(probs, devs, stats=st, return_parts=True)
    assert len(got) == len(probs) and np.all((parts >= 0) & (parts < len(devs)))
    if len(devs) > 1:
        assert len(set(parts.tolist())) == len(devs)
    assert st.kernel_launches >= 1 and st.total_ms > 0
    for prob, res in zip(probs, got):
        _assert_equal_results(res, chain_dp(prob))
        if prob.expect_chain is not None and len(prob.expect_chain):
            assert np.array_equal(res[0], prob.expect_chain)
    # the generated fill-in problems also against the oracle, independently of the GPU code (every piece count in the mix)
    n_fixed = len(probs) - 300
    for prob, res in list(zip(probs, got))[n_fixed: n_fixed + 12]:
        _assert_equal_results(res, chain_oracle(prob))
    assert chain_dp_batch_multi([], devs) == []
    from centrolign_b200.popoa import ClbError

    with pytest.raises(ClbError):
        chain_dp_batch_multi(probs[:2], [devs[0], devs[0]])
    with pytest.raises(ClbError):
        chain_dp_batch_multi(probs[:2], [len(devs)])


_SECOND_DEVICE = r"""
import os, sys
import numpy as np
sys.path[:0] = [{root!r}, {tests!r}]
from centrolign_b200.chain import ChainProblem, chain_dp, chain_dp_batch, synth_fill_in_problems
from checkers import chain_oracle
from golden_io import load_chain_golden
gold = load_chain_golden()
fixtures = [gold[c][k] for c in sorted(gold) for k in sorted(gold[c])]
src = gold["msa4_3k"]["affine"]
large = ChainProblem(src.num_pw, src.gap_open, src.gap_extend, src.scale, src.n_chain1, src.n_chain2, src.min_score, src.arrays)
fill_in = synth_fill_in_problems(40, seed=5)
res = {{}}
for d in (0, 1):
    batch = chain_dp_batch(fixtures + fill_in, device=d)  # chain_small_batch_kernel
    small = chain_dp(gold["pair600"]["gapfree"], device=d)  # chain_small_kernel
    # chain_kernel in a cluster of 16 CTAs; CLB_TIMING prints the cluster size the kernel was launched with
    os.environ["CLB_CHAIN_CLUSTER"], os.environ["CLB_CHAIN_NO_SMALL"], os.environ["CLB_TIMING"] = "16", "1", "1"
    cluster = chain_dp(large, device=d)
    del os.environ["CLB_CHAIN_CLUSTER"], os.environ["CLB_CHAIN_NO_SMALL"], os.environ["CLB_TIMING"]
    res[d] = batch + [small, cluster]
want = [chain_oracle(p) for p in fixtures] + [None] * len(fill_in) + [chain_oracle(gold["pair600"]["gapfree"]), chain_oracle(large)]
for k, w in enumerate(want):
    for d in (0, 1):
        chain, dp, bp, opt = res[d][k]
        ref = w if w is not None else res[0][k]
        assert np.array_equal(chain, ref[0]) and opt == ref[3], (d, k)
        assert np.array_equal(dp.view(np.uint32), ref[1].view(np.uint32)) and np.array_equal(bp, ref[2]), (d, k)
print("second device ok")
"""


@pytest.mark.gpu
def test_chaining_on_a_second_device():
    """In a fresh process: both shared-memory kernels and a cluster launch (CLB_CHAIN_CLUSTER=16) on device 0, then on
    device 1; the same results on both, equal to the oracle, and the cluster kernel launched with the same cluster size
    on both (a size the device cannot place falls back to a smaller one, which would give the same results).  Function
    attributes are per device, so the second device must get its own."""
    _need_two()
    code = _SECOND_DEVICE.format(root=ROOT, tests=os.path.join(ROOT, "tests"))
    res = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert res.returncode == 0 and "second device ok" in res.stdout, res.stdout
    launched = [int(c) for c in re.findall(r"\[clb\] chain: .*\(grid \d+, cluster (\d+),", res.stdout)]
    assert len(launched) == 2 and launched[0] > 1 and launched[0] == launched[1], res.stdout


@pytest.mark.gpu
def test_concurrent_chaining_on_two_devices():
    """Two host threads call clb_chain_dp at the same time on different devices: the results are those of serial calls."""
    from centrolign_b200.chain import chain_dp

    devs = _need_two()
    gold = load_chain_golden()
    probs = [gold[c][k] for c in sorted(gold) for k in sorted(gold[c])]
    serial = [chain_dp(p, device=0) for p in probs]
    got = {}
    errors = []

    def work(d):
        try:
            got[d] = [chain_dp(p, device=d) for p in probs]
        except Exception as e:  # handed to the main thread
            errors.append(e)

    threads = [threading.Thread(target=work, args=(d,)) for d in devs[:2]]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for d in devs[:2]:
        for res, want in zip(got[d], serial):
            _assert_equal_results(res, want)
    for p, want in zip(probs[:2], serial[:2]):
        _assert_equal_results(want, chain_oracle(p))
