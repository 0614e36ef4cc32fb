"""Whole-call time of the multi-device entry points on 1, 2, 4, ... and all visible GPUs:
  * pwfa: the windows of tools/bench_pwfa.py (the size the Stitcher routes to pwfa_po_poa) through clb_pwfa_batch_multi;
  * chain: a batch of fill-in-sized chaining problems (a few dozen matches each) through clb_chain_dp_batch_multi.
Results must be identical at every device count (asserted).  Prints one JSON line per (workload, device count).
    python tools/multi_device_bench.py [--windows 2000] [--problems 4000] [--reps 2]
There is no CPU path: without a CUDA device the calls raise."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from centrolign_b200.batch import AlignmentParameters, successor_form, synth_windows  # noqa: E402
from centrolign_b200.chain import ChainStats, chain_dp_batch_multi, synth_fill_in_problems  # noqa: E402
from centrolign_b200.popoa import PwfaStats, load_library, pwfa_po_poa_batch_multi  # noqa: E402


def device_counts(n):
    out, k = [], 1
    while k < n:
        out.append(k)
        k *= 2
    return out + [n]


def gpu_info():
    """Name and power limit of the GPUs the numbers were taken on (read-only query)."""
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=30)
        return sorted(set(line.strip() for line in res.stdout.splitlines() if line.strip()))
    except (OSError, subprocess.SubprocessError):
        return ["unknown"]


def timed(fn, reps):
    """Best wall time of `reps` calls after one warm-up call, and the last result."""
    out = fn()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=2000)
    ap.add_argument("--len-min", type=float, default=5600.0)
    ap.add_argument("--len-max", type=float, default=7600.0)
    ap.add_argument("--prune", type=int, default=50)
    ap.add_argument("--problems", type=int, default=4000)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    n_dev = load_library().clb_device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device: there is no CPU path to measure")
    gpus = gpu_info()

    p = AlignmentParameters()
    sb = successor_form(synth_windows(a.windows, first_index=0, seed=20261017, len_min=a.len_min, len_max=a.len_max))
    ref = None
    for nd in device_counts(n_dev):
        devs = list(range(nd))
        st = PwfaStats()
        wall, (scores, alns) = timed(lambda: pwfa_po_poa_batch_multi(sb, p, a.prune, devs, stats=st), a.reps)
        if ref is None:
            ref = (scores.copy(), [x.copy() for x in alns])
        same = bool(np.array_equal(scores, ref[0]) and all(np.array_equal(x, y) for x, y in zip(alns, ref[1])))
        assert same, f"pwfa results on {nd} devices differ from 1 device"
        print(json.dumps({"workload": "pwfa_batch_multi", "devices": nd, "windows": a.windows, "wall_ms": wall * 1e3,
                          "windows_per_s": a.windows / wall, "max_kernel_ms": st.kernel_ms, "identical_to_1_device": same,
                          "gpus": gpus}), flush=True)

    probs = synth_fill_in_problems(a.problems, seed=20261022)
    ref = None
    for nd in device_counts(n_dev):
        devs = list(range(nd))
        st = ChainStats()
        wall, res = timed(lambda: chain_dp_batch_multi(probs, devs, stats=st), a.reps)
        if ref is None:
            ref = res
        same = all(np.array_equal(c, rc) and np.array_equal(d.view(np.uint32), rd.view(np.uint32)) and np.array_equal(b, rb) and o == ro
                   for (c, d, b, o), (rc, rd, rb, ro) in zip(res, ref))
        assert same, f"chaining results on {nd} devices differ from 1 device"
        print(json.dumps({"workload": "chain_dp_batch_multi", "devices": nd, "problems": a.problems,
                          "matches": int(sum(q.n_match for q in probs)), "wall_ms": wall * 1e3, "problems_per_s": a.problems / wall,
                          "sum_kernel_ms": st.kernel_ms, "kernel_launches": st.kernel_launches, "identical_to_1_device": same,
                          "gpus": gpus}), flush=True)


if __name__ == "__main__":
    main()
