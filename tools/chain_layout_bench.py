"""Host layout against device layout of the chaining search structures (clb_chain_dp, CLB_CHAIN_LAYOUT=host|device).

Seeded synthetic problems (centrolign_b200.chain.synth_chain_problem) from 10^3 to 10^7 tree entries, gap-free and
affine, with one and with three chains per graph.  Per problem both layouts run in the same process, alternating, `reps`
times each after one warm-up call of each; the table reports the best `build_ms` (layout time: host threads, or device
kernels up to a synchronise) and the best whole-call time of either side.  Outputs of the two sides must be identical
(asserted).  Prints one JSON line per problem and writes them, with the card's name and power limit, to --out.
    python tools/chain_layout_bench.py [--reps 3] [--min-entries 0] [--max-entries 10000000] [--out chain_layout.json]
There is no CPU path: without a CUDA device the calls raise."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from centrolign_b200.chain import ChainStats, chain_dp, synth_chain_problem  # noqa: E402


def gpu_info():
    """Name and power limit of the GPUs the numbers were taken on (read-only query)."""
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                             stderr=subprocess.DEVNULL, text=True, timeout=30)
        return sorted(set(line.strip() for line in res.stdout.splitlines() if line.strip()))
    except (OSError, subprocess.SubprocessError):
        return ["unknown"]


def run(prob, side):
    os.environ["CLB_CHAIN_LAYOUT"] = side
    st = ChainStats()
    out = chain_dp(prob, stats=st)
    return out, st


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--min-entries", type=int, default=0)
    ap.add_argument("--max-entries", type=int, default=10_000_000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    rows = []
    sizes = [1_000, 3_000, 10_000, 30_000, 100_000, 300_000, 1_000_000, 3_000_000, 10_000_000]
    for entries in [s for s in sizes if args.min_entries <= s <= args.max_entries]:
        for chains in (1, 3):
            for num_pw in (0, 2):
                npm = chains * chains
                M = max(16, entries // npm)
                # a few thousand steps keep the DP itself short next to the layout at every size
                prob = synth_chain_problem(M, chains, chains, num_pw, seed=entries + chains + num_pw, shifts=256, offsets=1 << 20,
                                           n_step=min(M // 2, 4096))
                best = {"host": [1e30, 1e30], "device": [1e30, 1e30]}
                ref = None
                for rep in range(args.reps + 1):
                    for side in (("host", "device") if rep % 2 == 0 else ("device", "host")):
                        out, st = run(prob, side)
                        if ref is None:
                            ref = out
                        else:
                            assert np.array_equal(out[0], ref[0]) and out[3] == ref[3], f"{side}: chain differs"
                            assert np.array_equal(out[1].view(np.uint32), ref[1].view(np.uint32)), f"{side}: dp values differ"
                            assert np.array_equal(out[2], ref[2]), f"{side}: back-pointers differ"
                        if rep:  # rep 0 warms both sides up
                            best[side][0] = min(best[side][0], st.build_ms)
                            best[side][1] = min(best[side][1], st.total_ms)
                row = {"entries": int(prob.arrays["ins_off"][-1]), "matches": M, "chains": chains, "num_pw": num_pw,
                       "steps": prob.n_step, "host_build_ms": round(best["host"][0], 3), "device_build_ms": round(best["device"][0], 3),
                       "host_total_ms": round(best["host"][1], 3), "device_total_ms": round(best["device"][1], 3),
                       "identical": True}
                rows.append(row)
                print(json.dumps(row), flush=True)
    os.environ.pop("CLB_CHAIN_LAYOUT", None)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"gpu": info, "reps": args.reps, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
