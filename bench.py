#!/usr/bin/env python
"""bench.py -- GCUPS of the batched PO-to-PO gap-fill DP (BASELINE.json metric, configs[1]).

A "step" is one pass of the hot path (DP fill + traceback of every window) over one batch of
synthetic inter-anchor windows (SURVEY.md 8d, config 2: PO graph pairs, ~1-20 k nodes per side,
SNP + 171-node bubbles, production 3-piece parameters), `--windows` of them per GPU.

  value      device-resident throughput: cells of all ranks / max-over-ranks CUDA-event time of K
             `clb_batch_run` calls on a batch already in HBM
  e2e        the same K steps through the reference-facing call `clb_popoa_batch` with HOST buffers:
             host flattening, H2D, kernels, D2H and id translation all inside the timed region
  roofline   the dominant kernel (`popoa_kernel`, INT32/DPX issue bound -- SURVEY.md 8d) + HBM side
  cpu_baseline  the unmodified reference's po_poa (oracle/_ref/libclref.so) or the C port, one
             thread, on a bounded sample of the same windows, parity-checked against the GPU result

`--impl reference` times the reference's own CPU implementation on all host threads instead.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # tests/checkers.py: the CPU checkers of the cpu_baseline / reference legs

METRIC = "GCUPS (graph DP cell updates/s), batched PO-to-PO gap-fill windows"
UNIT = "GCUPS"
SEED = 20261017


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--windows", type=int, default=int(os.environ.get("CLB_BENCH_WINDOWS", "50000")),
                    help="windows per GPU per step (configs[1]: 50000)")
    ap.add_argument("--len-min", type=float, default=880.0)
    ap.add_argument("--len-max", type=float, default=17600.0)
    ap.add_argument("--alt-period", type=int, default=2000, help="one 171-node alternate-path bubble per this many bp (0 = none)")
    ap.add_argument("--snp-rate", type=float, default=0.05)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-other-paths", action="store_true", help="skip the short pwfa / chaining / end-to-end MSA measurements")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --windows per GPU (the driver's 1->8 run); strong: ONE batch of --windows windows dealt to the ranks "
                         "in cell-balanced bins (clb_balanced_partition, the rule of clb_popoa_batch_multi)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's windows) to DIR/<name>.npy, float64: "
                         "every window's score and the alignments of a fixed, seeded sample of windows")
    return ap.parse_args()


REFERENCE_SAMPLE = ("reference arm: per step max(4*cores, 64) windows of the same generator with backbone <= 3 kbp (so that one 28 B/cell "
                    "table per host thread fits in RAM), all host threads each running the single-threaded reference po_poa; the "
                    "reference's per-cell rate is size-independent within 0.020-0.035 GCUPS/thread (BASELINE.md section 2)")


def workload_config(args, world):
    per = "per GPU" if args.scaling == "weak" else f"in total, dealt to {world} rank(s) in cell-balanced bins"
    return {"workload": f"configs[1]: batched inter-anchor windows, {args.windows} synthetic PO-to-PO gap-fill problems {per}, "
                        f"backbone {args.len_min:.0f}-{args.len_max:.0f} bp log-uniform (~1-20 k nodes/side), 5% SNP bubbles, "
                        "171-node bubble per 2 kbp, NumPW=3 production parameters 20/80/{60,800,2500}/{30,5,1}",
            "windows_per_gpu": args.windows if args.scaling == "weak" else args.windows // max(1, world), "num_pw": 3, "seed": SEED,
            "sharding": f"independent windows, {world} rank(s), no collective ({args.scaling} scaling)",
            "reference_sample": REFERENCE_SAMPLE,
            "l2_policy": "inputs (GBs of CSR + workspace) exceed the 126 MB L2; no flush needed"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 8 for k in range(4) if r[4 + k].lower().startswith("active")})
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(sm)}


DUMP_SAMPLE_WINDOWS = 64
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, scores, alns):
    """What a caller of the resident path receives, for comparing two builds output for output: scores.npy (one per
    window), and for a seeded sample of windows (alignment_windows.npy, ascending) their alignments concatenated
    (alignment_pairs.npy, node-id pairs, -1 = gap) with alignment_offsets.npy.  Every value is an integer below 2^53,
    so float64 holds it exactly.  Sampled windows whose alignments would push the files past 64 MB are left out."""
    rng = np.random.default_rng(SEED)
    pick = np.sort(rng.choice(len(scores), min(DUMP_SAMPLE_WINDOWS, len(scores)), replace=False))
    budget = (DUMP_MAX_BYTES - 8 * len(scores) - 16 * (len(pick) + 1)) // 16
    keep = pick[np.cumsum([len(alns[w]) for w in pick]) <= budget]
    off = np.zeros(len(keep) + 1, np.int64)
    np.cumsum([len(alns[w]) for w in keep], out=off[1:])
    pairs = np.concatenate([alns[w] for w in keep]) if len(keep) else np.zeros((0, 2), np.int32)
    os.makedirs(path, exist_ok=True)
    for name, a in (("scores", scores), ("alignment_windows", keep), ("alignment_offsets", off), ("alignment_pairs", pairs)):
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, np.float64))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def cpu_sample(batch, cells, budget_cells, max_cells):
    """Bounded, size-stratified sample of window ids: evenly spaced in the size-sorted order."""
    order = np.argsort(cells, kind="stable")
    order = order[cells[order] <= max_cells]
    if len(order) == 0:
        order = np.argsort(cells, kind="stable")[:1]
    picks, total = [], 0
    for q in np.linspace(0.05, 0.95, 12):
        w = int(order[int(q * (len(order) - 1))])
        if w in picks:
            continue
        if total + int(cells[w]) > budget_cells and picks:
            continue
        picks.append(w)
        total += int(cells[w])
    return picks


def run_reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path, all host threads, bounded sample per step."""
    if rank != 0:
        return
    from concurrent.futures import ThreadPoolExecutor

    from centrolign_b200.batch import AlignmentParameters, select_windows, synth_windows

    from checkers import CpuChecker
    kind = "reference" if CpuChecker.available("reference") else "port"
    chk = CpuChecker(kind)
    cores = os.cpu_count() or 1
    params = AlignmentParameters()
    # bounded sample of the workload: windows small enough that `cores` tables fit in RAM (28 B/cell),
    # ~1.5 s of work per thread per step
    pool_n = max(4 * cores, 64)
    full = synth_windows(pool_n, first_index=0, seed=SEED, len_min=args.len_min, len_max=min(args.len_max, 3000.0))
    cells = full.cells()
    budget = int(0.03e9 * 1.5 * cores)
    order = np.argsort(-cells, kind="stable")
    picks, tot = [], 0
    for w in order:
        if tot >= budget:
            break
        picks.append(int(w))
        tot += int(cells[w])
    sample = select_windows(full, picks)
    scells = float(sample.cells().sum())

    def one(w):
        return chk.po_poa(sample, w, params)[0]

    def step():
        with ThreadPoolExecutor(max_workers=cores) as ex:
            list(ex.map(one, range(sample.n_windows)))

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = scells * args.steps / dt / 1e9
    sample_desc = (f"{sample.n_windows} windows of the same generator (backbone <= 3 kbp so {cores} concurrent 28 B/cell tables fit), "
                   f"{scells:.3g} cells per step, {cores} threads each running the single-threaded reference po_poa")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": workload_config(args, world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_desc},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def other_paths(device):
    """Short measurements of the two other hot-path kernels (outside the timed region of the headline metric),
    each next to the reference's CPU code on the same inputs and parity-checked: the wavefront variant
    pwfa_po_poa (clb_pwfa_batch) and the sparse anchor-chaining DP (clb_chain_dp)."""
    import tempfile

    from centrolign_b200.batch import AlignmentParameters, select_windows, successor_form, synth_windows
    from centrolign_b200.chain import ChainStats, chain_dp, read_chain_bin
    from centrolign_b200.popoa import PwfaStats, pwfa_po_poa_batch

    out = {}
    # ---- pwfa: windows of the size the Stitcher routes to it (4e7 < cells < 7.5e7, stitcher.hpp:327-339) ----
    params = AlignmentParameters()
    nw = 512
    sb = successor_form(synth_windows(nw, first_index=0, seed=SEED, len_min=5600.0, len_max=7600.0))
    pwfa_po_poa_batch(sb, params, 50, device=device)  # warm-up
    st = PwfaStats()
    t0 = time.perf_counter()
    scores, alns = pwfa_po_poa_batch(sb, params, 50, device=device, stats=st)
    wall = time.perf_counter() - t0
    from checkers import CpuChecker
    kind = "reference" if CpuChecker.available("reference") else "port"
    chk = CpuChecker(kind)
    idx = np.linspace(0, nw - 1, 6).astype(int)
    sub = select_windows(sb, idx)
    t0 = time.perf_counter()
    for k, w in enumerate(idx):
        s, a = chk.pwfa_po_poa(sub, k, params, 50)
        assert s == scores[w] and np.array_equal(a, alns[w]), f"pwfa: GPU result differs from the CPU {kind} on window {w}"
    cpu_s = (time.perf_counter() - t0) / len(idx)
    out["pwfa_po_poa"] = {"windows": nw, "nodes_per_side": "6.3-8.7 k", "prune_limit": 50, "kernel_ms": st.kernel_ms,
                          "windows_per_s": nw / (st.kernel_ms * 1e-3), "e2e_windows_per_s": nw / wall,
                          "search_states_per_s": st.states / (st.kernel_ms * 1e-3), "entries_per_warp_step": st.dequeued / max(1, st.steps),
                          "gpu_launches": int(st.kernel_launches),
                          "roofline": {"bound": "latency of the dependent global accesses of one warp step (hash probe -> node record -> "
                                                "FIFO append, ~3 L2 round trips), hidden by resident windows: one warp per window",
                                       "achieved": st.kernel_ms * 1e3 / max(1, st.steps) * min(nw, 148 * 16), "unit": "us per warp step x resident windows",
                                       "peak": 3 * 0.13, "peak_source": "3 dependent L2 round trips of ~250 cycles at 1.965 GHz (B300_MICROARCH.md L2 hit latency)",
                                       "frac": (3 * 0.13) / max(1e-9, st.kernel_ms * 1e3 / max(1, st.steps) * min(nw, 148 * 16)),
                                       "note": "issue slots and HBM are idle (profiles/r01_ncu_pwfa.md: issue 4 %, DRAM 0.7 %); throughput scales with the batch"},
                          "cpu_baseline": {"kind": kind, "cores": 1, "windows_per_s": 1.0 / cpu_s,
                                           "sample": f"{len(idx)} windows, each equal to the GPU result (score + alignment)"}}
    # ---- chaining: a pairwise HOR problem made by the reference's own match finder where its objects travelled ----
    shim = os.path.join(ROOT, "oracle", "_ref", "chain_fixture")
    probs, src = None, None
    if os.path.exists(shim):
        with tempfile.TemporaryDirectory() as tmp:
            fa, binp = os.path.join(tmp, "x.fa"), os.path.join(tmp, "x.bin")
            subprocess.run([sys.executable, os.path.join(ROOT, "integration", "make_hor_fasta.py"), fa, "2", "20000", "7", "0"], check=True)
            r = subprocess.run([shim, fa, binp, "pair", "100000", "1.0"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            if r.returncode == 0:
                probs, src = read_chain_bin(binp), "two 20 kbp HOR arrays, 100 k match pairs, reference timed in this run (1 thread)"
    if probs is None:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from golden_io import load_chain_golden

        probs, src = load_chain_golden()["pair8k_indels"], "tests/golden fixture pair8k_indels (reference time recorded where the fixture was made)"
    chain_out = {"problem": src}
    for kind_name in ("gapfree", "affine"):
        prob = probs[kind_name]
        chain_dp(prob, device=device)
        cst = ChainStats()
        t0 = time.perf_counter()
        chain, dp, bp, opt = chain_dp(prob, device=device, stats=cst)
        wall = (time.perf_counter() - t0) * 1e3
        assert np.array_equal(chain, prob.expect_chain), f"chaining ({kind_name}): GPU chain differs from the reference's"
        t0 = time.perf_counter()
        from checkers import chain_oracle
        ochain = chain_oracle(prob)[0]
        oracle_ms = (time.perf_counter() - t0) * 1e3
        assert np.array_equal(chain, ochain)
        chain_out[kind_name] = {"matches": prob.n_match, "steps": prob.n_step, "kernel_ms": cst.kernel_ms, "build_ms": cst.build_ms,
                                "e2e_ms": wall, "matches_per_s": prob.n_match / (cst.kernel_ms * 1e-3), "reference_cpu_ms": prob.ref_ms,
                                "oracle_cpu_ms": oracle_ms, "chain_len": int(len(chain)), "equal_to_reference": True,
                                "gpu_launches": int(cst.kernel_launches),
                                "roofline": {"bound": "dependent L2 round trips per step of the strictly sequential DP over graph-1 nodes "
                                                      "(insert -> barrier -> query -> barrier)",
                                             "achieved": cst.kernel_ms * 1e3 / max(1, prob.n_step), "unit": "us per step",
                                             "peak": 4 * 0.13, "peak_source": "4 dependent L2 round trips of ~250 cycles at 1.965 GHz per step "
                                                                             "(B300_MICROARCH.md L2 hit latency 234-262 cycles)",
                                             "frac": (4 * 0.13) / max(1e-9, cst.kernel_ms * 1e3 / max(1, prob.n_step))}}
    # ---- batched entry point: fill-in sized problems (anchorer.hpp:619-699 makes thousands of them per alignment) ----
    try:
        from centrolign_b200.chain import chain_dp_batch
        from golden_io import load_chain_golden

        gold = load_chain_golden()
        small = [gold[c][k] for c in sorted(gold) for k in sorted(gold[c]) if gold[c][k].n_match <= 2000]
        if small:
            reps = max(1, 2000 // len(small))
            many = small * reps
            chain_dp_batch(many[: len(small)], device=device)  # warm-up
            bst = ChainStats()
            t0 = time.perf_counter()
            got = chain_dp_batch(many, device=device, stats=bst)
            t_batch = time.perf_counter() - t0
            t0 = time.perf_counter()
            ones = [chain_dp(p, device=device) for p in many[: 4 * len(small)]]
            t_one = (time.perf_counter() - t0) / (4 * len(small)) * len(many)
            assert all(np.array_equal(a[0], b[0]) for a, b in zip(got, ones)), "batched chaining differs from the single calls"
            from centrolign_b200.chain import chain_dp_jobs

            n_threads = min(16, os.cpu_count() or 1)
            chain_dp_jobs(many[: len(small)], device=device, threads=n_threads)
            t0 = time.perf_counter()
            got_jobs = chain_dp_jobs(many, device=device, threads=n_threads)
            t_jobs = time.perf_counter() - t0
            assert all(np.array_equal(a[0], b[0]) for a, b in zip(got_jobs, got)), "threaded job creation changes the chains"
            chain_out["batched_fill_in"] = {"problems": len(many), "matches_total": int(sum(p.n_match for p in many)),
                                            "batch_call_ms": t_batch * 1e3, "kernel_ms": bst.kernel_ms, "gpu_launches": int(bst.kernel_launches),
                                            "jobs_call_ms": t_jobs * 1e3, "jobs_threads": n_threads,
                                            "one_by_one_ms_extrapolated": t_one * 1e3, "speedup": t_one / t_batch, "speedup_jobs": t_one / t_jobs,
                                            "what": "clb_chain_dp_batch: host layout per problem, ONE staging copy, ONE launch (a CTA per problem), "
                                                    "ONE read-back; jobs = clb_chain_job_create on host threads (what the drop-in Anchorer's fill-in pool "
                                                    "does) + ONE clb_chain_jobs_run; one_by_one = clb_chain_dp per problem (timed on a fifth of them)"}
    except Exception as exc:
        chain_out["batched_fill_in"] = {"error": str(exc)[:200]}
    out["chain_dp"] = chain_out
    return out


def pipeline_windows(device):
    """Windows of the size the reference's own Stitcher sends to po_poa (SURVEY.md section 6, 2 x 93 kbp HOR arrays:
    median 9 cells, p90 49, p99 169, max 18 549): windows/s through clb_popoa_batch with host buffers, with the
    warp-per-window kernel (popoa_small_kernels.cu) and, for comparison, with every window forced through the
    CTA-per-window strip kernel; the reference on one core on a sample, parity-checked."""
    from centrolign_b200.batch import AlignmentParameters, concat_batches, select_windows, synth_windows
    from centrolign_b200.popoa import DeviceBatch, po_poa_batch

    params = AlignmentParameters()
    nw = 200000
    mix = [(0.55, 2.0, 2.4), (0.35, 2.4, 7.0), (0.09, 7.0, 13.0), (0.01, 13.0, 135.0)]  # share, backbone length range per side
    batch = concat_batches([synth_windows(int(nw * f), first_index=k * 10 ** 7, seed=SEED + 1, len_min=lo, len_max=hi, alt_period=0)
                            for k, (f, lo, hi) in enumerate(mix)])
    cells = batch.cells()
    out = {"windows": int(batch.n_windows), "cells": float(cells.sum()), "cells_median": float(np.median(cells)),
           "cells_p90": float(np.percentile(cells, 90)), "cells_p99": float(np.percentile(cells, 99)), "cells_max": float(cells.max())}
    res = {}
    for name, env in (("warp_per_window", None), ("cta_per_window", "1")):
        if env:
            os.environ["CLB_NO_SMALL_WINDOWS"] = env
        try:
            po_poa_batch(batch, params, device=device)  # warm-up
            t0 = time.perf_counter()
            res[name] = po_poa_batch(batch, params, device=device)
            dt = time.perf_counter() - t0
        finally:
            os.environ.pop("CLB_NO_SMALL_WINDOWS", None)
        out[name] = {"seconds": dt, "windows_per_s": batch.n_windows / dt, "ns_per_cell": dt * 1e9 / float(cells.sum()),
                     "includes": "host flattening, H2D, kernels, D2H, id translation"}
        if env:
            os.environ["CLB_NO_SMALL_WINDOWS"] = env
        try:  # the kernels alone, on a batch resident in HBM (CUDA events of clb_batch_run)
            db = DeviceBatch(batch, params, device=device)
            db.upload()
            db.run()
            kms = []
            for _ in range(3):
                db.run()
                kms.append(db.stats().kernel_ms)
            out[name]["kernel_ms"] = float(np.median(kms))
            out[name]["kernel_windows_per_s"] = batch.n_windows / (float(np.median(kms)) * 1e-3)
            out[name]["kernel_launches"] = int(db.stats().kernel_launches)
            db.close()
        finally:
            os.environ.pop("CLB_NO_SMALL_WINDOWS", None)
    assert np.array_equal(res["warp_per_window"][0], res["cta_per_window"][0])
    assert all(np.array_equal(a, b) for a, b in zip(res["warp_per_window"][1], res["cta_per_window"][1])), "the two kernels disagree"
    out["speedup_over_cta_per_window"] = out["cta_per_window"]["seconds"] / out["warp_per_window"]["seconds"]
    out["kernel_speedup_over_cta_per_window"] = out["cta_per_window"]["kernel_ms"] / out["warp_per_window"]["kernel_ms"]
    from checkers import CpuChecker
    kind = "reference" if CpuChecker.available("reference") else "port"
    chk = CpuChecker(kind)
    idx = np.linspace(0, batch.n_windows - 1, 3000).astype(int)
    t0 = time.perf_counter()
    for w in idx:
        s, a = chk.po_poa(batch, int(w), params)
        assert s == res["warp_per_window"][0][w] and np.array_equal(a, res["warp_per_window"][1][w]), f"pipeline window {w} differs from the CPU {kind}"
    dt = time.perf_counter() - t0
    out["cpu_baseline"] = {"kind": kind, "cores": 1, "windows_per_s": len(idx) / dt, "ns_per_cell": dt * 1e9 / float(cells[idx].sum()),
                           "sample": f"{len(idx)} windows evenly spaced, each equal to the GPU result; includes the ctypes call per window",
                           "reference_in_pipeline_ns_per_cell": 134}
    return out


E2E_CASES = [  # (name in tests/golden/e2e.json, what it stands for)
    ("pair100k_default", "configs[0] at full size, default options: two 100 kbp HOR arrays -> CIGAR"),
    ("tree4_3k_default", "configs[2] scaled: four 3 kbp HOR arrays with HOR indels, Newick guide tree, default options -> GFA"),
    ("msa3_2k5_cyclic", "configs[4] scaled: three 2.5 kbp arrays with HOR indels, -c with cyclizing size 800 -> cyclic GFA"),
]
E2E_LIVE_REFERENCE_S = 150.0  # the unmodified CLI is run live if the fixture says it needs at most this long (else its recorded time is quoted)


def e2e_msa(device):
    """End-to-end MSA wall time and output identity (BASELINE.json metric, second half): the reference CLI built from its
    own unmodified sources (oracle/_ref/centrolign_ref) next to the same sources built with the shadow headers
    (oracle/_ref/centrolign_b200: chaining DP, po_poa and pwfa_po_poa on the GPU), same input, outputs compared by md5
    with each other and with the md5 recorded from the unmodified CLI in tests/golden/e2e.json."""
    import hashlib
    import tempfile

    clis = {k: os.path.join(ROOT, "oracle", "_ref", "centrolign_" + k) for k in ("ref", "b200")}
    if not all(os.path.exists(c) for c in clis.values()):
        return {"unavailable": "oracle/_ref/centrolign_{ref,b200} did not travel (built by `make -C integration` where /root/reference exists)"}
    sys.path.insert(0, os.path.join(ROOT, "integration"))
    from make_e2e_golden import run_cli

    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "e2e.json")))
    out = {"what": "wall seconds of the whole CLI run (process start to exit, GPU context creation included); the reference is single-threaded; "
                   "identical = md5 of stdout (CIGAR / GFA) equal"}
    env = dict(os.environ, CLB_COUNT_CALLS="1", CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(device)))
    with tempfile.TemporaryDirectory() as tmp:
        for name, what in E2E_CASES:
            case = gold[name]
            fa = os.path.join(tmp, name + ".fa")
            subprocess.run([sys.executable, os.path.join(ROOT, "integration", "make_hor_fasta.py"), fa] + [str(a) for a in case["fasta_args"]], check=True)
            row = {"what": what, "options": " ".join(case["options"]) or "(defaults)", "recorded_reference_md5": case["output_md5"],
                   "recorded_reference_seconds": case["reference_seconds"]}
            for k in ("b200", "ref"):
                if k == "ref" and case["reference_seconds"] > E2E_LIVE_REFERENCE_S:
                    row[k] = {"seconds": None, "note": f"not run live (needs {case['reference_seconds']} s where the fixture was made); see recorded_reference_*"}
                    continue
                t0 = time.perf_counter()
                res = run_cli(clis[k], case["options"], fa, case.get("config_overrides") or {}, tmp, env=env, tree=case.get("tree"))
                row[k] = {"seconds": round(time.perf_counter() - t0, 2), "returncode": res.returncode, "output_bytes": len(res.stdout),
                          "md5": hashlib.md5(res.stdout).hexdigest()}
                if k == "b200":
                    row[k]["gpu_calls"] = [l for l in res.stderr.decode().splitlines() if l.startswith("[clb]")]
            accepted = [case["output_md5"]] + case.get("reference_also_printed", [])
            if "md5" in row["ref"]:
                accepted.append(row["ref"]["md5"])
            row["identical"] = bool(row["b200"].get("returncode") == 0 and row["b200"]["md5"] in accepted)
            if case.get("reference_also_printed"):
                row["note"] = "the unmodified reference is not reproducible in -c mode (its output follows argv): tests/golden/e2e.json"
            ref_s = row["ref"].get("seconds") or case["reference_seconds"]
            row["speedup"] = round(ref_s / row["b200"]["seconds"], 2) if row["b200"].get("seconds") else None
            out[name] = row
    return out


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch

    from centrolign_b200.batch import AlignmentParameters, select_windows, synth_windows
    from centrolign_b200.popoa import DeviceBatch, load_library, po_poa_batch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the gap-fill path)")
    torch.cuda.set_device(local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = load_library()
    params = AlignmentParameters()

    # host-memory guard: ~0.8 MB of host RAM per window (raw arrays, pinned staging, outputs) and rank
    try:
        import psutil

        avail = psutil.virtual_memory().available / max(1, world)
        fit = int(avail * 0.6 / 0.8e6) * (world if args.scaling == "strong" else 1)
        if fit < args.windows:
            if args.dump_outputs:  # dumped outputs are compared across runs: the inputs must not depend on the host's free RAM
                raise SystemExit(f"bench.py: host RAM allows {fit} windows per rank, not {args.windows}; pass --windows {max(1000, fit)}")
            if rank == 0:
                print(f"[bench] host RAM allows {fit} windows per rank, not {args.windows}: reducing", file=sys.stderr)
            args.windows = max(1000, fit)
    except ImportError:
        pass
    if use_dist:
        t = torch.tensor([args.windows], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        args.windows = int(t.item())
    t_gen = time.perf_counter()
    if args.scaling == "strong" and world > 1:
        # ONE batch of args.windows windows: every rank computes the same cell-balanced assignment from the backbone
        # lengths (node counts are proportional to them) and generates only its own share
        from centrolign_b200.batch import synth_backbone_lengths
        from centrolign_b200.popoa import balanced_partition_c

        lens = synth_backbone_lengths(args.windows, 0, SEED, args.len_min, args.len_max)
        part = balanced_partition_c(lens * lens, world)
        batch = synth_windows(0, seed=SEED, len_min=args.len_min, len_max=args.len_max, snp_rate=args.snp_rate,
                              alt_period=args.alt_period, indices=np.nonzero(part == rank)[0])
    else:
        batch = synth_windows(args.windows, first_index=rank * args.windows, seed=SEED, len_min=args.len_min, len_max=args.len_max,
                              snp_rate=args.snp_rate, alt_period=args.alt_period)
    t_gen = time.perf_counter() - t_gen
    cells = batch.cells()
    my_cells = float(cells.sum())

    db = DeviceBatch(batch, params, device=local)
    db.upload()

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        db.run()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    kernel_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        db.run()
        kernel_ms += db.stats().kernel_ms  # CUDA events on the library's own stream
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if rank == 0 else None
    st = db.stats()
    launches_per_step = int(st.kernel_launches)

    # results of the resident run (for the parity check of the CPU sample)
    scores, alns = db.download()
    scores = scores.copy()
    if args.dump_outputs and rank == 0:  # before the e2e leg, which reuses db's alignment buffer
        dump_outputs(args.dump_outputs, scores, alns)
    st = db.stats()  # now includes the D2H byte count
    db.close()

    # ---- e2e: the reference-facing one-shot call with host buffers ----
    e2e_ms, h2d, d2h = None, int(st.h2d_bytes), int(st.d2h_bytes)
    if not args.no_e2e:
        out = (np.zeros(batch.n_windows, np.int64), db.aln_off, db.aln_pairs, np.zeros(batch.n_windows, np.uint32))
        po_poa_batch(batch, params, device=local, out=out)  # one warm-up pass (page-in, pinned pools)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            po_poa_batch(batch, params, device=local, out=out)
        torch.cuda.synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        assert np.array_equal(out[0], scores), "e2e scores differ from the resident run"

    def allmax(x):
        if not use_dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if not use_dist:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    kernel_ms_max = allmax(kernel_ms)
    total_cells = allsum(my_cells)
    e2e_ms_max = allmax(e2e_ms) if e2e_ms is not None else None
    value = total_cells * args.steps / (kernel_ms_max * 1e-3) / 1e9

    if rank == 0:
        # ---- roofline of the dominant kernel ----
        peak_dpx = lib.clb_int32_peak_tops(local, 1)
        peak_plain = lib.clb_int32_peak_tops(local, 0)
        peak = max(peak_dpx, peak_plain)
        step_s = kernel_ms / args.steps * 1e-3
        achieved = st.int_ops / step_s / 1e12
        peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
        hbm_peak, hbm_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        if os.path.exists(peaks_file):
            hbm_peak, hbm_src = float(json.load(open(peaks_file))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
        hbm_bytes = float(st.persist_bytes + st.h2d_bytes)
        roofline = {"bound": "int32", "kernel": "popoa_kernel<3> (fused DP fill + traceback, 1 launch per step)",
                    "achieved": achieved, "peak": peak, "unit": "TOP/s", "frac": achieved / peak if peak > 0 else None,
                    "traffic": hbm_bytes,
                    "ops_per_launch": int(st.int_ops), "ops_model": "SURVEY 8d: a*b+1+4P(a+b)+2P INT32 add/max per cell (32 for a linear cell at P=3)",
                    "peak_source": f"measured in this run by clb_int32_peak_tops: DPX viaddmax {peak_dpx:.1f}, add+max {peak_plain:.1f} TOP/s "
                                   "(nominal 148 SM x 128 lanes x 1.965 GHz = 37.2)",
                    "hbm": {"bound": "hbm", "achieved": hbm_bytes / step_s / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": hbm_bytes / step_s / 1e9 / hbm_peak, "traffic": hbm_bytes,
                            "bytes_model": "persisted rows/columns written once + flattened graph arrays read once", "peak_source": hbm_src,
                            "traffic_model": "bytes per launch = persisted rows {M,H_k} and columns {M,D_k}+E written once (persist_bytes) + "
                                             "flattened graph arrays read once (h2d_bytes); ncu cross-check on the 1480-window profile batch: "
                                             "dram read+write 27.2 GB per launch for 2.37e10 cells = 1.15 B/cell (profiles/r02_ncu_popoa.md)"}}
        # ---- CPU baseline on a bounded sample, parity-checked against the GPU result ----
        cpu = None
        if not args.no_cpu_baseline:
            from checkers import CpuChecker
            kind = "reference" if CpuChecker.available("reference") else "port"
            chk = CpuChecker(kind)
            picks = cpu_sample(batch, cells, budget_cells=int(5e8), max_cells=int(1.2e8))
            t_cpu, c_cpu = 0.0, 0.0
            for w in picks:
                t1 = time.perf_counter()
                s, a = chk.po_poa(batch, w, params)
                t_cpu += time.perf_counter() - t1
                c_cpu += float(cells[w])
                assert s == scores[w] and np.array_equal(a, alns[w]), f"GPU result differs from the CPU {kind} on window {w}"
            cpu = {"value": c_cpu / t_cpu / 1e9, "unit": UNIT, "cores": 1, "kind": kind,
                   "sample": f"{len(picks)} windows evenly spaced in the size-sorted batch (<=1.2e8 cells each), {c_cpu:.3g} cells, "
                             f"{t_cpu:.1f} s single-threaded; score+alignment of every sampled window equal to the GPU's",
                   "host_cores": os.cpu_count()}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": kernel_ms_max / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "int32", "data": "synthetic", "config": workload_config(args, world),
                "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
                "e2e": None if e2e_ms_max is None else {"value": total_cells * args.steps / (e2e_ms_max * 1e-3) / 1e9, "unit": UNIT,
                                                         "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                                         "ms_per_step": e2e_ms_max / args.steps,
                                                         "includes": "host topological flattening, pinned staging, H2D, kernels, D2H, id translation"},
                "gpu_launches": launches_per_step * args.steps,
                "wall_ms_per_step": wall_ms / args.steps, "cells_per_step": total_cells, "windows_gen_s": t_gen,
                "workspace_bytes": int(st.workspace_bytes)}
        if world == 1 and not args.no_other_paths:
            try:
                line["other_paths"] = other_paths(local)
            except Exception as exc:  # the headline metric stands on its own
                line["other_paths"] = {"error": str(exc)[:300]}
            try:
                line["other_paths"]["pipeline_windows"] = pipeline_windows(local)
            except Exception as exc:
                line["other_paths"]["pipeline_windows"] = {"error": str(exc)[:300]}
            try:
                line["other_paths"]["e2e_msa"] = e2e_msa(local)
            except Exception as exc:
                line["other_paths"]["e2e_msa"] = {"error": str(exc)[:300]}
        print(json.dumps(line), flush=True)
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
