"""Python front for ``clb_chain_dp`` (include/centrolign_b200.h) -- harness plumbing only.

The sparse anchor-chaining DP of the reference (``Anchorer::sparse_affine_chain_dp`` /
``Anchorer::sparse_chain_dp``, include/centrolign/anchorer.hpp:1812-2471 / :1511-1750) runs in
``libcentrolign_b200.so``; this module only moves the flat problem arrays (``clb_chain_problem``) across
ctypes.  The C++ host layer that produces such problems from the reference's own objects is
``centrolign_b200/hostcpp/chain_b200.hpp``.  There is no CPU path here.
"""
from __future__ import annotations

import ctypes
import struct
from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np

from .popoa import _check, load_library

_FIELDS = [("weight", np.float32), ("dp_init", np.float32), ("final_term", np.float32), ("end_off", np.int64),
           ("end_match", np.uint32), ("qry_off", np.int64), ("qry_match", np.uint32), ("qry_chain1", np.uint32),
           ("ins_off", np.int64), ("ins_p1", np.uint32), ("ins_p2", np.uint32), ("ins_shift", np.int32),
           ("ins_offset", np.uint32), ("ins_active", np.uint8), ("qa1", np.int32), ("qa2", np.int32), ("qoff", np.uint32)]


class _CProblem(ctypes.Structure):
    _fields_ = [("num_pw", ctypes.c_int32), ("gap_open", ctypes.c_double * 3), ("gap_extend", ctypes.c_double * 3),
                ("scale", ctypes.c_double), ("n_chain1", ctypes.c_int32), ("n_chain2", ctypes.c_int32),
                ("n_match", ctypes.c_int64), ("weight", ctypes.c_void_p), ("dp_init", ctypes.c_void_p),
                ("final_term", ctypes.c_void_p), ("min_score", ctypes.c_float), ("n_step", ctypes.c_int64),
                ("end_off", ctypes.c_void_p), ("end_match", ctypes.c_void_p), ("qry_off", ctypes.c_void_p),
                ("qry_match", ctypes.c_void_p), ("qry_chain1", ctypes.c_void_p), ("ins_off", ctypes.c_void_p),
                ("ins_p1", ctypes.c_void_p), ("ins_p2", ctypes.c_void_p), ("ins_shift", ctypes.c_void_p),
                ("ins_offset", ctypes.c_void_p), ("ins_active", ctypes.c_void_p), ("qa1", ctypes.c_void_p), ("qa2", ctypes.c_void_p), ("qoff", ctypes.c_void_p)]


class ChainStats(ctypes.Structure):
    _fields_ = [("build_ms", ctypes.c_double), ("kernel_ms", ctypes.c_double), ("total_ms", ctypes.c_double),
                ("steps", ctypes.c_int64), ("inserts", ctypes.c_int64), ("queries", ctypes.c_int64),
                ("tree_bytes", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64),
                ("kernel_launches", ctypes.c_int64)]


@dataclass
class ChainProblem:
    """Mirror of ``clb_chain_problem``; array meanings are documented in include/centrolign_b200.h."""

    num_pw: int
    gap_open: tuple
    gap_extend: tuple
    scale: float
    n_chain1: int
    n_chain2: int
    min_score: float
    arrays: Dict[str, np.ndarray]
    expect_chain: Optional[np.ndarray] = None  # fixture only: the chain the reference found (match ranks)
    ref_ms: float = 0.0  # fixture only: the reference's run time for this problem where the fixture was made
    meta: dict = field(default_factory=dict)

    @property
    def n_match(self) -> int:
        return len(self.arrays["weight"])

    @property
    def n_step(self) -> int:
        return len(self.arrays["end_off"]) - 1


def _bind(lib):
    if getattr(lib, "_chain_bound", False):
        return
    lib.clb_chain_dp.restype = ctypes.c_int
    lib.clb_chain_dp.argtypes = [ctypes.c_int, ctypes.POINTER(_CProblem), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                 ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ChainStats)]
    lib.clb_chain_job_create.restype = ctypes.c_int
    lib.clb_chain_job_create.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_void_p]
    lib.clb_chain_jobs_run.restype = ctypes.c_int
    lib.clb_chain_jobs_run.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.c_void_p]
    lib.clb_chain_job_destroy.restype = None
    lib.clb_chain_job_destroy.argtypes = [ctypes.c_void_p]
    lib.clb_chain_dp_batch.restype = ctypes.c_int
    lib.clb_chain_dp_batch.argtypes = [ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ChainStats)]
    lib.clb_chain_dp_batch_multi.restype = ctypes.c_int
    lib.clb_chain_dp_batch_multi.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.POINTER(ChainStats)]
    lib._chain_bound = True


def _c_problem(problem: ChainProblem):
    keep = {k: np.ascontiguousarray(problem.arrays[k], dt) for k, dt in _FIELDS}
    cp = _CProblem()
    cp.num_pw = problem.num_pw
    for k in range(3):
        cp.gap_open[k] = problem.gap_open[k] if k < len(problem.gap_open) else 0.0
        cp.gap_extend[k] = problem.gap_extend[k] if k < len(problem.gap_extend) else 0.0
    cp.scale, cp.n_chain1, cp.n_chain2 = problem.scale, problem.n_chain1, problem.n_chain2
    cp.n_match, cp.n_step, cp.min_score = problem.n_match, problem.n_step, problem.min_score
    for k, _ in _FIELDS:
        setattr(cp, k, keep[k].ctypes.data)
    return cp, keep


def chain_dp_batch(problems, device: int = 0, stats: Optional[ChainStats] = None):
    """``clb_chain_dp_batch``: many independent problems in one call (one launch for all that fit shared memory).
    Returns a list of (chain ranks, dp values, back-pointers, optimum), one per problem."""
    return _chain_batch(problems, stats, lambda lib, *args: lib.clb_chain_dp_batch(device, *args))


def chain_dp_batch_multi(problems, devices, stats: Optional[ChainStats] = None, return_parts: bool = False):
    """``clb_chain_dp_batch_multi``: the problems dealt to several GPUs of one box by their step, insert and query counts,
    ``clb_chain_dp_batch`` on each device's share.  ``devices`` is a list of distinct device ordinals.  Returns the list of
    ``chain_dp_batch``, plus the index into ``devices`` each problem ran on if ``return_parts``."""
    devs = np.ascontiguousarray(list(devices), np.int32)
    parts = np.zeros(max(1, len(problems)), np.int32)
    out = _chain_batch(problems, stats, lambda lib, n, *args: lib.clb_chain_dp_batch_multi(
        len(devs), devs.ctypes.data, n, *args[:-1], parts.ctypes.data, args[-1]))
    return (out, parts[: len(problems)]) if return_parts else out


def _chain_batch(problems, stats, call):
    lib = load_library()
    _bind(lib)
    n = len(problems)
    cps = [_c_problem(p) for p in problems]
    ms = [p.n_match for p in problems]
    dps = [np.zeros(max(1, m), np.float32) for m in ms]
    bps = [np.full(max(1, m), -1, np.int64) for m in ms]
    chains = [np.zeros(m + 1, np.int64) for m in ms]
    lens = np.zeros(max(1, n), np.int64)
    opts = np.zeros(max(1, n), np.float32)
    PP = ctypes.POINTER(_CProblem) * max(1, n)
    VP = ctypes.c_void_p * max(1, n)
    parr = PP(*[ctypes.pointer(c[0]) for c in cps]) if n else PP()
    _check(call(lib, n, parr, VP(*[a.ctypes.data for a in dps]), VP(*[a.ctypes.data for a in bps]),
                VP(*[a.ctypes.data for a in chains]), lens.ctypes.data, opts.ctypes.data,
                ctypes.byref(stats) if stats is not None else None))
    return [(chains[k][: int(lens[k])].copy(), dps[k][: ms[k]], bps[k][: ms[k]], float(opts[k])) for k in range(n)]


def chain_dp_jobs(problems, device: int = 0, threads: int = 4):
    """The batched call in two halves (``clb_chain_job_create`` on ``threads`` host threads, then ONE ``clb_chain_jobs_run``):
    what the drop-in Anchorer's fill-in pool does.  Returns the same list as chain_dp_batch."""
    from concurrent.futures import ThreadPoolExecutor

    lib = load_library()
    _bind(lib)
    n = len(problems)
    cps = [_c_problem(p) for p in problems]
    ms = [p.n_match for p in problems]
    dps = [np.zeros(max(1, m), np.float32) for m in ms]
    bps = [np.full(max(1, m), -1, np.int64) for m in ms]
    chains = [np.zeros(m + 1, np.int64) for m in ms]
    lens = [ctypes.c_int64(0) for _ in range(n)]
    opts = [ctypes.c_float(0) for _ in range(n)]
    jobs = [ctypes.c_void_p(None) for _ in range(n)]

    def create(k):  # ctypes releases the GIL: the layouts really run side by side
        return lib.clb_chain_job_create(device, ctypes.byref(cps[k][0]), dps[k].ctypes.data, bps[k].ctypes.data, chains[k].ctypes.data,
                                        ctypes.byref(lens[k]), ctypes.byref(opts[k]), ctypes.byref(jobs[k]))

    try:
        with ThreadPoolExecutor(max(1, threads)) as pool:
            for rc in pool.map(create, range(n)):
                _check(rc)
        live = [j for j in jobs if j.value]
        arr = (ctypes.c_void_p * max(1, len(live)))(*[j.value for j in live])
        _check(lib.clb_chain_jobs_run(device, len(live), arr))
    finally:
        for j in jobs:
            if j.value:
                lib.clb_chain_job_destroy(j)
    return [(chains[k][: int(lens[k].value)].copy(), dps[k][: ms[k]], bps[k][: ms[k]], float(opts[k].value)) for k in range(n)]


def chain_dp(problem: ChainProblem, device: int = 0, stats: Optional[ChainStats] = None):
    """Run the chaining DP + traceback on the GPU.  Returns (chain ranks, dp values, back-pointers, optimum)."""
    lib = load_library()
    _bind(lib)
    cp, keep = _c_problem(problem)
    m = problem.n_match
    dp = np.zeros(max(1, m), np.float32)
    bp = np.full(max(1, m), -1, np.int64)
    chain = np.zeros(m + 1, np.int64)
    n = ctypes.c_int64(0)
    opt = ctypes.c_float(0)
    _check(lib.clb_chain_dp(device, ctypes.byref(cp), dp.ctypes.data, bp.ctypes.data, chain.ctypes.data, ctypes.byref(n),
                            ctypes.byref(opt), ctypes.byref(stats) if stats is not None else None))
    return chain[: n.value].copy(), dp[:m], bp[:m], float(opt.value)


def synth_fill_in_problems(n_problems: int, seed: int = 0, matches=(20, 60), num_pw=(0, 1, 3)):
    """Independent random problems of the size the Anchorer's fill-in pass makes (a few dozen matches on one path per
    graph), for tests and benchmarks of the batched calls.  Every array is in range and every DP is well defined; the
    values mean nothing.  Problem k has ``num_pw[k % len(num_pw)]`` gap pieces."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n_problems):
        P = num_pw[k % len(num_pw)]
        M = int(rng.integers(matches[0], matches[1] + 1))
        n1 = 4 * M + 8  # nodes of graph 1 = steps
        ln = rng.integers(2, 6, M)
        s1 = rng.integers(0, n1 - 6, M)
        s2 = np.clip(s1 + rng.integers(-5, 6, M), 0, n1 - 6)
        e1, e2 = s1 + ln - 1, s2 + ln - 1
        ends = sorted(range(M), key=lambda m: (e1[m], m))
        starts = sorted((m for m in range(M) if s1[m] > 0), key=lambda m: (s1[m], m))  # queried from the edge s1-1 -> s1
        end_off = np.searchsorted(e1[ends], np.arange(n1 + 1), side="left").astype(np.int64)
        qry_off = np.searchsorted(s1[starts] - 1, np.arange(n1 + 1), side="left").astype(np.int64)
        w = ln.astype(np.float32)
        a = dict(weight=w, dp_init=(w - 0.1 * s1).astype(np.float32), final_term=(-0.05 * (n1 - e1)).astype(np.float32),
                 end_off=end_off, end_match=np.asarray(ends, np.uint32), qry_off=qry_off,
                 qry_match=np.asarray(starts, np.uint32), qry_chain1=np.zeros(len(starts), np.uint32),
                 ins_off=np.arange(M + 1, dtype=np.int64), ins_p1=np.zeros(M, np.uint32), ins_p2=np.zeros(M, np.uint32),
                 ins_shift=(e1 - e2).astype(np.int32), ins_offset=e2.astype(np.uint32), ins_active=np.ones(M, np.uint8),
                 qa1=(s1 - 1).astype(np.int32), qa2=(s2 - 1).astype(np.int32), qoff=s2.astype(np.uint32))
        kp = max(1, P)
        out.append(ChainProblem(P, (1.0, 2.0, 3.0)[:kp], (0.5, 0.2, 0.1)[:kp], 1.0, 1, 1, 0.0, a))
    return out


def synth_chain_problem(n_match: int, n_chain1: int = 1, n_chain2: int = 1, num_pw: int = 1, seed: int = 0, shifts: int = 16,
                        offsets: int = 64, inactive: float = 0.1, empty_pair: bool = False, n_step: Optional[int] = None):
    """One random problem with an entry per match on every (chain1, chain2) pair, for tests and benchmarks of the search
    structures: ``n_match * n_chain1 * n_chain2`` tree entries (one pair fewer per match with ``empty_pair``).  Shifts are
    drawn from ``shifts`` values and offsets from ``offsets`` values, so small ranges give many equal keys; a fraction
    ``inactive`` of the entries shape their trees without being entered.  Every match is queried on the step before its
    start, which precedes its end, on one of ``n_step`` steps (default n_match / 2); the values mean nothing."""
    rng = np.random.default_rng(seed)
    M, C1, C2 = n_match, n_chain1, n_chain2
    n1 = max(16, M // 2 if n_step is None else n_step)  # steps: several matches end on most of them
    ln = rng.integers(2, 6, M)
    s1 = rng.integers(1, n1 - 6, M)
    e1 = s1 + ln - 1
    ends = np.lexsort((np.arange(M), e1))
    starts = np.lexsort((np.arange(M), s1))
    pairs = [(p1, p2) for p1 in range(C1) for p2 in range(C2)]
    if empty_pair and len(pairs) > 1:
        pairs = pairs[:-1]
    npm = len(pairs)
    E = M * npm
    a = dict(weight=ln.astype(np.float32), dp_init=(ln - 0.01 * s1).astype(np.float32),
             final_term=(-0.001 * (n1 - e1)).astype(np.float32),
             end_off=np.searchsorted(e1[ends], np.arange(n1 + 1), side="left").astype(np.int64), end_match=ends.astype(np.uint32),
             qry_off=np.searchsorted(s1[starts] - 1, np.arange(n1 + 1), side="left").astype(np.int64),
             qry_match=starts.astype(np.uint32), qry_chain1=rng.integers(0, C1, M).astype(np.uint32),
             ins_off=(np.arange(M + 1, dtype=np.int64) * npm),
             ins_p1=np.tile(np.array([p for p, _ in pairs], np.uint32), M), ins_p2=np.tile(np.array([q for _, q in pairs], np.uint32), M),
             ins_shift=rng.integers(-shifts, shifts, E).astype(np.int32), ins_offset=rng.integers(0, offsets, E).astype(np.uint32),
             ins_active=(rng.random(E) >= inactive).astype(np.uint8),
             qa1=rng.integers(0, offsets + shifts, M * C1).astype(np.int32), qa2=rng.integers(0, offsets, M * C2).astype(np.int32),
             qoff=rng.integers(0, offsets + 1, M * C2).astype(np.uint32))
    k = max(1, num_pw)
    return ChainProblem(num_pw, (1.0, 2.0, 3.0)[:k], (0.5, 0.2, 0.1)[:k], 1.0, C1, C2, 0.0, a)


_DTYPES = {0: np.float32, 1: np.int32, 2: np.uint32, 3: np.int64, 4: np.float64}


def read_chain_bin(path: str) -> Dict[str, ChainProblem]:
    """Read a file written by oracle/_ref/chain_fixture (oracle/chain_shim.cpp): {'gapfree', 'affine', 'local'}."""
    raw: Dict[str, np.ndarray] = {}
    with open(path, "rb") as f:
        data = f.read()
    pos = 0
    while pos < len(data):
        (ln,) = struct.unpack_from("<I", data, pos)
        pos += 4
        name = data[pos: pos + ln].decode()
        pos += ln
        code, n = struct.unpack_from("<IQ", data, pos)
        pos += 12
        dt = np.dtype(_DTYPES[code])
        raw[name] = np.frombuffer(data, dt, n, pos).copy()
        pos += n * dt.itemsize
    return problems_from_arrays(raw)


def problems_from_arrays(raw, prefix: str = "") -> Dict[str, ChainProblem]:
    """Group ``<prefix><kind>.<field>`` arrays (kind = gapfree / affine / local) into ChainProblems."""
    out = {}
    kinds = sorted({k[len(prefix):].split(".")[0] for k in raw if k.startswith(prefix) and "." in k[len(prefix):]})
    meta = raw["meta"] if "meta" in raw else None
    for kind in kinds:
        pre = prefix + kind
        prm = raw[pre + ".params"]
        out[kind] = ChainProblem(int(prm[0]), tuple(prm[1:4]), tuple(prm[4:7]), float(prm[7]), int(prm[8]), int(prm[9]),
                                 float(raw[pre + ".min_score"][0]), {k: raw[f"{pre}.{k}"] for k, _ in _FIELDS},
                                 np.asarray(raw[pre + ".expect_chain"], np.int64), float(prm[10]),
                                 {} if meta is None else dict(zip(("nodes1", "nodes2", "chains1", "chains2", "match_sets", "pairs"),
                                                                  np.asarray(meta).tolist())))
    return out
