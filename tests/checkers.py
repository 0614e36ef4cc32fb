"""CPU checkers -- TEST INFRASTRUCTURE, not part of the product package.

ctypes fronts of ``oracle/libcloracle.so`` (the C restatements under oracle/) and, when it was built, of
``oracle/_ref/libclref.so`` (the unmodified reference).  Only tests/, ``__graft_entry__.smoke()`` and bench.py's CPU
legs import this module; nothing under centrolign_b200/ does, and the product path has no CPU fallback."""
import ctypes
import os

import numpy as np

from centrolign_b200.batch import AlignmentParameters, GraphSide, WindowBatch
from centrolign_b200.chain import _FIELDS, ChainProblem

_ORACLE_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle")

_u32p = ctypes.POINTER(ctypes.c_uint32)
_u8p = ctypes.POINTER(ctypes.c_uint8)
_SIDE_ARGS = [ctypes.c_uint32, _u8p, _u32p, _u32p, ctypes.c_uint32, _u32p, ctypes.c_uint32, _u32p]


def _bind_checker(lib, name, extra=(), tail=()):
    fn = getattr(lib, name)
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_int, _u32p, *extra, *_SIDE_ARGS, *_SIDE_ARGS, ctypes.POINTER(ctypes.c_int64),
                   ctypes.POINTER(ctypes.c_int32), _u32p, *tail]
    return fn


class CpuChecker:
    """ctypes front for ``oracle/libcloracle.so`` (kind='port') or
    ``oracle/_ref/libclref.so`` (kind='reference', the unmodified reference)."""

    def __init__(self, kind: str = "port"):
        self.kind = kind
        if kind == "port":
            path, sym = os.path.join(_ORACLE_DIR, "libcloracle.so"), "clo_po_poa"
        elif kind == "reference":
            path, sym = os.path.join(_ORACLE_DIR, "_ref", "libclref.so"), "clref_po_poa"
        else:
            raise ValueError(kind)
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.lib = ctypes.CDLL(path)
        self._po_poa = _bind_checker(self.lib, sym)
        self._pwfa = _bind_checker(self.lib, "clref_pwfa_po_poa", (ctypes.c_int64,)) if kind == "reference" else None
        self._pwfa_succ = _bind_checker(self.lib, "clo_pwfa_po_poa" if kind == "port" else "clref_pwfa_po_poa_succ",
                                        (ctypes.c_int64,), (ctypes.POINTER(ctypes.c_int64),))

    @staticmethod
    def available(kind: str) -> bool:
        p = os.path.join(_ORACLE_DIR, "libcloracle.so") if kind == "port" else os.path.join(_ORACLE_DIR, "_ref", "libclref.so")
        return os.path.exists(p)

    @staticmethod
    def _side(side: GraphSide, w: int):
        lab, po, pr, src, snk = (np.ascontiguousarray(a) for a in side.window(w))
        keep = (lab, po, pr, src, snk)

        def p32(a):
            return a.ctypes.data_as(_u32p)

        return keep, [len(lab), lab.ctypes.data_as(_u8p), p32(po), p32(pr), len(src), p32(src), len(snk), p32(snk)]

    def po_poa(self, batch: WindowBatch, w: int, params: AlignmentParameters, prune_limit=None):
        """Returns (score, alignment[int32 (len,2)], -1 = gap) for window ``w``."""
        k1, a1 = self._side(batch.g1, w)
        k2, a2 = self._side(batch.g2, w)
        pk = params.packed()
        score = ctypes.c_int64(0)
        cap = max(1, batch.g1.n(w) + batch.g2.n(w))
        aln = np.empty((cap, 2), np.int32)
        ln = ctypes.c_uint32(0)
        extra = [] if prune_limit is None else [ctypes.c_int64(prune_limit)]
        fn = self._po_poa if prune_limit is None else self._pwfa
        rc = fn(params.num_pw, pk.ctypes.data_as(_u32p), *extra, *a1, *a2, ctypes.byref(score),
                aln.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ctypes.byref(ln))
        if rc != 0:
            raise RuntimeError(f"{self.kind} checker failed with code {rc}")
        return int(score.value), aln[: ln.value].copy()

    def pwfa_po_poa(self, succ_batch: WindowBatch, w: int, params: AlignmentParameters, prune_limit: int, stats=None):
        """``pwfa_po_poa`` (alignment.hpp:2299-2338) on window ``w`` of a batch in ``successor_form``.
        Returns (score, alignment); ``stats`` (int64[3], port only) receives settled states, dequeued
        entries and the final WFA score."""
        k1, a1 = self._side(succ_batch.g1, w)
        k2, a2 = self._side(succ_batch.g2, w)
        pk = params.packed()
        score = ctypes.c_int64(0)
        cap = max(1, succ_batch.g1.n(w) + succ_batch.g2.n(w))
        aln = np.empty((cap, 2), np.int32)
        ln = ctypes.c_uint32(0)
        st = stats if stats is not None else np.zeros(3, np.int64)
        rc = self._pwfa_succ(params.num_pw, pk.ctypes.data_as(_u32p), ctypes.c_int64(prune_limit), *a1, *a2,
                             ctypes.byref(score), aln.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ctypes.byref(ln),
                             st.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)))
        if rc != 0:
            raise RuntimeError(f"{self.kind} pwfa checker failed with code {rc}")
        return int(score.value), aln[: ln.value].copy()

    def run(self, batch: WindowBatch, params: AlignmentParameters, prune_limit=None):
        """(scores, alignments) of every window: po_poa, or pwfa_po_poa on a batch in successor form when
        ``prune_limit`` is given."""
        res = [self.po_poa(batch, w, params) if prune_limit is None else self.pwfa_po_poa(batch, w, params, prune_limit)
               for w in range(batch.n_windows)]
        return [r[0] for r in res], [r[1] for r in res]


def chain_oracle(problem: ChainProblem):
    """The C restatement of the reference's chaining DP (oracle/libcloracle.so :: clo_chain_dp) on the same flat
    problem.  Returns (chain ranks, dp values, back-pointers, optimum)."""
    path = os.path.join(_ORACLE_DIR, "libcloracle.so")
    lib = ctypes.CDLL(path)
    vp = ctypes.c_void_p
    lib.clo_chain_dp.restype = ctypes.c_int
    lib.clo_chain_dp.argtypes = ([ctypes.c_int, vp, vp, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int64, vp, vp, vp,
                                  ctypes.c_float, ctypes.c_int64] + [vp] * 14 + [vp, vp, vp, ctypes.POINTER(ctypes.c_int64),
                                                                              ctypes.POINTER(ctypes.c_float)])
    keep = {k: np.ascontiguousarray(problem.arrays[k], dt) for k, dt in _FIELDS}
    go = np.asarray(list(problem.gap_open) + [0.0] * 3, np.float64)[:3].copy()
    ge = np.asarray(list(problem.gap_extend) + [0.0] * 3, np.float64)[:3].copy()
    m = problem.n_match
    dp = np.zeros(max(1, m), np.float32)
    bp = np.full(max(1, m), -1, np.int64)
    chain = np.zeros(m + 1, np.int64)
    n = ctypes.c_int64(0)
    opt = ctypes.c_float(0)
    order = ["end_off", "end_match", "qry_off", "qry_match", "qry_chain1", "ins_off", "ins_p1", "ins_p2", "ins_shift", "ins_offset",
             "ins_active", "qa1", "qa2", "qoff"]
    rc = lib.clo_chain_dp(problem.num_pw, go.ctypes.data, ge.ctypes.data, problem.scale, problem.n_chain1, problem.n_chain2, m,
                          keep["weight"].ctypes.data, keep["dp_init"].ctypes.data, keep["final_term"].ctypes.data,
                          problem.min_score, problem.n_step, *[keep[k].ctypes.data for k in order], dp.ctypes.data, bp.ctypes.data,
                          chain.ctypes.data, ctypes.byref(n), ctypes.byref(opt))
    if rc != 0:
        raise RuntimeError(f"chain oracle failed with code {rc}")
    return chain[: n.value].copy(), dp[:m], bp[:m], float(opt.value)
