"""Python front for the C ABI (include/centrolign_b200.h) -- harness plumbing only.

``po_poa_batch`` is the batched counterpart of the reference's ``po_poa``
(include/centrolign/alignment.hpp:78-85): same inputs (two PO graphs with source / sink sets,
``AlignmentParameters``), same outputs (optimal score, alignment as node-id pairs with a gap
sentinel), for many windows at once.  All compute happens in ``libcentrolign_b200.so``
(hand-written sm_100a kernels); there is no CPU path here -- if the library or a CUDA device
is missing these calls raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Tuple

import numpy as np

from .batch import AlignmentParameters, GraphSide, WindowBatch

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libcentrolign_b200.so")

EXPORTS = ["clb_popoa_batch", "clb_batch_create", "clb_batch_upload", "clb_batch_run", "clb_batch_download",
           "clb_batch_destroy", "clb_batch_get_stats", "clb_int32_peak_tops", "clb_last_error", "clb_device_count",
           "clb_release_cached_memory", "clb_pwfa_batch", "clb_chain_dp", "clb_topological_ranks", "clb_popoa_batch_multi",
           "clb_balanced_partition", "clb_chain_dp_batch", "clb_chain_job_create", "clb_chain_jobs_run", "clb_chain_job_destroy", "clb_warm_up",
           "clb_pwfa_batch_multi", "clb_chain_dp_batch_multi"]
ERROR_NAMES = {0: "CLB_OK", 1: "CLB_EINVAL", 2: "CLB_ECYCLE", 3: "CLB_ECUDA", 4: "CLB_ENOMEM", 5: "CLB_ESTATE"}


class ClbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {msg}")
        self.code = code


class _Params(ctypes.Structure):
    _fields_ = [("num_pw", ctypes.c_int32), ("match", ctypes.c_uint32), ("mismatch", ctypes.c_uint32),
                ("gap_open", ctypes.c_uint32 * 3), ("gap_extend", ctypes.c_uint32 * 3)]


class _GraphBatch(ctypes.Structure):
    _fields_ = [("node_off", ctypes.c_void_p), ("label", ctypes.c_void_p), ("edge_off", ctypes.c_void_p),
                ("pred_off", ctypes.c_void_p), ("pred", ctypes.c_void_p), ("src_off", ctypes.c_void_p),
                ("src", ctypes.c_void_p), ("snk_off", ctypes.c_void_p), ("snk", ctypes.c_void_p)]


class BatchStats(ctypes.Structure):
    _fields_ = [("cells", ctypes.c_double), ("kernel_ms", ctypes.c_double), ("fill_ms", ctypes.c_double),
                ("kernel_launches", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64),
                ("workspace_bytes", ctypes.c_int64), ("int_ops", ctypes.c_int64), ("persist_bytes", ctypes.c_int64)]


class PwfaStats(ctypes.Structure):
    _fields_ = [("kernel_ms", ctypes.c_double), ("kernel_launches", ctypes.c_int64), ("retries", ctypes.c_int64),
                ("states", ctypes.c_int64), ("dequeued", ctypes.c_int64), ("steps", ctypes.c_int64),
                ("h2d_bytes", ctypes.c_int64), ("d2h_bytes", ctypes.c_int64), ("workspace_bytes", ctypes.c_int64)]


_lib = None


def load_library() -> ctypes.CDLL:
    """Load ``libcentrolign_b200.so`` (built in-tree by ``__graft_entry__.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("CLB_LIBRARY", _LIB_PATH)  # A/B runs of kernel variants load another build of the same library
    if not os.path.exists(path):
        raise ClbError(3, f"{_LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
                          "there is no CPU fallback for the gap-fill path")
    lib = ctypes.CDLL(path)
    vp, i32 = ctypes.c_void_p, ctypes.c_int32
    gp, pp = ctypes.POINTER(_GraphBatch), ctypes.POINTER(_Params)
    lib.clb_popoa_batch.restype = ctypes.c_int
    lib.clb_popoa_batch.argtypes = [ctypes.c_int, i32, gp, gp, pp, vp, vp, vp, vp]
    lib.clb_batch_create.restype = ctypes.c_int
    lib.clb_batch_create.argtypes = [ctypes.c_int, i32, gp, gp, pp, ctypes.POINTER(vp)]
    for name in ("clb_batch_upload", "clb_batch_run"):
        getattr(lib, name).restype = ctypes.c_int
        getattr(lib, name).argtypes = [vp]
    lib.clb_batch_download.restype = ctypes.c_int
    lib.clb_batch_download.argtypes = [vp, vp, vp, vp, vp]
    lib.clb_batch_destroy.restype = None
    lib.clb_batch_destroy.argtypes = [vp]
    lib.clb_batch_get_stats.restype = ctypes.c_int
    lib.clb_batch_get_stats.argtypes = [vp, ctypes.POINTER(BatchStats)]
    lib.clb_popoa_batch_multi.restype = ctypes.c_int
    lib.clb_popoa_batch_multi.argtypes = [ctypes.c_int, vp, i32, gp, gp, pp, vp, vp, vp, vp, vp]
    lib.clb_balanced_partition.restype = ctypes.c_int
    lib.clb_balanced_partition.argtypes = [i32, vp, ctypes.c_int, vp]
    lib.clb_topological_ranks.restype = ctypes.c_int
    lib.clb_topological_ranks.argtypes = [ctypes.c_uint32, vp, vp, vp]
    lib.clb_int32_peak_tops.restype = ctypes.c_double
    lib.clb_int32_peak_tops.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.clb_last_error.restype = ctypes.c_char_p
    lib.clb_device_count.restype = ctypes.c_int
    lib.clb_release_cached_memory.restype = None
    lib.clb_pwfa_batch.restype = ctypes.c_int
    lib.clb_pwfa_batch.argtypes = [ctypes.c_int, i32, gp, gp, pp, ctypes.c_int64, vp, vp, vp, vp, ctypes.POINTER(PwfaStats)]
    lib.clb_pwfa_batch_multi.restype = ctypes.c_int
    lib.clb_pwfa_batch_multi.argtypes = [ctypes.c_int, vp, i32, gp, gp, pp, ctypes.c_int64, vp, vp, vp, vp, vp,
                                         ctypes.POINTER(PwfaStats)]
    _lib = lib
    return lib


def _check(rc: int):
    if rc != 0:
        raise ClbError(rc, load_library().clb_last_error().decode())


def _c_params(p: AlignmentParameters) -> _Params:
    if not 1 <= p.num_pw <= 3 or len(p.gap_extend) != p.num_pw:
        raise ClbError(1, "NumPW must be 1..3 with matching open/extend lists")
    cp = _Params()
    cp.num_pw, cp.match, cp.mismatch = p.num_pw, p.match, p.mismatch
    for k in range(p.num_pw):
        cp.gap_open[k], cp.gap_extend[k] = p.gap_open[k], p.gap_extend[k]
    return cp


def _c_side(side: GraphSide):
    arrs = [np.ascontiguousarray(side.node_off, np.int64), np.ascontiguousarray(side.label, np.uint8),
            np.ascontiguousarray(side.edge_off, np.int64), np.ascontiguousarray(side.pred_off, np.uint32),
            np.ascontiguousarray(side.pred, np.uint32), np.ascontiguousarray(side.src_off, np.int64),
            np.ascontiguousarray(side.src, np.uint32), np.ascontiguousarray(side.snk_off, np.int64),
            np.ascontiguousarray(side.snk, np.uint32)]
    gb = _GraphBatch(*[a.ctypes.data for a in arrs])
    return gb, arrs  # keep arrs alive


class DeviceBatch:
    """Staged form of the call (create -> upload -> run -> download); bench.py keeps one of
    these resident in HBM and times ``run`` alone."""

    def __init__(self, batch: WindowBatch, params: AlignmentParameters, device: int = 0):
        self.lib = load_library()
        self.batch = batch
        self.params = params
        self.handle = ctypes.c_void_p()
        self._p = _c_params(params)
        self._g1, self._k1 = _c_side(batch.g1)
        self._g2, self._k2 = _c_side(batch.g2)
        _check(self.lib.clb_batch_create(device, batch.n_windows, ctypes.byref(self._g1), ctypes.byref(self._g2),
                                         ctypes.byref(self._p), ctypes.byref(self.handle)))
        cap = batch.aln_capacity()
        self.aln_off = np.zeros(batch.n_windows + 1, np.int64)
        np.cumsum(cap, out=self.aln_off[1:])
        self.score = np.zeros(batch.n_windows, np.int64)
        self.aln_len = np.zeros(batch.n_windows, np.uint32)
        self.aln_pairs = np.empty((max(1, int(self.aln_off[-1])), 2), np.int32)

    def upload(self):
        _check(self.lib.clb_batch_upload(self.handle))

    def run(self):
        _check(self.lib.clb_batch_run(self.handle))

    def download(self):
        _check(self.lib.clb_batch_download(self.handle, self.score.ctypes.data, self.aln_off.ctypes.data,
                                           self.aln_pairs.ctypes.data, self.aln_len.ctypes.data))
        return self.score, self.alignments()

    def alignments(self) -> List[np.ndarray]:
        return [self.aln_pairs[int(self.aln_off[w]): int(self.aln_off[w]) + int(self.aln_len[w])]
                for w in range(self.batch.n_windows)]

    def stats(self) -> BatchStats:
        st = BatchStats()
        _check(self.lib.clb_batch_get_stats(self.handle, ctypes.byref(st)))
        return st

    def close(self):
        if getattr(self, "handle", None):
            self.lib.clb_batch_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def po_poa_batch(batch: WindowBatch, params: AlignmentParameters, device: int = 0,
                 out: Optional[Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]] = None):
    """One-shot ``clb_popoa_batch``: host arrays in, (scores, [alignment per window]) out."""
    lib = load_library()
    p = _c_params(params)
    g1, k1 = _c_side(batch.g1)
    g2, k2 = _c_side(batch.g2)
    nw = batch.n_windows
    if out is None:
        aln_off = np.zeros(nw + 1, np.int64)
        np.cumsum(batch.aln_capacity(), out=aln_off[1:])
        score = np.zeros(nw, np.int64)
        aln_len = np.zeros(nw, np.uint32)
        pairs = np.empty((max(1, int(aln_off[-1])), 2), np.int32)
    else:
        score, aln_off, pairs, aln_len = out
    _check(lib.clb_popoa_batch(device, nw, ctypes.byref(g1), ctypes.byref(g2), ctypes.byref(p), score.ctypes.data,
                               aln_off.ctypes.data, pairs.ctypes.data, aln_len.ctypes.data))
    del k1, k2
    return score, [pairs[int(aln_off[w]): int(aln_off[w]) + int(aln_len[w])] for w in range(nw)]


def po_poa_batch_multi(batch: WindowBatch, params: AlignmentParameters, devices, return_parts: bool = False):
    """``clb_popoa_batch_multi``: the windows dealt to several GPUs of one box in cell-balanced bins (one host thread
    per device inside the library), results in window order.  ``devices`` is a list of device ordinals."""
    lib = load_library()
    p = _c_params(params)
    g1, k1 = _c_side(batch.g1)
    g2, k2 = _c_side(batch.g2)
    nw = batch.n_windows
    aln_off = np.zeros(nw + 1, np.int64)
    np.cumsum(batch.aln_capacity(), out=aln_off[1:])
    score = np.zeros(nw, np.int64)
    aln_len = np.zeros(nw, np.uint32)
    pairs = np.empty((max(1, int(aln_off[-1])), 2), np.int32)
    devs = np.ascontiguousarray(list(devices), np.int32)
    parts = np.zeros(max(1, nw), np.int32)
    _check(lib.clb_popoa_batch_multi(len(devs), devs.ctypes.data, nw, ctypes.byref(g1), ctypes.byref(g2), ctypes.byref(p),
                                     score.ctypes.data, aln_off.ctypes.data, pairs.ctypes.data, aln_len.ctypes.data, parts.ctypes.data))
    del k1, k2
    alns = [pairs[int(aln_off[w]): int(aln_off[w]) + int(aln_len[w])] for w in range(nw)]
    return (score, alns, parts[:nw]) if return_parts else (score, alns)


def balanced_partition_c(cells, n_parts: int) -> np.ndarray:
    """``clb_balanced_partition`` (host only): part index per window, longest-processing-time-first by cell count."""
    lib = load_library()
    c = np.ascontiguousarray(cells, np.int64)
    out = np.zeros(max(1, len(c)), np.int32)
    _check(lib.clb_balanced_partition(len(c), c.ctypes.data, n_parts, out.ctypes.data))
    return out[: len(c)]


def po_poa(graph1, graph2, params: AlignmentParameters, device: int = 0):
    """Single-window convenience with the reference's argument order:
    ``graph = (labels, predecessor lists, sources, sinks)``; returns (alignment, score)."""
    from .batch import batch_from_graph_pairs

    score, alns = po_poa_batch(batch_from_graph_pairs([(graph1, graph2)]), params, device)
    return alns[0], int(score[0])


def pwfa_po_poa_batch(succ_batch: WindowBatch, params: AlignmentParameters, prune_limit: int, device: int = 0,
                      stats: Optional[PwfaStats] = None):
    """Batched ``pwfa_po_poa`` (include/centrolign/alignment.hpp:117-125, body :2299-2338) through
    ``clb_pwfa_batch``.  ``succ_batch`` holds SUCCESSOR lists in ``next()`` order (``batch.successor_form``).
    Returns (scores, [alignment per window])."""
    lib = load_library()
    p = _c_params(params)
    g1, k1 = _c_side(succ_batch.g1)
    g2, k2 = _c_side(succ_batch.g2)
    nw = succ_batch.n_windows
    aln_off = np.zeros(nw + 1, np.int64)
    np.cumsum(succ_batch.aln_capacity(), out=aln_off[1:])
    score = np.zeros(nw, np.int64)
    aln_len = np.zeros(nw, np.uint32)
    pairs = np.empty((max(1, int(aln_off[-1])), 2), np.int32)
    _check(lib.clb_pwfa_batch(device, nw, ctypes.byref(g1), ctypes.byref(g2), ctypes.byref(p), int(prune_limit),
                              score.ctypes.data, aln_off.ctypes.data, pairs.ctypes.data, aln_len.ctypes.data,
                              ctypes.byref(stats) if stats is not None else None))
    del k1, k2
    return score, [pairs[int(aln_off[w]): int(aln_off[w]) + int(aln_len[w])] for w in range(nw)]


def pwfa_po_poa_batch_multi(succ_batch: WindowBatch, params: AlignmentParameters, prune_limit: int, devices,
                            return_parts: bool = False, stats: Optional[PwfaStats] = None):
    """``clb_pwfa_batch_multi``: the windows of ``pwfa_po_poa_batch`` dealt to several GPUs of one box by
    (n1+1)+(n2+1) (one host thread per device inside the library), results in window order.  ``devices`` is a list of
    distinct device ordinals.  Returns (scores, [alignment per window]), plus the index into ``devices`` each window ran
    on if ``return_parts``.  ``stats``: the longest kernel time over the devices, the counters summed."""
    lib = load_library()
    p = _c_params(params)
    g1, k1 = _c_side(succ_batch.g1)
    g2, k2 = _c_side(succ_batch.g2)
    nw = succ_batch.n_windows
    aln_off = np.zeros(nw + 1, np.int64)
    np.cumsum(succ_batch.aln_capacity(), out=aln_off[1:])
    score = np.zeros(nw, np.int64)
    aln_len = np.zeros(nw, np.uint32)
    pairs = np.empty((max(1, int(aln_off[-1])), 2), np.int32)
    devs = np.ascontiguousarray(list(devices), np.int32)
    parts = np.zeros(max(1, nw), np.int32)
    _check(lib.clb_pwfa_batch_multi(len(devs), devs.ctypes.data, nw, ctypes.byref(g1), ctypes.byref(g2), ctypes.byref(p),
                                    int(prune_limit), score.ctypes.data, aln_off.ctypes.data, pairs.ctypes.data,
                                    aln_len.ctypes.data, parts.ctypes.data, ctypes.byref(stats) if stats is not None else None))
    del k1, k2
    alns = [pairs[int(aln_off[w]): int(aln_off[w]) + int(aln_len[w])] for w in range(nw)]
    return (score, alns, parts[:nw]) if return_parts else (score, alns)


def topological_ranks(pred_lists) -> "np.ndarray":
    """Matrix index (1-based topological rank) the library's flattening code gives every node of a graph whose
    predecessor lists are ``pred_lists`` (host only, no device needed; ``clb_topological_ranks``)."""
    lib = load_library()
    n = len(pred_lists)
    off = np.zeros(n + 1, dtype=np.uint32)
    off[1:] = np.cumsum([len(p) for p in pred_lists])
    pred = np.asarray([q for p in pred_lists for q in p], dtype=np.uint32)
    if pred.size == 0:
        pred = np.zeros(1, dtype=np.uint32)
    out = np.zeros(max(n, 1), dtype=np.uint32)
    rc = lib.clb_topological_ranks(n, off.ctypes.data, pred.ctypes.data, out.ctypes.data)
    if rc != 0:
        lib.clb_last_error.restype = ctypes.c_char_p
        raise ClbError(rc, (lib.clb_last_error() or b"").decode())
    return out[:n]
