"""ctypes binding of ``libxtrack_b200.so`` (C ABI declared in ``include/xtrack.h``).

There is no CPU fallback: importing this module raises if the shared library has not been
built (``python -c 'import __graft_entry__ as g; g.build()'`` or ``python -m extrack_b200.build``),
and creating an :class:`Engine` raises if no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np

XT_MAX_HEADS = 128
XT_MAX_STATES = 8
XT_MAX_DIMS = 3
XT_FLAG_INT8_WRAP = 1
XT_FLAG_VAR_LOC = 2
XT_FLAG_VAR_DT = 4
XT_FLAG_LOC_AFFINE = 8

XT_ERR_CUDA, XT_ERR_ARG, XT_ERR_GROUPING, XT_ERR_CAPACITY, XT_ERR_STATE, XT_ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6

LIB_NAME = "libxtrack_b200.so"
# XT_LIB_PATH: another build of the same engine (A/B timing of kernel variants); never a fallback
LIB_PATH = os.environ.get("XT_LIB_PATH") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)


class XtParams(C.Structure):
    _fields_ = [
        ("nS", C.c_int32),
        ("nsub", C.c_int32),
        ("d", C.c_int32),
        ("n_loc", C.c_int32),
        ("frame_len", C.c_int32),
        ("min_len", C.c_int32),
        ("max_nb_states", C.c_int32),
        ("flags", C.c_uint32),
        ("threshold", C.c_double),
        ("l2", C.c_double * XT_MAX_DIMS),
        ("dd", C.c_double * XT_MAX_HEADS),
        ("LT", C.c_double * XT_MAX_HEADS),
        ("LF", C.c_double * XT_MAX_HEADS),
        ("Lp_stay", C.c_double * XT_MAX_HEADS),
        ("L_leave", C.c_double * XT_MAX_HEADS),
        ("twoD", C.c_double * XT_MAX_STATES),
        ("loc_slope", C.c_double),
        ("loc_offset", C.c_double),
    ]


class XtStats(C.Structure):
    _fields_ = [
        ("n_tracks", C.c_int64),
        ("track_steps", C.c_int64),
        ("seq_updates", C.c_int64),
        ("seq_groups", C.c_int64),
        ("max_nB_in", C.c_int32),
        ("n_chunks", C.c_int32),
        ("k1_launches", C.c_int32),
        ("k2_launches", C.c_int32),
        ("ms_plan", C.c_float),
        ("ms_replay", C.c_float),
        ("pipelined", C.c_int32),
        ("ms_predict", C.c_float),
        ("k3_launches", C.c_int32),
        ("k3_cap", C.c_int32),
        ("fp32", C.c_int32),
        ("plan_verified", C.c_int32),
        ("replanned", C.c_int32),
    ]


# every symbol include/xtrack.h declares (tests check the library exports all of them)
EXPORTS = (
    "xt_device_count",
    "xt_create",
    "xt_destroy",
    "xt_last_error",
    "xt_upload",
    "xt_upload_aux",
    "xt_set_stay_tables",
    "xt_sum_logp",
    "xt_sum_logp_host",
    "xt_sum_logp_async",
    "xt_chunk_logp",
    "xt_eval_frozen",
    "xt_score_outer",
    "xt_plan_dump",
    "xt_predict",
    "xt_predict_pairs",
    "xt_predict_residuals",
    "xt_predict_path",
    "xt_predict_samples",
    "xt_refine_positions",
    "xt_get_stats",
    "xt_seglen_hist",
    "xt_seglen_last_ms",
    "xt_set_option",
    "xt_fp64_peak_tflops",
    "xt_host_alloc",
    "xt_host_free",
    "xt_multi_create",
    "xt_multi_destroy",
    "xt_multi_last_error",
    "xt_multi_n_devices",
    "xt_multi_upload",
    "xt_multi_upload_aux",
    "xt_multi_set_stay_tables",
    "xt_multi_sum_logp",
    "xt_multi_chunk_logp",
    "xt_multi_eval_frozen",
    "xt_multi_score_outer",
    "xt_multi_set_option",
    "xt_multi_device_load",
    "xt_multi_get_stats",
)

_lib = None


def load_library() -> C.CDLL:
    """Load the CUDA engine; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_NAME} not found at {LIB_PATH}: the CUDA engine is not built. "
            "Run `python -m extrack_b200.build` (needs nvcc). There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    P = C.POINTER
    lib.xt_device_count.argtypes = []
    lib.xt_create.argtypes = [C.c_int, P(vp)]
    lib.xt_destroy.argtypes = [vp]
    lib.xt_destroy.restype = None
    lib.xt_last_error.argtypes = [vp]
    lib.xt_last_error.restype = C.c_char_p
    lib.xt_upload.argtypes = [vp, i32, P(i32), P(i64), P(i32), P(vp), i32, i32]
    lib.xt_upload_aux.argtypes = [vp, i32, P(vp), P(vp)]
    lib.xt_set_stay_tables.argtypes = [vp, i32, i32, i32, P(dbl), P(dbl)]
    lib.xt_sum_logp.argtypes = [vp, P(XtParams), P(dbl)]
    lib.xt_sum_logp_host.argtypes = [vp, i32, P(i32), P(i64), P(i32), P(vp), i32, i32, P(XtParams), P(dbl)]
    lib.xt_sum_logp_async.argtypes = [vp, P(XtParams), vp, vp]
    lib.xt_chunk_logp.argtypes = [vp, i32, P(XtParams), P(dbl)]
    lib.xt_eval_frozen.argtypes = [vp, i32, P(XtParams), P(dbl), P(vp)]
    lib.xt_score_outer.argtypes = [vp, i32, P(XtParams), P(XtParams), P(dbl), P(dbl), P(dbl), P(dbl), P(dbl)]
    lib.xt_multi_eval_frozen.argtypes = [vp, i32, P(XtParams), P(dbl)]
    lib.xt_multi_score_outer.argtypes = [vp, i32, P(XtParams), P(XtParams), P(dbl), P(dbl), P(dbl), P(dbl), P(dbl)]
    lib.xt_plan_dump.argtypes = [vp, i32, i32, P(i32), P(i32), P(i32), i32, P(dbl)]
    lib.xt_predict.argtypes = [vp, P(XtParams), P(vp)]
    lib.xt_predict_pairs.argtypes = [vp, P(XtParams), P(vp), P(vp)]
    lib.xt_predict_residuals.argtypes = [vp, P(XtParams), P(vp), P(vp), P(vp)]
    lib.xt_predict_path.argtypes = [vp, P(XtParams), P(vp), P(vp), P(vp)]
    lib.xt_predict_samples.argtypes = [vp, P(XtParams), i32, C.c_uint64, P(i64), P(vp), P(vp), P(vp)]
    lib.xt_refine_positions.argtypes = [vp, P(XtParams), P(XtParams), P(vp), P(vp)]
    lib.xt_get_stats.argtypes = [vp, P(XtStats)]
    lib.xt_seglen_hist.argtypes = [vp, P(XtParams), P(dbl), P(dbl), i32, i32, vp, vp, P(i32)]
    lib.xt_seglen_last_ms.argtypes = [vp, P(C.c_float)]
    lib.xt_set_option.argtypes = [vp, C.c_char_p, C.c_int]
    lib.xt_fp64_peak_tflops.argtypes = [vp, P(dbl)]
    lib.xt_host_alloc.argtypes = [P(vp), C.c_uint64]
    lib.xt_host_free.argtypes = [vp]
    lib.xt_multi_create.argtypes = [P(i32), i32, P(vp)]
    lib.xt_multi_destroy.argtypes = [vp]
    lib.xt_multi_destroy.restype = None
    lib.xt_multi_last_error.argtypes = [vp]
    lib.xt_multi_last_error.restype = C.c_char_p
    lib.xt_multi_n_devices.argtypes = [vp]
    lib.xt_multi_upload.argtypes = [vp, i32, P(i32), P(i64), P(i32), P(vp), i32, i32]
    lib.xt_multi_upload_aux.argtypes = [vp, i32, P(i32), P(i64), i32, P(vp), P(vp)]
    lib.xt_multi_set_stay_tables.argtypes = [vp, i32, i32, P(dbl), P(dbl)]
    lib.xt_multi_sum_logp.argtypes = [vp, P(XtParams), P(dbl)]
    lib.xt_multi_chunk_logp.argtypes = [vp, i32, P(XtParams), P(dbl)]
    lib.xt_multi_set_option.argtypes = [vp, C.c_char_p, C.c_int]
    lib.xt_multi_device_load.argtypes = [vp, i32, P(i32), P(i32), P(i64)]
    lib.xt_multi_get_stats.argtypes = [vp, P(XtStats)]
    for name in EXPORTS:
        if name not in ("xt_destroy", "xt_last_error", "xt_multi_destroy", "xt_multi_last_error"):
            getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"xtrack error {code}: {msg}")
        self.code = code
        self.msg = msg


def _raise(code: int, msg: str):
    # error conventions of the reference (SURVEY.md §8b): malformed input / grouping -> ValueError
    if code in (XT_ERR_ARG, XT_ERR_GROUPING, XT_ERR_CAPACITY):
        raise ValueError(msg)
    if code == XT_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise EngineError(code, msg)


XT_MAX_SCORE_DIRS = 32


def _param_array(ps: Sequence[XtParams]):
    arr = (XtParams * len(ps))()
    for k, p in enumerate(ps):
        arr[k] = p
    return arr


def _score_outer(fn, h, p_plus: Sequence[XtParams], p_minus: Sequence[XtParams], inv_2h) -> dict:
    """Shared body of Engine.score_outer / MultiEngine.score_outer (``fn`` = the C entry point)."""
    n = len(p_plus)
    if len(p_minus) != n or len(inv_2h) != n:
        raise ValueError("score_outer: p_plus, p_minus and inv_2h need the same length")
    dp = C.POINTER(C.c_double)
    inv = np.ascontiguousarray(inv_2h, dtype=np.float64)
    sp, sm, gs = np.empty(n), np.empty(n), np.empty(n)
    gram = np.empty((n, n))
    rc = fn(h, n, _param_array(p_plus), _param_array(p_minus), inv.ctypes.data_as(dp), sp.ctypes.data_as(dp),
            sm.ctypes.data_as(dp), gs.ctypes.data_as(dp), gram.ctypes.data_as(dp))
    return rc, {"sum_plus": sp, "sum_minus": sm, "gsum": gs, "gram": gram}


class Engine:
    """One context = one GPU.  Owns all device memory; freed on ``close()`` / garbage collection."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.xt_create(int(device), C.byref(self._h))
        if rc != 0:
            msg = self._lib.xt_last_error(None).decode()
            self._h = None
            raise EngineError(rc, f"cannot create a CUDA context on device {device}: {msg} (no CPU fallback)")
        self.device = int(device)
        self.segments = []  # (L, n) per uploaded segment

    # -- lifetime ------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.xt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            _raise(rc, self._lib.xt_last_error(self._h).decode())

    # -- data ----------------------------------------------------------------------------
    def upload(self, segments: Sequence[np.ndarray], isBL: Sequence[int], chunk_size: int):
        """segments: float64 arrays [n, L, d] (made C-contiguous here if they are not)."""
        segs = [np.ascontiguousarray(s, dtype=np.float64) for s in segments]
        if len(segs) == 0:
            raise ValueError("No track could be detected. The loaded tracks seem empty.")
        d = segs[0].shape[2]
        for s in segs:
            if s.ndim != 3 or s.shape[2] != d:
                raise ValueError("all track arrays must have shape [n, L, d] with the same d")
        n = len(segs)
        Ls = (C.c_int32 * n)(*[s.shape[1] for s in segs])
        ns = (C.c_int64 * n)(*[s.shape[0] for s in segs])
        bl = (C.c_int32 * n)(*[int(b) for b in isBL])
        ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in segs])
        self._check(self._lib.xt_upload(self._h, n, Ls, ns, bl, ptrs, d, int(chunk_size)))
        self.segments = [(s.shape[1], s.shape[0]) for s in segs]
        self.chunk_size = int(chunk_size)
        self.d = d

    def upload_aux(self, sigma: Optional[Sequence[np.ndarray]] = None, dt: Optional[Sequence[np.ndarray]] = None):
        """Per-localisation inputs of the uploaded segments: ``sigma[s]`` float64 [n, L, k] peak-wise
        localisation errors (k = 1 or d), ``dt[s]`` float64 [n, L] time steps."""
        n = len(self.segments)
        k = 0
        sp = dp = None
        keep = []
        if sigma is not None:
            sg = [np.ascontiguousarray(a, dtype=np.float64) for a in sigma]
            k = sg[0].shape[2] if sg[0].ndim == 3 else -1
            for a, (L, cnt) in zip(sg, self.segments):
                if a.ndim != 3 or a.shape != (cnt, L, k):
                    raise ValueError("Localization error is not specified correctly: input_LocErr arrays must have shape "
                                     "[n, L, 1] or [n, L, d] matching all_tracks")
            if len(sg) != n:
                raise ValueError("input_LocErr must hold one array per track-length bucket")
            sp = (C.c_void_p * n)(*[a.ctypes.data for a in sg])
            keep.append(sg)
        if dt is not None:
            ds_ = [np.ascontiguousarray(a, dtype=np.float64) for a in dt]
            if len(ds_) != n:
                raise ValueError("dt must hold one array per track-length bucket")
            for a, (L, cnt) in zip(ds_, self.segments):
                if a.shape != (cnt, L):
                    raise ValueError("dt is not informed properly. It must either be a float number or a dictionary of same "
                                     "structure than `all_tracks` with each element being an array of dims (nb_tracks, track_len)")
            dp = (C.c_void_p * n)(*[a.ctypes.data for a in ds_])
            keep.append(ds_)
        self._check(self._lib.xt_upload_aux(self._h, int(k), sp, dp))

    def set_stay_tables(self, per_track: bool, Lp_stay: Optional[np.ndarray], L_leave: Optional[np.ndarray]):
        """Per-chunk (objective) or per-track (predict) field-of-view tables, float64 [rows, K] / [rows, H]."""
        if Lp_stay is None:
            self._check(self._lib.xt_set_stay_tables(self._h, int(per_track), 0, 0, None, None))
            return
        a = np.ascontiguousarray(Lp_stay, dtype=np.float64)
        b = np.ascontiguousarray(L_leave, dtype=np.float64)
        pd = C.POINTER(C.c_double)
        self._check(self._lib.xt_set_stay_tables(self._h, int(per_track), a.shape[1], b.shape[1], a.ctypes.data_as(pd),
                                                 b.ctypes.data_as(pd)))

    # -- evaluation ----------------------------------------------------------------------
    def sum_logp_host(self, segments: Sequence[np.ndarray], isBL: Sequence[int], chunk_size: int, p: XtParams) -> float:
        """Objective on host arrays: upload (overlapped with the kernels) + evaluation in one call."""
        segs = [np.ascontiguousarray(s, dtype=np.float64) for s in segments]
        if len(segs) == 0:
            raise ValueError("No track could be detected. The loaded tracks seem empty.")
        d = segs[0].shape[2]
        for s in segs:
            if s.ndim != 3 or s.shape[2] != d:
                raise ValueError("all track arrays must have shape [n, L, d] with the same d")
        n = len(segs)
        Ls = (C.c_int32 * n)(*[s.shape[1] for s in segs])
        ns = (C.c_int64 * n)(*[s.shape[0] for s in segs])
        bl = (C.c_int32 * n)(*[int(b) for b in isBL])
        ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in segs])
        out = C.c_double()
        self._check(self._lib.xt_sum_logp_host(self._h, n, Ls, ns, bl, ptrs, d, int(chunk_size), C.byref(p), C.byref(out)))
        self.segments = [(s.shape[1], s.shape[0]) for s in segs]
        self.chunk_size = int(chunk_size)
        self.d = d
        return out.value

    def sum_logp(self, p: XtParams) -> float:
        out = C.c_double()
        self._check(self._lib.xt_sum_logp(self._h, C.byref(p), C.byref(out)))
        return out.value

    def sum_logp_async(self, p: XtParams, d_out_ptr: int, stream_ptr: Optional[int] = None):
        self._check(self._lib.xt_sum_logp_async(self._h, C.byref(p), C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr or 0)))

    def chunk_logp(self, chunk: int, nT: int, p: XtParams) -> np.ndarray:
        out = np.empty(nT, dtype=np.float64)
        self._check(self._lib.xt_chunk_logp(self._h, int(chunk), C.byref(p), out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def eval_frozen(self, ps: Sequence[XtParams], per_track: bool = False):
        """Sums of log P for every parameter set along the resident plan (``xt_eval_frozen``); with ``per_track`` also
        float64[len(ps), n_tracks] per-track values in upload order.  Returns ``sums`` or ``(sums, per_track)``."""
        sums = np.empty(len(ps))
        n_tracks = sum(n for (_, n) in self.segments)
        lps = np.empty((len(ps), n_tracks)) if per_track else None
        ptrs = (C.c_void_p * len(ps))(*[r.ctypes.data for r in lps]) if per_track else None
        self._check(self._lib.xt_eval_frozen(self._h, len(ps), _param_array(ps), sums.ctypes.data_as(C.POINTER(C.c_double)),
                                             ptrs))
        return (sums, lps) if per_track else sums

    def score_outer(self, p_plus: Sequence[XtParams], p_minus: Sequence[XtParams], inv_2h) -> dict:
        """Central-difference scores along the resident plan (``xt_score_outer``): dict of ``sum_plus``, ``sum_minus``,
        ``gsum`` [n] and ``gram`` [n, n]."""
        rc, out = _score_outer(self._lib.xt_score_outer, self._h, p_plus, p_minus, inv_2h)
        self._check(rc)
        return out

    def plan_dump(self, chunk: int, step: int, cap: int = 4096):
        nB, nG, th = C.c_int32(), C.c_int32(), C.c_double()
        gid = np.empty(cap, dtype=np.int32)
        self._check(
            self._lib.xt_plan_dump(
                self._h, int(chunk), int(step), C.byref(nB), C.byref(nG), gid.ctypes.data_as(C.POINTER(C.c_int32)), cap, C.byref(th)
            )
        )
        return nB.value, nG.value, gid[: nB.value].copy(), th.value

    def predict(self, p: XtParams, nS: int) -> List[np.ndarray]:
        outs = [np.empty((n, L, nS), dtype=np.float64) for (L, n) in self.segments]
        ptrs = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
        self._check(self._lib.xt_predict(self._h, C.byref(p), ptrs))
        return outs

    def predict_pairs(self, p: XtParams, nS: int) -> Tuple[List[np.ndarray], List[np.ndarray]]:
        """``predict`` plus the two-slice posteriors [n, L - 1, nS, nS] per uploaded segment (``xt_predict_pairs``)."""
        outs = [np.empty((n, L, nS), dtype=np.float64) for (L, n) in self.segments]
        pairs = [np.empty((n, L - 1, nS, nS), dtype=np.float64) for (L, n) in self.segments]
        ptrs = (C.c_void_p * len(outs))(*[o.ctypes.data for o in outs])
        pptrs = (C.c_void_p * len(pairs))(*[o.ctypes.data for o in pairs])
        self._check(self._lib.xt_predict_pairs(self._h, C.byref(p), ptrs, pptrs))
        return outs, pairs

    def predict_residuals(self, p: XtParams, nS: int) -> Tuple[List[np.ndarray], List[np.ndarray], List[np.ndarray]]:
        """``predict`` plus the one-step-ahead log predictive densities [n, L] and PIT values [n, L, d] per uploaded
        segment (``xt_predict_residuals``; localisation 0 is NaN)."""
        outs = [np.empty((n, L, nS), dtype=np.float64) for (L, n) in self.segments]
        lps = [np.empty((n, L), dtype=np.float64) for (L, n) in self.segments]
        pits = [np.empty((n, L, self.d), dtype=np.float64) for (L, n) in self.segments]
        arr = lambda xs: (C.c_void_p * len(xs))(*[o.ctypes.data for o in xs])
        self._check(self._lib.xt_predict_residuals(self._h, C.byref(p), arr(outs), arr(lps), arr(pits)))
        return outs, lps, pits

    def predict_path(self, p: XtParams, nS: int) -> Tuple[List[np.ndarray], List[np.ndarray], List[np.ndarray]]:
        """``predict`` plus the MAP state paths int8[n, L] and their log posterior probabilities float64[n] per uploaded
        segment (``xt_predict_path``)."""
        outs = [np.empty((n, L, nS), dtype=np.float64) for (L, n) in self.segments]
        paths = [np.empty((n, L), dtype=np.int8) for (L, n) in self.segments]
        logps = [np.empty(n, dtype=np.float64) for (L, n) in self.segments]
        arr = lambda xs: (C.c_void_p * len(xs))(*[o.ctypes.data for o in xs])
        self._check(self._lib.xt_predict_path(self._h, C.byref(p), arr(outs), arr(paths), arr(logps)))
        return outs, paths, logps

    def predict_samples(self, p: XtParams, nS: int, n_samples: int, seed: int, row0: Optional[Sequence[int]] = None):
        """``predict`` plus ``n_samples`` posterior draws of whole state paths per track: int8[n, n_samples, L] labels
        and float64[n, n_samples] log route weights per uploaded segment (``xt_predict_samples``).  ``row0[s]``: the
        caller's row of segment s's first track, the Philox counter of the draws (None: all 0)."""
        outs = [np.empty((n, L, nS), dtype=np.float64) for (L, n) in self.segments]
        smp = [np.empty((n, int(n_samples), L), dtype=np.int8) for (L, n) in self.segments]
        logps = [np.empty((n, int(n_samples)), dtype=np.float64) for (L, n) in self.segments]
        arr = lambda xs: (C.c_void_p * len(xs))(*[o.ctypes.data for o in xs])
        r0 = None
        if row0 is not None:
            if len(row0) != len(self.segments):
                raise ValueError("row0 needs one entry per uploaded segment")
            r0 = (C.c_int64 * len(row0))(*[int(r) for r in row0])
        self._check(self._lib.xt_predict_samples(self._h, C.byref(p), int(n_samples), C.c_uint64(int(seed)), r0, arr(outs),
                                                 arr(smp), arr(logps)))
        return outs, smp, logps

    def refine_positions(self, p_rev: XtParams, p_fwd: XtParams):
        """Refined positions [n, L, d] and their standard deviations [n, L] per uploaded segment (every segment
        uploaded as one chunk); see ``xt_refine_positions``."""
        mus = [np.empty((n, L, self.d), dtype=np.float64) for (L, n) in self.segments]
        sigmas = [np.empty((n, L), dtype=np.float64) for (L, n) in self.segments]
        pm = (C.c_void_p * len(mus))(*[o.ctypes.data for o in mus])
        ps = (C.c_void_p * len(sigmas))(*[o.ctypes.data for o in sigmas])
        self._check(self._lib.xt_refine_positions(self._h, C.byref(p_rev), C.byref(p_fwd), pm, ps))
        return mus, sigmas

    def seglen_hist(self, p: XtParams, leave_LL: np.ndarray, Lmax: int, nS: int, n_chunks: int, dbg_chunk: int = -1,
                    dbg_shape=None):
        """Per-chunk segment-length histograms [n_chunks, Lmax, nS] (histograms.py:26-258 per chunk); with
        ``dbg_chunk`` >= 0 and ``dbg_shape = (nT, L)`` also that chunk's final LP [nT, nBf] and histories [nT, nBf, L]."""
        hist = np.zeros((n_chunks, Lmax, nS), dtype=np.float64)
        lv = np.ascontiguousarray(leave_LL, dtype=np.float64)
        dp = C.POINTER(C.c_double)
        nf = C.c_int32(0)
        if dbg_chunk < 0:
            self._check(self._lib.xt_seglen_hist(self._h, C.byref(p), lv.ctypes.data_as(dp), hist.ctypes.data_as(dp), int(Lmax),
                                                 -1, None, None, C.byref(nf)))
            return hist
        nT, L = dbg_shape
        # first call sizes the outputs (n_final), second call fills them
        self._check(self._lib.xt_seglen_hist(self._h, C.byref(p), lv.ctypes.data_as(dp), hist.ctypes.data_as(dp), int(Lmax),
                                             int(dbg_chunk), None, None, C.byref(nf)))
        LP = np.empty((nT, nf.value), dtype=np.float64)
        Bs = np.empty((nT, nf.value, L), dtype=np.int8)
        self._check(self._lib.xt_seglen_hist(self._h, C.byref(p), lv.ctypes.data_as(dp), hist.ctypes.data_as(dp), int(Lmax),
                                             int(dbg_chunk), C.c_void_p(LP.ctypes.data), C.c_void_p(Bs.ctypes.data), C.byref(nf)))
        return hist, LP, Bs

    def seglen_last_ms(self) -> float:
        ms = C.c_float()
        self._check(self._lib.xt_seglen_last_ms(self._h, C.byref(ms)))
        return ms.value

    def stats(self) -> dict:
        st = XtStats()
        self._check(self._lib.xt_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in XtStats._fields_}

    def set_option(self, name: str, value: int):
        self._check(self._lib.xt_set_option(self._h, name.encode(), int(value)))

    def fp64_peak_tflops(self) -> float:
        out = C.c_double()
        self._check(self._lib.xt_fp64_peak_tflops(self._h, C.byref(out)))
        return out.value


def device_count() -> int:
    """Visible CUDA devices (0 without a driver / GPU)."""
    return int(load_library().xt_device_count())


class MultiEngine:
    """Several GPUs driven from one Python thread (``xt_multi_*``): the chunk list is dealt to the devices
    longest-processing-time-first, every device keeps its chunks resident, and the objective is the sum of
    the per-chunk sums in global chunk order (same bits for any number of devices)."""

    def __init__(self, devices: Sequence[int]):
        self._lib = load_library()
        self._h = C.c_void_p()
        devs = [int(d) for d in devices]
        arr = (C.c_int32 * len(devs))(*devs)
        rc = self._lib.xt_multi_create(arr, len(devs), C.byref(self._h))
        if rc != 0:
            msg = self._lib.xt_multi_last_error(None).decode()
            self._h = None
            raise EngineError(rc, f"cannot create CUDA contexts on devices {devs}: {msg} (no CPU fallback)")
        self.devices = devs
        self.segments = []

    def close(self):
        if getattr(self, "_h", None):
            self._lib.xt_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            _raise(rc, self._lib.xt_multi_last_error(self._h).decode())

    def upload(self, segments: Sequence[np.ndarray], isBL: Sequence[int], chunk_size: int):
        segs = [np.ascontiguousarray(s, dtype=np.float64) for s in segments]
        if len(segs) == 0:
            raise ValueError("No track could be detected. The loaded tracks seem empty.")
        d = segs[0].shape[2]
        for s in segs:
            if s.ndim != 3 or s.shape[2] != d:
                raise ValueError("all track arrays must have shape [n, L, d] with the same d")
        n = len(segs)
        self._Ls = (C.c_int32 * n)(*[s.shape[1] for s in segs])
        self._ns = (C.c_int64 * n)(*[s.shape[0] for s in segs])
        bl = (C.c_int32 * n)(*[int(b) for b in isBL])
        ptrs = (C.c_void_p * n)(*[s.ctypes.data for s in segs])
        self._check(self._lib.xt_multi_upload(self._h, n, self._Ls, self._ns, bl, ptrs, d, int(chunk_size)))
        self.segments = [(s.shape[1], s.shape[0]) for s in segs]
        self.chunk_size = int(chunk_size)
        self.d = d

    def upload_aux(self, sigma: Optional[Sequence[np.ndarray]] = None, dt: Optional[Sequence[np.ndarray]] = None):
        n = len(self.segments)
        k = 0
        sp = dp = None
        keep = []
        if sigma is not None:
            sg = [np.ascontiguousarray(a, dtype=np.float64) for a in sigma]
            k = sg[0].shape[2] if sg[0].ndim == 3 else -1
            for a, (L, cnt) in zip(sg, self.segments):
                if a.ndim != 3 or a.shape != (cnt, L, k):
                    raise ValueError("Localization error is not specified correctly: input_LocErr arrays must have shape "
                                     "[n, L, 1] or [n, L, d] matching all_tracks")
            sp = (C.c_void_p * n)(*[a.ctypes.data for a in sg])
            keep.append(sg)
        if dt is not None:
            ds_ = [np.ascontiguousarray(a, dtype=np.float64) for a in dt]
            for a, (L, cnt) in zip(ds_, self.segments):
                if a.shape != (cnt, L):
                    raise ValueError("dt is not informed properly. It must either be a float number or a dictionary of same "
                                     "structure than `all_tracks` with each element being an array of dims (nb_tracks, track_len)")
            dp = (C.c_void_p * n)(*[a.ctypes.data for a in ds_])
            keep.append(ds_)
        self._check(self._lib.xt_multi_upload_aux(self._h, n, self._Ls, self._ns, int(k), sp, dp))

    def set_stay_tables(self, per_track: bool, Lp_stay: Optional[np.ndarray], L_leave: Optional[np.ndarray]):
        if per_track:
            raise NotImplementedError("per-track field-of-view tables belong to predict_Bs (single-device contexts)")
        if Lp_stay is None:
            self._check(self._lib.xt_multi_set_stay_tables(self._h, 0, 0, None, None))
            return
        a = np.ascontiguousarray(Lp_stay, dtype=np.float64)
        b = np.ascontiguousarray(L_leave, dtype=np.float64)
        pd = C.POINTER(C.c_double)
        self._check(self._lib.xt_multi_set_stay_tables(self._h, a.shape[1], b.shape[1], a.ctypes.data_as(pd), b.ctypes.data_as(pd)))

    def sum_logp(self, p: XtParams) -> float:
        out = C.c_double()
        self._check(self._lib.xt_multi_sum_logp(self._h, C.byref(p), C.byref(out)))
        return out.value

    def chunk_logp(self, chunk: int, nT: int, p: XtParams) -> np.ndarray:
        out = np.empty(nT, dtype=np.float64)
        self._check(self._lib.xt_multi_chunk_logp(self._h, int(chunk), C.byref(p), out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def eval_frozen(self, ps: Sequence[XtParams]) -> np.ndarray:
        """Sums of log P along every device's resident plan (``xt_multi_eval_frozen``), global chunk order."""
        sums = np.empty(len(ps))
        self._check(self._lib.xt_multi_eval_frozen(self._h, len(ps), _param_array(ps), sums.ctypes.data_as(C.POINTER(C.c_double))))
        return sums

    def score_outer(self, p_plus: Sequence[XtParams], p_minus: Sequence[XtParams], inv_2h) -> dict:
        """``xt_multi_score_outer``: same result, with the same bits, as one context holding all chunks."""
        rc, out = _score_outer(self._lib.xt_multi_score_outer, self._h, p_plus, p_minus, inv_2h)
        self._check(rc)
        return out

    def set_option(self, name: str, value: int):
        self._check(self._lib.xt_multi_set_option(self._h, name.encode(), int(value)))

    def device_load(self):
        """[(CUDA ordinal, chunks, track-steps)] per device slot."""
        out = []
        for g in range(len(self.devices)):
            dev, nch, steps = C.c_int32(), C.c_int32(), C.c_int64()
            self._check(self._lib.xt_multi_device_load(self._h, g, C.byref(dev), C.byref(nch), C.byref(steps)))
            out.append((dev.value, nch.value, steps.value))
        return out

    def stats(self) -> dict:
        st = XtStats()
        self._check(self._lib.xt_multi_get_stats(self._h, C.byref(st)))
        return {k: getattr(st, k) for k, _ in XtStats._fields_}


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """numpy array backed by pinned host memory (for end-to-end timing with host buffers)."""
    lib = load_library()
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    if lib.xt_host_alloc(C.byref(p), max(nbytes, 8)) != 0:
        raise EngineError(XT_ERR_CUDA, "cudaMallocHost failed")
    buf = (C.c_char * max(nbytes, 8)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    return arr
