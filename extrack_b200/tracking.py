"""Drop-in mirror of ``extrack.tracking``'s fit / predict API on top of the sm_100a CUDA engine.

Same names, argument meaning and error behaviour as the reference (ExTrack 1.6.3,
``extrack/tracking.py``): ``param_fitting`` (:1299), ``cum_Proba_Cs`` (:991), ``Proba_Cs`` (:769),
``predict_Bs`` (:792), ``extract_params`` (:913), ``generate_params`` (:1214), ``get_params``
(:1090) and the legacy ``get_2DSPT_params`` (``old_tracking.py:585``).  Host code stays
Python: parameter extraction, the parameter guard and the tiny per-evaluation tables
(incl. ``scipy.stats.norm.cdf`` for the field-of-view term) are computed here exactly as the
reference does; everything per track runs in hand-written CUDA kernels reached through the C
ABI in ``include/xtrack.h``.  There is no CPU fallback.

Tracks are packed and uploaded once per ``param_fitting`` / ``predict_Bs`` call (or once per
distinct list of arrays handed to ``cum_Proba_Cs``) and stay resident on the GPU.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _native
from ._lmfit_compat import Parameters, minimize

MAX_TRACKS_PER_CHUNK = 2000  # tracking.py:991 max_number_of_tracks_per_matrix


# --------------------------------------------------------------------------------------
# parameters -> model quantities (host; tracking.py:913-986)
# --------------------------------------------------------------------------------------
def _extract_scalars(params, nb_substeps, Matrix_type=1):
    """lmfit ``Parameters`` -> ``(LocErr values, Ds, Fs, TrMat, pBL)`` (tracking.py:918-975)."""
    # one pass over the sorted names (every `.value` of a constrained parameter evaluates its expression)
    names = tuple(params.keys())
    plan = _NAME_PLAN.get(names)
    if plan is None:  # classification of the (sorted) names: the same at every evaluation of a fit
        plan = []
        for n in sorted(names):
            c = n[0]
            if c == "L" and n.startswith("LocErr"):
                plan.append((n, 0, 0, 0))
            elif c == "D" and len(n) < 3:
                plan.append((n, 1, 0, 0))
            elif c == "F":
                plan.append((n, 2, 0, 0))
            elif c == "p":
                plan.append((n, 4, 0, 0) if n == "pBL" else (n, 3, int(n[1]), int(n[2])))
        if len(_NAME_PLAN) > 32:
            _NAME_PLAN.clear()
        _NAME_PLAN[names] = plan
    loc, Dv, Fv, rates, pBL = [], [], [], [], None
    for n, kind, i, j in plan:
        v = params[n].value
        if kind == 0:
            loc.append(v)
        elif kind == 1:
            Dv.append(v)
        elif kind == 2:
            Fv.append(v)
        elif kind == 3:
            rates.append((i, j, v))
        else:
            pBL = v
    Ds = np.array(Dv, dtype=float)
    Fs = np.array(Fv, dtype=float)
    nS = len(Ds)
    TrMat = np.zeros((nS, nS))
    for i, j, v in rates:
        TrMat[i, j] = v
    TrMat = TrMat / nb_substeps
    diag = np.arange(nS)
    if Matrix_type == 0:
        TrMat[diag, diag] = 1 - np.sum(TrMat, 1)
    if Matrix_type == 1:
        TrMat = 1 - np.exp(-TrMat)
        TrMat[diag, diag] = 1 - np.sum(TrMat, 1)
    elif Matrix_type in (2, 3, 4):
        from scipy import linalg

        if Matrix_type == 2:
            TrMat[diag, diag] = -np.sum(TrMat, 1)
            TrMat = linalg.expm(TrMat)
        else:
            TrMat[diag, diag] = 0
            G = np.copy(TrMat)
            TrMat[diag, diag] = 1 - np.sum(TrMat, 1)
            G[diag, diag] = -np.sum(G, 1)
            TrMatG = linalg.expm(G)
            TrMat = np.mean([TrMat, TrMatG], axis=0) if Matrix_type == 3 else (TrMat * TrMatG) ** 0.5
    return np.array(loc, dtype=float), Ds, Fs, TrMat, pBL


def _has_slope(params) -> bool:
    return any(k == "slope_LocErr" for k in params.keys())


def extract_params(params, dt, nb_states, nb_substeps, input_LocErr=None, Matrix_type=1):
    """lmfit ``Parameters`` -> ``(LocErr, ds, Fs, TrMat, pBL)`` with the reference's conventions
    (tracking.py:913-986).

    ``LocErr`` is ``[array(1,1,k)]``, or with peak-wise ``input_LocErr`` (a list of ``[n, L, k]``
    arrays, one per bucket) that list, transformed by ``slope_LocErr`` / ``offset_LocErr`` when
    these parameters exist (:926-932).  ``ds = sqrt(2 D dt)``; with a list of per-track ``dt``
    arrays ``[n, L]`` it is the list of ``[n, L, nS]`` arrays (:979-982).  ``TrMat`` holds
    per-sub-step transition probabilities.
    """
    loc, Ds, Fs, TrMat, pBL = _extract_scalars(params, nb_substeps, Matrix_type)
    LocErr = [loc[None, None]]
    if input_LocErr is not None:
        if _has_slope(params):
            LocErr = [np.clip(a * params["slope_LocErr"].value + params["offset_LocErr"].value, 0.000001, np.inf)
                      for a in input_LocErr]
        else:
            LocErr = input_LocErr
    if type(dt) == list:
        ds = [np.sqrt(2 * Ds[None, None] * t[:, :, None]) for t in dt]
    else:
        ds = np.sqrt(2 * Ds * dt)
    return LocErr, ds, Fs, TrMat, pBL


_P_STAY_MEMO: dict = {}
_FOV_GRID: dict = {}
_FOV_COLS: dict = {}
_FOV_LIN: dict = {}
_DIGITS: dict = {}
_NAME_PLAN: dict = {}


def _p_stay(ds, nS, nsub, cell_dims):
    """P(stay in the field of view) per sub-step state tuple (tracking.py:508-523).

    ``ds``: ``[nS]`` -> ``[K]``; or ``[rows, nS]`` (one row per chunk / track when dt is per track,
    :501-506) -> ``[rows, K]``, each row computed with the operations (and the summation order of
    ``np.mean(.., 0)``) the reference applies to a single chunk.
    """
    from scipy.special import ndtr  # what scipy.stats.norm.cdf evaluates (same bits, without the 0.1 ms wrapper)

    ds = np.asarray(ds, dtype=float)
    one = ds.ndim == 1
    if one:  # memo: most evaluations of a fit perturb a parameter that leaves ds unchanged (LocErr, F, p_ij, pBL)
        key = (ds.tobytes(), nS, nsub, tuple(float(c) for c in cell_dims))
        hit = _P_STAY_MEMO.get(key)
        if hit is not None:
            return hit.copy()
    K = nS**nsub
    tup = _DIGITS.get((nS, nsub, "tuples"))
    if tup is None:
        tup = _DIGITS[(nS, nsub, "tuples")] = np.arange(K)[:, None] // nS ** np.arange(nsub)[None, :] % nS
    if one:
        # One column per distinct diffusion length, memoised: a finite-difference step of a fit moves one D, so one
        # column is new.  np.mean(.., 0) of the reference's [1000, 1, K] array accumulates every column sequentially
        # over the grid points (the reduction runs over the outer axis), which np.cumsum reproduces bit for bit
        # (tests/test_host.py::test_p_stay_columns_reproduce_the_array_formula); a plain 1-D sum would be pairwise.
        sub_ds = np.mean(ds[tup] ** 2, axis=1) ** 0.5  # [K]
        out1 = np.ones(K)
        for cell_len in cell_dims:
            grid = _FOV_GRID.get(cell_len)
            if grid is None:
                xs = np.linspace(0 + cell_len / 2000, cell_len - cell_len / 2000, 1000)
                grid = _FOV_GRID[cell_len] = ((cell_len - xs[:, None, None]), -xs[:, None, None])
            cols = _FOV_COLS.setdefault(cell_len, {})
            for k in range(K):
                sk = float(sub_ds[k])
                cur = cols.get(sk)
                if cur is None:
                    lin = _FOV_LIN.get(cell_len)
                    if lin is None:
                        lin = _FOV_LIN[cell_len] = (np.ascontiguousarray(grid[0][:, 0, 0]), np.ascontiguousarray(grid[1][:, 0, 0]))
                    den1 = sub_ds[k] + 1e-200
                    cur = np.cumsum(ndtr(lin[0] / den1) - ndtr(lin[1] / den1))[-1] / 1000
                    if len(cols) > 256:
                        cols.clear()
                    cols[sk] = cur
                out1[k] = out1[k] * cur
        if len(_P_STAY_MEMO) > 64:
            _P_STAY_MEMO.clear()
        _P_STAY_MEMO[key] = out1.copy()
        return out1
    ds2 = ds
    out = np.ones((len(ds2), K))
    for r0 in range(0, len(ds2), 512):
        sub_ds = np.mean(ds2[r0 : r0 + 512][:, tup] ** 2, axis=2) ** 0.5  # [rows, K]
        p_stay = np.ones(sub_ds.shape)
        den = sub_ds + 1e-200
        for cell_len in cell_dims:
            grid = _FOV_GRID.get(cell_len)
            if grid is None:  # (cell_len - x) and -x on the 1000-point grid: the same arrays at every evaluation
                xs = np.linspace(0 + cell_len / 2000, cell_len - cell_len / 2000, 1000)
                grid = _FOV_GRID[cell_len] = ((cell_len - xs[:, None, None]), -xs[:, None, None])
            cur = np.mean(ndtr(grid[0] / den) - ndtr(grid[1] / den), 0)
            p_stay = p_stay * cur
        out[r0 : r0 + 512] = p_stay
    return out


def _head_tables(ds, Fs, TrMat, nS, nsub):
    """digits, dd, LT, LF per head (tracking.py:487-488,549-555,759-767); head h: digit k (base nS) =
    state k sub-steps ago, digit nsub = newest state of the parent."""
    dig = _DIGITS.get((nS, nsub))
    if dig is None:  # (the same small index table at every evaluation of a fit)
        nH0 = nS ** (nsub + 1)
        dig = _DIGITS[(nS, nsub)] = np.arange(nH0)[:, None] // nS ** np.arange(nsub + 1)[None, :] % nS
    nH = len(dig)
    d2 = ds[dig] ** 2
    dd = np.mean((d2[:, 1:] + d2[:, :-1]) / 2, axis=1)
    Tt = TrMat.T
    LT = np.zeros(nH)
    for k in range(nsub):
        LT += np.log(Tt[dig[:, k], dig[:, k + 1]])
    LF = np.log(Fs[dig[:, nsub]])
    return dig, dd, LT, LF


def _mid2(x):
    """The two middle order statistics of x (equal for an odd count): np.median = their mean."""
    x = np.sort(np.asarray(x, dtype=float).ravel())
    return x[(len(x) - 1) // 2], x[len(x) // 2]


def _median_ds(Ds, mids):
    """median over tracks of sqrt(2 D dt) per state from the two middle dt values (sqrt is monotone)."""
    mids = np.asarray(mids, dtype=float)
    a = np.sqrt(2 * Ds[None] * mids[..., 0:1].reshape(-1, 1))
    b = np.sqrt(2 * Ds[None] * mids[..., 1:2].reshape(-1, 1))
    return (a + b) / 2


def stay_tables(Ds, mids, TrMat, pBL, cell_dims, nb_substeps):
    """Per-row (chunk or track) ``Lp_stay [rows, K]`` and ``L_leave [rows, H]`` when dt is per track:
    the reference derives p_stay from the median diffusion length of the chunk's first time step
    (tracking.py:501-506,515-524,630-631).  ``mids``: ``[rows, 2]`` middle order statistics of
    ``dt[:, 0]`` per row."""
    Ds = np.asarray(Ds, dtype=float)
    nS, nsub = len(Ds), int(nb_substeps)
    uniq, inv = np.unique(np.asarray(mids, dtype=float).reshape(-1, 2), axis=0, return_inverse=True)
    inv = np.asarray(inv).reshape(-1)
    p_stay = _p_stay(_median_ds(Ds, uniq), nS, nsub, cell_dims)  # [U, K]
    dig, _, LT, _ = _head_tables(np.zeros(nS), np.ones(nS), np.asarray(TrMat, dtype=float), nS, nsub)
    Lp_stay = np.log(p_stay * (1 - pBL))
    e = p_stay[:, dig[:, 0]]
    L_leave = np.log(pBL + (1 - e) - pBL * (1 - e)) + LT[None]
    return Lp_stay[inv], L_leave[inv]


def build_tables(LocErr, ds, Fs, TrMat, pBL, cell_dims, nb_substeps, frame_len, min_len, threshold,
                 max_nb_states, nb_dims, int8_wrap=True, var_loc_k=0, var_dt=False, Ds=None,
                 slope_offset=None) -> _native.XtParams:
    """Model quantities -> the engine's per-evaluation POD (``xt_params`` in include/xtrack.h).

    Restates the table-building half of ``P_Cs_inter_bound_stats_th`` (tracking.py:474-524,
    549-555, 630-631) once per evaluation instead of once per chunk.  ``var_loc_k`` > 0: the
    localisation errors are the resident peak-wise ones (k components, ``LocErr`` is ignored,
    optionally ``slope_offset``); ``var_dt``: dt is resident per localisation (``Ds`` required, ``ds``
    = the guard's median diffusion lengths).
    """
    ds = np.asarray(ds, dtype=float)
    Fs = np.asarray(Fs, dtype=float)
    TrMat = np.asarray(TrMat, dtype=float)
    nS, nsub = len(ds), int(nb_substeps)
    loc = np.asarray(LocErr, dtype=float).reshape(-1)
    if var_loc_k:
        loc = np.zeros(int(var_loc_k))
    if len(loc) not in (1, nb_dims):
        raise ValueError(
            "Localization error is not specified correctly, in case of unique localization error specify a float "
            "number in estimated_vals['LocErr'].\n If one localization error per dimension, specify a list or 1D "
            "array of elements the localization error for each dimension."
        )
    K = nS**nsub
    nH = K * nS
    if nH > _native.XT_MAX_HEADS or nS > _native.XT_MAX_STATES:
        raise ValueError(f"nb_states**(nb_substeps+1) = {nH} exceeds the engine limit {_native.XT_MAX_HEADS}")
    p = _native.XtParams()
    p.nS, p.nsub, p.d, p.n_loc = nS, nsub, int(nb_dims), len(loc)
    p.frame_len, p.min_len, p.max_nb_states = int(frame_len), int(min_len), int(min(max_nb_states, 2**31 - 1))
    p.flags = _native.XT_FLAG_INT8_WRAP if int8_wrap else 0
    if var_loc_k:
        p.flags |= _native.XT_FLAG_VAR_LOC
        if slope_offset is not None:
            p.flags |= _native.XT_FLAG_LOC_AFFINE
            p.loc_slope, p.loc_offset = float(slope_offset[0]), float(slope_offset[1])
    if var_dt:
        p.flags |= _native.XT_FLAG_VAR_DT
    if Ds is not None:
        for k, v in enumerate(2 * np.asarray(Ds, dtype=float)):
            p.twoD[k] = v
    p.threshold = float(threshold)
    for k, v in enumerate(loc**2):
        p.l2[k] = v
    dig, dd, LT, LF = _head_tables(ds, Fs, TrMat, nS, nsub)
    p_stay = _p_stay(ds, nS, nsub, cell_dims)
    Lp_stay = np.log(p_stay * (1 - pBL))
    e = p_stay[dig[:, 0]]  # indexed by the newest *state value* (reference quirk, tracking.py:630)
    L_leave = np.log(pBL + (1 - e) - pBL * (1 - e)) + LT
    for field, vals in (("dd", dd), ("LT", LT), ("LF", LF), ("L_leave", L_leave), ("Lp_stay", Lp_stay)):
        v = np.ascontiguousarray(vals, dtype=np.float64)
        ctypes.memmove(ctypes.addressof(getattr(p, field)), v.ctypes.data, v.nbytes)  # one copy per table, no Python loop
    return p


# --------------------------------------------------------------------------------------
# resident data set
# --------------------------------------------------------------------------------------
def _sorted_buckets(all_tracks: Dict[str, np.ndarray]):
    """Numerically sorted, non-empty length buckets (tracking.py:1346-1359, :822-833)."""
    keys = np.sort(np.array(list(all_tracks.keys())).astype(int)).astype(str)
    return [all_tracks[k] for k in keys if len(all_tracks[k]) > 0], [k for k in keys]


def chunk_table(sorted_tracks: Sequence[np.ndarray], chunk: int, reverse: bool = True):
    """Reference chunk list: ``(bucket, start, stop, isBL)`` (tracking.py:1024-1044)."""
    max_len = sorted_tracks[-1].shape[1]
    out = []
    for b, arr in enumerate(sorted_tracks):
        for n in range(int(np.ceil(len(arr) / chunk))):
            out.append((b, n * chunk, min((n + 1) * chunk, len(arr)), 0 if arr.shape[1] == max_len else 1))
    if reverse:
        out.reverse()
    return out


def shard_chunks(chunks, sorted_tracks, world_size: int) -> List[List[int]]:
    """Longest-processing-time-first assignment of chunks to ranks; cost = nT*(L-1).

    Chunks are the atomic unit (the grouping plan is decided per chunk, tracking.py:677-691),
    so shards are sets of whole chunks and the result is independent of ``world_size``.
    """
    cost = [(z - a) * (sorted_tracks[b].shape[1] - 1) for (b, a, z, _) in chunks]
    order = sorted(range(len(chunks)), key=lambda i: (-cost[i], i))
    load = [0] * world_size
    owner: List[List[int]] = [[] for _ in range(world_size)]
    for i in order:
        r = min(range(world_size), key=lambda k: (load[k], k))
        owner[r].append(i)
        load[r] += cost[i]
    for r in range(world_size):
        owner[r].sort()
    return owner


class TrackSet:
    """Tracks of one fit, packed and resident on this process's GPU.

    With ``torch.distributed`` initialised (one process per GPU) each rank uploads only its
    shard of the chunk list and ``sum_logp`` all-reduces the partial sums (one 8-byte
    all-reduce per objective call, NCCL over NVLink).
    """

    def __init__(self, sorted_tracks: Sequence[np.ndarray], chunk: int = MAX_TRACKS_PER_CHUNK, device: Optional[int] = None,
                 rank: Optional[int] = None, world_size: Optional[int] = None, reverse: bool = True,
                 input_LocErr: Optional[Sequence[np.ndarray]] = None, dt_list: Optional[Sequence[np.ndarray]] = None,
                 precision: Optional[str] = None, devices: Optional[Sequence[int]] = None):
        if len(sorted_tracks) < 1:
            raise ValueError("No track could be detected. The loaded tracks seem empty. Errors often come from wrong input paths.")
        for a in sorted_tracks:
            if a.shape[1] < 2:
                raise ValueError("minimal track length = 2, here track length = %s" % a.shape[1])
        self.sorted_tracks = list(sorted_tracks)
        self.min_len = sorted_tracks[0].shape[1]
        self.max_len = sorted_tracks[-1].shape[1]
        self.nb_dims = sorted_tracks[0].shape[2]
        self.chunk = int(chunk)
        self.rank, self.world_size = _dist_info(rank, world_size)
        self.chunks = chunk_table(sorted_tracks, self.chunk, reverse)
        mine = shard_chunks(self.chunks, sorted_tracks, self.world_size)[self.rank] if self.world_size > 1 else list(range(len(self.chunks)))
        self.my_chunks = mine
        if device is None:
            device = _default_device()
        # several GPUs driven from this one process (`devices`, see resolve_devices): the engine deals the chunk list
        # to them; the objective keeps the bits of the one-GPU evaluation.  Not combined with one-process-per-GPU runs.
        self.devices = [int(x) for x in devices] if (devices is not None and len(devices) > 1 and self.world_size == 1) else None
        self.engine = _native.MultiEngine(self.devices) if self.devices else _native.Engine(device)
        self.device = device
        self.precision = _check_precision(precision if precision is not None else _PRECISION)
        if self.precision == "fp32":
            self.engine.set_option("fp32_replay", 1)
        segs = [self.sorted_tracks[b][a:z] for (b, a, z, _) in (self.chunks[i] for i in mine)]
        bl = [self.chunks[i][3] for i in mine]
        self.n_local_chunks = len(segs)
        if segs:
            self.engine.upload(segs, bl, self.chunk)
        self._dist_buf = None
        # peak-wise localisation errors [n, L, k] / per-localisation dt [n, L] per bucket (sorted like the tracks)
        self.loc_k = 0
        self.has_dt = dt_list is not None
        self.dt_mids = self.dt_mid0 = None
        if input_LocErr is not None or dt_list is not None:
            cut = lambda arrs: [np.asarray(arrs[b])[a:z] for (b, a, z, _) in (self.chunks[i] for i in mine)]
            if input_LocErr is not None:
                for a, c in zip(input_LocErr, self.sorted_tracks):
                    a = np.asarray(a)
                    if a.ndim != 3 or a.shape[:2] != c.shape[:2] or a.shape[2] not in (1, c.shape[2]):
                        raise ValueError(
                            "Localization error is not specified correctly, in case of unique localization error specify "
                            "a float number in estimated_vals['LocErr'].\n If one localization error per dimension, "
                            "specify a list or 1D array of elements the localization error for each dimension.\n If "
                            "localization error is predetermined by another method for each position the argument "
                            "input_LocErr should be a dict for each track length of the 3D arrays corresponding to "
                            "all_tracks (can be obtained from the reader functions using the opt_colname argument)")
                self.loc_k = int(np.asarray(input_LocErr[0]).shape[2])
            if dt_list is not None:
                for a, c in zip(dt_list, self.sorted_tracks):
                    if np.asarray(a).shape != c.shape[:2]:
                        raise ValueError(
                            "dt is not informed properly. It must either be a float number or a dictionary of same "
                            "structure than `all_tracks` with each element being an array of dims (nb_tracks, track_len)")
                dts = cut(dt_list)
                # field-of-view term: median over the chunk of ds[:, 0] (tracking.py:501-506); guard: median of
                # the first bucket's ds (:1012-1013).  sqrt is monotone: keep the middle order statistics of dt
                self.dt_mids = np.array([_mid2(a[:, 0]) for a in dts]).reshape(-1, 2)
                self.dt_mid0 = np.array(_mid2(np.asarray(dt_list[0])))
            if segs:
                self.engine.upload_aux(cut(input_LocErr) if input_LocErr is not None else None,
                                       dts if dt_list is not None else None)

    # local chunk index of global chunk i (or None when another rank owns it)
    def local_index(self, i: int) -> Optional[int]:
        try:
            return self.my_chunks.index(i)
        except ValueError:
            return None

    def sum_logp(self, p: _native.XtParams) -> float:
        if self.world_size == 1:
            return self.engine.sum_logp(p)
        import torch
        import torch.distributed as dist

        if self._dist_buf is None:
            dev = torch.device("cuda", self.device) if dist.get_backend() == "nccl" else torch.device("cpu")
            self._dist_buf = torch.zeros(2, dtype=torch.float64, device=dev)  # [sum, error flag]
        buf = self._dist_buf
        # a rank whose engine fails must still enter the collective (the others would wait for ever): the
        # second element carries an error flag and every rank raises after the all-reduce
        err = None
        buf[1] = 0.0
        try:
            if buf.is_cuda and self.n_local_chunks:
                # result stays on the device; the all-reduce is chained on torch's current stream
                self.engine.sum_logp_async(p, buf.data_ptr(), torch.cuda.current_stream(buf.device).cuda_stream)
            else:
                buf[0] = self.engine.sum_logp(p) if self.n_local_chunks else 0.0
        except Exception as e:  # noqa: BLE001 - re-raised below on every rank
            err = e
            buf[0] = 0.0
            buf[1] = 1.0
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        total, flag = (float(x) for x in buf.tolist())
        if err is not None:
            raise err
        if flag != 0.0:
            raise _native.EngineError(_native.XT_ERR_STATE, "the likelihood evaluation failed on another rank")
        return total

    def _all_reduce(self, compute, size: int) -> np.ndarray:
        """``compute()`` -> float64[size] on this rank's shard, summed over the ranks in one all-reduce that also carries
        the error flag (as ``sum_logp``)."""
        if self.world_size == 1:
            return compute()
        import torch
        import torch.distributed as dist

        dev = torch.device("cuda", self.device) if dist.get_backend() == "nccl" else torch.device("cpu")
        buf = torch.zeros(size + 1, dtype=torch.float64, device=dev)
        err = None
        try:
            if self.n_local_chunks:
                buf[:size] = torch.from_numpy(np.ascontiguousarray(compute(), dtype=np.float64)).to(dev)
        except Exception as e:  # noqa: BLE001 - re-raised below on every rank
            err = e
            buf.zero_()
            buf[size] = 1.0
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        out = buf.cpu().numpy()
        if err is not None:
            raise err
        if out[size] != 0.0:
            raise _native.EngineError(_native.XT_ERR_STATE, "the frozen-plan evaluation failed on another rank")
        return out[:size]

    def eval_frozen(self, ps: Sequence[_native.XtParams]) -> np.ndarray:
        """Sums of log P over the data set for every parameter set, along the plan of the last ``sum_logp``."""
        return self._all_reduce(lambda: self.engine.eval_frozen(ps), len(ps))

    def score_outer(self, p_plus: Sequence[_native.XtParams], p_minus: Sequence[_native.XtParams], inv_2h) -> dict:
        """Central-difference scores along the plan of the last ``sum_logp``: ``sum_plus``, ``sum_minus``, ``gsum``,
        ``gram`` (see ``xt_score_outer``)."""
        n = len(p_plus)

        def compute():
            r = self.engine.score_outer(p_plus, p_minus, inv_2h)
            return np.concatenate([r["sum_plus"], r["sum_minus"], r["gsum"], r["gram"].reshape(-1)])

        v = self._all_reduce(compute, 3 * n + n * n)
        return {"sum_plus": v[:n], "sum_minus": v[n:2 * n], "gsum": v[2 * n:3 * n], "gram": v[3 * n:].reshape(n, n)}

    def close(self):
        self.engine.close()


def _dist_info(rank, world_size):
    if rank is not None and world_size is not None:
        return int(rank), int(world_size)
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    return 0, 1


def _default_device() -> int:
    import os

    return int(os.environ.get("LOCAL_RANK", "0"))


def resolve_devices(workers: int = 1) -> Optional[List[int]]:
    """GPUs one process drives for a fit, as a list of CUDA ordinals (None = the single default device).

    The reference's ``workers`` is the width of its process pool over chunks (tracking.py:1061-1063); here
    ``workers = N > 1`` asks for up to N GPUs of this box; ``EXTRACK_B200_GPUS`` (a count or ``all``)
    overrides it and ``EXTRACK_B200_DEVICES`` (comma-separated ordinals) names the devices explicitly.  Under ``torch.distributed`` (one process per GPU) every process keeps its own device.
    """
    import os

    if _dist_info(None, None)[1] > 1:
        return None
    explicit = os.environ.get("EXTRACK_B200_DEVICES", "").strip()  # explicit ordinals, e.g. "0,1,2,3" (may repeat: logical shards)
    if explicit:
        devs = [int(x) for x in explicit.split(",")]
        return devs if len(devs) > 1 else None
    env = os.environ.get("EXTRACK_B200_GPUS", "").strip().lower()
    want = int(workers) if workers else 1
    if env:
        want = 10**6 if env == "all" else int(env)
    if want <= 1:
        return None
    n = min(want, _native.device_count())
    return list(range(n)) if n > 1 else None


# Arithmetic of the replay kernel: "fp64" (reference precision, default) or "fp32" (optional path of the
# north star: total log-likelihood within 1e-4 relative of the FP64 result; the fusion plan stays FP64).
# The reference signatures have no such argument, so it is a module switch (or EXTRACK_B200_PRECISION).
import os as _os

_PRECISION = _os.environ.get("EXTRACK_B200_PRECISION", "fp64")


def _check_precision(name: str) -> str:
    if name not in ("fp64", "fp32"):
        raise ValueError("precision must be 'fp64' or 'fp32', got %r" % (name,))
    return name


def set_precision(name: str) -> None:
    """Select the replay arithmetic of the data sets created from now on (``param_fitting`` /
    ``cum_Proba_Cs``); ``predict_Bs`` always runs in FP64."""
    global _PRECISION
    _PRECISION = _check_precision(name)
    for _, _, old in _TRACKSET_CACHE:
        old.close()
    del _TRACKSET_CACHE[:]


def get_precision() -> str:
    return _PRECISION


_TRACKSET_CACHE: List = []  # [(key, refs, TrackSet)] most recent first


def _fingerprint(a) -> tuple:
    """Identity + a cheap content sample of one caller array: (id, shape, data pointer, strided-sample sum).  The
    sample (<= 4096 elements spread over the whole array, O(microseconds)) catches in-place edits of the tracks
    between objective calls without re-reading the data set."""
    arr = np.asarray(a)
    flat = arr.reshape(-1)
    step = max(1, flat.size // 4096)
    return (id(a), arr.shape, arr.__array_interface__["data"][0], float(np.sum(flat[::step], dtype=np.float64)))


def _trackset_for(all_tracks: Sequence[np.ndarray], chunk: int, input_LocErr=None, dt_list=None, workers: int = 1) -> TrackSet:
    """Resident data for the arrays handed to ``cum_Proba_Cs`` (upload once per fit, not once per call).

    Contract: the data set of a distinct list of caller arrays stays resident on the GPU(s) and is reused by
    later calls with the same arrays; it is keyed on the caller's own objects (identity, shape, data pointer)
    plus a strided content sample, so replacing or editing an array uploads again.  An in-place edit that the
    sample misses is not seen: call ``invalidate_cache()`` after mutating tracks in place (the reference
    re-reads its arrays on every call).  At most two data sets are kept; ``invalidate_cache()`` /
    ``set_precision()`` free them."""
    sig = lambda arrs: tuple(_fingerprint(a) for a in arrs)
    devices = resolve_devices(workers)
    key = sig(all_tracks) + (chunk, tuple(devices or ())) + (sig(input_LocErr) if input_LocErr is not None else (None,)) + (
        sig(dt_list) if dt_list is not None else (None,))
    for k, refs, ts in _TRACKSET_CACHE:
        if k == key:
            return ts
    loc = [np.asarray(a, dtype=np.float64) for a in input_LocErr] if input_LocErr is not None else None
    ts = TrackSet(all_tracks, chunk, input_LocErr=loc, dt_list=dt_list, devices=devices)
    _TRACKSET_CACHE.insert(0, (key, [list(all_tracks), input_LocErr, dt_list], ts))
    while len(_TRACKSET_CACHE) > 2:
        _, _, old = _TRACKSET_CACHE.pop()
        old.close()
    return ts


def invalidate_cache() -> None:
    """Free the data sets ``cum_Proba_Cs`` keeps resident between calls (GPU and pinned host memory)."""
    for _, _, old in _TRACKSET_CACHE:
        old.close()
    del _TRACKSET_CACHE[:]


# --------------------------------------------------------------------------------------
# objective (tracking.py:991-1088)
# --------------------------------------------------------------------------------------
def _objective_tables(params, ts: TrackSet, dt, cell_dims, nb_substeps, frame_len, threshold, max_nb_states, Matrix_type):
    """Parameters -> the objective's validity guard -> ``build_tables``: ``(p, (Ds, TrMat, pBL))``, ``p`` = None when
    the guard rejects the parameters (the objective is then +inf)."""
    loc, Ds, Fs, TrMat, pBL = _extract_scalars(params, nb_substeps, Matrix_type)
    if type(dt) == list:
        ds = _median_ds(Ds, ts.dt_mid0)[0]  # avg_ds = np.median(ds[0], axis=(0, 1)), tracking.py:1012-1013
    else:
        ds = np.sqrt(2 * Ds * dt)
    # validity guard of the reference (tracking.py:1017: all transition probabilities and fractions positive, diffusion
    # lengths ascending); minima instead of three np.all passes - NaN fails either way
    if not (TrMat.min() > 0 and Fs.min() > 0 and (len(ds) < 2 or (ds[1:] - ds[:-1]).min() >= 0)):
        return None, (Ds, TrMat, pBL)
    slope = (params["slope_LocErr"].value, params["offset_LocErr"].value) if (ts.loc_k and _has_slope(params)) else None
    p = build_tables(loc, ds, Fs, TrMat, pBL, cell_dims, nb_substeps, frame_len, ts.min_len, threshold,
                     max_nb_states, ts.nb_dims, var_loc_k=ts.loc_k, var_dt=ts.has_dt, Ds=Ds, slope_offset=slope)
    return p, (Ds, TrMat, pBL)


def cum_Proba_Cs(params, all_tracks, dt, cell_dims, input_LocErr, nb_states, nb_substeps, frame_len, verbose=1,
                 workers=1, Matrix_type=1, threshold=0.2, max_nb_states=120, max_number_of_tracks_per_matrix=2000,
                 _trackset: Optional[TrackSet] = None):
    """-sum log L over all tracks for ``params`` (``np.inf`` for invalid parameters).

    ``all_tracks`` is the sorted list of ``[n, L, d]`` arrays (as ``param_fitting`` builds it);
    ``input_LocErr`` (optional) the matching list of peak-wise localisation errors ``[n, L, k]`` and
    ``dt`` a float or the matching list of ``[n, L]`` time steps (tracking.py:1024-1044).
    ``workers`` > 1 asks for that many GPUs of this box (``resolve_devices``); the GPUs replace the process pool.
    """
    dt_list = dt if type(dt) == list else None
    ts = _trackset if _trackset is not None else _trackset_for(all_tracks, max_number_of_tracks_per_matrix, input_LocErr,
                                                               dt_list, workers)
    quiet = ts.rank != 0
    p, (Ds, TrMat, pBL) = _objective_tables(params, ts, dt, cell_dims, nb_substeps, frame_len, threshold, max_nb_states,
                                            Matrix_type)
    if p is not None:
        if ts.has_dt and ts.n_local_chunks:
            ts.engine.set_stay_tables(False, *stay_tables(Ds, ts.dt_mids, TrMat, pBL, cell_dims, nb_substeps))
        ts._last_p = p
        Cum_P = ts.sum_logp(p)
        if not quiet:
            if verbose == 1:
                q = [param + " = " + str(np.round(params[param].value, 6)) for param in params]
                print(Cum_P, q)
            else:
                print(".", end="")
        out = -Cum_P
    else:
        out = np.inf
        if not quiet:
            print("x", end="")
            if verbose == 1:
                q = [param + " = " + str(np.round(params[param].value, 4)) for param in params]
                print(q)
    if np.isnan(out):
        out = np.inf
        if not quiet:
            print("input parameters give nans, you may want to pick more suitable parameter initial values")
    return out


def Proba_Cs(Cs, LocErr, ds, Fs, TrMat, pBL, isBL, cell_dims, nb_substeps, frame_len, min_len, threshold, max_nb_states):
    """log P(track) for every track of one chunk (tracking.py:769-787). Test / parity seam."""
    Cs = np.asarray(Cs, dtype=np.float64)
    if Cs.shape[1] < 2:
        raise ValueError("minimal track length = 2, here track length = %s" % Cs.shape[1])
    p = build_tables(LocErr, ds, Fs, TrMat, pBL, cell_dims, nb_substeps, frame_len, min_len, threshold, max_nb_states,
                     Cs.shape[2])
    eng = _native.Engine(_default_device())
    try:
        eng.upload([Cs], [isBL], max(len(Cs), 1))
        return eng.chunk_logp(0, len(Cs), p)
    finally:
        eng.close()


# --------------------------------------------------------------------------------------
# state annotation (tracking.py:792-906)
# --------------------------------------------------------------------------------------
def _gather_predictions(preds_local, sorted_tracks, world, row_shape, nb_max=1):
    """All ranks' slices of every bucket -> full arrays in input order (rank r holds rows predict_shard(n, r, world)).
    ``row_shape(L)``: the shape of one track's entry in the slices of a bucket of length L."""
    import torch
    import torch.distributed as dist

    dev = torch.device("cuda", _default_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    out = []
    for a, mine in zip(sorted_tracks, preds_local):
        n, L = a.shape[0], a.shape[1]
        rows = [predict_shard(n, r, world, nb_max) for r in range(world)]
        pad = max(hi - lo for lo, hi in rows)
        buf = torch.zeros((pad,) + row_shape(L), dtype=torch.float64, device=dev)
        buf[: len(mine)] = torch.from_numpy(np.ascontiguousarray(mine)).to(dev)
        parts = [torch.empty_like(buf) for _ in range(world)]
        dist.all_gather(parts, buf)
        out.append(np.concatenate([parts[r][: hi - lo].cpu().numpy() for r, (lo, hi) in enumerate(rows)]))
    return out


def predict_shard(n: int, rank: int, world_size: int, nb_max: int = 1):
    """Rows ``[lo, hi)`` of an ``n``-track bucket annotated by ``rank``: contiguous, balanced, and cut at multiples of
    ``nb_max`` so that every rank holds whole chunks of the reference's chunk list (tracking.py:866-867)."""
    nch = -(-n // nb_max)
    return min(n, (nch * rank // world_size) * nb_max), min(n, (nch * (rank + 1) // world_size) * nb_max)


def predict_Bs(all_tracks, dt, params, cell_dims=[1], nb_states=4, frame_len=5, max_nb_states=200, threshold=0.1,
               workers=1, input_LocErr=None, verbose=0, nb_max=1, gather=True):
    """Per-localisation state posteriors, ``{str(L): float64[n, L, nb_states]}`` (forward time).

    ``nb_max`` tracks share one grouping plan, decided from the first 30 tracks of their chunk exactly as the
    reference does (tracking.py:803,866-867; "higher numbers ... might affect the predictions quality"); with the
    default ``nb_max = 1`` every track gets its own plan.  ``nb_max > 1`` is implemented for scalar ``LocErr`` /
    ``dt`` (``NotImplementedError`` with peak-wise ``input_LocErr`` or a ``dt`` dictionary).
    ``workers`` is accepted and ignored.

    With ``torch.distributed`` initialised (one process per GPU) every rank annotates a contiguous
    slice of each length bucket (``predict_shard``); tracks are independent, so the data path has no
    collective.  ``gather=True`` (default) reassembles the full dictionary on every rank in input
    order (one all-gather per bucket); ``gather=False`` returns only this rank's rows.
    """
    return _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max,
                     gather, "preds")[0]


def predict_transitions(all_tracks, dt, params, cell_dims=[1], nb_states=4, frame_len=5, max_nb_states=200, threshold=0.1,
                        workers=1, input_LocErr=None, verbose=0, nb_max=1, gather=True):
    """``predict_Bs`` plus the two-slice (transition) posteriors of the same recursion: ``(preds, pairs)``, two
    ``{str(L): array}`` dictionaries.  ``preds[k]`` is ``predict_Bs``'s float64[n, L, nb_states];
    ``pairs[k]`` is float64[n, L - 1, nb_states, nb_states] with ``pairs[k][t, i, a, b]`` = P(state a at localisation
    i, state b at localisation i + 1 | track t), forward time.  ``pairs.sum(-1) == preds[:, :-1]`` and
    ``pairs.sum(-2) == preds[:, 1:]`` to rounding.  The probability that track t switches state between localisations
    i and i + 1 is ``1 - trace(pairs[t, i])``; ``transition_summary`` aggregates them.

    Arguments, validation, ``nb_max`` rules and errors, ``torch.distributed`` sharding and ``gather`` are those of
    ``predict_Bs`` (the pairs take one more all-gather per bucket).
    """
    return _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max,
                     gather, "pairs")


def predict_residuals(all_tracks, dt, params, cell_dims=[1], nb_states=4, frame_len=5, max_nb_states=200, threshold=0.1,
                      workers=1, input_LocErr=None, verbose=0, nb_max=1, gather=True):
    """``predict_Bs`` plus the one-step-ahead residuals of the same recursion: ``(preds, logpred, pit)``, three
    ``{str(L): array}`` dictionaries.  ``preds[k]`` is ``predict_Bs``'s float64[n, L, nb_states].

    At the step that consumes localisation ``c_i`` (i >= 1), the live state sequences of the recursion form a Gaussian
    mixture: the model's predictive distribution of ``c_i`` given ``c_0 .. c_i-1``.  ``logpred[k]`` is float64[n, L]:
    the log density of that mixture at ``c_i``.  A mislinked localisation, or a jump no state explains, is a deep
    minimum inside its track.  ``pit[k]`` is float64[n, L, d]: the mixture's cumulative distribution at ``c_i``, per
    dimension (probability integral transform).  When the model describes the data these values are Uniform(0, 1); a
    skewed histogram shows where it does not (for example a missing state).  Localisation 0 has no predictive: its
    entries are NaN.

    Arguments, validation, ``nb_max`` rules and errors, ``torch.distributed`` sharding and ``gather`` are those of
    ``predict_Bs`` (logpred and pit take one more all-gather per bucket each).
    """
    return _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max,
                     gather, "resid")


def predict_path(all_tracks, dt, params, cell_dims=[1], nb_states=4, frame_len=5, max_nb_states=200, threshold=0.1,
                 workers=1, input_LocErr=None, verbose=0, nb_max=1, gather=True):
    """``predict_Bs`` plus the most probable state path (MAP / Viterbi path) of every track: ``(preds, paths,
    path_logp)``, three ``{str(L): array}`` dictionaries.  ``preds[k]`` is ``predict_Bs``'s float64[n, L, nb_states];
    ``paths[k]`` is int8[n, L], one state label per localisation (forward time); ``path_logp[k]`` is float64[n].

    The annotation recursion is a lattice: every expansion gives each child one parent, every fusion gives each member
    a normalised merge weight inside its group, and the final sequences get softmax(LP).  A route from an initial to a
    final sequence weighs its final weight times the product of the merge weights along it; the route weights sum to 1,
    and summed by label they are ``preds``.  ``paths`` is the label sequence of the heaviest route (ties: the lowest
    member / sequence index) and ``path_logp`` the log of its weight, so ``path_logp <= log preds[t, k, paths[t, k]]``
    for every k.  Without fusion (tracks no longer than ``frame_len``) the path is the exact most probable state
    sequence and ``path_logp`` its posterior log-probability.  Unlike ``argmax(preds, -1)``, which maximises the
    expected number of correct frames, the path is one consistent segmentation: it does not dither where the
    posteriors are near 0.5.  ``path_segments`` turns the paths into dwell-time histograms.  Labels are those of
    ``preds`` (with the reference's int8 label wrap, which only matters for 3, 5, ... states past 128 sequences).

    Arguments, validation, ``nb_max`` rules and errors, ``torch.distributed`` sharding and ``gather`` are those of
    ``predict_Bs`` (paths and path_logp take one more all-gather per bucket each).
    """
    return _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max,
                     gather, "path")


def sample_paths(all_tracks, dt, params, cell_dims=[1], nb_states=4, frame_len=5, max_nb_states=200, threshold=0.1,
                 workers=1, input_LocErr=None, verbose=0, nb_max=1, gather=True, n_samples=100, seed=0):
    """``predict_Bs`` plus ``n_samples`` posterior draws of the whole state path of every track: ``(preds, samples,
    sample_logp)``, three ``{str(L): array}`` dictionaries.  ``preds[k]`` is ``predict_Bs``'s float64[n, L,
    nb_states]; ``samples[k]`` is int8[n, n_samples, L], one state label per localisation and draw (forward time);
    ``sample_logp[k]`` is float64[n, n_samples].

    The draws run on the lattice of ``predict_path`` (forward filtering, backward sampling): a draw picks a route with
    probability equal to its weight, from the end backwards (the final sequence with the final softmax weights, then at
    every fusion one member of the parent group with its normalised merge weight).  ``sample_logp`` is the log of the
    drawn route's weight, so it never exceeds ``predict_path``'s ``path_logp``.  Over the draws, the frequency of label
    i at localisation k converges to ``preds[t, k, i]`` and that of consecutive labels to ``predict_transitions``'
    pairs; without fusion (tracks no longer than ``frame_len``) every draw is an exact sample of the posterior
    P(s_0..s_L-1 | track).  The mean over draws of any path statistic (dwell times, switches per track, time to the
    first switch) is its posterior expectation and the spread over draws its credible interval; ``sample_segments``
    gives the dwell-time histogram of every draw.  Labels are those of ``preds`` (with the reference's int8 label wrap).

    The draws are reproducible: they depend only on ``seed``, the bucket length, the track's row in its bucket and the
    draw index, so draw d is the same whatever ``n_samples`` (>= d + 1), ``torch.distributed`` sharding or launch
    shape.  ``n_samples`` must be an int in [1, 65535] and ``seed`` an int in [0, 2^64).  Other arguments, validation,
    ``nb_max`` rules and errors, sharding and ``gather`` are those of ``predict_Bs`` (the samples and their log weights
    take one more all-gather per bucket each).
    """
    _int = lambda x: isinstance(x, (int, np.integer)) and not isinstance(x, (bool, np.bool_))
    if not _int(n_samples) or not 1 <= int(n_samples) <= 65535:
        raise ValueError("n_samples must be an int in [1, 65535]")
    if not _int(seed) or not 0 <= int(seed) < 2**64:
        raise ValueError("seed must be an int in [0, 2^64)")
    return _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max,
                     gather, "samples", int(n_samples), int(seed))


def _segments(a):
    """Maximal runs of equal labels in the rows of a [n, L] (int64): (row, length, state, censored) of every run, in
    row-major order.  A run is censored when it touches the first or the last localisation of its row."""
    n, L = a.shape
    change = a[:, 1:] != a[:, :-1]  # [n, L - 1]: a segment ends at localisation k and the next starts at k + 1
    t_e, k_e = np.nonzero(np.concatenate([change, np.ones((n, 1), dtype=bool)], axis=1))
    _, k_s = np.nonzero(np.concatenate([np.ones((n, 1), dtype=bool), change], axis=1))
    # (row-major order: the i-th start and the i-th end belong to the same segment)
    return t_e, k_e - k_s + 1, a[t_e, k_e], (k_s == 0) | (k_e == L - 1)


def sample_segments(samples, nb_states):
    """Dwell-time histograms of ``sample_paths``' draws (host only): ``(interior, censored)``, two int64 arrays
    [n_samples, L_max, nb_states].  Slice d is ``path_segments`` of draw d over all tracks: row ``n - 1`` counts the
    segments of n localisations by state, ``interior`` those with both ends observed inside the track, ``censored``
    those touching its first or last localisation.  The mean over the first axis is the posterior expectation of the
    histogram and its quantiles over that axis are credible bands."""
    items = [np.asarray(a) for a in (samples.values() if isinstance(samples, dict) else samples)]
    items = [a for a in items if a.ndim == 3]
    L_max = max((a.shape[2] for a in items), default=0)
    S = items[0].shape[1] if items else 0
    if any(a.shape[1] != S for a in items):
        raise ValueError("every bucket must hold the same number of draws")
    interior = np.zeros((S, L_max, nb_states), dtype=np.int64)
    censored = np.zeros((S, L_max, nb_states), dtype=np.int64)
    for a in items:
        if a.size == 0:
            continue
        n, _, L = a.shape
        row, length, state, cens = _segments(a.astype(np.int64).reshape(n * S, L))
        draw = row % S
        np.add.at(interior, (draw[~cens], length[~cens] - 1, state[~cens]), 1)
        np.add.at(censored, (draw[cens], length[cens] - 1, state[cens]), 1)
    return interior, censored


def path_segments(paths, nb_states):
    """Run lengths of the MAP segments of ``predict_path``'s paths (host only): ``(interior, censored)``, two int64
    arrays [L_max, nb_states] (L_max: the longest bucket's length).  Row ``n - 1`` counts the segments of n
    localisations, by state (the layout of ``xt_seglen_hist``).  ``interior`` holds the segments whose both ends are
    observed inside the track: the dwell-time histogram to fit.  ``censored`` holds those that touch the first or the
    last localisation of their track, whose true length is unknown (a track without a switch is one censored segment of
    its full length)."""
    items = [np.asarray(a) for a in (paths.values() if isinstance(paths, dict) else paths)]
    L_max = max((a.shape[1] for a in items if a.ndim == 2), default=0)
    interior = np.zeros((L_max, nb_states), dtype=np.int64)
    censored = np.zeros((L_max, nb_states), dtype=np.int64)
    for a in items:
        if a.size == 0:
            continue
        _, length, state, cens = _segments(a.astype(np.int64))
        np.add.at(interior, (length[~cens] - 1, state[~cens]), 1)
        np.add.at(censored, (length[cens] - 1, state[cens]), 1)
    return interior, censored


def transition_summary(preds, pairs):
    """Switching statistics from ``predict_transitions``' outputs (host only).

    Returns ``(expected, TrMat_emp)``: ``expected`` = ``{str(L): float64[n]}``, the expected number of state changes
    of every track (sum over its steps of ``1 - trace(pairs)``); ``TrMat_emp`` = float64[nS, nS], the empirical
    per-step transition matrix ``sum xi[i, j] / sum_(steps) P(s = i)`` over all steps of all tracks, to hold against
    the fitted transition probabilities (rows sum to 1; a state never occupied gives a row of NaN)."""
    expected = {}
    num = den = None
    for k, q in pairs.items():
        q = np.asarray(q, dtype=np.float64)
        nS = q.shape[-1]
        expected[k] = (1.0 - np.trace(q, axis1=-2, axis2=-1)).sum(axis=1)
        if num is None:
            num, den = np.zeros((nS, nS)), np.zeros(nS)
        num += q.sum(axis=(0, 1))
        den += np.asarray(preds[k], dtype=np.float64)[:, :-1].sum(axis=(0, 1))
    if num is None:
        raise ValueError("no tracks")
    with np.errstate(invalid="ignore", divide="ignore"):
        return expected, num / den[:, None]


def _annotate(all_tracks, dt, params, cell_dims, nb_states, frame_len, max_nb_states, threshold, input_LocErr, nb_max, gather,
              kind, n_samples=0, seed=0):
    """Body of predict_Bs ("preds"), predict_transitions ("pairs"), predict_residuals ("resid"), predict_path
    ("path") and sample_paths ("samples", with n_samples and seed): the posteriors and the arrays of that output kind,
    each as a {str(L): array} dictionary."""
    sorted_tracks, l_list = _sorted_buckets(all_tracks)
    keys = [k for k in l_list if len(all_tracks[k]) > 0]
    sorted_LocErrs = [np.asarray(input_LocErr[k], dtype=np.float64) for k in keys] if input_LocErr is not None else None
    sorted_dt = [np.asarray(dt[k], dtype=np.float64) for k in keys] if type(dt) == dict else None
    nb_substeps = 1  # substeps should not impact the step labelling (tracking.py:839)
    if not isinstance(params, Parameters):
        raise TypeError("params must be either of the class 'lmfit.parameter.Parameters' or a dictionary of the relevant parameters")
    nb_max = int(nb_max)
    if nb_max < 1:
        raise ValueError("nb_max must be a positive integer")
    if nb_max > 1 and (input_LocErr is not None or type(dt) == dict):
        raise NotImplementedError("predict_Bs with nb_max > 1 is implemented for scalar LocErr / dt; use nb_max = 1 with "
                                  "peak-wise localisation errors or per-track time steps")
    loc, Ds, Fs, TrMat, pBL = _extract_scalars(params, nb_substeps)
    if len(Ds) != nb_states:
        raise ValueError("nb_states (%d) must equal the number of D parameters (%d)" % (nb_states, len(Ds)))
    d = next((np.shape(a)[2] for a in all_tracks.values() if np.ndim(a) == 3), 0)
    # one track's entry of every returned array, by bucket length
    row_shapes = [lambda L: (L, nb_states)] + {
        "preds": [],
        "pairs": [lambda L: (L - 1, nb_states, nb_states)],
        "resid": [lambda L: (L,), lambda L: (L, d)],
        "path": [lambda L: (L,), lambda L: ()],
        "samples": [lambda L: (n_samples, L), lambda L: (n_samples,)],
    }[kind]
    # the paths and samples are int8 labels (gathered as float64, exact for labels < 2^53, and cast back)
    dtypes = [np.int8 if (kind in ("path", "samples") and i == 1) else np.float64 for i in range(len(row_shapes))]
    outs = [{l: np.empty((0,) + rs(int(l)), dtype=dt_) for l in l_list} for rs, dt_ in zip(row_shapes, dtypes)]
    if not sorted_tracks:
        return tuple(outs)
    for a in sorted_tracks:
        if a.shape[1] < 2:
            raise ValueError("minimal track length = 2, here track length = %s" % a.shape[1])
    min_len, max_len = int(l_list[0]), int(l_list[-1])
    loc_k = 0
    if sorted_LocErrs is not None:
        for a, c in zip(sorted_LocErrs, sorted_tracks):
            if a.ndim != 3 or a.shape[:2] != c.shape[:2] or a.shape[2] not in (1, c.shape[2]):
                raise ValueError("Localization error is not specified correctly: input_LocErr arrays must have shape "
                                 "[n, L, 1] or [n, L, d] matching all_tracks")
        loc_k = sorted_LocErrs[0].shape[2]
    if sorted_dt is not None:
        # one track per chunk (nb_max = 1): every track's own dt[0] sets its field-of-view term (:501-506)
        ds = _median_ds(Ds, np.array(_mid2(sorted_dt[0])))[0]
    else:
        ds = np.sqrt(2 * Ds * dt)
    slope = (params["slope_LocErr"].value, params["offset_LocErr"].value) if (loc_k and _has_slope(params)) else None
    p = build_tables(loc, ds, Fs, TrMat, pBL, cell_dims, nb_substeps, frame_len, min_len, threshold, max_nb_states,
                     sorted_tracks[0].shape[2], var_loc_k=loc_k, var_dt=sorted_dt is not None, Ds=Ds, slope_offset=slope)
    rank, world = _dist_info(None, None)
    cuts = [predict_shard(len(a), rank, world, nb_max) for a in sorted_tracks]
    mine = [b for b, (lo, hi) in enumerate(cuts) if hi > lo]
    loc = lambda arrs: [arrs[b][cuts[b][0]:cuts[b][1]] for b in mine] if arrs is not None else None
    local = [[np.empty((0,) + rs(a.shape[1]), dtype=dt_) for a in sorted_tracks] for rs, dt_ in zip(row_shapes, dtypes)]
    if mine:
        eng = _native.Engine(_default_device())
        try:
            # nb_max = 1: plans are per track and the chunk size only shapes the device layout; nb_max > 1: the chunks
            # of nb_max tracks are the reference's (tracking.py:866-867) and share one plan each
            eng.upload(loc(sorted_tracks), [0 if sorted_tracks[b].shape[1] == max_len else 1 for b in mine],
                       MAX_TRACKS_PER_CHUNK if nb_max == 1 else nb_max)
            eng.set_option("predict_shared_plans", int(nb_max > 1))
            if sorted_LocErrs is not None or sorted_dt is not None:
                eng.upload_aux(loc(sorted_LocErrs), loc(sorted_dt))
            if sorted_dt is not None:
                t0 = np.concatenate([a[:, 0] for a in loc(sorted_dt)])
                eng.set_stay_tables(True, *stay_tables(Ds, np.stack([t0, t0], 1), TrMat, pBL, cell_dims, nb_substeps))
            if kind == "pairs":
                res = eng.predict_pairs(p, nb_states)
            elif kind == "resid":
                res = eng.predict_residuals(p, nb_states)
            elif kind == "path":
                res = eng.predict_path(p, nb_states)
            elif kind == "samples":
                # the draws' Philox counter is the track's row in its whole bucket, not in this rank's slice
                res = eng.predict_samples(p, nb_states, n_samples, seed, [cuts[b][0] for b in mine])
            else:
                res = (eng.predict(p, nb_states),)
            for lo, arrs in zip(local, res):
                for b, x in zip(mine, arrs):
                    lo[b] = x
        finally:
            eng.close()
    for out, lo, rs, dt_ in zip(outs, local, row_shapes, dtypes):
        full = lo if (world == 1 or not gather) else _gather_predictions(lo, sorted_tracks, world, rs, nb_max)
        for a, x in zip(sorted_tracks, full):
            out[str(a.shape[1])] = np.asarray(x).astype(dt_, copy=False)
    return tuple(outs)


# --------------------------------------------------------------------------------------
# parameter builders (host only; tracking.py:1090-1290) and the fit driver (:1299-1386)
# --------------------------------------------------------------------------------------
def generate_params(nb_states=3, LocErr_type=1, nb_dims=3, LocErr_bounds=[0.005, 0.1], D_max=10,
                    Fractions_bounds=[0.001, 0.99], estimated_LocErr=None, estimated_Ds=None, estimated_Fs=None,
                    estimated_transition_rates=0.1, slope_offsets_estimates=None):
    """lmfit ``Parameters`` for an ``nb_states`` model (same names / bounds / exprs as tracking.py:1214-1290)."""
    params = Parameters()
    for s in range(nb_states):
        v = 0.5 * s**2 * D_max / (nb_states - 1) ** 2 if estimated_Ds is None else estimated_Ds[s]
        params.add("D" + str(s), value=v, min=0, max=D_max, vary=True)
    geo = (LocErr_bounds[0] * LocErr_bounds[1]) ** 0.5
    lo, hi = LocErr_bounds
    if LocErr_type == 1:
        params.add("LocErr", value=geo if estimated_LocErr is None else estimated_LocErr[0], min=lo, max=hi, vary=True)
    elif LocErr_type == 2:
        for d in range(nb_dims):
            params.add("LocErr" + str(d), value=geo if estimated_LocErr is None else estimated_LocErr[d], min=lo, max=hi, vary=True)
    elif LocErr_type == 3:
        params.add("LocErr0", value=geo if estimated_LocErr is None else estimated_LocErr[0], min=lo, max=hi, vary=True)
        params.add("LocErr1", expr="LocErr0")
        params.add("LocErr2", value=geo if estimated_LocErr is None else estimated_LocErr[-1], min=lo, max=hi, vary=True)
    if LocErr_type == 4:
        params.add("slope_LocErr", value=slope_offsets_estimates[0], min=-1, max=20, vary=True)
        params.add("offset_LocErr", value=slope_offsets_estimates[1], min=-1, max=1, vary=True)
    F_expr = "1"
    for s in range(nb_states - 1):
        v = 1 / nb_states if estimated_Fs is None else estimated_Fs[s]
        params.add("F" + str(s), value=v, min=Fractions_bounds[0], max=Fractions_bounds[1], vary=True)
        F_expr += " - F" + str(s)
    params.add("F" + str(nb_states - 1), expr=F_expr)
    if not isinstance(estimated_transition_rates, (np.ndarray, list)):
        estimated_transition_rates = [estimated_transition_rates] * (nb_states * (nb_states - 1))
    idx = 0
    for i in range(nb_states):
        for j in range(nb_states):
            if i != j:
                params.add("p" + str(i) + str(j), value=estimated_transition_rates[idx], min=0.0001, max=1, vary=True)
                idx += 1
    params.add("pBL", value=0.1, min=0.0001, max=1, vary=True)
    return params


def get_params(nb_states=2, steady_state=False,
               vary_params={"LocErr": True, "D0": True, "D1": True, "F0": True, "p01": True, "p10": True, "pBL": True},
               estimated_vals={"LocErr": 0.025, "D0": 1e-20, "D1": 0.05, "F0": 0.45, "p01": 0.05, "p10": 0.05, "pBL": 0.1},
               min_values={"LocErr": 0.007, "D0": 1e-12, "D1": 0.00001, "F0": 0.001, "p01": 0.01, "p10": 0.01, "pBL": 0.01},
               max_values={"LocErr": 0.6, "D0": 1, "D1": 10, "F0": 0.999, "p01": 1.0, "p10": 1.0, "pBL": 0.99}):
    """lmfit ``Parameters`` from dictionaries (generic live branch of tracking.py:1164-1212).

    ``nb_states`` and ``steady_state`` are accepted and ignored, as in the reference.
    """
    params = Parameters()
    keys = list(estimated_vals.keys())
    if "slope_LocErr" in keys:
        for n in ("slope_LocErr", "offset_LocErr"):
            params.add(n, value=estimated_vals[n], min=min_values[n], max=max_values[n], vary=vary_params[n])
    if "LocErr" in keys:
        LocErr = estimated_vals["LocErr"]
        if type(LocErr) == float:
            params.add("LocErr", value=LocErr, min=min_values["LocErr"], max=max_values["LocErr"], vary=vary_params["LocErr"])
        elif isinstance(LocErr, (np.ndarray, list)):
            for s in range(len(LocErr)):
                params.add("LocErr" + str(s), value=LocErr[s], min=min_values["LocErr"][s], max=max_values["LocErr"][s],
                           vary=vary_params["LocErr"][s])
    Dn = [k for k in vary_params if k.startswith("D")]
    Fn = [k for k in vary_params if k.startswith("F")]
    params.add("D0", value=estimated_vals["D0"], min=min_values["D0"], max=0.3, brute_step=0.04, vary=vary_params["D0"])
    last_D, sum_Ds, expr = "D0", estimated_vals["D0"], "D0"
    for D in Dn[1:]:
        nm = D + "_minus_" + last_D
        params.add(nm, value=estimated_vals[D] - sum_Ds, min=0, max=max_values[D], vary=vary_params[D])
        expr = expr + "+" + nm
        params.add(D, expr=expr)
        last_D = D
        sum_Ds += estimated_vals[D]
    params.add("F0", value=estimated_vals["F0"], min=min_values["F0"], max=max_values["F0"], brute_step=0.04, vary=vary_params["F0"])
    expr = "1-F0"
    for F in Fn[1 : len(Dn) - 1]:
        params.add(F, value=estimated_vals[F], min=0.001, max=0.99, vary=vary_params[F])
        expr = expr + "-" + F
    params.add("F" + str(len(Dn) - 1), expr=expr)
    for k in vary_params:
        if k.startswith("p"):
            params.add(k, value=estimated_vals[k], min=min_values[k], max=max_values[k], vary=vary_params[k])
    return params


def param_fitting(all_tracks, dt, params=None, nb_states=2, nb_substeps=1, frame_len=6, verbose=1, workers=1,
                  Matrix_type=1, method="bfgs", steady_state=False, cell_dims=[1], input_LocErr=None, threshold=0.2,
                  max_nb_states=120):
    """Maximum-likelihood fit of the model parameters; returns the lmfit result (tracking.py:1299-1386).

    The tracks are packed and uploaded to the GPU once; every objective evaluation then runs
    the plan / replay kernels on the resident data.
    """
    if params is None:
        params = generate_params(nb_states=nb_states, LocErr_type=1, LocErr_bounds=[0.005, 0.1], D_max=3,
                                 Fractions_bounds=[0.001, 0.99], estimated_transition_rates=0.1)
    sorted_tracks, l_list = _sorted_buckets(all_tracks)
    if len(sorted_tracks) < 1:
        raise ValueError("No track could be detected. The loaded tracks seem empty. Errors often come from wrong input paths.")
    keys = [k for k in l_list if len(all_tracks[k]) > 0]
    if input_LocErr is not None:  # dict like all_tracks -> list sorted like the tracks (tracking.py:1351-1366)
        input_LocErr = [np.asarray(input_LocErr[k], dtype=np.float64) for k in keys]
    if type(dt) == dict:
        dt = [np.asarray(dt[k], dtype=np.float64) for k in keys]
    print("cell_dims", cell_dims)
    ts = TrackSet(sorted_tracks, MAX_TRACKS_PER_CHUNK, input_LocErr=input_LocErr, dt_list=dt if type(dt) == list else None,
                  devices=resolve_devices(workers))
    try:
        fit = minimize(cum_Proba_Cs, params,
                       args=(sorted_tracks, dt, cell_dims, input_LocErr, nb_states, nb_substeps, frame_len, verbose, workers,
                             Matrix_type, threshold, max_nb_states),
                       kws={"_trackset": ts}, method=method, nan_policy="propagate")
    finally:
        ts.close()
    if verbose == 0:
        print("")
    return fit


def get_2DSPT_params(all_tracks, dt, nb_substeps=1, nb_states=2, frame_len=8, verbose=1, workers=1, method="powell",
                     steady_state=False, cell_dims=[1],
                     vary_params={"LocErr": True, "D0": True, "D1": True, "F0": True, "p01": True, "p10": True, "pBL": True},
                     estimated_vals={"LocErr": 0.025, "D0": 1e-20, "D1": 0.05, "F0": 0.45, "p01": 0.05, "p10": 0.05, "pBL": 0.1},
                     min_values={"LocErr": 0.007, "D0": 1e-12, "D1": 0.00001, "F0": 0.001, "p01": 0.01, "p10": 0.01, "pBL": 0.01},
                     max_values={"LocErr": 0.6, "D0": 1, "D1": 10, "F0": 0.999, "p01": 1.0, "p10": 1.0, "pBL": 0.99}):
    """Legacy entry point (``old_tracking.py:585-674``) kept as a wrapper: builds the parameters
    with ``get_params`` and runs ``param_fitting`` on the current likelihood engine."""
    params = get_params(nb_states, steady_state, vary_params, estimated_vals, min_values, max_values)
    return param_fitting(all_tracks, dt, params=params, nb_states=nb_states, nb_substeps=nb_substeps, frame_len=frame_len,
                         verbose=verbose, workers=workers, method=method, steady_state=steady_state, cell_dims=cell_dims)


# --------------------------------------------------------------------------------------
# standard errors of fitted parameters (frozen-plan scores and observed information)
# --------------------------------------------------------------------------------------
@dataclass
class ParamUncertainty:
    """Result of ``param_uncertainty``.  Matrices are over ``names`` (free parameters with a usable step), in order.

    ``hessian``: observed information H (Hessian of -log L); ``opg``: J = sum over tracks of g g^T (per-track scores g);
    ``gradient``: sum of g (gradient of log L); ``newton_decrement``: g^T H^-1 g (near 0 at a converged fit);
    ``covar`` = H^-1, ``covar_robust`` = H^-1 J H^-1 (sandwich, valid under misspecification); ``stderr`` /
    ``stderr_robust``: per parameter name (NaN for ``at_bound``, None for ``vary=False``; ``expr`` parameters by the
    delta method); ``correl``: correlation matrix of ``covar``; ``params``: a copy with ``.stderr`` / ``.correl`` set."""

    names: List[str]
    at_bound: List[str]
    hessian: np.ndarray
    opg: np.ndarray
    gradient: np.ndarray
    newton_decrement: float
    covar: np.ndarray
    covar_robust: np.ndarray
    stderr: Dict[str, Optional[float]]
    stderr_robust: Dict[str, Optional[float]]
    correl: np.ndarray
    params: object
    n_evaluations: int = 0


class InvalidPoint(Exception):
    """Raised by an uncertainty backend when parameter list entry ``index`` fails the objective's validity guard."""

    def __init__(self, index: int):
        super().__init__(index)
        self.index = index


def uncertainty_from_backend(params, totals, score_outer, rel_step: float = 1e-4) -> ParamUncertainty:
    """Standard errors by central differences of a smooth log-likelihood surface, given by two callables:

    * ``totals(thetas)`` -> float64[len(thetas)]: sum of log P at every free-parameter vector;
    * ``score_outer(th_plus, th_minus, inv_2h)`` -> dict ``sum_plus``, ``sum_minus``, ``gsum``, ``gram`` (see
      ``xt_score_outer``).

    Either may raise ``InvalidPoint(index)``.  Vectors are over the free parameters with a usable step (``names``).
    The engine along a frozen plan is the production backend; tests drive this with oracles and synthetic surfaces."""
    import warnings

    names_all = list(params.keys())
    free = [n for n in names_all if params[n].vary and params[n].expr is None]
    act, held, h = [], [], []
    for n in free:
        if _held(params[n], rel_step):
            held.append(n)
        else:
            act.append(n)
            h.append(rel_step * abs(float(params[n].value)))
    m = len(act)
    if m > _native.XT_MAX_SCORE_DIRS:
        raise ValueError("param_uncertainty: at most %d free parameters" % _native.XT_MAX_SCORE_DIRS)
    h = np.array(h, dtype=float)
    theta = np.array([float(params[n].value) for n in act])
    E = np.eye(m) * h[:, None] if m else np.zeros((0, 0))

    def run(fn, describe, *args):
        try:
            return fn(*args)
        except InvalidPoint as e:
            raise ValueError("param_uncertainty: the step of %s leaves the region the objective accepts (the "
                             "parameter guard rejects the perturbed point)" % describe(e.index)) from None

    plus, minus = [theta + E[i] for i in range(m)], [theta - E[i] for i in range(m)]
    sc = run(score_outer, lambda k: act[k % m], plus, minus, 1.0 / (2.0 * h)) if m else None
    pts, who = [theta], [None]
    for i in range(m):
        for j in range(i + 1, m):
            for si, sj in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                pts.append(theta + si * E[i] + sj * E[j])
                who.append((i, j))
    S = run(totals, lambda k: "%s / %s" % (act[who[k][0]], act[who[k][1]]) if who[k] else "the estimate", pts)
    S0 = S[0]
    H = np.zeros((m, m))
    k = 1
    for i in range(m):
        H[i, i] = -(sc["sum_plus"][i] - 2.0 * S0 + sc["sum_minus"][i]) / (h[i] * h[i])
        for j in range(i + 1, m):
            spp, spm, smp, smm = S[k:k + 4]
            H[i, j] = H[j, i] = -(spp - spm - smp + smm) / (4.0 * h[i] * h[j])
            k += 4
    J = np.array(sc["gram"], dtype=float) if m else np.zeros((0, 0))
    g = np.array(sc["gsum"], dtype=float) if m else np.zeros(0)
    try:
        np.linalg.cholesky(H)
        cov = np.linalg.inv(H)
        cov = (cov + cov.T) / 2
        newton = float(g @ cov @ g)
    except np.linalg.LinAlgError:
        warnings.warn("param_uncertainty: the observed information is not positive definite (not at a maximum, or "
                      "a parameter is not identified); covariances are NaN", RuntimeWarning, stacklevel=2)
        cov = np.full((m, m), np.nan)
        newton = float("nan")
    rob = cov @ J @ cov
    out_params = params.copy()

    def delta(C):
        """stderr of every parameter from the covariance C of ``act``; expr parameters by the delta method."""
        se: Dict[str, Optional[float]] = {}
        for n in names_all:
            p = params[n]
            if n in act:
                se[n] = float(np.sqrt(C[act.index(n), act.index(n)]))
            elif n in held:
                se[n] = float("nan")
            elif p.expr is None:
                se[n] = None
            else:
                jac = np.zeros(m)
                for i, a in enumerate(act):  # numerical Jacobian of the expression (held parameters stay fixed)
                    q = params.copy()
                    q[a].value = theta[i] + h[i]
                    vp = float(q[n].value)
                    q[a].value = theta[i] - h[i]
                    jac[i] = (vp - float(q[n].value)) / (2.0 * h[i])
                se[n] = float(np.sqrt(jac @ C @ jac))
        return se

    se, se_r = delta(cov), delta(rob)
    sd = np.sqrt(np.diag(cov))
    correl = cov / np.outer(sd, sd) if m else np.zeros((0, 0))
    for n in names_all:
        out_params[n].stderr = se[n]
        if n in act:
            i = act.index(n)
            out_params[n].correl = {b: float(correl[i, j]) for j, b in enumerate(act) if j != i}
    return ParamUncertainty(act, held, H, J, g, newton, cov, rob, se, se_r, correl, out_params, 1 + 2 * m + len(pts))


def param_uncertainty(all_tracks, dt, params, nb_states=2, nb_substeps=1, frame_len=6, workers=1, Matrix_type=1,
                      cell_dims=[1], input_LocErr=None, threshold=0.2, max_nb_states=120, rel_step=1e-4) -> ParamUncertainty:
    """Standard errors of fitted parameters (``params`` = ``fit.params`` or the ``param_fitting`` result itself).

    Takes ``param_fitting``'s data arguments.  The objective is evaluated once at the estimate to build the grouping
    plan; everything else runs along that frozen plan, where log P of every track is a smooth function of the
    parameters.  Central differences (step ``rel_step * |value|``) give per-track scores and the observed information;
    see ``ParamUncertainty`` and DESIGN.md §9.  A parameter whose value is 0, or within two steps of a bound, is held
    fixed (listed in ``at_bound``, stderr NaN).  A ``dt`` dictionary is not supported: its field-of-view tables depend
    on D and are per-chunk state of the engine."""
    params = getattr(params, "params", params)
    if isinstance(params, dict) and not hasattr(params, "valuesdict"):
        raise TypeError("params must be lmfit Parameters or a fit result")
    if type(dt) in (dict, list):
        raise NotImplementedError("param_uncertainty: per-localisation dt (a dt dictionary) is not supported: the "
                                  "field-of-view tables it needs depend on D and are per-chunk engine state")
    sorted_tracks, l_list = _sorted_buckets(all_tracks)
    if len(sorted_tracks) < 1:
        raise ValueError("No track could be detected. The loaded tracks seem empty. Errors often come from wrong input paths.")
    keys = [k for k in l_list if len(all_tracks[k]) > 0]
    if input_LocErr is not None:
        input_LocErr = [np.asarray(input_LocErr[k], dtype=np.float64) for k in keys]
    ts = TrackSet([np.asarray(a, dtype=np.float64) for a in sorted_tracks], MAX_TRACKS_PER_CHUNK,
                  input_LocErr=input_LocErr, precision="fp64", devices=resolve_devices(workers))
    try:
        # the free parameters the assembly steps (same rule, _held) name the entries of its vectors
        act = [n for n in params.keys() if params[n].vary and params[n].expr is None and not _held(params[n], rel_step)]

        def tables(thetas):
            out = []
            for k, th in enumerate(thetas):
                q = params.copy()
                for n, v in zip(act, th):
                    q[n].value = float(v)
                p, _ = _objective_tables(q, ts, dt, cell_dims, nb_substeps, frame_len, threshold, max_nb_states, Matrix_type)
                if p is None:
                    raise InvalidPoint(k)
                out.append(p)
            return out

        p_hat, _ = _objective_tables(params, ts, dt, cell_dims, nb_substeps, frame_len, threshold, max_nb_states, Matrix_type)
        if p_hat is None:
            raise ValueError("param_uncertainty: the parameters fail the objective's validity guard")
        ts.sum_logp(p_hat)  # the grouping plan at the estimate (every later evaluation runs along it)
        totals = lambda thetas: ts.eval_frozen(tables(thetas))
        score = lambda plus, minus, inv_2h: ts.score_outer(tables(plus), tables(minus), inv_2h)
        return uncertainty_from_backend(params, totals, score, rel_step)
    finally:
        ts.close()


def _held(p, rel_step) -> bool:
    v = float(p.value)
    step = rel_step * abs(v)
    return v == 0.0 or v - 2 * step < p.min or v + 2 * step > p.max
