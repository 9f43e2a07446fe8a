"""TEST INFRASTRUCTURE ONLY — CPU (numpy, FP64) two-slice state posteriors along ExTrack's annotation recursion.

``extrack_oracle.chunk_recursion(do_preds=1)`` carries, for every live sequence, a history ``hist[nT, nB, L, nS]``:
one-hot rows prepended at every expansion (with the int8 label wrap of tracking.py:543), rows averaged with the merge
weights at every fusion, and ``preds = sum P * hist / sum P``.  This module restates that recursion with a second,
*pair* history ``hist2[nT, nB, L - 1, nS, nS]`` carried through exactly the same operations:

* expansion: prepend ``outer(hist[:, parent, 0, :], onehot(label(child)))`` (the parent's newest row, which may be a
  mixture after a fusion, paired with the child's new label);
* fusion: the same weighted average as ``hist`` (``extrack_oracle._merge``), a copy for one-member groups;
* end of track with ``isBL``: the newest pair row is dropped as ``hist[:, :, 1:]`` drops the newest row;
* output: ``pairs = sum P * hist2 / sum P`` with the same ``max(LP) > 600`` shift as ``preds``, in forward time.

``pairs[t, k, i, j]`` is then P(state i at localisation k, state j at localisation k + 1 | track); its sums over ``j``
and ``i`` are ``preds[:, :-1]`` and ``preds[:, 1:]``.  Only ``nb_substeps = 1`` exists here (predict_Bs forces it,
tracking.py:839).  The product (``extrack_b200``) never imports this module.
"""
from __future__ import annotations

from typing import List

import numpy as np

from oracle.extrack_oracle import HeadTables, Model, _label, _merge, _plan_groups


def _onehot(labels: np.ndarray, nS: int) -> np.ndarray:
    return (labels[..., None] == np.arange(nS)).astype(np.float64)


def chunk_recursion_pairs(C, model: Model, isBL: int, tables=None, sig=None, ds3=None):
    """``extrack_oracle.chunk_recursion(C, model, isBL, do_preds=1, ...)`` plus the pair history.

    Returns (LP [nT, nB], preds [nT, L, nS], pairs [nT, L - 1, nS, nS]), forward time."""
    C = np.asarray(C, dtype=np.float64)
    nT, L, d = C.shape
    if L < 2:
        raise ValueError("minimal track length = 2, here track length = %s" % L)
    if model.nb_substeps != 1:
        raise ValueError("state annotation runs with nb_substeps = 1 (tracking.py:839)")
    nS = model.nS
    if ds3 is not None:
        ds3 = np.asarray(ds3, dtype=np.float64)
        tb = HeadTables(model, np.median(ds3[:, 0], axis=0))
    else:
        tb = tables if tables is not None else HeadTables(model)
    K = tb.K
    if sig is not None:
        sig2 = np.asarray(sig, dtype=np.float64) ** 2
        if sig2.ndim != 3 or sig2.shape[1] != L or sig2.shape[2] not in (1, d):
            raise ValueError("Localization error is not specified correctly")
        l2_at = lambda j: sig2[:, None, j, :]
    else:
        l2c = (np.asarray(model.loc_err, dtype=np.float64).reshape(-1) ** 2)[None, None, :]
        if l2c.shape[2] not in (1, d):
            raise ValueError("Localization error is not specified correctly")
        l2_at = lambda j: l2c

    def dd_at(col, head):
        if ds3 is None:
            return tb.dd[head][None, :, None]
        d2 = ds3[:, col, :][:, tb.digits[head]] ** 2
        pair = (d2[:, :, 1:] + d2[:, :, :-1]) / 2
        return np.mean(pair, axis=2)[:, :, None]

    l2 = l2_at(0)
    th = float(model.threshold)
    frame_len = int(model.frame_len)

    # ---- first localisation: two states per sequence, row 0 = newest (digit 0), row 1 = digit 1 ----
    nB = K * nS
    head = np.arange(nB)
    cur = tb.digits[head, 0].copy()
    hist = _onehot(tb.digits[head], nS)[None]  # [1, nB, 2, nS] (per track from the first fusion on, as in chunk_recursion)
    hist2 = (hist[:, :, 1, :, None] * hist[:, :, 0, None, :])[:, :, None]  # [1, nB, 1, nS, nS]: (older, newer)
    LP = np.repeat((tb.LT[head] + tb.LF[head])[None], nT, axis=0)
    s2 = l2 + dd_at(L - 1, head)
    m = np.repeat(C[:, None, 0, :], nB, axis=1)

    def expand(cur, hist, hist2):
        n = len(cur) * nS
        new_row = np.repeat(_onehot(_label(np.arange(n), nS, model.int8_wrap), nS)[None, :, None, :], hist.shape[0], 0)
        par_new = np.repeat(hist[:, :, 0, :], nS, 1)  # [nT, n, nS]: the parent's newest row
        new_pair = (par_new[:, :, :, None] * new_row[:, :, 0, None, :])[:, :, None]
        hist = np.concatenate((new_row, np.repeat(hist, nS, 1)), -2)
        hist2 = np.concatenate((new_pair, np.repeat(hist2, nS, 1)), -3)
        child = np.arange(n)
        return (child % K) + K * cur[child // K], child % nS, hist, hist2

    def merge_pairs(LP, hist2, groups):
        # the weighted average of _merge over the flattened (i, j) axis (history rows are merged with trailing dims [R, S])
        R = hist2.shape[2]
        flat = hist2.reshape(hist2.shape[:3] + (nS * nS,))
        return _merge(m, s2, LP, cur, flat, groups, nT, frame_len, 1)[4].reshape(nT, len(groups), R, nS, nS)

    for step in range(2, L):
        head, cur, hist, hist2 = expand(cur, hist, hist2)
        dd = dd_at(L - step, head)
        l2 = l2_at(step - 1)
        m = np.repeat(m, K, axis=1)
        s2 = np.repeat(s2, K, axis=1)
        LP = np.repeat(LP, K, axis=1)
        c = C[:, None, step - 1, :]
        q = l2 + s2
        new_m = (m * l2 + c * s2) / (l2 + s2)
        new_s2 = (dd * l2 + dd * s2 + l2 * s2) / q
        if s2.shape[2] == 1:
            LC = d * -0.5 * np.log(2 * np.pi * q[:, :, 0]) - np.sum((c - m) ** 2 / (2 * q), axis=2)
        else:
            LC = np.sum(-0.5 * np.log(2 * np.pi * q), 2) - np.sum((c - m) ** 2 / (2 * q), axis=2)
        m, s2 = new_m, new_s2
        LL = tb.Lp_stay[head % K] if step >= model.min_len else 0
        LP = LP + (tb.LT[head][None] + LC + LL)
        nB = len(cur)
        if nB > model.max_nb_states:
            th = th * 1.2
        if step < L - 1:
            groups = _plan_groups(m, s2, hist, frame_len, th)
            hist2 = merge_pairs(LP, hist2, groups)
            m, s2, LP, cur, hist = _merge(m, s2, LP, cur, hist, groups, nT, frame_len, 1)

    # ---- end of track (tracking.py:613-639) ----
    if isBL:
        head, cur, hist, hist2 = expand(cur, hist, hist2)
        m = np.repeat(m, K, axis=1)
        s2 = np.repeat(s2, K, axis=1)
        LP = np.repeat(LP, K, axis=1)
        LL = tb.L_leave[head][None]
        hist = hist[:, :, 1:]
        hist2 = hist2[:, :, 1:]
    else:
        LL = 0
    l2 = l2_at(L - 1)
    q = s2 + l2
    term = np.sum(-0.5 * np.log(2 * np.pi * q) - (C[:, None, L - 1, :] - m) ** 2 / (2 * q), axis=2)
    LP = LP + (term + LL)

    pLP = LP
    if np.max(LP) > 600:
        pLP = LP - (np.max(LP) - 600)
    P = np.exp(pLP)
    sP = np.sum(P, axis=1, keepdims=True)[:, :, None]
    preds = np.sum(P[:, :, None, None] * hist, axis=1) / sP
    pairs = np.sum(P[:, :, None, None, None] * hist2, axis=1) / sP[:, :, :, None]
    return LP, preds[:, ::-1], pairs[:, ::-1]


def predict_pairs(sorted_tracks: List[np.ndarray], model: Model, nb_max: int = 1, sigs=None, ds_list=None):
    """``extrack_oracle.predict_states`` with the two-slice posteriors: per bucket ``(preds [n, L, nS],
    pairs [n, L - 1, nS, nS])``."""
    max_len = sorted_tracks[-1].shape[1]
    tables = HeadTables(model)
    out = []
    for b, arr in enumerate(sorted_tracks):
        isBL = 0 if arr.shape[1] == max_len else 1
        ps, qs = [], []
        for n in range(int(np.ceil(len(arr) / nb_max))):
            sl = slice(n * nb_max, (n + 1) * nb_max)
            _, p, q = chunk_recursion_pairs(arr[sl], model, isBL, tables, None if sigs is None else sigs[b][sl],
                                            None if ds_list is None else ds_list[b][sl])
            ps.append(p)
            qs.append(q)
        L = arr.shape[1]
        out.append((np.concatenate(ps) if ps else np.empty((0, L, model.nS)),
                    np.concatenate(qs) if qs else np.empty((0, L - 1, model.nS, model.nS))))
    return out
