"""TEST INFRASTRUCTURE ONLY — CPU (numpy, FP64) one-step-ahead residuals along ExTrack's annotation recursion.

``extrack_oracle.chunk_recursion(do_preds=1)`` consumes localisation ``c_k`` (k >= 1) at one step: the loop step
``k + 1`` for ``k <= L - 2``, the end of the track for ``k = L - 1``.  After that step's expansion and update, before any
fusion, every live sequence ``j`` has

* ``LC_j``: the Gaussian term of ``c_k`` the step adds (the reference's ``LC`` / end ``term``), with variance
  ``q_j = l2 + s2_j`` around its parent's mean ``m_j``;
* ``A_j``: its log-weight after the step minus ``LC_j`` (the parent's fused log-weight plus ``LT[head]`` plus the
  field-of-view term, or at a bleaching end ``L_leave[head]``).

The mixture ``sum_j softmax(A)_j N(m_j, q_j)`` is the model's predictive distribution of ``c_k`` given
``c_0 .. c_k-1``, so

    logpred[t, k] = logsumexp_j(A_j + LC_j) - logsumexp_j(A_j)
    pit[t, k, x]  = sum_j softmax(A)_j Phi((c_k,x - m_j,x) / sqrt(q_j,kappa(x)))

with ``kappa(x) = 0`` for one LocErr component and ``x`` otherwise; entry ``k = 0`` is NaN.  This module runs the same
steps as ``chunk_recursion`` (its tables, label wrap, ``_plan_groups`` and ``_merge``, operation for operation, so the
posteriors are bitwise equal to ``predict_states``) and reads the residuals off each step.  Only ``nb_substeps = 1``
exists here (predict_Bs forces it, tracking.py:839).  The product (``extrack_b200``) never imports this module.
"""
from __future__ import annotations

from typing import List

import numpy as np
from scipy.special import logsumexp, ndtr

from oracle.extrack_oracle import HeadTables, Model, _label, _merge, _plan_groups


def _residual(c, m, q, A, LC):
    """logpred [nT] and pit [nT, d] of localisation c [nT, 1, d] under the sequences (m [nT, nB, d], q [., nB, k],
    A / LC [nT, nB])."""
    d = m.shape[2]
    lp = logsumexp(A + LC, axis=1) - logsumexp(A, axis=1)
    w = np.exp(A - logsumexp(A, axis=1, keepdims=True))
    qx = q if q.shape[2] == d else np.repeat(q, d, axis=2)
    pit = np.sum(w[:, :, None] * ndtr((c - m) / np.sqrt(qx)), axis=1)
    return lp, pit


def chunk_recursion_resid(C, model: Model, isBL: int, tables=None, sig=None, ds3=None):
    """``extrack_oracle.chunk_recursion(C, model, isBL, do_preds=1, ...)`` plus the residuals.

    Returns (LP [nT, nB], preds [nT, L, nS], logpred [nT, L], pit [nT, L, d]), forward time."""
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

    logpred = np.full((nT, L), np.nan)
    pit = np.full((nT, L, d), np.nan)
    l2 = l2_at(0)
    th = float(model.threshold)
    frame_len = int(model.frame_len)

    nB = K * nS
    head = np.arange(nB)
    cur = tb.digits[head, 0].copy()
    hist = (tb.digits[head][None, :, :, None] == np.arange(nS)[None, None, None, :]).astype(np.float64)
    LP = np.repeat((tb.LT[head] + tb.LF[head])[None], nT, axis=0)
    s2 = l2 + dd_at(L - 1, head)
    m = np.repeat(C[:, None, 0, :], nB, axis=1)

    def expand(cur, hist):
        n = len(cur) * nS
        lab = _label(np.arange(n), nS, model.int8_wrap)
        new_row = np.repeat((lab[None, :, None, None] == np.arange(nS)[None, None, None, :]).astype(np.float64), hist.shape[0], 0)
        hist = np.concatenate((new_row, np.repeat(hist, nS, 1)), -2)
        child = np.arange(n)
        return (child % K) + K * cur[child // K], child % nS, hist

    for step in range(2, L):  # consumes localisation step - 1
        head, cur, hist = expand(cur, hist)
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
        LL = tb.Lp_stay[head % K] if step >= model.min_len else 0
        logpred[:, step - 1], pit[:, step - 1] = _residual(c, m, q, LP + tb.LT[head][None] + LL, LC)
        m, s2 = new_m, new_s2
        LP = LP + (tb.LT[head][None] + LC + LL)
        nB = len(cur)
        if nB > model.max_nb_states:
            th = th * 1.2
        if step < L - 1:
            groups = _plan_groups(m, s2, hist, frame_len, th)
            m, s2, LP, cur, hist = _merge(m, s2, LP, cur, hist, groups, nT, frame_len, 1)

    if isBL:
        head, cur, hist = expand(cur, hist)
        m = np.repeat(m, K, axis=1)
        s2 = np.repeat(s2, K, axis=1)
        LP = np.repeat(LP, K, axis=1)
        LL = tb.L_leave[head][None]
        hist = hist[:, :, 1:]
    else:
        LL = 0
    l2 = l2_at(L - 1)
    q = s2 + l2
    term = np.sum(-0.5 * np.log(2 * np.pi * q) - (C[:, None, L - 1, :] - m) ** 2 / (2 * q), axis=2)
    logpred[:, L - 1], pit[:, L - 1] = _residual(C[:, None, L - 1, :], m, q, LP + LL, term)
    LP = LP + (term + LL)

    pLP = LP
    if np.max(LP) > 600:
        pLP = LP - (np.max(LP) - 600)
    P = np.exp(pLP)
    sP = np.sum(P, axis=1, keepdims=True)[:, :, None]
    preds = np.sum(P[:, :, None, None] * hist, axis=1) / sP
    return LP, preds[:, ::-1], logpred, pit


def predict_residuals(sorted_tracks: List[np.ndarray], model: Model, nb_max: int = 1, sigs=None, ds_list=None):
    """``extrack_oracle.predict_states`` with the residuals: per bucket ``(preds [n, L, nS], logpred [n, L],
    pit [n, L, d])``."""
    max_len = sorted_tracks[-1].shape[1]
    tables = HeadTables(model)
    out = []
    for b, arr in enumerate(sorted_tracks):
        isBL = 0 if arr.shape[1] == max_len else 1
        parts = []
        for n in range(int(np.ceil(len(arr) / nb_max))):
            sl = slice(n * nb_max, (n + 1) * nb_max)
            parts.append(chunk_recursion_resid(arr[sl], model, isBL, tables, None if sigs is None else sigs[b][sl],
                                               None if ds_list is None else ds_list[b][sl])[1:])
        n, L, d = arr.shape
        out.append(tuple(np.concatenate(x) for x in zip(*parts)) if parts
                   else (np.empty((0, L, model.nS)), np.empty((0, L)), np.empty((0, L, d))))
    return out
