"""TEST INFRASTRUCTURE ONLY — CPU (numpy, FP64) most probable state paths (MAP / Viterbi paths) of ExTrack's
annotation recursion.

``extrack_oracle.chunk_recursion(do_preds=1)`` is a lattice:

* every expansion gives each child one parent;
* every fusion gives each member a normalised merge weight ``w`` inside its group (``_merge``);
* the final sequences get ``softmax(LP)`` (the bleaching end sums each sequence's hidden heads, the engine's ``Lsum``).

A *route* is a path from an initial sequence to a final one.  Its weight is the final softmax weight times the product
of the member weights ``w`` along it.  Route weights sum to 1, and summed by label they are ``predict_states``'
posteriors.  **The MAP path of a track is the label sequence of its heaviest route**, and ``path_logp`` is the log of
that route's weight.

As a forward recursion: every live sequence carries a score ``V``, updated exactly like its log-weight ``LP``, except
that a fusion sets the group's ``V`` to the *maximum* of its members' ``V`` (``LP``: their log-sum-exp), ties to the
first member.  At the end of the track the route is chosen by ``V`` plus the end term ``LP`` receives (the bleaching
end's log-sum over hidden heads included), ties to the lowest index, and ``path_logp = V* - logsumexp(final LP)``.  By
telescoping (``LP_group - LP_member = -log w_member``) this is the log route weight above.  Hence:

* without fusion ``V = LP`` for every sequence: the path is the exact argmax over all state sequences and ``path_logp``
  its exact posterior log-probability;
* ``path_logp <= 0`` and ``path_logp <= log preds[t, k, path[t, k]]`` for every k (a route's weight never exceeds the
  marginal of a label on it).

Labels are the history labels of the posteriors: the child index mod nS with the int8 wrap of tracking.py:543 in the
default bug-compatible mode.  The *decision margin* of a track is the smallest gap in score between the chosen
candidate and the runner-up over the argmax decisions on its chosen route (every fusion it passes through with two or
more members, and the final choice); a test comparing paths computed in another arithmetic needs it well above the
rounding.  This module runs the same steps as ``chunk_recursion`` (its tables, label wrap, ``_plan_groups`` and
``_merge``, operation for operation, so the posteriors are bitwise equal to ``predict_states``).  Only
``nb_substeps = 1`` exists here (predict_Bs forces it, tracking.py:839).  The product (``extrack_b200``) never imports
this module.
"""
from __future__ import annotations

from typing import List

import numpy as np

from oracle.extrack_oracle import HeadTables, Model, _label, _merge, _plan_groups


def _lse(x, axis):
    """log-sum-exp as the engine computes it: max + log(sum(exp(x - max)))."""
    mx = np.max(x, axis=axis, keepdims=True)
    return (np.log(np.sum(np.exp(x - mx), axis=axis, keepdims=True)) + mx).squeeze(axis)


def _best(score):
    """Per row of score [nT, n]: the argmax (first on ties), its value and the gap to the runner-up (inf for n = 1)."""
    j = np.argmax(score, axis=1)
    top = score[np.arange(len(score)), j]
    if score.shape[1] < 2:
        return j, top, np.full(len(score), np.inf)
    return j, top, top - np.sort(score, axis=1)[:, -2]


def chunk_recursion_path(C, model: Model, isBL: int, tables=None, sig=None, ds3=None):
    """``extrack_oracle.chunk_recursion(C, model, isBL, do_preds=1, ...)`` plus the MAP paths.

    Returns (LP [nT, nB], preds [nT, L, nS], path int8 [nT, L], path_logp [nT], margin [nT]), forward time."""
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
    rows = np.arange(nT)

    # ---- first localisation: initial sequence h = h0 + nS*h1, forward-time labels (h1, h0) ----
    nB = K * nS
    head = np.arange(nB)
    cur = tb.digits[head, 0].copy()
    hist = (tb.digits[head][None, :, :, None] == np.arange(nS)[None, None, None, :]).astype(np.float64)
    LP = np.repeat((tb.LT[head] + tb.LF[head])[None], nT, axis=0)
    s2 = l2 + dd_at(L - 1, head)
    m = np.repeat(C[:, None, 0, :], nB, axis=1)
    V = LP.copy()
    route = np.repeat(tb.digits[head][:, ::-1][None], nT, axis=0)  # [nT, nB, rows so far]
    margin = np.full((nT, nB), np.inf)  # smallest decision gap along each sequence's best route

    def expand(cur, hist):
        n = len(cur) * nS
        lab = _label(np.arange(n), nS, model.int8_wrap)
        new_row = np.repeat((lab[None, :, None, None] == np.arange(nS)[None, None, None, :]).astype(np.float64), hist.shape[0], 0)
        hist = np.concatenate((new_row, np.repeat(hist, nS, 1)), -2)
        child = np.arange(n)
        return (child % K) + K * cur[child // K], child % nS, hist, lab

    for step in range(2, L):  # consumes localisation step - 1
        head, cur, hist, lab = expand(cur, hist)
        dd = dd_at(L - step, head)
        l2 = l2_at(step - 1)
        m = np.repeat(m, K, axis=1)
        s2 = np.repeat(s2, K, axis=1)
        LP = np.repeat(LP, K, axis=1)
        V = np.repeat(V, K, axis=1)
        route = np.concatenate((np.repeat(route, K, axis=1), np.broadcast_to(lab[None, :, None], (nT, len(lab), 1))), 2)
        margin = np.repeat(margin, K, axis=1)
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
        V = V + (tb.LT[head][None] + LC + LL)
        nB = len(cur)
        if nB > model.max_nb_states:
            th = th * 1.2
        if step < L - 1:
            groups = _plan_groups(m, s2, hist, frame_len, th)
            gV = np.empty((nT, len(groups)))
            groute = np.empty((nT, len(groups), route.shape[2]), dtype=route.dtype)
            gmar = np.empty((nT, len(groups)))
            for g, mem in enumerate(groups):  # the group keeps its best member's route
                j, gV[:, g], gap = _best(V[:, mem])
                groute[:, g] = route[rows, mem[j]]
                gmar[:, g] = np.minimum(margin[rows, mem[j]], gap)
            V, route, margin = gV, groute, gmar
            m, s2, LP, cur, hist = _merge(m, s2, LP, cur, hist, groups, nT, frame_len, 1)

    # ---- end of track (tracking.py:613-639); the route choice sums the bleaching end's hidden heads ----
    l2e = l2_at(L - 1)
    qe = s2 + l2e
    term_seq = np.sum(-0.5 * np.log(2 * np.pi * qe) - (C[:, None, L - 1, :] - m) ** 2 / (2 * qe), axis=2)
    score = V + term_seq
    if isBL:
        child = np.arange(len(cur) * K)
        leave = tb.L_leave[(child % K) + K * cur[child // K]].reshape(len(cur), K)
        score = score + _lse(leave, 1)[None]
        head, cur, hist, _ = expand(cur, hist)
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
    LP = LP + (term + LL)

    pLP = LP
    if np.max(LP) > 600:
        pLP = LP - (np.max(LP) - 600)
    P = np.exp(pLP)
    sP = np.sum(P, axis=1, keepdims=True)[:, :, None]
    preds = np.sum(P[:, :, None, None] * hist, axis=1) / sP

    j, top, gap = _best(score)
    path = route[rows, j].astype(np.int8)
    path_logp = top - _lse(LP, 1)
    return LP, preds[:, ::-1], path, path_logp, np.minimum(margin[rows, j], gap)


def predict_path(sorted_tracks: List[np.ndarray], model: Model, nb_max: int = 1, sigs=None, ds_list=None):
    """``extrack_oracle.predict_states`` with the MAP paths: per bucket ``(preds [n, L, nS], path int8 [n, L],
    path_logp [n], margin [n])``."""
    max_len = sorted_tracks[-1].shape[1]
    tables = HeadTables(model)
    out = []
    for b, arr in enumerate(sorted_tracks):
        isBL = 0 if arr.shape[1] == max_len else 1
        parts = []
        for n in range(int(np.ceil(len(arr) / nb_max))):
            sl = slice(n * nb_max, (n + 1) * nb_max)
            parts.append(chunk_recursion_path(arr[sl], model, isBL, tables, None if sigs is None else sigs[b][sl],
                                              None if ds_list is None else ds_list[b][sl])[1:])
        L = arr.shape[1]
        out.append(tuple(np.concatenate(x) for x in zip(*parts)) if parts
                   else (np.empty((0, L, model.nS)), np.empty((0, L), dtype=np.int8), np.empty(0), np.empty(0)))
    return out
