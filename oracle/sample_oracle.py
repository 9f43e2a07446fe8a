"""TEST INFRASTRUCTURE ONLY — CPU (numpy, FP64) posterior samples of whole state paths along ExTrack's annotation
recursion (forward filtering, backward sampling).

``extrack_oracle.chunk_recursion(do_preds=1)`` is a lattice (see ``path_oracle``): every expansion gives each child one
parent (child c of the sequences before it has parent c // K), every fusion gives each member a normalised merge weight
``w`` inside its group (``_merge``), and the final sequences get ``softmax(LP)`` (the bleaching end sums each sequence's
hidden heads, the engine's ``Lsum``).  A route from an initial to a final sequence weighs its final weight times the
product of the ``w`` along it; the route weights sum to 1.

A draw picks a route with probability equal to its weight, from the end backwards:

1. the final sequence c, among the final sequences in ascending index, with the final weights;
2. for s = L-1 down to 3: label(c) at localisation s, then one member of the parent group c // K of the fusion at step
   s - 1, with the members' normalised weights, in member order (``_plan_groups``' order);
3. at s = 2: label(c) at localisation 2; the parent c // K is the initial sequence h0 + nS*h1 (h0 at localisation 1, h1
   at 0).  With L = 2 the final choice picks the initial sequence directly.

A choice among n >= 2 candidates of weights w_0..w_n-1 takes the first k with ``u * S < cum_k`` (cum: the running FP64
sums in that order, S = cum_n-1); if rounding leaves none, the last candidate of positive weight.  A single candidate
consumes no random number.  ``u`` is ``((x0 << 32 | x1) >> 11) * 2^-53`` from Philox4x32-10 (``philox4x32_10``) with
key ``{seed & 0xffffffff, seed >> 32}`` and counter ``{row, L, draw, level}``: ``row`` is the track's row in its bucket,
``level`` is ``L - 1`` for the final choice and ``s - 1`` for a member choice.  ``sample_logp`` is the log final weight
plus the logs of the member weights along the route, in that order.

The *margin* of a draw is the smallest ``|u * S - cum_k| / S`` over all its choices: a test comparing draws computed in
another arithmetic (the engine's) needs it well above the rounding.  Labels are the history labels of the posteriors
(the child index mod nS with the int8 wrap of tracking.py:543).  This module runs the same steps as ``chunk_recursion``
(its tables, label wrap, ``_plan_groups`` and ``_merge``, operation for operation, so the posteriors are bitwise equal to
``predict_states``) and keeps the lattice records.  Only ``nb_substeps = 1`` exists here (predict_Bs forces it,
tracking.py:839).  The product (``extrack_b200``) never imports this module.
"""
from __future__ import annotations

import itertools
from typing import List

import numpy as np

from oracle.extrack_oracle import HeadTables, Model, _label, _merge, _plan_groups, chunk_recursion

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 of counters ``ctr`` (4 arrays or ints, 32-bit words) under ``key`` (2 words): 4 uint64 arrays
    holding the 32-bit output words."""
    c = [np.asarray(x, dtype=np.uint64) & _MASK for x in ctr]
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(_W0)) & _MASK
            k1 = (k1 + np.uint64(_W1)) & _MASK
        p0 = np.uint64(_M0) * c[0]
        p1 = np.uint64(_M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
    return c


def uniforms(seed: int, row: int, L: int, draws: np.ndarray, level: int) -> np.ndarray:
    """u in [0, 1) of the given draws at one choice level of one track."""
    x = philox4x32_10([row, L, draws, level], [seed & 0xFFFFFFFF, seed >> 32])
    return ((x[0] << np.uint64(32) | x[1]) >> np.uint64(11)).astype(np.float64) * 2.0**-53


def _choose(w, u):
    """The choice rule for candidates of weights w [n] and uniforms u [S]: (index [S], margin [S])."""
    n = len(w)
    if n == 1:
        return np.zeros(len(u), dtype=np.int64), np.full(len(u), np.inf)
    cum = np.cumsum(w)  # running sums in order (sequential)
    S = cum[-1]
    x = u * S
    k = np.searchsorted(cum, x, side="right")  # first k with x < cum_k
    # cum is non-decreasing: the nearest running sums to x are cum_k-1 <= x and cum_k > x
    margin = np.minimum(np.abs(x - cum[np.maximum(k - 1, 0)]), np.abs(x - cum[np.minimum(k, n - 1)])) / S
    pos = np.nonzero(w > 0)[0]
    k[k == n] = pos[-1]
    return k, margin


def chunk_recursion_sample(C, model: Model, isBL: int, n_samples: int, seed: int, row0: int = 0, tables=None, sig=None,
                           ds3=None):
    """``extrack_oracle.chunk_recursion(C, model, isBL, do_preds=1, ...)`` plus ``n_samples`` posterior draws per track;
    track t has the row ``row0 + t`` of its bucket.

    Returns (preds [nT, L, nS], samples int8 [nT, S, L], sample_logp [nT, S], margin [nT, S]), forward time."""
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

    # ---- first localisation: initial sequence h = h0 + nS*h1, forward-time labels (h1, h0) ----
    nB = K * nS
    head = np.arange(nB)
    init_digits = tb.digits[head].copy()  # [nB, 2]: (h0, h1)
    cur = tb.digits[head, 0].copy()
    hist = (tb.digits[head][None, :, :, None] == np.arange(nS)[None, None, None, :]).astype(np.float64)
    LP = np.repeat((tb.LT[head] + tb.LF[head])[None], nT, axis=0)
    s2 = l2 + dd_at(L - 1, head)
    m = np.repeat(C[:, None, 0, :], nB, axis=1)
    rec = {}  # fusion step -> (groups, normalised member weights [nT, nC])

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
        m, s2 = new_m, new_s2
        LL = tb.Lp_stay[head % K] if step >= model.min_len else 0
        LP = LP + (tb.LT[head][None] + LC + LL)
        nB = len(cur)
        if nB > model.max_nb_states:
            th = th * 1.2
        if step < L - 1:
            groups = _plan_groups(m, s2, hist, frame_len, th)
            rw = np.empty_like(LP)
            for mem in groups:  # the weights _merge averages with, normalised
                w = np.exp(LP[:, mem] - LP[:, mem].max(axis=1, keepdims=True))
                rw[:, mem] = w / np.sum(w, 1, keepdims=True)
            rec[step] = (groups, rw)
            m, s2, LP, cur, hist = _merge(m, s2, LP, cur, hist, groups, nT, frame_len, 1)

    # ---- end of track (tracking.py:613-639); the final weights sum the bleaching end's hidden heads ----
    n_final = len(cur) if L > 2 else nB
    l2e = l2_at(L - 1)
    qe = s2 + l2e
    v = LP + np.sum(-0.5 * np.log(2 * np.pi * qe) - (C[:, None, L - 1, :] - m) ** 2 / (2 * qe), axis=2)
    if isBL:
        child = np.arange(len(cur) * K)
        leave = tb.L_leave[(child % K) + K * cur[child // K]].reshape(len(cur), K)
        mx = np.max(leave, axis=1, keepdims=True)
        v = v + (np.log(np.sum(np.exp(leave - mx), axis=1, keepdims=True)) + mx)[:, 0][None]
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
    LP = LP + (term + LL)

    pLP = LP
    if np.max(LP) > 600:
        pLP = LP - (np.max(LP) - 600)
    P = np.exp(pLP)
    sP = np.sum(P, axis=1, keepdims=True)[:, :, None]
    preds = np.sum(P[:, :, None, None] * hist, axis=1) / sP

    # ---- the draws ----
    e = np.exp(v - np.max(v, axis=1, keepdims=True))
    final_w = e * (1.0 / np.sum(e, axis=1, keepdims=True))  # [nT, n_final]
    assert final_w.shape[1] == n_final
    S = int(n_samples)
    draws = np.arange(S, dtype=np.uint64)
    samples = np.empty((nT, S, L), dtype=np.int8)
    logp = np.empty((nT, S))
    margin = np.empty((nT, S))
    for t in range(nT):
        row = row0 + t
        c, mar = _choose(final_w[t], uniforms(seed, row, L, draws, L - 1))
        lp = np.log(final_w[t, c])
        for s in range(L - 1, 2, -1):
            samples[t, :, s] = _label(c, nS, model.int8_wrap)
            groups, rw = rec[s - 1]
            p = c // K
            nxt = np.empty_like(c)
            u = uniforms(seed, row, L, draws, s - 1)
            for g in np.unique(p):
                sel = p == g
                mem = groups[g]
                k, mg = _choose(rw[t, mem], u[sel])
                nxt[sel] = mem[k]
                mar[sel] = np.minimum(mar[sel], mg)
            c = nxt
            lp = lp + np.log(rw[t, c])
        if L >= 3:
            samples[t, :, 2] = _label(c, nS, model.int8_wrap)
            c = c // K
        samples[t, :, 1] = init_digits[c, 0]
        samples[t, :, 0] = init_digits[c, 1]
        logp[t] = lp
        margin[t] = mar
    return preds[:, ::-1], samples, logp, margin


def predict_samples(sorted_tracks: List[np.ndarray], model: Model, n_samples: int, seed: int, nb_max: int = 1, sigs=None,
                    ds_list=None):
    """``extrack_oracle.predict_states`` with the posterior draws: per bucket ``(preds [n, L, nS], samples int8
    [n, S, L], sample_logp [n, S], margin [n, S])``."""
    max_len = sorted_tracks[-1].shape[1]
    tables = HeadTables(model)
    out = []
    for b, arr in enumerate(sorted_tracks):
        isBL = 0 if arr.shape[1] == max_len else 1
        parts = []
        for n in range(int(np.ceil(len(arr) / nb_max))):
            sl = slice(n * nb_max, (n + 1) * nb_max)
            parts.append(chunk_recursion_sample(arr[sl], model, isBL, n_samples, seed, n * nb_max, tables,
                                                None if sigs is None else sigs[b][sl],
                                                None if ds_list is None else ds_list[b][sl]))
        L = arr.shape[1]
        out.append(tuple(np.concatenate(x) for x in zip(*parts)) if parts
                   else (np.empty((0, L, model.nS)), np.empty((0, n_samples, L), dtype=np.int8),
                         np.empty((0, n_samples)), np.empty((0, n_samples))))
    return out


def enumerate_posterior(C, model: Model, isBL: int):
    """Exact posterior of every full state sequence of tracks too short for any fusion, by direct enumeration of the
    recursion's surviving sequences (every history one-hot).  At a bleaching end the K children of a sequence differ
    only in the hidden state after the last localisation, which no label shows: they are summed.

    Returns (labels int8 [n_seq, L] forward time, log posterior [nT, n_seq])."""
    LP, hist, _ = chunk_recursion(C, model, isBL, 1)
    h = np.broadcast_to(hist, (len(C),) + hist.shape[1:])[:, :, ::-1]  # [nT, nB, L, nS], forward time
    if not set(np.unique(h)) <= {0.0, 1.0}:
        raise ValueError("a fusion happened: the posterior is not enumerable this way")
    mx = np.max(LP, axis=1, keepdims=True)
    logZ = np.log(np.sum(np.exp(LP - mx), axis=1, keepdims=True)) + mx
    if isBL:
        r = LP.reshape(len(C), -1, model.nS)
        rm = np.max(r, axis=2, keepdims=True)
        LPs = (np.log(np.sum(np.exp(r - rm), axis=2, keepdims=True)) + rm)[:, :, 0]
        h = h[:, :: model.nS]
    else:
        LPs = LP
    labels = np.argmax(h[0], axis=-1).astype(np.int8)
    n_seq = model.nS ** C.shape[1]
    assert labels.shape[0] == n_seq and len({tuple(x) for x in labels}) == n_seq, "every sequence exactly once"
    assert set(map(tuple, labels)) == set(itertools.product(range(model.nS), repeat=C.shape[1]))
    return labels, LPs - logZ
