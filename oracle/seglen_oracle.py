"""TEST INFRASTRUCTURE ONLY — CPU restatement of the reference's segment-length histogram
(``extrack/histograms.py:26-258`` ``P_segment_len`` and ``:265-373`` ``len_hist``), SURVEY.md §8(f) N2.

Only ``tests/``, ``tests/golden/make_golden.py`` and ``__graft_entry__.smoke()`` may import it.

Own structure (the reference carries the whole state history ``cur_Bs[nT, nB, L]`` of every live
sequence and re-gathers it at every pruning step): per step one *lattice record* (parent index,
newest state) per surviving sequence, histories are recovered by walking the records back.
Restated behaviour, ``nb_substeps = 1``, scalar / per-dimension ``LocErr``:

* expansion: child ``j`` of a step has parent ``j // nS`` and newest state ``j % nS`` (``:146``);
* Gaussian-product update in the reference's operation order (``tracking.py:87-98``);
* ``LL`` gains ``Lp_stay[newest]`` from step ``min_l`` on (``:133,:172``);
* literal top-``max_nb_states`` pruning (``:183-206``): key = ``LP`` + log-density of the *next*
  localisation, sorted descending; moments, ``LP`` and histories keep the first ``k`` ranks, **``LL``
  keeps the last ``k`` ranks of the same order** (``:202`` slices ``[-max_nb_states:]`` — reproduced);
* end of track (``:211-234``): optional leave expansion whose ``end_p_stay`` is ``p_stay[s]`` only
  when newest and previous state are both ``s`` and ``p_stay[0]`` otherwise (``:224`` broadcasts a
  two-column comparison), transition term *not* added (``:220``);
* weights ``P = exp(LP + LL)`` normalised per track; every maximal run of ``k`` equal states in a
  sequence's history adds its weight to ``hist[k-1, state]`` (``:248-258``), runs of length ``L`` are
  not counted (``k`` ranges ``1..L-1``).

Tie-break of the sort (the reference uses ``argsort()[:, ::-1]`` with numpy's unstable default sort,
so its order among equal keys is unspecified): descending key, equal keys by descending index — what
a stable ascending sort followed by the reversal gives.  The reference sorts ``exp(key - shift)``;
keys that underflow to zero there are in unspecified order, here they keep the order of their keys.
The ``> 600`` rescale of the final ``LP`` (``:243-244``) is per *column* over the tracks of the chunk
(``np.max(LP, axis=0)``), which changes the relative weights of a track's sequences — reproduced.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np

from .extrack_oracle import HeadTables, Model

NB_MAX = 50  # histograms.py:319  tracks per chunk


def _logdens_next(Cn, m, s2, l2):
    """sum_dims(-0.5 log(2 pi (s2 + l2)) - (Cn - m)^2 / (2 (s2 + l2)))  (histograms.py:187-188, :238-239)"""
    ns2 = s2 + l2
    return np.sum(-0.5 * np.log(2 * np.pi * ns2) - (Cn - m) ** 2 / (2 * ns2), axis=2)


def _min_rel_gap(key: np.ndarray) -> np.ndarray:
    """Per row: the smallest non-zero relative gap between adjacent finite keys of the sorted row (inf if none)."""
    s = np.sort(key, axis=1)
    a, b = s[:, :-1], s[:, 1:]
    with np.errstate(invalid="ignore"):
        g = np.abs(b - a) / np.maximum(np.maximum(np.abs(a), np.abs(b)), 1e-300)
    g = np.where(np.isfinite(a) & np.isfinite(b) & (g > 0), g, np.inf)
    return g.min(axis=1) if g.shape[1] else np.full(len(key), np.inf)


def segment_len_chunk(C: np.ndarray, model: Model, isBL: int, max_nb_states: int = 1000, min_l: int = 3,
                      want_histories: bool = False, ties_ascending: bool = False, want_gaps: bool = False):
    """One chunk ``C[nT, L, d]`` (forward time).  Returns ``(LP[nT, nB], hist[L-1, nS])`` and, if
    asked, the state histories ``[nT, nB, L]`` (column 0 = newest, like the reference's ``cur_Bs``).

    Test-only options: ``ties_ascending`` orders equal sort keys by *ascending* index (the reverse of
    the documented rule), which shows whether a case has ties that change the result; ``want_gaps``
    appends, per track, the smallest non-zero relative gap between adjacent sort keys over all pruning
    steps (``inf`` without pruning) — where a last-bit difference of a library ``log`` could reorder keys."""
    if model.nb_substeps != 1:
        raise NotImplementedError("segment-length oracle: nb_substeps = 1 only")
    C = np.asarray(C, dtype=float)
    nT, L, d = C.shape
    if L < 2:
        raise NotImplementedError("segment-length oracle: L >= 2")
    nS = model.nS
    tb = HeadTables(model)
    l2 = (np.asarray(model.loc_err, dtype=float) ** 2).reshape(1, 1, -1)  # [1, 1, k]
    head = np.arange(nS * nS)
    newest, parent_state = head % nS, head // nS

    # first localisation: nS^2 sequences (newest, oldest)
    LP = np.repeat((tb.LT + tb.LF)[None], nT, 0)
    LL = np.zeros((nT, nS * nS))
    step = 1
    if step >= min_l:
        LL = LL + tb.Lp_stay[newest][None]
    m = np.repeat(C[:, None, 0, :], nS * nS, axis=1)
    s2 = np.repeat(l2 + tb.dd[None, :, None], nT, 0)
    state = np.repeat(newest[None], nT, 0)            # newest state per live sequence
    lattice = [(np.repeat((parent_state)[None], nT, 0), state.copy())]  # (oldest state as "parent", newest)
    gaps = np.full(nT, np.inf)
    step = 2
    while step <= L - 1:
        nB = state.shape[1]
        j = np.arange(nB * nS)
        par, new = j // nS, j % nS
        hd = new[None] + nS * state[:, par]            # head = newest + nS * previous
        mp, sp = m[:, par], s2[:, par]
        Ci = C[:, None, step - 1, :]
        q = l2 + sp
        nm = (mp * l2 + Ci * sp) / (l2 + sp)
        dd = tb.dd[hd][:, :, None]
        ns2 = (dd * l2 + dd * sp + l2 * sp) / q
        if sp.shape[2] == 1:
            LC = d * -0.5 * np.log(2 * np.pi * q[:, :, 0]) - np.sum((Ci - mp) ** 2 / (2 * q), axis=2)
        else:
            LC = np.sum(-0.5 * np.log(2 * np.pi * q), 2) - np.sum((Ci - mp) ** 2 / (2 * q), axis=2)
        LLn = LL[:, par]
        if step >= min_l:
            LLn = LLn + tb.Lp_stay[new][None]
        LPn = LP[:, par] + (tb.LT[hd] + LC)
        m, s2, LP, LL = nm, ns2, LPn, LLn
        state = np.repeat(new[None], nT, 0)
        parent = np.repeat(par[None], nT, 0)
        if step < L - 1 and nB * nS > max_nb_states:
            key = LP + _logdens_next(C[:, None, step, :], m, s2, l2)
            if ties_ascending:  # descending key, ties by ascending index
                order = np.argsort(-key, axis=1, kind="stable")
            else:  # descending key, ties by descending index
                order = np.argsort(key, axis=1, kind="stable")[:, ::-1]
            if want_gaps:
                gaps = np.minimum(gaps, _min_rel_gap(key))
            k = max_nb_states
            top = order[:, :k]
            m = np.take_along_axis(m, top[:, :, None], 1)
            s2 = np.take_along_axis(s2, top[:, :, None], 1)
            LP = np.take_along_axis(LP, top, 1)
            LL = np.take_along_axis(LL, order[:, -k:], 1)   # histograms.py:202
            state = np.take_along_axis(state, top, 1)
            parent = np.take_along_axis(parent, top, 1)
        lattice.append((parent, state))
        step += 1

    nB = state.shape[1]
    dropped_newest = False
    if isBL:
        j = np.arange(nB * nS)
        par, new = j // nS, j % nS
        prev = state[:, par]
        e = np.where(new[None] == prev, tb.p_stay[prev], tb.p_stay[0])
        LL = LL[:, par] + np.log(model.pBL + (1 - e) - model.pBL * (1 - e))
        LP, m, s2 = LP[:, par], m[:, par], s2[:, par]
        lattice.append((np.repeat(par[None], nT, 0), None))   # history of a child = history of its parent
        dropped_newest = True
    LP = LP + _logdens_next(C[:, None, L - 1, :], m, s2, l2)
    if np.max(LP) > 600:  # histograms.py:243-244: per column, over the tracks of the chunk
        LP = LP - (np.max(LP, axis=0, keepdims=True) - 600)
    P = np.exp(LP + LL)
    Pn = P / np.sum(P, axis=1, keepdims=True)

    # histories by walking the lattice back: hist_states[t, j, c], column 0 = newest
    nBf = LP.shape[1]
    idx = np.repeat(np.arange(nBf)[None], nT, 0)
    cols = []
    recs = lattice[::-1]
    if dropped_newest:
        idx = np.take_along_axis(recs[0][0], idx, 1)
        recs = recs[1:]
    for parent, st in recs[:-1]:
        cols.append(np.take_along_axis(st, idx, 1))
        idx = np.take_along_axis(parent, idx, 1)
    oldest, st0 = recs[-1]
    cols.append(np.take_along_axis(st0, idx, 1))
    cols.append(np.take_along_axis(oldest, idx, 1))
    H = np.stack(cols, axis=2)                           # [nT, nBf, L]
    assert H.shape[2] == L

    hist = np.zeros((L - 1, nS))
    run = np.ones((nT, nBf), dtype=int)
    cur = H[:, :, 0]
    counted = np.zeros((nT, nBf), dtype=int)
    for c in range(1, L):
        tr = cur != H[:, :, c]
        run = run + (~tr)
        if tr.any():                                      # runs that end here: length run, state cur
            np.add.at(hist, (run[tr] - 1, cur[tr]), Pn[tr])
        counted += run * tr
        run[tr] = 1
        cur = H[:, :, c]
    last = L - counted                                    # the oldest run; a run of L (no transition) is not counted
    sel = last <= L - 1
    np.add.at(hist, (last[sel] - 1, cur[sel]), Pn[sel])
    return (LP, hist) + ((H,) if want_histories else ()) + ((gaps,) if want_gaps else ())


def len_hist(sorted_tracks: Sequence[np.ndarray], model: Model, max_nb_states: int = 500) -> np.ndarray:
    """Sum over chunks of <= 50 tracks (histograms.py:306-360); the longest bucket has isBL = 0."""
    min_l = int(min(a.shape[1] for a in sorted_tracks))
    Lmax = int(sorted_tracks[-1].shape[1])
    out = np.zeros((Lmax, model.nS))
    for b, arr in enumerate(sorted_tracks):
        isBL = 0 if b == len(sorted_tracks) - 1 else 1
        for a in range(0, len(arr), NB_MAX):
            _, h = segment_len_chunk(arr[a:a + NB_MAX], model, isBL, max_nb_states, min_l)
            out[:h.shape[0]] += h
    return out
