"""TEST INFRASTRUCTURE ONLY — CPU (numpy, FP64) log-likelihood along a FROZEN grouping plan.

``extrack_oracle.chunk_recursion`` decides a grouping at every fusion step from the current parameters.  Along a
frozen plan the groups are those recorded (``plan_out``) by one run at theta0; any theta is then replayed with the
recorded groups, and the threshold escalation is implied by them.  log P of every track is then a smooth function of
theta (Gaussian products and log-sum-exps over a fixed lattice): the surface ``param_uncertainty`` differentiates.

``frozen_chunk_logp`` runs the steps of ``chunk_recursion`` operation for operation (``HeadTables``, ``_label``,
``_merge``), only the call of ``_plan_groups`` is replaced by the recorded groups.  So at theta0, and at any theta whose
own plan equals theta0's, it is bitwise ``chunk_logp``.  Peak-wise localisation errors (``sig``) are covered; per-track
dt is not (``param_uncertainty`` does not support it).  The product (``extrack_b200``) never imports this module.
"""
from __future__ import annotations

from typing import List, Optional

import numpy as np

from .extrack_oracle import HeadTables, Model, _label, _merge, chunk_recursion, make_chunks


def record_plan(C, model: Model, isBL: int, sig=None) -> list:
    """The grouping plan of one chunk at ``model`` (one dict per fusion step, see ``chunk_recursion``)."""
    plan: list = []
    chunk_recursion(C, model, isBL, 0, plan, None, sig)
    return plan


def frozen_chunk_logp(C, model: Model, isBL: int, plan: list, sig=None) -> np.ndarray:
    """log P per track of one chunk at ``model``, fusing with the recorded groups of ``plan``."""
    C = np.asarray(C, dtype=np.float64)
    nT, L, d = C.shape
    nS, nsub = model.nS, model.nb_substeps
    tb = HeadTables(model)
    K = tb.K
    if sig is not None:
        sig2 = np.asarray(sig, dtype=np.float64) ** 2
        l2_at = lambda j: sig2[:, None, j, :]
    else:
        l2c = (np.asarray(model.loc_err, dtype=np.float64).reshape(-1) ** 2)[None, None, :]
        l2_at = lambda j: l2c
    frame_len = int(model.frame_len)
    nB = K * nS
    head = np.arange(nB)
    cur = tb.digits[head, 0].copy()
    hist = (tb.digits[head][None, :, :, None] == np.arange(nS)[None, None, None, :]).astype(np.float64)
    LP = np.repeat((tb.LT[head] + tb.LF[head])[None], nT, axis=0)
    s2 = l2_at(0) + tb.dd[head][None, :, None]
    m = np.repeat(C[:, None, 0, :], nB, axis=1)

    def expand(cur, hist):
        nB0 = len(cur)
        n = nB0
        for _ in range(nsub):
            n = n * nS
            lab = _label(np.arange(n), nS, model.int8_wrap)
            new_row = (lab[None, :, None, None] == np.arange(nS)[None, None, None, :]).astype(np.float64)
            new_row = np.repeat(new_row, hist.shape[0], 0)
            hist = np.concatenate((new_row, np.repeat(hist, nS, 1)), -2)
        child = np.arange(nB0 * K)
        return (child % K) + K * cur[child // K], child % nS, hist

    rec = iter(plan)
    for step in range(2, L):
        head, cur, hist = expand(cur, hist)
        dd = tb.dd[head][None, :, None]
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
        if step < L - 1:
            r = next(rec)
            assert r["step"] == step and r["nB_in"] == len(cur), "plan does not match the chunk"
            m, s2, LP, cur, hist = _merge(m, s2, LP, cur, hist, r["groups"], nT, frame_len, 0)
    if isBL:
        head, cur, hist = expand(cur, hist)
        m = np.repeat(m, K, axis=1)
        s2 = np.repeat(s2, K, axis=1)
        LP = np.repeat(LP, K, axis=1)
        LL = tb.L_leave[head][None]
    else:
        LL = 0
    l2 = l2_at(L - 1)
    q = s2 + l2
    term = np.sum(-0.5 * np.log(2 * np.pi * q) - (C[:, None, L - 1, :] - m) ** 2 / (2 * q), axis=2)
    LP = LP + (term + LL)
    top = np.max(LP, axis=1, keepdims=True)
    return np.log(np.sum(np.exp(LP - top), axis=1)) + top[:, 0]


class FrozenDataSet:
    """A data set with the plans of all its chunks recorded at ``model0`` (chunks as ``make_chunks``: the engine's
    upload order).  ``logp(model)`` = per-track log P along those plans, concatenated in that order."""

    def __init__(self, sorted_tracks: List[np.ndarray], model0: Model, chunk: int = 2000,
                 sigs: Optional[List[np.ndarray]] = None):
        self.jobs = [(sorted_tracks[b][a:z], isBL, None if sigs is None else sigs[b][a:z])
                     for (b, a, z, isBL) in make_chunks(sorted_tracks, chunk)]
        self.plans = [record_plan(C, model0, isBL, sg) for (C, isBL, sg) in self.jobs]

    def logp(self, model: Model) -> np.ndarray:
        return np.concatenate([frozen_chunk_logp(C, model, isBL, pl, sg) for (C, isBL, sg), pl in zip(self.jobs, self.plans)])
