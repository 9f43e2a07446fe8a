"""Grouping decisions placed exactly on the threshold, and the plan-verification paths such ties drive.

Leader i captures sequence j when ``fl(mean|m_j - m_i| / s_j) < th`` (and the same for the standard deviations) for
more than 80 % of the leader-track votes (tracking.py:689-691, ``oracle.extrack_oracle._plan_groups``).  The kernels
decide most comparisons with two products against ``th (1 -+ 1e-14)`` and divide only near the boundary, so random
data never exercise the exact half of the predicate.  Here ``th`` itself is set to one of the ratios the oracle
compares (``th = r``: ``r < r`` is false; ``nextafter(r, inf)``: true), at a vote that sits on its 80 % margin, so
the plan at ``th = r`` differs from the plan one ulp above.  The tie finder proves on the CPU that each fixture flips
the oracle plan before any GPU test relies on it.
"""
from __future__ import annotations

import contextlib
import functools
import io

import numpy as np
import pytest

from helpers import engine_params, gid_from_groups, make_model, random_walk_tracks
from oracle import extrack_oracle as orc
from oracle import ref_loader

TT = orc.TEST_TRACKS
RTOL_LOGL = 1e-9
RTOL_FP32 = 1e-4


def up(x):
    return float(np.nextafter(x, np.inf))


def at(model, th):
    """The oracle model with another threshold."""
    return orc.Model(**{**vars(model), "threshold": th})


# ---------------------------------------------------------------------------------------------------------------
# tie finder (CPU)
# ---------------------------------------------------------------------------------------------------------------
def oracle_steps(C, model, isBL, do_preds=0):
    """Per fusion step of one oracle recursion: the arguments of ``_plan_groups`` (m, s2, hist, threshold used) and the
    groups it returned."""
    steps = []
    plan = orc._plan_groups

    def spy(m, s2, hist, frame_len, th):
        groups = plan(m, s2, hist, frame_len, th)
        steps.append((m, s2, hist, th, groups))
        return groups

    orc._plan_groups = spy
    try:
        orc.chunk_recursion(C, model, isBL, do_preds)
    finally:
        orc._plan_groups = plan
    return steps


def oracle_plan(C, model, isBL, do_preds=0):
    """Per fusion step: (nB_in, groups, threshold used)."""
    return [(m.shape[1], groups, th) for m, _, _, th, groups in oracle_steps(C, model, isBL, do_preds)]


def same_groups(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def same_plan(a, b):
    """Same step of two oracle plans: live sequences and groups (the thresholds differ by construction)."""
    return a[0] == b[0] and same_groups(a[1], b[1])


def first_difference(pa, pb):
    """First step (2-based) at which two oracle plans differ, None if they are equal."""
    for k, (a, b) in enumerate(zip(pa, pb)):
        if not same_plan(a, b):
            return k + 2
    return None


def min_votes(n):
    """Smallest count c of passing votes with fl(c / n) > 0.8 (``np.mean(..) > 0.8``)."""
    return next(c for c in range(n + 1) if c / n > 0.8)


def margin_ratios(m, s2, hist, frame_len, lo, hi):
    """Ratios of ``_plan_groups`` (its expressions, shapes and operation order) that sit on a vote's margin: for a pair
    (i, j) with the other vote passing, the ratio r with ``count(ratio < r) < need <= count(ratio <= r)``.  Returns
    {r: whether some x / s = r has x < fl(r s)}, i.e. whether deciding ``x < fl(th s)`` in product form errs at r."""
    nB = m.shape[1]
    s = s2**0.5
    mK, sK, hK = m[:TT], s[:TT], hist[:TT]
    newest = np.argmax(hist[0, :, 0], axis=1)
    use_window = hist.shape[2] > frame_len
    if use_window:
        win = np.argmax(hK[:, :, :frame_len], axis=-1)
    out = {}
    for i in range(nB):
        xm = np.mean(np.abs(mK - mK[:, i : i + 1]), axis=2, keepdims=True)
        xs = np.mean(np.abs(sK - sK[:, i : i + 1]), axis=2, keepdims=True)
        dm, dsd = xm / sK, xs / sK
        cand = newest == newest[i]
        cand[i] = False
        if use_window:
            cand &= ~(np.mean(np.all(win == win[:, i : i + 1], axis=2), axis=0) > 0.999)
        for a, x, b in ((dm, xm, dsd), (dsd, xs, dm)):
            # (s2 has one row while no merge has mixed tracks: the standard-deviation vote then has KS voters)
            va = np.sort(np.moveaxis(a, 1, 0).reshape(nB, -1), axis=1)[:, min_votes(a.shape[0] * a.shape[2]) - 1]
            for j in np.nonzero(cand)[0]:
                r = float(va[j])
                if lo < r < hi and np.mean(b[:, j] < r) > 0.8:
                    xj, sj = np.broadcast_arrays(x[:, j], sK[:, j])
                    out[r] = out.get(r, False) or bool(np.any((a[:, j] == r) & (xj < r * sj)))
    return out


def model_threshold_for(r, escalations):
    """Model threshold t with fl(t 1.2 .. 1.2) = r and fl(nextafter(t) 1.2 .. 1.2) > r (``th *= 1.2`` sticky
    escalation applied ``escalations`` times), or None when no double maps onto r."""
    if escalations == 0:
        return r

    def f(t):
        for _ in range(escalations):
            t = t * 1.2
        return t

    t = r / 1.2**escalations
    for _ in range(8):
        t = float(np.nextafter(t, -np.inf))
    for _ in range(16):
        if f(t) == r and f(up(t)) > r:
            return t
        t = up(t)
    return None


def tie_thresholds(C30, model, step, isBL=1, do_preds=0, lo=0.02, hi=1.0, budget=60, want=3):
    """Model thresholds t at which the oracle plan of the 30-track chunk ``C30`` at ``threshold = t`` differs from the
    plan at ``nextafter(t, inf)``, with every step before ``step`` planned identically.  Candidates are the margin
    ratios of ``step`` in the recursion at ``model.threshold``; later steps only see the same inputs at a candidate
    threshold while the earlier plans stay, hence the nearest candidates first."""
    steps = oracle_steps(C30, model, isBL, do_preds)
    if len(steps) < step - 1:
        return []
    m, s2, hist, th_used, _ = steps[step - 2]
    esc = int(round(np.log(th_used / model.threshold) / np.log(1.2)))
    # the ones a product-form decision gets wrong first, then nearest to the threshold used
    ratios = margin_ratios(m, s2, hist, model.frame_len, lo, hi)
    cands = sorted(ratios, key=lambda r: (not ratios[r], abs(np.log(r / th_used))))
    found = []
    for r in cands[:budget]:
        # cheap screen on this step's inputs, then the whole recursion at both thresholds
        if same_groups(orc._plan_groups(m, s2, hist, model.frame_len, r), orc._plan_groups(m, s2, hist, model.frame_len, up(r))):
            continue
        t = model_threshold_for(r, esc)
        if t is None:
            continue
        pa, pb = (oracle_plan(C30, at(model, th), isBL, do_preds) for th in (t, up(t)))
        if first_difference(pa, pb) == step:
            found.append(t)
            if len(found) >= want:
                break
    return found


def groups_product_form(m, s2, hist, frame_len, th):
    """``_plan_groups`` with ``x / s < th`` decided as ``x < fl(th s)`` unless the two are equal (a plan kernel that
    lost the exact division of its near-boundary fallback)."""
    nB = m.shape[1]
    s = s2**0.5
    mK, sK, hK = m[:TT], s[:TT], hist[:TT]
    newest = np.argmax(hist[0, :, 0], axis=1)
    use_window = hist.shape[2] > frame_len
    if use_window:
        win = np.argmax(hK[:, :, :frame_len], axis=-1)

    def lt(x):
        p = th * sK
        return np.where(x < p, True, np.where(x > p, False, x / sK < th))

    grouped = np.zeros(nB, dtype=bool)
    groups = []
    for i in range(nB):
        if grouped[i]:
            continue
        m_ok = np.mean(lt(np.mean(np.abs(mK - mK[:, i : i + 1]), axis=2, keepdims=True)), axis=(0, 2)) > 0.8
        s_ok = np.mean(lt(np.mean(np.abs(sK - sK[:, i : i + 1]), axis=2, keepdims=True)), axis=(0, 2)) > 0.8
        sel = m_ok & s_ok & (newest == newest[i])
        if use_window:
            sel = sel | (np.mean(np.all(win == win[:, i : i + 1], axis=2), axis=0) > 0.999)
        sel &= ~grouped
        groups.append(np.nonzero(sel)[0])
        grouped[groups[-1]] = True
    return groups


def product_form_differs(C30, model, t, step, isBL=1):
    """Does the product-form predicate give another plan than the exact one at ``t`` or one ulp above (at ``step``)?"""
    for th in (t, up(t)):
        m, s2, hist, th_used, groups = oracle_steps(C30, at(model, th), isBL)[step - 2]
        if not same_groups(groups, groups_product_form(m, s2, hist, model.frame_len, th_used)):
            return True
    return False


# ---------------------------------------------------------------------------------------------------------------
# families: a 30-track tie block, its model and the ties found in it
# ---------------------------------------------------------------------------------------------------------------
FAMILIES = {
    # name: model keywords, dimensions, track length, steps searched for ties
    "s2_2d": dict(model=dict(nS=2, frame_len=4), d=2, L=9, steps=(2, 3)),
    "s3_3d": dict(model=dict(nS=3, frame_len=3), d=3, L=8, steps=(2,)),
    "s2_locdim": dict(model=dict(nS=2, frame_len=4, loc_err=(0.02, 0.03)), d=2, L=9, steps=(2,)),
    "s2_1d": dict(model=dict(nS=2, frame_len=4), d=1, L=9, steps=(2,)),
    "s3_nsub2": dict(model=dict(nS=3, nsub=2, frame_len=6, max_nb_states=500), d=2, L=6, steps=(2,)),
    "s2_escalate": dict(model=dict(nS=2, frame_len=4, max_nb_states=3), d=2, L=9, steps=(2,)),
}


@functools.lru_cache(maxsize=None)
def family(name):
    """The first seed whose 30-track block has a tie at every searched step; ties[(step)] = model thresholds, the
    ones at which the product-form predicate also goes wrong first."""
    f = FAMILIES[name]
    model = make_model(**f["model"])
    for seed in range(20):
        C = random_walk_tracks(TT, f["L"], f["d"], np.random.default_rng(1000 + seed), Ds=model.ds**2 / 0.04)
        ties = {}
        for step in f["steps"]:
            ts = tie_thresholds(C, model, step)
            if not ts:
                break
            prod = [t for t in ts if product_form_differs(C, model, t, step)]
            ties[step] = prod + [t for t in ts if t not in prod]
        if len(ties) == len(f["steps"]):
            return dict(C=C, model=model, ties=ties, seed=seed)
    return None


def pairs_of(fam):
    """(step, model threshold at the tie) of a family, every searched step."""
    return [(step, t) for step, ts in fam["ties"].items() for t in ts]


@pytest.mark.parametrize("name", list(FAMILIES))
def test_tie_fixtures_flip_the_oracle_plan(name):
    """Every family has a tie at each searched step, and the oracle plans at th = t and nextafter(t) agree before that
    step and differ at it: the GPU tests below compare the engine against two different plans."""
    fam = family(name)
    if fam is None and name == "s2_escalate":
        pytest.skip("no threshold whose escalation fl(th * 1.2) lands on a margin ratio of these tracks")
    assert fam is not None, "no tie found"
    C, model = fam["C"], fam["model"]
    for step, t in pairs_of(fam):
        pa, pb = oracle_plan(C, at(model, t), 1), oracle_plan(C, at(model, up(t)), 1)
        assert first_difference(pa, pb) == step
        nB, _, th_used = pa[step - 2]
        if name == "s3_nsub2":
            assert nB > 64  # batch / split mode of the plan kernel, not the matrix mode
        if name == "s2_escalate":
            assert th_used == t * 1.2 and pb[step - 2][2] == up(t) * 1.2  # the escalated threshold decides
        else:
            assert th_used == t
    if name == "s2_2d":
        assert 3 in fam["ties"]  # a later step too: verification records are per step


def test_some_ties_defeat_a_product_form_decision():
    """Deciding fl(x / s) < th as x < fl(th s) (no exact fallback) gives another plan at some of the fixtures' ties."""
    hits = [name for name in FAMILIES if family(name) is not None
            and product_form_differs(family(name)["C"], family(name)["model"], *reversed(pairs_of(family(name))[0]))]
    assert {"s3_3d", "s3_nsub2"} <= set(hits)


def test_product_form_twin_agrees_with_the_oracle_away_from_ties():
    """The product-form twin of _plan_groups differs from it only at ties: at thresholds no ratio sits on, both give
    the same plan at every step (so the twin's disagreements above are the boundary's, not the twin's own)."""
    for name in ("s2_2d", "s3_3d", "s2_locdim"):
        fam = family(name)
        for th in (0.05, 0.2, 0.5):
            for m, s2, hist, th_used, groups in oracle_steps(fam["C"], at(fam["model"], th), 1):
                assert same_groups(groups_product_form(m, s2, hist, fam["model"].frame_len, th_used), groups)


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not present")
@pytest.mark.parametrize("name", list(FAMILIES))
def test_tie_plans_match_the_reference(name):
    """The unmodified reference takes the same decision at both thresholds: log P equals the oracle's."""
    fam = family(name)
    if fam is None:
        pytest.skip("no tie in this family")
    trk = ref_loader.load_tracking()
    C, model = fam["C"], fam["model"]
    for _, t in pairs_of(fam):
        for th in (t, up(t)):
            m = at(model, th)
            with contextlib.redirect_stdout(io.StringIO()):
                ref = trk.Proba_Cs(C, np.asarray(m.loc_err)[None, None], m.ds, m.Fs, m.TrMat, m.pBL, 1, m.cell_dims,
                                   m.nb_substeps, m.frame_len, m.min_len, m.threshold, m.max_nb_states)
            np.testing.assert_allclose(orc.chunk_logp(C, m, 1), ref, rtol=1e-13)


# ---------------------------------------------------------------------------------------------------------------
# plan construction at the tie (GPU)
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def native():
    from extrack_b200 import _native

    return _native


@pytest.fixture(scope="module")
def xt():
    from extrack_b200 import tracking

    return tracking


def gpu_family(name):
    fam = family(name)
    if fam is None:
        pytest.skip("no tie in this family")
    return fam


def assert_plan_is_oracle(eng, chunk, C, model, isBL=1):
    """plan_dump of every fusion step of ``chunk`` equals the oracle's groups for the tracks C."""
    for step, (nB, groups, th) in enumerate(oracle_plan(C, model, isBL), start=2):
        got_nB, nG, gid, th_used = eng.plan_dump(chunk, step)
        assert (got_nB, nG, th_used) == (nB, len(groups), th), step
        np.testing.assert_array_equal(gid, gid_from_groups(groups, nB), err_msg="step %d" % step)


PLAN_OPTS = [dict(k1_threads=nt, k1_smem_scratch=ss) for nt in (256, 512, 1024) for ss in (0, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FAMILIES))
def test_plan_at_the_tie_is_the_oracle_plan(name, native):
    """Plan construction (plan_verify off) at th = t and nextafter(t): every step's groups equal the oracle's and log P
    is within 1e-9, for each thread count and scratch placement of the plan kernel; above 64 live sequences also for
    the batched and the one-leader-at-a-time (split) grouping."""
    fam = gpu_family(name)
    C, model = fam["C"], fam["model"]
    opts = PLAN_OPTS + ([dict(o, k1_batch=0) for o in PLAN_OPTS] if name == "s3_nsub2" else [])
    ref = {th: orc.chunk_logp(C, at(model, th), 1) for _, t in pairs_of(fam) for th in (t, up(t))}
    for o in opts:
        eng = native.Engine(0)
        try:
            eng.upload([C], [1], len(C))
            eng.set_option("plan_verify", 0)
            for k, v in o.items():
                eng.set_option(k, v)
            for _, t in pairs_of(fam):
                for th in (t, up(t)):
                    got = eng.chunk_logp(0, len(C), engine_params(at(model, th), C.shape[2]))
                    assert_plan_is_oracle(eng, 0, C, at(model, th))
                    np.testing.assert_allclose(got, ref[th], rtol=RTOL_LOGL, err_msg=str(o))
        finally:
            eng.close()


@pytest.mark.gpu
def test_plan_at_the_tie_under_fp32_replay(native):
    """The FP32 replay runs on the same FP64 plan: the plan is the oracle's, log P within the FP32 tolerance."""
    fam = gpu_family("s2_2d")
    C, model = fam["C"], fam["model"]
    eng = native.Engine(0)
    try:
        eng.upload([C], [1], len(C))
        eng.set_option("plan_verify", 0)
        eng.set_option("fp32_replay", 1)
        for _, t in pairs_of(fam):
            for th in (t, up(t)):
                got = eng.chunk_logp(0, len(C), engine_params(at(model, th), C.shape[2]))
                assert eng.stats()["fp32"] == 1
                assert_plan_is_oracle(eng, 0, C, at(model, th))
                np.testing.assert_allclose(got, orc.chunk_logp(C, at(model, th), 1), rtol=RTOL_FP32)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------
# plan verification driven by ties (GPU)
# ---------------------------------------------------------------------------------------------------------------
CHUNK = 64


def tie_data(xt, fam, n_chunks, flipped, step=2, seed=5):
    """One bucket of n_chunks * 64 random tracks; the family's tie block (30 tracks: the leaders) heads the chunks
    ``flipped`` (indices into the chunk list).  Returns (tracks, chunk list)."""
    C, model = fam["C"], fam["model"]
    X = random_walk_tracks(n_chunks * CHUNK, C.shape[1], C.shape[2], np.random.default_rng(seed), Ds=model.ds**2 / 0.04)
    chunks = xt.chunk_table([X], CHUNK)
    for c in flipped:
        a = chunks[c][1]
        X[a : a + TT] = C
    return [X], chunks


VERIFY_VARIANTS = {
    "default": dict(family="s2_2d"),
    "k1_threads_1024": dict(family="s2_2d", opts=dict(k1_threads=1024)),
    "verify_fork_k2": dict(family="s2_2d", opts=dict(verify_fork_k2=1)),
    "s3_3d": dict(family="s3_3d"),
    "locerr_per_dim": dict(family="s2_locdim"),
    "fp32_replay": dict(family="s2_2d", opts=dict(fp32_replay=1)),
    "three_shards": dict(family="s2_2d", devices=[0, 0, 0]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VERIFY_VARIANTS))
def test_verification_catches_a_single_flipped_decision(variant, xt, native):
    """Engine A (plan verification on) against engine B (every evaluation plans from scratch), threshold moved by one
    ulp across a tie that sits in chosen chunks.  After every evaluation: the objective bits, every chunk's per-track
    values and the statistics that say which path ran (construction, verified, chunks planned again)."""
    v = VERIFY_VARIANTS[variant]
    fam = gpu_family(v["family"])
    model, d = fam["model"], fam["C"].shape[2]
    opts = v.get("opts", {})
    devices = v.get("devices")
    # three shards of 8 chunks: two flipped chunks stay a partial re-plan wherever they land; all flipped: fallback.
    # One context of 8 chunks: 2 flipped chunks are re-planned, 3 exceed (8 + 3) / 4 and fall back to construction.
    n_chunks = 24 if devices else 8
    layouts = [(2, [2], 1), (2, [2, 5], 2), (2, list(range(n_chunks)) if devices else [1, 2, 5], None)]
    if 3 in fam["ties"]:
        layouts.append((3, [2], 1))

    def engines(st):
        a = xt.TrackSet(st, CHUNK, devices=devices)
        one = xt.TrackSet(st, CHUNK) if devices else None
        b = xt.TrackSet(st, CHUNK)
        b.engine.set_option("plan_verify", 0)
        for ts in (a, one, b):
            if ts is not None:
                for k, val in opts.items():
                    ts.engine.set_option(k, val)
        return a, one, b

    for step, flipped, n_replanned in layouts:
        t = fam["ties"][step][0]
        p_tie, p_hi = (engine_params(at(model, th), d) for th in (t, up(t)))
        st, chunks = tie_data(xt, fam, n_chunks, flipped, step)
        a, one, b = engines(st)
        try:
            def both(p):
                va, vb = a.sum_logp(p), b.sum_logp(p)
                assert va == vb
                if one is not None:
                    assert one.sum_logp(p) == va
                assert b.engine.stats()["plan_verified"] == 0
                for c, (_, lo, hi, _) in enumerate(chunks):
                    np.testing.assert_array_equal(a.engine.chunk_logp(c, hi - lo, p), b.engine.chunk_logp(c, hi - lo, p))
                s = a.engine.stats()
                return s["plan_verified"], s["replanned"]

            assert both(p_hi) == (0, 0)          # construction
            assert both(p_hi) == (1, 0)          # along the resident plan, nothing changed
            if n_replanned is None:              # too many changed chunks: construction from scratch
                assert both(p_tie)[0] == 0
                continue
            assert both(p_tie) == (1, n_replanned)
            eng = one.engine if devices else a.engine
            lo = chunks[flipped[0]][1]
            assert_plan_is_oracle(eng, flipped[0], st[0][lo : lo + CHUNK], at(model, t), chunks[flipped[0]][3])
            # the frozen-plan entry points see the re-planned chunks' plans
            if opts.get("fp32_replay"):
                with pytest.raises(NotImplementedError):  # frozen-plan evaluations run the FP64 replay only
                    a.engine.eval_frozen([p_tie])
            elif devices:
                np.testing.assert_array_equal(a.engine.eval_frozen([p_tie]), b.engine.eval_frozen([p_tie]))
            else:
                sa, ta = a.engine.eval_frozen([p_tie], per_track=True)
                sb, tb = b.engine.eval_frozen([p_tie], per_track=True)
                np.testing.assert_array_equal(sa, sb)
                np.testing.assert_array_equal(ta, tb)
            assert both(p_hi) == (1, n_replanned)  # back across the tie
            assert both(p_hi) == (1, 0)            # the re-planned chunks' verification records hold again
        finally:
            for ts in (a, one, b):
                if ts is not None:
                    ts.close()


# ---------------------------------------------------------------------------------------------------------------
# state annotation at the tie (GPU)
# ---------------------------------------------------------------------------------------------------------------
PRED_ATOL = 1e-10
ANNOTATION_FAMILIES = ("s2_2d", "s3_3d", "s2_locdim")


@functools.lru_cache(maxsize=None)
def own_plan_ties(name, n=40, want=4):
    """Tracks whose own plan (one-track chunk, posteriors kept) flips at a tie that moves the oracle posteriors by more
    than 1e-8: (tracks, model, [(track, model threshold)])."""
    f = FAMILIES[name]
    model = make_model(**f["model"])
    C = random_walk_tracks(n, f["L"], f["d"], np.random.default_rng(77), Ds=model.ds**2 / 0.04)
    out = []
    for i in range(n):
        for t in tie_thresholds(C[i : i + 1], model, 2, do_preds=1, want=1):
            pa = orc.chunk_recursion(C[i : i + 1], at(model, t), 1, 1)[2]
            pb = orc.chunk_recursion(C[i : i + 1], at(model, up(t)), 1, 1)[2]
            if np.max(np.abs(pa - pb)) > 1e-8:
                out.append((i, t))
        if len(out) >= want:
            break
    return C, model, out


@pytest.mark.parametrize("name", ANNOTATION_FAMILIES)
def test_own_plan_tie_fixtures_move_the_posteriors(name):
    C, model, ties = own_plan_ties(name)
    assert ties, "no track with a posterior-moving tie"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ANNOTATION_FAMILIES)
def test_own_plan_annotation_at_the_tie(name, native):
    """predict_Bs with nb_max = 1 (every track planned from its own numbers): at th = t and nextafter(t) the posteriors
    of the tie's track equal the oracle's (which differ by more than 1e-8 between the two thresholds); the transition,
    residual and path instantiations return the same posteriors bit for bit."""
    C, model, ties = own_plan_ties(name)
    assert ties
    nS, d = model.nS, C.shape[2]
    eng = native.Engine(0)
    try:
        eng.upload([C], [1], 2000)
        for i, t in ties:
            want = {th: orc.chunk_recursion(C[i : i + 1], at(model, th), 1, 1)[2][0] for th in (t, up(t))}
            assert np.max(np.abs(want[t] - want[up(t)])) > 1e-8
            for th in (t, up(t)):
                p = engine_params(at(model, th), d)
                got = eng.predict(p, nS)[0]
                np.testing.assert_allclose(got[i], want[th], rtol=0, atol=PRED_ATOL)
                for other in (eng.predict_pairs(p, nS)[0], eng.predict_residuals(p, nS)[0], eng.predict_path(p, nS)[0]):
                    assert np.array_equal(other[0], got)
    finally:
        eng.close()


@functools.lru_cache(maxsize=None)
def shared_plan_ties(name):
    """The family's 30-track block, ties found with the posteriors kept (do_preds), that move them by more than 1e-8.
    One bucket is the longest one: no end-of-track expansion (isBL = 0), as predict_states has it."""
    fam = family(name)
    C, model = fam["C"], fam["model"]
    out = []
    for t in tie_thresholds(C, model, 2, isBL=0, do_preds=1, want=3):
        pa = orc.chunk_recursion(C, at(model, t), 0, 1)[2]
        pb = orc.chunk_recursion(C, at(model, up(t)), 0, 1)[2]
        if np.max(np.abs(pa - pb)) > 1e-8:
            out.append(t)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("nb_max", [30, 50])
@pytest.mark.parametrize("name", ANNOTATION_FAMILIES)
def test_shared_plan_annotation_at_the_tie(name, nb_max, native):
    """predict_Bs with nb_max > 1: the tie block forms the first 30 tracks (the leaders) of the first chunk; posteriors
    of every track equal the oracle's at th = t and nextafter(t)."""
    fam = family(name)
    ties = shared_plan_ties(name)
    assert ties
    model = fam["model"]
    extra = random_walk_tracks(20, fam["C"].shape[1], fam["C"].shape[2], np.random.default_rng(3), Ds=model.ds**2 / 0.04)
    X = np.concatenate([fam["C"], extra])
    eng = native.Engine(0)
    try:
        eng.upload([X], [0], nb_max)
        eng.set_option("predict_shared_plans", 1)
        for t in ties:
            want = {th: orc.predict_states([X], at(model, th), nb_max=nb_max)[0] for th in (t, up(t))}
            assert np.max(np.abs(want[t][:TT] - want[up(t)][:TT])) > 1e-8
            for th in (t, up(t)):
                got = eng.predict(engine_params(at(model, th), X.shape[2]), model.nS)[0]
                np.testing.assert_allclose(got, want[th], rtol=0, atol=PRED_ATOL)
    finally:
        eng.close()
