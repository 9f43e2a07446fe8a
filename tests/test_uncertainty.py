"""Standard errors along the frozen grouping plan: the frozen oracle against the oracle (CPU), the assembly on a
synthetic quadratic surface (CPU), the information equality on exact data (CPU oracle, GPU engine), the engine's frozen
evaluations and scores against the oracle and numpy, their absence of side effects and their errors (GPU), and the
calibration of ``param_uncertainty`` over repeated fits (GPU)."""
import os
import warnings

import numpy as np
import pytest

from helpers import engine_params, make_model, random_walk_tracks
from oracle import extrack_oracle as orc
from oracle import score_oracle as so

DT = 0.02


# ----------------------------------------------------------------------------------------------------------------------
# fixtures: exact generator and parameter sets
# ----------------------------------------------------------------------------------------------------------------------
def truth_params(D0=0.005, D1=0.25, LocErr=0.02, p01=0.1, p10=0.2, pBL=0.1):
    """2-state parameters with F0 = stationary law of the per-step transition matrix; pBL held fixed."""
    from extrack_b200._lmfit_compat import Parameters

    T01, T10 = 1 - np.exp(-p01), 1 - np.exp(-p10)
    prm = Parameters()
    prm.add("D0", value=D0, min=0, max=3)
    prm.add("D1", value=D1, min=0, max=3)
    prm.add("LocErr", value=LocErr, min=0.005, max=0.1)
    prm.add("F0", value=T10 / (T01 + T10), min=0.001, max=0.999)
    prm.add("F1", expr="1 - F0")
    prm.add("p01", value=p01, min=0.0001, max=1)
    prm.add("p10", value=p10, min=0.0001, max=1)
    prm.add("pBL", value=pBL, min=0.0001, max=1, vary=False)
    return prm


def exact_tracks(prm, n, L, d, rng):
    """Tracks drawn from the model: a stationary 2-state chain (reversible, so the direction of the recursion does not
    matter), step variance (ds[s_k]^2 + ds[s_k+1]^2) / 2 per dimension, Gaussian localisation noise."""
    Ds = np.array([prm["D0"].value, prm["D1"].value])
    T01, T10 = 1 - np.exp(-prm["p01"].value), 1 - np.exp(-prm["p10"].value)
    T = np.array([[1 - T01, T01], [T10, 1 - T10]])
    s = np.empty((n, L), dtype=int)
    s[:, 0] = (rng.random(n) >= prm["F0"].value).astype(int)
    for k in range(1, L):
        s[:, k] = (rng.random(n) < T[s[:, k - 1], 1]).astype(int)
    d2 = 2 * Ds * DT
    var = (d2[s[:, :-1]] + d2[s[:, 1:]]) / 2
    steps = rng.normal(size=(n, L - 1, d)) * np.sqrt(var)[:, :, None]
    pos = np.concatenate([np.zeros((n, 1, d)), np.cumsum(steps, 1)], 1) + 10 * rng.random((n, 1, d))
    return pos + rng.normal(size=(n, L, d)) * prm["LocErr"].value


EXACT = dict(frame_len=8, threshold=1e-12, max_nb_states=10**6, cell_dims=[1000.0])  # no group has two members


def oracle_model(prm, L, frame_len, threshold, max_nb_states, cell_dims):
    from extrack_b200 import tracking as xt

    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(prm, DT, 2, 1)
    return orc.Model(np.asarray(LocErr[0]).reshape(-1), ds, Fs, TrMat, pBL, cell_dims, 1, frame_len, L, threshold, max_nb_states)


def oracle_backend(prm, fds, act, cfg, L):
    """``uncertainty_from_backend`` callables on the frozen oracle."""
    from extrack_b200 import tracking as xt

    def lp(th, k):
        q = prm.copy()
        for n, v in zip(act, th):
            q[n].value = float(v)
        m = oracle_model(q, L, **cfg)
        if not orc.model_valid(m):
            raise xt.InvalidPoint(k)
        return fds.logp(m)

    totals = lambda ths: np.array([np.sum(lp(t, k)) for k, t in enumerate(ths)])

    def score(plus, minus, inv_2h):
        P = np.array([lp(t, k) for k, t in enumerate(plus)])
        M = np.array([lp(t, k) for k, t in enumerate(minus)])
        g = ((P - M) * np.asarray(inv_2h)[:, None]).T
        return {"sum_plus": P.sum(1), "sum_minus": M.sum(1), "gsum": g.sum(0), "gram": g.T @ g}

    return totals, score


def free_names(prm, rel_step=1e-4):
    from extrack_b200 import tracking as xt

    return [n for n in prm.keys() if prm[n].vary and prm[n].expr is None and not xt._held(prm[n], rel_step)]


def check_information_equality(u, tol):
    assert np.all(np.abs(u.gradient) <= 4 * np.sqrt(np.diag(u.opg))), (u.gradient, np.sqrt(np.diag(u.opg)))
    rel = np.linalg.norm(u.opg - u.hessian) / np.linalg.norm(u.hessian)
    assert rel <= tol, rel


# ----------------------------------------------------------------------------------------------------------------------
# CPU
# ----------------------------------------------------------------------------------------------------------------------
def fusion_data(rng):
    return [random_walk_tracks(n, L, 2, rng) for n, L in ((300, 6), (250, 12), (120, 20))]


def test_frozen_oracle_bitwise():
    rng = np.random.default_rng(3)
    st = fusion_data(rng)
    m0 = make_model(frame_len=8, min_len=6)
    fds = so.FrozenDataSet(st, m0, chunk=200)
    assert any(len(g) > 1 for pl in fds.plans for r in pl for g in r["groups"]), "no fusion in the data"
    ref = np.concatenate([orc.chunk_logp(C, m0, isBL, sig=sg) for (C, isBL, sg) in fds.jobs])
    assert np.array_equal(fds.logp(m0), ref)
    m1 = make_model(frame_len=8, min_len=6)
    m1.ds = m1.ds * (1 + 1e-9)
    plans1 = [so.record_plan(C, m1, isBL, sg) for (C, isBL, sg) in fds.jobs]
    for a, b in zip(fds.plans, plans1):
        assert len(a) == len(b)
        for ra, rb in zip(a, b):
            assert ra["nB_in"] == rb["nB_in"] and ra["threshold"] == rb["threshold"]
            assert all(np.array_equal(x, y) for x, y in zip(ra["groups"], rb["groups"])) and len(ra["groups"]) == len(rb["groups"])
    ref1 = np.concatenate([orc.chunk_logp(C, m1, isBL, sig=sg) for (C, isBL, sg) in fds.jobs])
    assert np.array_equal(fds.logp(m1), ref1)


def test_frozen_oracle_peakwise_bitwise():
    rng = np.random.default_rng(4)
    st = [random_walk_tracks(80, 9, 2, rng)]
    sig = [0.015 + 0.01 * rng.random((80, 9, 1))]
    m0 = make_model(frame_len=6, min_len=9)
    fds = so.FrozenDataSet(st, m0, chunk=50, sigs=sig)
    ref = np.concatenate([orc.chunk_logp(C, m0, isBL, sig=sg) for (C, isBL, sg) in fds.jobs])
    assert np.array_equal(fds.logp(m0), ref)


def synthetic_params():
    from extrack_b200._lmfit_compat import Parameters

    prm = Parameters()
    prm.add("D0", value=0.5, min=0, max=1)
    prm.add("D1_minus_D0", value=0.3, min=0, max=10)
    prm.add("D1", expr="D0+D1_minus_D0")
    prm.add("F0", value=0.4, min=0.001, max=0.999)
    prm.add("F1", expr="1-F0")
    prm.add("p01", value=0.01, min=0.01, max=1)  # at its lower bound: held
    prm.add("pBL", value=0.1, min=0.01, max=0.99, vary=False)
    return prm


def test_assembly_synthetic_quadratic():
    """log P_t(theta) = g_t . (theta - theta0) - (theta - theta0)^T A (theta - theta0) / (2 T): H = A, J = sum g g^T."""
    from extrack_b200 import tracking as xt

    prm = synthetic_params()
    act = free_names(prm)
    assert act == ["D0", "D1_minus_D0", "F0"]
    th0 = np.array([prm[n].value for n in act])
    rng = np.random.default_rng(0)
    T = 500
    G = rng.normal(size=(T, 3)) * np.array([30.0, 20.0, 50.0])
    B = rng.normal(size=(3, 3))
    A = B @ B.T * 1e3 + np.diag([5e3, 4e3, 9e3])

    def lp(th):
        x = np.asarray(th) - th0
        return G @ x - 0.5 * (x @ A @ x) / T

    totals = lambda ths: np.array([np.sum(lp(t)) for t in ths])

    def score(plus, minus, inv_2h):
        P = np.array([lp(t) for t in plus])
        M = np.array([lp(t) for t in minus])
        g = ((P - M) * np.asarray(inv_2h)[:, None]).T
        return {"sum_plus": P.sum(1), "sum_minus": M.sum(1), "gsum": g.sum(0), "gram": g.T @ g}

    u = xt.uncertainty_from_backend(prm, totals, score)
    J = G.T @ G
    cov = np.linalg.inv(A)
    assert u.names == act and u.at_bound == ["p01"]
    np.testing.assert_allclose(u.hessian, A, rtol=1e-8)
    np.testing.assert_allclose(u.opg, J, rtol=1e-8)
    np.testing.assert_allclose(u.covar, cov, rtol=1e-8)
    np.testing.assert_allclose(u.covar_robust, cov @ J @ cov, rtol=1e-8)
    np.testing.assert_allclose(u.gradient, G.sum(0), rtol=1e-8)
    np.testing.assert_allclose(u.newton_decrement, G.sum(0) @ cov @ G.sum(0), rtol=1e-8)
    np.testing.assert_allclose(u.stderr["F1"], u.stderr["F0"], rtol=1e-8)
    np.testing.assert_allclose(u.stderr["D1"], np.sqrt(cov[0, 0] + cov[1, 1] + 2 * cov[0, 1]), rtol=1e-8)
    rob = cov @ J @ cov
    np.testing.assert_allclose(u.stderr_robust["D1"], np.sqrt(rob[0, 0] + rob[1, 1] + 2 * rob[0, 1]), rtol=1e-8)
    assert np.isnan(u.stderr["p01"]) and u.stderr["pBL"] is None
    assert u.params["D0"].stderr == u.stderr["D0"] and "F0" in u.params["D0"].correl
    sd = np.sqrt(np.diag(cov))
    np.testing.assert_allclose(u.correl, cov / np.outer(sd, sd), rtol=1e-8)


def test_assembly_not_positive_definite_warns():
    from extrack_b200 import tracking as xt

    prm = synthetic_params()
    totals = lambda ths: np.array([float(np.sum((np.asarray(t) - 0.5) ** 2)) for t in ths])  # a minimum, not a maximum

    def score(plus, minus, inv_2h):
        n = len(plus)
        return {"sum_plus": totals(plus), "sum_minus": totals(minus), "gsum": np.zeros(n), "gram": np.eye(n)}

    with pytest.warns(RuntimeWarning, match="positive definite"):
        u = xt.uncertainty_from_backend(prm, totals, score)
    assert np.all(np.isnan(u.covar)) and np.isnan(u.stderr["D0"])


def test_assembly_names_invalid_step():
    from extrack_b200 import tracking as xt

    prm = synthetic_params()

    def score(plus, minus, inv_2h):
        raise xt.InvalidPoint(len(plus) + 2)  # the - step of the third parameter

    with pytest.raises(ValueError, match="F0"):
        xt.uncertainty_from_backend(prm, lambda ths: np.zeros(len(ths)), score)


def test_information_equality_oracle():
    from extrack_b200 import tracking as xt

    prm = truth_params()
    L = 6
    st = [exact_tracks(prm, 10**4, L, 2, np.random.default_rng(11))]
    fds = so.FrozenDataSet(st, oracle_model(prm, L, **EXACT), chunk=2000)
    assert all(len(g) == 1 for pl in fds.plans for r in pl for g in r["groups"])
    act = free_names(prm)
    assert "pBL" not in act and len(act) == 6
    totals, score = oracle_backend(prm, fds, act, EXACT, L)
    u = xt.uncertainty_from_backend(prm, totals, score)
    check_information_equality(u, 0.1)


# ----------------------------------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------------------------------
def _engine_for(st, chunk, sigma=None):
    from extrack_b200 import _native

    jobs = orc.make_chunks(st, chunk)
    eng = _native.Engine(0)
    eng.upload([st[b][a:z] for (b, a, z, _) in jobs], [bl for (_, _, _, bl) in jobs], chunk)
    if sigma is not None:
        eng.upload_aux([sigma[b][a:z] for (b, a, z, _) in jobs], None)
    return eng


def _scaled(m, f):
    m2 = orc.Model(m.loc_err * f, m.ds * f, m.Fs, m.TrMat, m.pBL, m.cell_dims, m.nb_substeps, m.frame_len, m.min_len,
                   m.threshold, m.max_nb_states, m.int8_wrap)
    return m2


def _case(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "fusion":
        st = [random_walk_tracks(n, L, 2, rng) for n, L in ((300, 6), (2100, 12), (150, 20))]
        return st, make_model(frame_len=8, min_len=6), None, None
    if name == "3state_3d":
        st = [random_walk_tracks(200, 8, 3, rng, Ds=(1e-5, 0.04, 0.25))]
        return st, make_model(nS=3, loc_err=(0.02, 0.025, 0.03), frame_len=5, min_len=8), None, None
    if name == "substeps2":
        st = [random_walk_tracks(300, 7, 2, rng)]
        return st, make_model(nsub=2, frame_len=5, min_len=7), None, None
    if name == "peakwise":
        st = [random_walk_tracks(250, 8, 2, rng)]
        return st, make_model(frame_len=6, min_len=8), [0.01 + 0.02 * rng.random((250, 8, 1))], (1.1, 0.002)
    if name == "many_sequences":
        st = [random_walk_tracks(100, 12, 2, rng, Ds=(1e-5, 0.04, 0.25))]
        return st, make_model(nS=3, frame_len=9, min_len=12, threshold=0.02, max_nb_states=400), None, None
    raise KeyError(name)


def _engine_p(m, d, peak):
    from extrack_b200 import tracking as xt

    if peak is None:
        return engine_params(m, d)
    return xt.build_tables(m.loc_err, m.ds, m.Fs, m.TrMat, m.pBL, m.cell_dims, m.nb_substeps, m.frame_len, m.min_len,
                           m.threshold, m.max_nb_states, d, m.int8_wrap, var_loc_k=1, slope_offset=peak)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fusion", "3state_3d", "substeps2", "peakwise", "many_sequences"])
def test_eval_frozen_matches_oracle(name):
    st, m0, sigma, peak = _case(name)
    d = st[0].shape[2]
    chunk = 2000
    eng = _engine_for(st, chunk, sigma)
    try:
        sig = None if sigma is None else [np.clip(a * peak[0] + peak[1], 1e-6, np.inf) for a in sigma]
        fds = so.FrozenDataSet(st, m0, chunk=chunk, sigs=sig)
        p0 = _engine_p(m0, d, peak)
        total = eng.sum_logp(p0)
        models = [m0, _scaled(m0, 1 + 1e-4), _scaled(m0, 1 - 1e-4)]
        sums, per = eng.eval_frozen([_engine_p(m, d, peak) for m in models], per_track=True)
        for k, m in enumerate(models):
            ref = fds.logp(m)
            np.testing.assert_allclose(per[k], ref, rtol=1e-9, atol=0)
        assert sums[0] == total  # the objective's bits at the plan's own parameters
        if name == "many_sequences":
            assert eng.stats()["max_nB_in"] > 64
    finally:
        eng.close()


@pytest.mark.gpu
def test_frozen_calls_have_no_side_effects():
    from extrack_b200 import _native

    st, m0, _, _ = _case("fusion")
    p1, p2 = engine_params(m0, 2), engine_params(_scaled(m0, 1.01), 2)
    fresh = _engine_for(st, 2000)
    eng = _engine_for(st, 2000)
    try:
        ref2 = fresh.sum_logp(p2)
        ref_chunk = fresh.chunk_logp(2, 2000, p2)
        ref_plan = fresh.plan_dump(2, 5)
        eng.sum_logp(p1)
        eng.eval_frozen([p1, p2, engine_params(_scaled(m0, 0.99), 2)], per_track=True)
        eng.score_outer([p2], [p1], [1.0])
        got = eng.sum_logp(p2)
        assert got == ref2
        assert np.array_equal(eng.chunk_logp(2, 2000, p2), ref_chunk)
        a, b = eng.plan_dump(2, 5), ref_plan
        assert a[0] == b[0] and a[1] == b[1] and np.array_equal(a[2], b[2]) and a[3] == b[3]
        st_ = eng.stats()
        assert st_["plan_verified"] == 1 and st_["replanned"] == 0
        eng.set_option("fp32_replay", 1)
        eng.sum_logp(p1)
        with pytest.raises(NotImplementedError, match="fp32_replay"):  # XT_ERR_UNSUPPORTED
            eng.eval_frozen([p1])
    finally:
        eng.close()
        fresh.close()


@pytest.mark.gpu
def test_score_outer_gram_and_shards():
    from extrack_b200 import _native

    st, m0, _, _ = _case("fusion")
    models_p = [_scaled(m0, 1 + 1e-4), _scaled(m0, 1 + 2e-4)]
    models_m = [_scaled(m0, 1 - 1e-4), _scaled(m0, 1 - 2e-4)]
    pp, pm = [engine_params(m, 2) for m in models_p], [engine_params(m, 2) for m in models_m]
    inv = np.array([1 / 2e-4, 1 / 4e-4])
    p0 = engine_params(m0, 2)
    eng = _engine_for(st, 2000)
    try:
        eng.sum_logp(p0)
        r = eng.score_outer(pp, pm, inv)
        _, P = eng.eval_frozen(pp, per_track=True)
        _, M = eng.eval_frozen(pm, per_track=True)
        g = ((P - M) * inv[:, None]).T
        np.testing.assert_allclose(r["gsum"], g.sum(0), rtol=1e-12)
        np.testing.assert_allclose(r["gram"], g.T @ g, rtol=1e-12)
        np.testing.assert_allclose(r["sum_plus"], P.sum(1), rtol=1e-12)
    finally:
        eng.close()
    # one context holding all chunks (whole buckets uploaded as segments) vs logical and physical shards
    isBL = [1, 1, 0]
    one = _native.Engine(0)
    one.upload(st, isBL, 2000)
    one.sum_logp(p0)
    ref = one.score_outer(pp, pm, inv)
    ref_s = one.eval_frozen(pp + pm)
    one.close()
    devsets = [[0, 0]]
    if _native.device_count() > 1:
        devsets.append(list(range(_native.device_count())))
    for devs in devsets:
        me = _native.MultiEngine(devs)
        try:
            me.upload(st, isBL, 2000)
            me.sum_logp(p0)
            r = me.score_outer(pp, pm, inv)
            for k in ref:
                assert np.array_equal(r[k], ref[k]), (devs, k)
            assert np.array_equal(me.eval_frozen(pp + pm), ref_s)
        finally:
            me.close()


@pytest.mark.gpu
def test_frozen_errors():
    from extrack_b200 import _native, tracking as xt

    st, m0, _, _ = _case("3state_3d")
    eng = _engine_for(st, 2000)
    try:
        p0 = engine_params(m0, 3)
        with pytest.raises(_native.EngineError) as e:
            eng.eval_frozen([p0])
        assert e.value.code == _native.XT_ERR_STATE
        eng.sum_logp(p0)
        other = make_model(nS=3, loc_err=(0.02, 0.025, 0.03), frame_len=6, min_len=8)
        with pytest.raises(ValueError, match="differ in structure"):  # XT_ERR_ARG
            eng.eval_frozen([engine_params(other, 3)])
        with pytest.raises(ValueError, match="n_dir"):  # XT_ERR_ARG
            eng.score_outer([p0] * 33, [p0] * 33, np.ones(33))
        eng.upload_aux([np.full((200, 8, 1), 0.02)], None)
        with pytest.raises(_native.EngineError) as e:
            eng.eval_frozen([p0])
        assert e.value.code == _native.XT_ERR_STATE
    finally:
        eng.close()
    with pytest.raises(NotImplementedError):
        xt.param_uncertainty({"8": st[0][:, :, :2]}, {"8": np.full((200, 8), DT)}, truth_params())


@pytest.mark.gpu
def test_information_equality_engine():
    from extrack_b200 import tracking as xt

    prm = truth_params()
    tr = exact_tracks(prm, 10**5, 6, 2, np.random.default_rng(12))
    u = xt.param_uncertainty({"6": tr}, DT, prm, **EXACT)
    assert "pBL" not in u.names
    check_information_equality(u, 0.05)


def _fit(prm, tracks, **kw):
    from extrack_b200 import tracking as xt

    fit = xt.param_fitting(tracks, DT, params=prm.copy(), verbose=0, **kw)
    return fit


@pytest.mark.gpu
def test_calibration():
    """40 seeded data sets of 5000 exact tracks, each fitted from the truth, then param_uncertainty."""
    from extrack_b200 import tracking as xt

    prm = truth_params()
    names = free_names(prm)
    kw = dict(frame_len=6, cell_dims=[1000.0], threshold=0.2, max_nb_states=120)
    est, se, se_r = [], [], []
    u1 = None
    for seed in range(40):
        tracks = {"6": exact_tracks(prm, 5000, 6, 2, np.random.default_rng(1000 + seed))}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            fit = _fit(prm, tracks, **kw)
        u = xt.param_uncertainty(tracks, DT, fit, **kw)
        est.append([fit.params[n].value for n in names])
        se.append([u.stderr[n] for n in names])
        se_r.append([u.stderr_robust[n] for n in names])
        if seed == 0:
            u1, tracks1, fit1 = u, tracks, fit
    est, se, se_r = np.array(est), np.array(se), np.array(se_r)
    truth = np.array([prm[n].value for n in names])
    ratio = est.std(0, ddof=1) / se_r.mean(0)
    assert np.all((ratio >= 0.7) & (ratio <= 1.4)), dict(zip(names, ratio))
    cover = np.mean(np.abs(est - truth) <= 1.96 * se)
    assert cover >= 0.85, cover
    # 4x the tracks: stderr halves
    big = {"6": exact_tracks(prm, 20000, 6, 2, np.random.default_rng(999))}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        fit4 = _fit(prm, big, **kw)
    u4 = xt.param_uncertainty(big, DT, fit4, **kw)
    r4 = np.array([u4.stderr[n] for n in names]) / np.array([u1.stderr[n] for n in names])
    assert np.all((r4 >= 0.45) & (r4 <= 0.55)), dict(zip(names, r4))
    u3 = xt.param_uncertainty(tracks1, DT, fit1, rel_step=3e-4, **kw)
    for n in names:
        np.testing.assert_allclose(u3.stderr[n], u1.stderr[n], rtol=1e-3)
