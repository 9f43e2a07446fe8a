"""One-step-ahead residuals of the state annotation: the residual oracle against the pinned likelihood and against
``predict_states`` (CPU), and ``predict_residuals`` against the residual oracle, its calibration on data drawn from the
model and its response to mislinked localisations (GPU)."""
import glob
import os

import numpy as np
import pytest

from helpers import engine_params, load_var_case, make_model, random_walk_tracks, var_oracle_inputs
from oracle import extrack_oracle as orc
from oracle import resid_oracle as ro

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "s*.npz")) if "seglen_" not in f)
NBMAX_CASES = sorted(glob.glob(os.path.join(GOLDEN, "nbmax_*.npz")))
VAR_CASES = sorted(glob.glob(os.path.join(GOLDEN, "var_*.npz")))
_ids = lambda paths: [os.path.basename(p)[:-4] for p in paths]
LP_TOL, PIT_TOL = 1e-9, 1e-10


def golden_case(path):
    z = np.load(path, allow_pickle=False)
    if z["ref_preds"].size == 0:
        pytest.skip("nb_substeps > 1: predict_Bs forces nb_substeps = 1")
    m = orc.Model(z["loc_err"], z["ds"], z["Fs"], z["TrMat"], float(z["pBL"]), list(z["cell_dims"]), 1, int(z["frame_len"]),
                  int(z["min_len"]), 0.1, 200)  # predict_Bs' defaults (threshold 0.1, max_nb_states 200, nb_substeps 1)
    n = z["ref_preds"].shape[0]
    return z["C"][:n], int(z["isBL"]), m


def nbmax_case(path):
    from test_oracle import load_nbmax_case

    from extrack_b200 import tracking as xt

    tracks, _, params, nS, fl, nb_max = load_nbmax_case(path)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, 0.02, nS, 1)
    keys = sorted(tracks, key=int)
    m = orc.Model(np.asarray(LocErr[0]).reshape(-1), ds, Fs, TrMat, pBL, [1], 1, fl, tracks[keys[0]].shape[1], 0.1, 200)
    return tracks, keys, params, nS, fl, nb_max, m


def simulate(n, L, d, Ds, Fs, TrMat, loc_err, dt, rng):
    """Tracks drawn from the annotation model itself: s_0 ~ Fs, s_k ~ TrMat[s_k-1], the increment k-1 -> k Gaussian with
    the variance dd of its head, (ds[s_k-1]^2 + ds[s_k]^2) / 2 per dimension, and Gaussian localisation errors."""
    d2 = 2 * np.asarray(Ds, dtype=float) * dt
    cum = np.cumsum(TrMat, axis=1)
    s = np.empty((n, L), dtype=int)
    s[:, 0] = np.searchsorted(np.cumsum(Fs), rng.random(n) * np.sum(Fs), side="right")
    for k in range(1, L):
        s[:, k] = np.minimum((rng.random(n)[:, None] > cum[s[:, k - 1]]).sum(1), len(Fs) - 1)
    var = (d2[s[:, 1:]] + d2[s[:, :-1]]) / 2
    steps = rng.normal(size=(n, L - 1, d)) * np.sqrt(var)[:, :, None]
    x0 = rng.random((n, 1, d))
    x = np.concatenate([x0, x0 + np.cumsum(steps, 1)], axis=1)
    return x + rng.normal(size=x.shape) * loc_err


def lmfit_params(Ds, Fs, TrMat, loc_err, pBL):
    """Parameters whose extract_params gives back (Ds, Fs, TrMat) with rows summing to 1."""
    from extrack_b200._lmfit_compat import Parameters

    nS = len(Ds)
    p = Parameters()
    for i in range(nS):
        p.add("D%d" % i, value=float(Ds[i]))
        p.add("F%d" % i, value=float(Fs[i]))
        for j in range(nS):
            if i != j:
                p.add("p%d%d" % (i, j), value=float(-np.log(1 - TrMat[i, j])) if TrMat[i, j] > 0 else 0.0)
    p.add("LocErr", value=loc_err)
    p.add("pBL", value=pBL)
    return p


# ---------------------------------------------------------------- CPU: the residual oracle
@pytest.mark.parametrize("nS,d", [(2, 1), (2, 3), (3, 1), (3, 3)])
def test_resid_oracle_matches_pinned_likelihood(nS, d):
    """No fusion (tracks no longer than frame_len, a vanishing threshold), p_stay = 1 (a huge cell) and pBL ~ 0: every
    field-of-view and bleaching term is 0, so the predictive of c_k is the ratio of the likelihoods of two prefixes."""
    L = 7
    m = make_model(nS=nS, frame_len=L, threshold=1e-9, max_nb_states=10**6, min_len=3, pBL=1e-18, cell_dims=(1e6,), rates=0.3)
    assert np.allclose(m.TrMat.sum(1), 1) and np.isclose(m.Fs.sum(), 1)
    C = random_walk_tracks(5, L, d, np.random.default_rng(40 + nS + d), Ds=m.ds**2 / 0.04)
    _, _, logpred, pit = ro.chunk_recursion_resid(C, m, 0)
    assert np.all(np.isnan(logpred[:, 0])) and np.all(np.isnan(pit[:, 0]))
    assert np.all((pit[:, 1:] > 0) & (pit[:, 1:] < 1))
    ll = [None, None] + [orc.chunk_logp(C[:, :n], m, 0) for n in range(2, L + 1)]
    np.testing.assert_allclose(logpred[:, 1], ll[2], rtol=0, atol=1e-10)
    for k in range(2, L):
        np.testing.assert_allclose(logpred[:, k], ll[k + 1] - ll[k], rtol=0, atol=1e-10)


@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_resid_oracle_posteriors_equal_predict_states(path):
    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    for i in range(len(C)):
        _, preds, logpred, pit = ro.chunk_recursion_resid(C[i : i + 1], m, isBL, tb)
        assert np.array_equal(preds, orc.chunk_recursion(C[i : i + 1], m, isBL, 1, None, tb)[2])
        assert np.all(np.isfinite(logpred[:, 1:])) and np.all((pit[:, 1:] >= 0) & (pit[:, 1:] <= 1))


@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_resid_oracle_with_shared_plans_posteriors_equal_predict_states(path):
    tracks, keys, _, _, _, nb_max, m = nbmax_case(path)
    st = [tracks[k] for k in keys]
    for w, (preds, logpred, pit) in zip(orc.predict_states(st, m, nb_max=nb_max), ro.predict_residuals(st, m, nb_max=nb_max)):
        assert np.array_equal(preds, w)
        assert logpred.shape == preds.shape[:2] and pit.shape == preds.shape[:2] + (st[0].shape[2],)


@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_resid_oracle_with_peakwise_inputs_posteriors_equal_predict_states(path):
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    for w, (preds, _, _) in zip(orc.predict_states(st, m, 1, sigs, ds_list), ro.predict_residuals(st, m, 1, sigs, ds_list)):
        assert np.array_equal(preds, w)


# ---------------------------------------------------------------- GPU: predict_residuals
@pytest.fixture(scope="module")
def xt():
    from extrack_b200 import tracking

    return tracking


def check_close(logpred, pit, want_lp, want_pit):
    assert np.array_equal(np.isnan(logpred), np.isnan(want_lp)) and np.array_equal(np.isnan(pit), np.isnan(want_pit))
    np.testing.assert_allclose(logpred, want_lp, rtol=0, atol=LP_TOL)
    np.testing.assert_allclose(pit, want_pit, rtol=0, atol=PIT_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_engine_residuals_match_oracle_on_golden_tracks(path):
    """nb_max = 1 (own plans, NSC 2 / 3 and generic instantiations): 2, 3 and 4 states, 2-D and 3-D."""
    from extrack_b200 import _native

    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    want = [ro.chunk_recursion_resid(C[i : i + 1], m, isBL, tb) for i in range(len(C))]
    eng = _native.Engine(0)
    try:
        eng.upload([C], [isBL], 2000)
        p = engine_params(m, C.shape[2])
        preds_only = eng.predict(p, m.nS)[0]
        (preds,), (logpred,), (pit,) = eng.predict_residuals(p, m.nS)
    finally:
        eng.close()
    assert np.array_equal(preds, preds_only)
    check_close(logpred, pit, np.concatenate([w[2] for w in want]), np.concatenate([w[3] for w in want]))


@pytest.mark.gpu
@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_predict_residuals_with_shared_plans_matches_oracle(path, xt):
    """nb_max > 1 (plans shared per chunk, the FOLLOW instantiation)."""
    tracks, keys, params, nS, fl, nb_max, m = nbmax_case(path)
    preds, logpred, pit = xt.predict_residuals(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    ref = xt.predict_Bs(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    assert set(preds) == set(logpred) == set(pit) == set(tracks)
    for k, (_, wl, wp) in zip(keys, ro.predict_residuals([tracks[k] for k in keys], m, nb_max=nb_max)):
        assert np.array_equal(preds[k], ref[k])
        check_close(logpred[k], pit[k], wl, wp)


@pytest.mark.gpu
@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_predict_residuals_with_peakwise_inputs_matches_oracle(path, xt):
    """Peak-wise LocErr (with slope / offset in some cases) and per-track dt, nb_max = 1."""
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    tr = {str(a.shape[1]): a for a in st}
    ild = None if il is None else {str(a.shape[1]): x for a, x in zip(st, il)}
    dtd = 0.02 if dts is None else {str(a.shape[1]): x for a, x in zip(st, dts)}
    kw = dict(cell_dims=[1], nb_states=cfg["nS"], frame_len=cfg["fl"], input_LocErr=ild)
    preds, logpred, pit = xt.predict_residuals(tr, dtd, params, **kw)
    only = xt.predict_Bs(tr, dtd, params, **kw)
    for a, (_, wl, wp) in zip(st, ro.predict_residuals(st, m, 1, sigs, ds_list)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], only[k])
        check_close(logpred[k], pit[k], wl, wp)


def _api_case():
    from extrack_b200._lmfit_compat import Parameters

    rng = np.random.default_rng(21)
    tracks = {str(L): random_walk_tracks(n, L, 2, rng) for L, n in ((2, 3), (3, 4), (7, 40), (15, 70), (31, 33))}
    tracks["9"] = np.zeros((0, 9, 2))
    p = Parameters()
    for k, v in dict(D0=1e-5, D1=0.25, LocErr=0.02, F0=0.6, p01=0.1, p10=0.12, pBL=0.05).items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    return tracks, p


@pytest.mark.gpu
def test_predict_residuals_api_buckets_and_errors(xt):
    """L = 2 and 3, bleaching buckets and the longest bucket, an empty bucket, and predict_Bs' errors."""
    tracks, p = _api_case()
    preds, logpred, pit = xt.predict_residuals(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    assert set(preds) == set(logpred) == set(pit) == set(tracks)
    assert preds["9"].shape == (0, 9, 2) and logpred["9"].shape == (0, 9) and pit["9"].shape == (0, 9, 2)
    st, _ = xt._sorted_buckets(tracks)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    m = orc.Model(LocErr[0].reshape(-1), ds, Fs, TrMat, pBL, [1], 1, 8, 2, 0.1, 200)
    ref = xt.predict_Bs(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    for a, (_, wl, wp) in zip(st, ro.predict_residuals(st, m, nb_max=1)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], ref[k])
        check_close(logpred[k], pit[k], wl, wp)
    with pytest.raises(NotImplementedError):
        xt.predict_residuals(tracks, 0.02, p, nb_states=2, nb_max=50,
                             input_LocErr={k: np.full(v.shape[:2] + (1,), 0.02) for k, v in tracks.items()})
    with pytest.raises(NotImplementedError):
        xt.predict_residuals(tracks, {k: np.full(v.shape[:2], 0.02) for k, v in tracks.items()}, p, nb_states=2, nb_max=50)
    with pytest.raises(TypeError):
        xt.predict_residuals(tracks, 0.02, {"D0": 1.0}, nb_states=2)
    with pytest.raises(ValueError):
        xt.predict_residuals(tracks, 0.02, p, nb_states=3)


@pytest.mark.gpu
def test_engine_residuals_identical_after_capacity_retry():
    """A small first capacity makes most tracks run again with more: outputs are those of one run."""
    from extrack_b200 import _native

    m = make_model(nS=3, frame_len=7, threshold=0.05, max_nb_states=200, min_len=5)
    C = random_walk_tracks(300, 16, 2, np.random.default_rng(8), Ds=m.ds**2 / 0.04)
    res = []
    for cap0 in (None, 27):
        eng = _native.Engine(0)
        try:
            eng.upload([C], [1], 2000)
            if cap0:
                eng.set_option("k3_cap0", cap0)
            res.append(eng.predict_residuals(engine_params(m, 2), 3))
            if cap0:
                assert eng.stats()["k3_launches"] > 1
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a[0], b[0], equal_nan=True)


@pytest.mark.gpu
def test_engine_residuals_identical_with_and_without_pieces():
    """Large enough for the launch in pieces with the read-back of a piece under the next: same outputs as one launch."""
    from extrack_b200 import _native

    m = make_model(nS=2, frame_len=6, threshold=0.1, max_nb_states=200, min_len=4)
    rng = np.random.default_rng(9)
    segs = [random_walk_tracks(90_000, L, 2, rng) for L in (4, 5, 6, 8)]
    res = []
    for pieces in (1, None):
        eng = _native.Engine(0)
        try:
            eng.upload(segs, [1, 1, 1, 0], 2000)
            if pieces:
                eng.set_option("k3_pieces", pieces)
            res.append(eng.predict_residuals(engine_params(m, 2), 2))
            launches = eng.stats()["k3_launches"]
            assert (launches == 1) if pieces else (launches > 1)
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("nS", [2, 3])
def test_pit_is_uniform_on_tracks_drawn_from_the_model(nS, xt):
    """Data from the model's own law, annotated at the true parameters without fusion (length 6, frame_len 8, a
    vanishing threshold) in a huge cell: the pooled PIT values of every dimension pass a Kolmogorov-Smirnov test."""
    from scipy.stats import kstest

    Ds = [1e-5, 0.25] if nS == 2 else [1e-5, 0.04, 0.25]
    Fs = np.full(nS, 1.0 / nS)
    TrMat = np.full((nS, nS), 0.15 / (nS - 1))
    np.fill_diagonal(TrMat, 0.85)
    p = lmfit_params(Ds, Fs, TrMat, 0.02, 1e-12)
    np.testing.assert_allclose(xt.extract_params(p, 0.02, nS, 1)[3], TrMat, rtol=1e-12)
    tracks = {"6": simulate(25_000, 6, 2, Ds, Fs, TrMat, 0.02, 0.02, np.random.default_rng(100 + nS))}
    _, logpred, pit = xt.predict_residuals(tracks, 0.02, p, cell_dims=[1e6], nb_states=nS, frame_len=8, threshold=1e-9,
                                           max_nb_states=10**6)
    assert np.all(np.isnan(pit["6"][:, 0])) and np.all(np.isfinite(logpred["6"][:, 1:]))
    for x in range(2):
        u = pit["6"][:, 1:, x].ravel()
        assert u.size >= 100_000
        stat = kstest(u, "uniform").statistic
        assert stat < 1.95 / np.sqrt(u.size), (x, stat)


@pytest.mark.gpu
def test_logpred_finds_mislinked_localisations(xt):
    """One interior localisation per track moved by 20 fast-state step lengths: the track's lowest log predictive
    density is at that localisation or the next one (the jump away and the jump back), under the normal approximate
    recursion (frame_len 5: sequences fuse)."""
    Ds, Fs = [1e-5, 0.25], np.array([0.6, 0.4])
    TrMat = np.array([[0.9, 0.1], [0.1, 0.9]])
    p = lmfit_params(Ds, Fs, TrMat, 0.02, 0.05)
    rng = np.random.default_rng(12)
    L, n = 20, 1000
    C = simulate(n, L, 2, Ds, Fs, TrMat, 0.02, 0.02, rng)
    j = rng.integers(1, L - 1, size=n)
    phi = rng.random(n) * 2 * np.pi
    C[np.arange(n), j] += 20 * np.sqrt(2 * Ds[1] * 0.02) * np.stack([np.cos(phi), np.sin(phi)], 1)
    _, logpred, _ = xt.predict_residuals({str(L): C}, 0.02, p, cell_dims=[1], nb_states=2, frame_len=5)
    k = np.nanargmin(logpred[str(L)], axis=1)
    rate = np.mean((k == j) | (k == j + 1))
    assert rate >= 0.99, rate
