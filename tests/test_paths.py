"""Most probable state paths (MAP / Viterbi paths) of the state annotation: the path oracle against brute-force
enumeration and against ``predict_states`` (CPU), ``path_segments``, the paths' agreement with simulated states (CPU),
and ``predict_path`` against the path oracle (GPU)."""
import glob
import os

import numpy as np
import pytest

from helpers import engine_params, load_var_case, make_model, random_walk_tracks, var_oracle_inputs
from oracle import extrack_oracle as orc
from oracle import path_oracle as pa

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "s*.npz")) if "seglen_" not in f)
NBMAX_CASES = sorted(glob.glob(os.path.join(GOLDEN, "nbmax_*.npz")))
VAR_CASES = sorted(glob.glob(os.path.join(GOLDEN, "var_*.npz")))
_ids = lambda paths: [os.path.basename(p)[:-4] for p in paths]
LOGP_TOL = 1e-10  # GPU vs oracle (FP64, different summation orders)
MARGIN = 1e-8  # smallest decision gap a GPU comparison accepts in its data (a near-tie is a property of the data)


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


def lse(x, axis):
    mx = np.max(x, axis=axis, keepdims=True)
    return (np.log(np.sum(np.exp(x - mx), axis=axis, keepdims=True)) + mx).squeeze(axis)


def enumerated_path(C, model, isBL):
    """The MAP path by direct enumeration over the surviving sequences (no fusion: every sequence's history is one-hot),
    from the oracle's final log-probabilities and histories.  At a bleaching end the K children of a sequence differ
    only in the hidden state after the last localisation, which no label shows: they are summed."""
    LP, hist, _ = orc.chunk_recursion(C, model, isBL, 1)
    h = np.broadcast_to(hist, (len(C),) + hist.shape[1:])[:, :, ::-1]  # [nT, nB, L, nS], forward time
    assert set(np.unique(h)) <= {0.0, 1.0}, "a fusion happened"
    LPs = lse(LP.reshape(len(C), -1, model.nS), 2) if isBL else LP
    if isBL:
        h = h[:, :: model.nS]
    j = np.argmax(LPs, axis=1)
    rows = np.arange(len(C))
    return np.argmax(h[rows, j], axis=-1).astype(np.int8), LPs[rows, j] - lse(LP, 1)


def check_bounds(preds, path, path_logp, tol=1e-12):
    """path_logp <= 0 and <= log preds[t, k, path[t, k]] for every k: a route never outweighs a label on it."""
    assert path.dtype == np.int8 and path.shape == preds.shape[:2] and path_logp.shape == preds.shape[:1]
    assert np.all(path_logp <= tol)
    on_path = np.take_along_axis(preds, path.astype(np.int64)[:, :, None], 2)[:, :, 0]
    with np.errstate(divide="ignore"):
        assert np.all(path_logp[:, None] <= np.log(on_path) + tol)


# ---------------------------------------------------------------- CPU: the path oracle
@pytest.mark.parametrize("nS,L,d,isBL", [(2, 7, 2, 1), (2, 6, 1, 0), (4, 4, 2, 1), (3, 2, 2, 1), (3, 3, 3, 0)])
def test_path_oracle_equals_enumeration_without_fusion(nS, L, d, isBL):
    m = make_model(nS=nS, frame_len=max(L, 2), threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(6, L, d, np.random.default_rng(100 + L), Ds=m.ds**2 / 0.04)
    _, preds, path, logp, _ = pa.chunk_recursion_path(C, m, isBL)
    want_path, want_logp = enumerated_path(C, m, isBL)
    assert np.array_equal(path, want_path)
    np.testing.assert_allclose(logp, want_logp, rtol=0, atol=1e-13)
    check_bounds(preds, path, logp)


def test_path_oracle_three_states_past_the_int8_label_wrap():
    # 3^6 = 729 sequences at the last step: children >= 128 carry the int8-wrapped labels of tracking.py:543
    m = make_model(nS=3, frame_len=6, threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(4, 6, 2, np.random.default_rng(7), Ds=m.ds**2 / 0.04)
    for isBL in (0, 1):
        _, preds, path, logp, _ = pa.chunk_recursion_path(C, m, isBL)
        want_path, want_logp = enumerated_path(C, m, isBL)
        assert np.array_equal(path, want_path)
        np.testing.assert_allclose(logp, want_logp, rtol=0, atol=1e-13)
        check_bounds(preds, path, logp)


@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_path_oracle_posteriors_equal_predict_states(path):
    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    for i in range(len(C)):
        _, preds, p, logp, margin = pa.chunk_recursion_path(C[i : i + 1], m, isBL, tb)
        assert np.array_equal(preds, orc.chunk_recursion(C[i : i + 1], m, isBL, 1, None, tb)[2])
        check_bounds(preds, p, logp)
        assert np.all(margin > 0)


@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_path_oracle_with_shared_plans_posteriors_equal_predict_states(path):
    tracks, keys, _, _, _, nb_max, m = nbmax_case(path)
    st = [tracks[k] for k in keys]
    for w, (preds, p, logp, _) in zip(orc.predict_states(st, m, nb_max=nb_max), pa.predict_path(st, m, nb_max=nb_max)):
        assert np.array_equal(preds, w)
        check_bounds(preds, p, logp)


@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_path_oracle_with_peakwise_inputs_posteriors_equal_predict_states(path):
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    for w, (preds, p, logp, _) in zip(orc.predict_states(st, m, 1, sigs, ds_list), pa.predict_path(st, m, 1, sigs, ds_list)):
        assert np.array_equal(preds, w)
        check_bounds(preds, p, logp)


# ---------------------------------------------------------------- CPU: path_segments
def test_path_segments_splits_interior_and_censored_runs():
    from extrack_b200.tracking import path_segments

    paths = {
        "5": np.array([[0, 0, 1, 1, 0],  # censored 0 x2, interior 1 x2, censored 0 x1
                       [1, 1, 1, 1, 1],  # no switch: one censored segment of 5
                       [0, 1, 0, 1, 0]],  # censored 0 x1, interior 1, 0, 1 of one localisation, censored 0 x1
                      dtype=np.int8),
        "3": np.array([[1, 0, 1]], dtype=np.int8),  # censored 1 x1, interior 0 x1, censored 1 x1
        "4": np.zeros((0, 4), dtype=np.int8),
    }
    interior, censored = path_segments(paths, 2)
    assert interior.dtype == censored.dtype == np.int64 and interior.shape == censored.shape == (5, 2)
    want_i = np.zeros((5, 2), dtype=np.int64)
    want_i[0] = [2, 2]
    want_i[1, 1] = 1
    want_c = np.zeros((5, 2), dtype=np.int64)
    want_c[0] = [3, 2]
    want_c[1, 0] = 1
    want_c[4, 1] = 1
    assert np.array_equal(interior, want_i) and np.array_equal(censored, want_c)
    # every localisation is in exactly one segment
    n_loc = sum(a.size for a in paths.values())
    assert ((interior + censored) * np.arange(1, 6)[:, None]).sum() == n_loc


# ---------------------------------------------------------------- CPU: MAP paths on simulated tracks
def test_map_paths_recover_simulated_states_with_fewer_switches():
    """Two well-separated states (D 0 and 0.25 um^2/s, LocErr 0.02 um), 300 tracks of 10-20 localisations drawn by
    ``sim_FOV`` with a fixed seed, annotated by the path oracle at the true parameters (frame_len 5: sequences fuse).
    The MAP paths match the true states at most localisations, and they switch state less often than the frame-wise
    argmax of the posteriors (which dithers where the posteriors are near 0.5)."""
    from extrack_b200.simulate import sim_FOV

    Ds, Fs, TrMat, dt = (0.0, 0.25), (0.6, 0.4), np.array([[0.9, 0.1], [0.1, 0.9]]), 0.02
    tracks, states = sim_FOV(nb_tracks=300, max_track_len=20, min_track_len=10, LocErr=0.02, Ds=Ds, nb_dims=2,
                             initial_fractions=Fs, TrMat=TrMat, dt=dt, pBL=0.05, cell_dims=(100.0,), seed=5,
                             return_states=True)
    keys = sorted((k for k in tracks if len(tracks[k])), key=int)
    m = orc.Model(np.array([0.02]), np.sqrt(2 * np.array(Ds) * dt), np.array(Fs), TrMat, 0.05, [100.0], 1, 5,
                  int(keys[0]), 0.1, 200)
    res = pa.predict_path([tracks[k] for k in keys], m)
    truth = [np.asarray(states[k]) for k in keys]
    n_loc = sum(s.size for s in truth)
    ok_path = sum(int(np.sum(p == s)) for (_, p, _, _), s in zip(res, truth))
    ok_argmax = sum(int(np.sum(np.argmax(pr, -1) == s)) for (pr, _, _, _), s in zip(res, truth))
    switches = lambda x: int(np.sum(x[:, 1:] != x[:, :-1]))
    sw_path = sum(switches(p) for (_, p, _, _) in res)
    sw_argmax = sum(switches(np.argmax(pr, -1)) for (pr, _, _, _) in res)
    sw_true = sum(switches(s) for s in truth)
    print("localisations %d; agreement MAP %.4f argmax %.4f; switches MAP %d argmax %d true %d"
          % (n_loc, ok_path / n_loc, ok_argmax / n_loc, sw_path, sw_argmax, sw_true))
    assert n_loc >= 2500
    # (this run: 2913 localisations, agreement 0.950 MAP / 0.954 argmax, switches 211 MAP / 226 argmax / 251 true)
    assert ok_path / n_loc >= 0.93
    assert sw_path < sw_argmax


# ---------------------------------------------------------------- GPU: predict_path
@pytest.fixture(scope="module")
def xt():
    from extrack_b200 import tracking

    return tracking


def check_paths(path, logp, want_path, want_logp, margin):
    assert np.all(margin > MARGIN), "near-tie in the test data (smallest decision margin %g)" % np.min(margin)
    assert path.dtype == np.int8 and path.shape == want_path.shape
    assert np.array_equal(path, want_path)
    np.testing.assert_allclose(logp, want_logp, rtol=0, atol=LOGP_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_engine_paths_match_oracle_on_golden_tracks(path):
    """nb_max = 1 (own plans, NSC 2 / 3 and generic instantiations): 2, 3 and 4 states, 2-D and 3-D."""
    from extrack_b200 import _native

    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    want = [pa.chunk_recursion_path(C[i : i + 1], m, isBL, tb) for i in range(len(C))]
    eng = _native.Engine(0)
    try:
        eng.upload([C], [isBL], 2000)
        p = engine_params(m, C.shape[2])
        preds_only = eng.predict(p, m.nS)[0]
        (preds,), (paths,), (logp,) = eng.predict_path(p, m.nS)
    finally:
        eng.close()
    assert np.array_equal(preds, preds_only)
    check_paths(paths, logp, *(np.concatenate([w[k] for w in want]) for k in (2, 3, 4)))


@pytest.mark.gpu
def test_engine_paths_three_states_past_the_int8_label_wrap():
    """729 sequences at the last step without fusion (generic and NSC = 3 instantiations): the exact MAP paths, with
    the int8-wrapped labels of the posteriors."""
    from extrack_b200 import _native

    m = make_model(nS=3, frame_len=6, threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(64, 6, 2, np.random.default_rng(70), Ds=m.ds**2 / 0.04)
    for isBL in (0, 1):
        _, _, want_path, want_logp, margin = pa.chunk_recursion_path(C, m, isBL)
        assert np.array_equal(want_path, enumerated_path(C, m, isBL)[0])
        eng = _native.Engine(0)
        try:
            eng.upload([C], [isBL], 2000)
            p = engine_params(m, 2)
            preds_only = eng.predict(p, 3)[0]
            (preds,), (paths,), (logp,) = eng.predict_path(p, 3)
        finally:
            eng.close()
        assert np.array_equal(preds, preds_only)
        check_paths(paths, logp, want_path, want_logp, margin)


@pytest.mark.gpu
@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_predict_path_with_shared_plans_matches_oracle(path, xt):
    """nb_max > 1 (plans shared per chunk, the FOLLOW instantiation)."""
    tracks, keys, params, nS, fl, nb_max, m = nbmax_case(path)
    preds, paths, logp = xt.predict_path(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    ref = xt.predict_Bs(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    assert set(preds) == set(paths) == set(logp) == set(tracks)
    for k, (_, wp, wl, mar) in zip(keys, pa.predict_path([tracks[k] for k in keys], m, nb_max=nb_max)):
        assert np.array_equal(preds[k], ref[k])
        check_paths(paths[k], logp[k], wp, wl, mar)


@pytest.mark.gpu
@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_predict_path_with_peakwise_inputs_matches_oracle(path, xt):
    """Peak-wise LocErr (with slope / offset in some cases) and per-track dt, nb_max = 1."""
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    tr = {str(a.shape[1]): a for a in st}
    ild = None if il is None else {str(a.shape[1]): x for a, x in zip(st, il)}
    dtd = 0.02 if dts is None else {str(a.shape[1]): x for a, x in zip(st, dts)}
    kw = dict(cell_dims=[1], nb_states=cfg["nS"], frame_len=cfg["fl"], input_LocErr=ild)
    preds, paths, logp = xt.predict_path(tr, dtd, params, **kw)
    only = xt.predict_Bs(tr, dtd, params, **kw)
    for a, (_, wp, wl, mar) in zip(st, pa.predict_path(st, m, 1, sigs, ds_list)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], only[k])
        check_paths(paths[k], logp[k], wp, wl, mar)


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
def test_predict_path_api_buckets_and_errors(xt):
    """L = 2 and 3, bleaching buckets and the longest bucket, an empty bucket, and predict_Bs' errors."""
    tracks, p = _api_case()
    preds, paths, logp = xt.predict_path(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    assert set(preds) == set(paths) == set(logp) == set(tracks)
    assert preds["9"].shape == (0, 9, 2) and paths["9"].shape == (0, 9) and logp["9"].shape == (0,)
    assert paths["9"].dtype == np.int8
    st, _ = xt._sorted_buckets(tracks)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    m = orc.Model(LocErr[0].reshape(-1), ds, Fs, TrMat, pBL, [1], 1, 8, 2, 0.1, 200)
    ref = xt.predict_Bs(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    for a, (_, wp, wl, mar) in zip(st, pa.predict_path(st, m, nb_max=1)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], ref[k])
        check_paths(paths[k], logp[k], wp, wl, mar)
        check_bounds(preds[k], paths[k], logp[k])
    with pytest.raises(NotImplementedError):
        xt.predict_path(tracks, 0.02, p, nb_states=2, nb_max=50,
                        input_LocErr={k: np.full(v.shape[:2] + (1,), 0.02) for k, v in tracks.items()})
    with pytest.raises(NotImplementedError):
        xt.predict_path(tracks, {k: np.full(v.shape[:2], 0.02) for k, v in tracks.items()}, p, nb_states=2, nb_max=50)
    with pytest.raises(TypeError):
        xt.predict_path(tracks, 0.02, {"D0": 1.0}, nb_states=2)
    with pytest.raises(ValueError):
        xt.predict_path(tracks, 0.02, p, nb_states=3)
    with pytest.raises(ValueError):
        xt.predict_path(tracks, 0.02, p, nb_states=2, nb_max=0)


@pytest.mark.gpu
def test_engine_paths_identical_after_capacity_retry():
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
            res.append(eng.predict_path(engine_params(m, 2), 3))
            if cap0:
                assert eng.stats()["k3_launches"] > 1
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a[0], b[0])


@pytest.mark.gpu
def test_engine_paths_identical_with_and_without_pieces():
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
            res.append(eng.predict_path(engine_params(m, 2), 2))
            launches = eng.stats()["k3_launches"]
            assert (launches == 1) if pieces else (launches > 1)
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    preds, paths, logp = res[0]
    for pr, pt, lp in zip(preds, paths, logp):
        check_bounds(pr, pt, lp, tol=1e-9)
