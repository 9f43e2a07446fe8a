"""Oracle pinning (CPU): the numpy restatement vs the committed golden vectors (reference outputs)
and, where /root/reference exists, vs the unmodified reference run in-process."""
import contextlib
import glob
import io
import os

import numpy as np
import pytest

from helpers import load_var_case, make_model, random_walk_tracks, var_oracle_inputs
from oracle import extrack_oracle as orc
from oracle import ref_loader

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "*.npz"))
               if "objective" not in f and "var_" not in f and "fit_" not in f and "seglen_" not in f and "window_" not in f and "nbmax_" not in f and "refine_" not in f)
VAR_CASES = sorted(glob.glob(os.path.join(GOLDEN, "var_*.npz")))
WINDOW_CASES = sorted(glob.glob(os.path.join(GOLDEN, "window_*.npz")))


def load_case(path):
    z = np.load(path, allow_pickle=False)
    model = orc.Model(z["loc_err"], z["ds"], z["Fs"], z["TrMat"], float(z["pBL"]), list(z["cell_dims"]), int(z["nsub"]),
                      int(z["frame_len"]), int(z["min_len"]), float(z["threshold"]), int(z["max_nb_states"]))
    return z, model


def test_golden_files_present():
    assert len(CASES) >= 10
    assert len(VAR_CASES) >= 6


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_oracle_matches_golden_logp(path):
    z, model = load_case(path)
    got = orc.chunk_logp(z["C"], model, int(z["isBL"]))
    # the oracle uses the same numpy reductions as the reference: agreement is at the ulp level
    np.testing.assert_allclose(got, z["ref_logp"], rtol=1e-13, atol=0)


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_oracle_matches_golden_predictions(path):
    z, model = load_case(path)
    if z["ref_preds"].size == 0:
        pytest.skip("nb_substeps > 1: predict_Bs forces nb_substeps = 1")
    model.threshold, model.max_nb_states = 0.1, 200
    n = z["ref_preds"].shape[0]
    got = np.concatenate([orc.chunk_recursion(z["C"][i : i + 1], model, int(z["isBL"]), 1)[2] for i in range(n)])
    np.testing.assert_allclose(got, z["ref_preds"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(got.sum(-1), 1.0, atol=1e-12)


def test_oracle_objective_multibucket_golden():
    z = np.load(os.path.join(GOLDEN, "objective_multibucket.npz"))
    st = [z["C" + k] for k in z["keys"]]
    Ds = np.array([1e-5, 0.25])
    rates = np.array([[0, 0.1], [0.12, 0]])
    Tr = 1 - np.exp(-rates)
    Tr[[0, 1], [0, 1]] = 1 - Tr.sum(1)
    for fl, want in zip(z["fl"], z["neglogl"]):
        model = orc.Model(np.array([0.02]), np.sqrt(2 * Ds * 0.02), np.array([0.6, 1 - 0.6]), Tr, 0.05, [1], 1, int(fl),
                          st[0].shape[1], 0.2, 120)
        got = orc.neg_log_likelihood(st, model)
        assert abs(got - want) / abs(want) < 1e-13


@pytest.mark.parametrize("path", VAR_CASES, ids=[os.path.basename(p)[:-4] for p in VAR_CASES])
def test_oracle_matches_golden_var_inputs(path):
    """Peak-wise input_LocErr / per-track dt: objective and predictions of the reference's
    cum_Proba_Cs / predict_Bs (golden) vs the oracle."""
    st, il, dts, params, preds, cfg = load_var_case(path)
    model, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg)
    got = orc.neg_log_likelihood(st, model, chunk=cfg["chunk"], sigs=sigs, ds_list=ds_list)
    assert abs(got - cfg["neglogl"]) <= 1e-13 * abs(cfg["neglogl"])
    if preds is not None:
        m2, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
        gp = orc.predict_states(st, m2, 1, sigs, ds_list)
        for a, b in zip(gp, preds):
            np.testing.assert_allclose(a, b, rtol=0, atol=1e-12)


def test_oracle_reproduces_reference_fit_objective_on_tutorial_tracks():
    """BASELINE config 1 (golden: tests/golden/make_golden.py:make_fit_case): at the parameters the
    reference's own param_fitting converged to on Tutorials/tracks.csv, the oracle's objective equals
    the reference's final objective."""
    path = os.path.join(GOLDEN, "fit_tracks_csv.npz")
    if not os.path.isfile(path):
        pytest.skip("fit golden not generated")
    z = np.load(path)
    st = [z["C" + k] for k in z["keys"]]
    assert sum(len(a) for a in st) == 613
    v = dict(zip([str(n) for n in z["names"]], z["fitted"]))
    Ds = np.array([v["D0"], v["D1"]])
    R = np.array([[0, v["p01"]], [v["p10"], 0]])
    Tr = 1 - np.exp(-R)
    Tr[[0, 1], [0, 1]] = 0
    Tr[[0, 1], [0, 1]] = 1 - Tr.sum(1)
    model = orc.Model(np.array([v["LocErr"]]), np.sqrt(2 * Ds * 0.02), np.array([v["F0"], v["F1"]]), Tr, v["pBL"], [1], 1, 6,
                      st[0].shape[1], 0.2, 120)
    got = orc.neg_log_likelihood(st, model)
    assert abs(got - float(z["neglogl"])) <= 1e-12 * abs(float(z["neglogl"]))


def test_oracle_chunk_order_and_workers():
    rng = np.random.default_rng(0)
    st = [random_walk_tracks(n, L, 2, rng) for L, n in ((6, 50), (9, 2300))]
    model = make_model(frame_len=5, min_len=6)
    chunks = orc.make_chunks(st, 2000)
    assert chunks == [(1, 2000, 2300, 0), (1, 0, 2000, 0), (0, 0, 50, 1)]
    a = orc.neg_log_likelihood(st, model, workers=1)
    b = orc.neg_log_likelihood(st, model, workers=2)
    assert a == b


def test_oracle_invalid_params_give_inf():
    model = make_model()
    model.Fs = np.array([1.0, 0.0])
    assert orc.neg_log_likelihood([np.zeros((3, 5, 2))], model) == np.inf


def test_int8_wrap_matters_for_three_states():
    rng = np.random.default_rng(3)
    C = random_walk_tracks(20, 10, 2, rng, Ds=(1e-5, 0.04, 0.25))
    a = orc.chunk_logp(C, make_model(nS=3, nsub=2, max_nb_states=500, int8_wrap=True), 1)
    b = orc.chunk_logp(C, make_model(nS=3, nsub=2, max_nb_states=500, int8_wrap=False), 1)
    assert np.max(np.abs(a - b)) > 1e-6


needs_ref = pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not present on this box")


@needs_ref
@pytest.mark.parametrize("cfg", [
    dict(nS=2, nsub=1, d=2, fl=7, L=15, nT=60, isBL=1),
    dict(nS=3, nsub=2, d=2, fl=5, L=9, nT=30, isBL=0, max_nb_states=300),
    dict(nS=2, nsub=1, d=3, fl=6, L=11, nT=35, isBL=1, loc_err=(0.02, 0.025, 0.03)),
])
def test_oracle_vs_live_reference(cfg):
    trk = ref_loader.load_tracking()
    kw = {k: cfg[k] for k in ("loc_err", "max_nb_states") if k in cfg}
    model = make_model(nS=cfg["nS"], nsub=cfg["nsub"], frame_len=cfg["fl"], **kw)
    C = random_walk_tracks(cfg["nT"], cfg["L"], cfg["d"], np.random.default_rng(42), Ds=model.ds**2 / 0.04)
    with contextlib.redirect_stdout(io.StringIO()):
        ref = trk.Proba_Cs(C, np.asarray(model.loc_err)[None, None], model.ds, model.Fs, model.TrMat, model.pBL, cfg["isBL"],
                           model.cell_dims, model.nb_substeps, model.frame_len, model.min_len, model.threshold, model.max_nb_states)
    got = orc.chunk_logp(C, model, cfg["isBL"])
    np.testing.assert_allclose(got, ref, rtol=1e-13)


@pytest.mark.parametrize("fl,ref", [(4, -16372.353108152653), (6, -16372.631616957766), (8, -16373.513684485983)])
def test_oracle_matches_reference_known_answers_on_tutorial_tracks(fl, ref):
    """Known-answer values of SURVEY.md §6: the unmodified reference's cum_Proba_Cs on Tutorials/tracks.csv at fixed
    parameters.  The tracks are the ones the reference's own reader produced from that file (stored in
    fit_tracks_csv.npz by tests/golden/make_golden.py:make_fit_case, same reader arguments)."""
    z = np.load(os.path.join(GOLDEN, "fit_tracks_csv.npz"))
    st = [z["C" + k] for k in z["keys"]]
    assert sum(len(a) for a in st) == 613
    from extrack_b200 import tracking as xt
    from extrack_b200._lmfit_compat import Parameters

    p = Parameters()
    for k, v in dict(D0=1e-5, D1=0.35, LocErr=0.02, F0=0.54, p01=0.077, p10=0.138, pBL=0.11).items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    model = orc.Model(LocErr[0].reshape(-1), ds, Fs, TrMat, pBL, [1], 1, fl, st[0].shape[1], 0.2, 120)
    got = orc.neg_log_likelihood(st, model)
    assert abs(got - ref) / abs(ref) < 1e-13


@pytest.mark.parametrize("path", WINDOW_CASES, ids=[os.path.basename(p)[:-4] for p in WINDOW_CASES])
def test_oracle_window_only_mode_matches_reference_window_function(path):
    """Window-only mode (the north star's `P_Cs_inter_bound_stats`, tracking.py:109-318): golden = the
    unmodified reference function (tests/golden/make_golden_window.py); the oracle runs the threshold
    recursion at threshold 1e-12 with no sequence limit, which groups by the sliding window alone."""
    z = np.load(path)
    m = orc.Model(z["loc_err"], z["ds"], z["Fs"], z["TrMat"], float(z["pBL"]), list(z["cell_dims"]), int(z["nsub"]),
                  int(z["frame_len"]), int(z["min_len"]), 1e-12, 10**9)
    got = orc.chunk_logp(z["C"], m, int(z["isBL"]))
    np.testing.assert_allclose(got, z["ref_logp"], rtol=1e-12)


NBMAX_CASES = sorted(glob.glob(os.path.join(GOLDEN, "nbmax_*.npz")))


def load_nbmax_case(path):
    from extrack_b200._lmfit_compat import Parameters

    z = np.load(path, allow_pickle=False)
    keys = [str(k) for k in z["keys"]]
    tracks = {k: z["C" + k] for k in keys}
    preds = {k: z["P" + k] for k in keys}
    params = Parameters()
    for k, v in zip(z["param_names"], z["param_values"]):
        params.add(str(k), value=float(v))
    return tracks, preds, params, int(z["nS"]), int(z["fl"]), int(z["nb_max"])


@pytest.mark.parametrize("path", NBMAX_CASES, ids=[os.path.basename(p)[:-4] for p in NBMAX_CASES])
def test_oracle_predict_with_shared_plans_matches_reference(path):
    """predict_Bs(nb_max > 1): golden = the unmodified reference (tests/golden/make_golden_nbmax.py)."""
    from extrack_b200 import tracking as xt

    tracks, preds, params, nS, fl, nb_max = load_nbmax_case(path)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, 0.02, nS, 1)
    keys = sorted(tracks, key=int)
    st = [tracks[k] for k in keys]
    m = orc.Model(np.asarray(LocErr[0]).reshape(-1), ds, Fs, TrMat, pBL, [1], 1, fl, st[0].shape[1], 0.1, 200)
    got = orc.predict_states(st, m, nb_max=nb_max)
    for k, g in zip(keys, got):
        np.testing.assert_allclose(g, preds[k], atol=1e-10)


REFINE_CASES = sorted(glob.glob(os.path.join(GOLDEN, "refine_*.npz")))


def load_refine_case(path):
    z = np.load(path, allow_pickle=False)
    keys = [str(k) for k in z["keys"]]
    return ({k: z["C" + k] for k in keys}, {k: z["M" + k] for k in keys}, {k: z["S" + k] for k in keys},
            dict(LocErr=float(z["loc_err"]), ds=z["ds"], Fs=z["Fs"], TrMat=z["TrMat"], frame_len=int(z["frame_len"]),
                 threshold=float(z["threshold"]), max_nb_states=int(z["max_nb_states"])))


@pytest.mark.parametrize("path", REFINE_CASES, ids=[os.path.basename(p)[:-4] for p in REFINE_CASES])
def test_refinement_oracle_matches_reference_golden(path):
    """Position refinement (refined_localization.py:304-338): golden = the unmodified reference (make_golden_refine.py)."""
    from oracle import refine_oracle

    tracks, mus, sigmas, kw = load_refine_case(path)
    got_mu, got_sig = refine_oracle.position_refinement(tracks, kw["LocErr"], kw["ds"], kw["Fs"], kw["TrMat"], kw["frame_len"],
                                                        kw["threshold"], kw["max_nb_states"])
    for k in tracks:
        np.testing.assert_allclose(got_mu[k], mus[k], atol=1e-12)
        np.testing.assert_allclose(got_sig[k], sigmas[k], atol=1e-12)


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not present")
def test_refinement_oracle_vs_live_reference():
    import contextlib
    import io

    from oracle import refine_oracle

    rl = ref_loader.load_refined_localization()
    rng = np.random.default_rng(12)
    m = make_model(nS=2, frame_len=5)
    tracks = {"7": random_walk_tracks(33, 7, 2, rng), "10": random_walk_tracks(31, 10, 2, rng)}
    with contextlib.redirect_stdout(io.StringIO()):
        mus, sig = rl.position_refinement(tracks, 0.02, m.ds, m.Fs, m.TrMat, frame_len=5, threshold=0.15, max_nb_states=1000)
    omus, osig = refine_oracle.position_refinement(tracks, 0.02, m.ds, m.Fs, m.TrMat, 5, 0.15, 1000)
    for k in tracks:
        np.testing.assert_allclose(omus[k], mus[k], atol=1e-12)
        np.testing.assert_allclose(osig[k], sig[k], atol=1e-12)
