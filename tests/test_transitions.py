"""Transition (two-slice) posteriors of the state annotation: the pair oracle against the reference's stored
posteriors and against direct enumeration (CPU), and ``predict_transitions`` against the pair oracle (GPU)."""
import glob
import os

import numpy as np
import pytest

from helpers import engine_params, load_var_case, make_model, random_walk_tracks, var_oracle_inputs
from oracle import extrack_oracle as orc
from oracle import pair_oracle as po

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "s*.npz")) if "seglen_" not in f)
NBMAX_CASES = sorted(glob.glob(os.path.join(GOLDEN, "nbmax_*.npz")))
VAR_CASES = sorted(glob.glob(os.path.join(GOLDEN, "var_*.npz")))
_ids = lambda paths: [os.path.basename(p)[:-4] for p in paths]


def golden_case(path):
    z = np.load(path, allow_pickle=False)
    if z["ref_preds"].size == 0:
        pytest.skip("nb_substeps > 1: predict_Bs forces nb_substeps = 1")
    m = orc.Model(z["loc_err"], z["ds"], z["Fs"], z["TrMat"], float(z["pBL"]), list(z["cell_dims"]), 1, int(z["frame_len"]),
                  int(z["min_len"]), 0.1, 200)  # predict_Bs' defaults (threshold 0.1, max_nb_states 200, nb_substeps 1)
    n = z["ref_preds"].shape[0]
    return z["C"][:n], int(z["isBL"]), m, z["ref_preds"]


def nbmax_case(path):
    from test_oracle import load_nbmax_case

    from extrack_b200 import tracking as xt

    tracks, preds, params, nS, fl, nb_max = load_nbmax_case(path)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, 0.02, nS, 1)
    keys = sorted(tracks, key=int)
    m = orc.Model(np.asarray(LocErr[0]).reshape(-1), ds, Fs, TrMat, pBL, [1], 1, fl, tracks[keys[0]].shape[1], 0.1, 200)
    return tracks, keys, preds, params, nS, fl, nb_max, m


def check_marginals(preds, pairs, tol=1e-12):
    assert pairs.shape == (preds.shape[0], preds.shape[1] - 1, preds.shape[2], preds.shape[2])
    np.testing.assert_allclose(pairs.sum(-1), preds[:, :-1], rtol=0, atol=tol)
    np.testing.assert_allclose(pairs.sum(-2), preds[:, 1:], rtol=0, atol=tol)


def enumerated_pairs(C, model, isBL):
    """Two-slice posteriors by direct enumeration over the surviving sequences (no fusion: every sequence's history
    is one-hot), from the oracle's final log-probabilities and histories."""
    LP, hist, _ = orc.chunk_recursion(C, model, isBL, 1)
    if np.max(LP) > 600:
        LP = LP - (np.max(LP) - 600)
    P = np.exp(LP)
    P /= P.sum(1, keepdims=True)
    h = np.broadcast_to(hist, (len(C),) + hist.shape[1:])[:, :, ::-1]  # [nT, nB, L, nS], forward time
    assert set(np.unique(h)) <= {0.0, 1.0}, "a fusion happened"
    return np.einsum("tb,tbki,tbkj->tkij", P, h[:, :, :-1], h[:, :, 1:])


# ---------------------------------------------------------------- CPU: the pair oracle
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_pair_oracle_marginals_match_reference_posteriors(path):
    C, isBL, m, ref = golden_case(path)
    tb = orc.HeadTables(m)
    for i in range(len(C)):
        _, preds, pairs = po.chunk_recursion_pairs(C[i : i + 1], m, isBL, tb)
        assert np.array_equal(preds, orc.chunk_recursion(C[i : i + 1], m, isBL, 1, None, tb)[2])
        np.testing.assert_allclose(pairs.sum(-1), ref[i : i + 1, :-1], rtol=0, atol=1e-12)
        np.testing.assert_allclose(pairs.sum(-2), ref[i : i + 1, 1:], rtol=0, atol=1e-12)
        assert pairs.min() >= 0


@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_pair_oracle_with_shared_plans_matches_reference_posteriors(path):
    tracks, keys, ref, _, _, _, nb_max, m = nbmax_case(path)
    st = [tracks[k] for k in keys]
    want = orc.predict_states(st, m, nb_max=nb_max)
    for k, w, (preds, pairs) in zip(keys, want, po.predict_pairs(st, m, nb_max=nb_max)):
        assert np.array_equal(preds, w)
        # (the oracle itself meets these stored posteriors to ~1e-11 in this mode: test_oracle uses 1e-10)
        np.testing.assert_allclose(pairs.sum(-1), ref[k][:, :-1], rtol=0, atol=1e-10)
        np.testing.assert_allclose(pairs.sum(-2), ref[k][:, 1:], rtol=0, atol=1e-10)
        check_marginals(preds, pairs)


@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_pair_oracle_with_peakwise_inputs_matches_reference_posteriors(path):
    st, il, dts, params, ref, cfg = load_var_case(path)
    if ref is None:
        pytest.skip("no stored posteriors in this case")
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    want = orc.predict_states(st, m, 1, sigs, ds_list)
    for w, r, (preds, pairs) in zip(want, ref, po.predict_pairs(st, m, 1, sigs, ds_list)):
        assert np.array_equal(preds, w)
        np.testing.assert_allclose(pairs.sum(-1), r[:, :-1], rtol=0, atol=1e-12)
        np.testing.assert_allclose(pairs.sum(-2), r[:, 1:], rtol=0, atol=1e-12)


@pytest.mark.parametrize("nS,L,d,isBL", [(2, 7, 2, 1), (2, 6, 1, 0), (4, 4, 2, 1), (3, 2, 2, 1), (3, 3, 3, 0)])
def test_pair_oracle_equals_enumeration_without_fusion(nS, L, d, isBL):
    m = make_model(nS=nS, frame_len=max(L, 2), threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(6, L, d, np.random.default_rng(100 + L), Ds=m.ds**2 / 0.04)
    _, preds, pairs = po.chunk_recursion_pairs(C, m, isBL)
    np.testing.assert_allclose(pairs, enumerated_pairs(C, m, isBL), rtol=0, atol=1e-13)
    check_marginals(preds, pairs)


def test_pair_oracle_three_states_past_the_int8_label_wrap():
    # 3^6 = 729 sequences at the last step: children >= 128 carry the int8-wrapped labels of tracking.py:543
    m = make_model(nS=3, frame_len=6, threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(4, 6, 2, np.random.default_rng(7), Ds=m.ds**2 / 0.04)
    for isBL in (0, 1):
        _, preds, pairs = po.chunk_recursion_pairs(C, m, isBL)
        np.testing.assert_allclose(pairs, enumerated_pairs(C, m, isBL), rtol=0, atol=1e-13)
        check_marginals(preds, pairs)
    m.int8_wrap = False  # the wrap really changes the labels of this case
    assert not np.allclose(po.chunk_recursion_pairs(C, m, 0)[2], pairs)


def test_transition_summary_counts_switches():
    from extrack_b200.tracking import transition_summary

    # track 0: certain switch 0 -> 1 at the second step; track 1: stays in 0; track 2: half-certain dithering
    pairs = np.zeros((3, 2, 2, 2))
    pairs[0, 0] = [[1, 0], [0, 0]]
    pairs[0, 1] = [[0, 1], [0, 0]]
    pairs[1, :] = [[1, 0], [0, 0]]
    pairs[2, :] = [[0.25, 0.25], [0.25, 0.25]]
    preds = np.concatenate([pairs.sum(-1), pairs[:, -1:].sum(-2)], axis=1)
    expected, tr = transition_summary({"3": preds}, {"3": pairs})
    np.testing.assert_allclose(expected["3"], [1.0, 0.0, 1.0])
    np.testing.assert_allclose(tr, [[3.5 / 5, 1.5 / 5], [0.5, 0.5]])
    np.testing.assert_allclose(tr.sum(1), 1.0)


# ---------------------------------------------------------------- GPU: predict_transitions
@pytest.fixture(scope="module")
def xt():
    from extrack_b200 import tracking

    return tracking


@pytest.mark.gpu
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_engine_pairs_match_pair_oracle_on_golden_tracks(path):
    """nb_max = 1 (own plans, NSC 2 / 3 and generic instantiations): 2, 3 and 4 states, 2-D and 3-D."""
    from extrack_b200 import _native

    C, isBL, m, _ = golden_case(path)
    tb = orc.HeadTables(m)
    want = [po.chunk_recursion_pairs(C[i : i + 1], m, isBL, tb) for i in range(len(C))]
    eng = _native.Engine(0)
    try:
        eng.upload([C], [isBL], 2000)
        p = engine_params(m, C.shape[2])
        preds_only = eng.predict(p, m.nS)[0]
        (preds,), (pairs,) = eng.predict_pairs(p, m.nS)
    finally:
        eng.close()
    assert np.array_equal(preds, preds_only)
    np.testing.assert_allclose(pairs, np.concatenate([w[2] for w in want]), rtol=0, atol=1e-9)
    check_marginals(preds, pairs)


@pytest.mark.gpu
def test_engine_pairs_three_states_many_sequences(xt):
    from extrack_b200 import _native

    m = make_model(nS=3, nsub=1, frame_len=7, threshold=0.05, max_nb_states=200, min_len=5)
    C = random_walk_tracks(24, 22, 3, np.random.default_rng(5), Ds=m.ds**2 / 0.04)
    want = np.concatenate([po.chunk_recursion_pairs(C[i : i + 1], m, 1)[2] for i in range(len(C))])
    eng = _native.Engine(0)
    try:
        eng.upload([C], [1], 2000)
        (preds,), (pairs,) = eng.predict_pairs(engine_params(m, 3), 3)
    finally:
        eng.close()
    np.testing.assert_allclose(pairs, want, rtol=0, atol=1e-9)
    check_marginals(preds, pairs)


@pytest.mark.gpu
@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_predict_transitions_with_shared_plans_matches_pair_oracle(path, xt):
    """nb_max 7, 40, 50 and 2000 (plans shared per chunk), 2 and 3 states, 2-D and 3-D."""
    tracks, keys, _, params, nS, fl, nb_max, m = nbmax_case(path)
    preds, pairs = xt.predict_transitions(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    ref = xt.predict_Bs(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    assert set(preds) == set(pairs) == set(tracks)
    for k, (_, want) in zip(keys, po.predict_pairs([tracks[k] for k in keys], m, nb_max=nb_max)):
        assert np.array_equal(preds[k], ref[k])
        np.testing.assert_allclose(pairs[k], want, rtol=0, atol=1e-9)
        check_marginals(preds[k], pairs[k])


@pytest.mark.gpu
@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_predict_transitions_with_peakwise_inputs_matches_pair_oracle(path, xt):
    st, il, dts, params, ref, cfg = load_var_case(path)
    if ref is None:
        pytest.skip("no stored posteriors in this case")
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    tr = {str(a.shape[1]): a for a in st}
    ild = None if il is None else {str(a.shape[1]): x for a, x in zip(st, il)}
    dtd = 0.02 if dts is None else {str(a.shape[1]): x for a, x in zip(st, dts)}
    kw = dict(cell_dims=[1], nb_states=cfg["nS"], frame_len=cfg["fl"], input_LocErr=ild)
    preds, pairs = xt.predict_transitions(tr, dtd, params, **kw)
    only = xt.predict_Bs(tr, dtd, params, **kw)
    for a, (_, want) in zip(st, po.predict_pairs(st, m, 1, sigs, ds_list)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], only[k])
        np.testing.assert_allclose(pairs[k], want, rtol=0, atol=1e-9)
        check_marginals(preds[k], pairs[k])


@pytest.mark.gpu
def test_predict_transitions_api_buckets_and_errors(xt):
    from extrack_b200._lmfit_compat import Parameters

    rng = np.random.default_rng(21)
    tracks = {str(L): random_walk_tracks(n, L, 2, rng) for L, n in ((2, 3), (3, 4), (7, 40), (15, 70), (31, 33))}
    tracks["9"] = np.zeros((0, 9, 2))
    p = Parameters()
    for k, v in dict(D0=1e-5, D1=0.25, LocErr=0.02, F0=0.6, p01=0.1, p10=0.12, pBL=0.05).items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    preds, pairs = xt.predict_transitions(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    assert set(preds) == set(pairs) == set(tracks)
    assert preds["9"].shape == (0, 9, 2) and pairs["9"].shape == (0, 8, 2, 2)
    st, _ = xt._sorted_buckets(tracks)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    m = orc.Model(LocErr[0].reshape(-1), ds, Fs, TrMat, pBL, [1], 1, 8, 2, 0.1, 200)
    ref = xt.predict_Bs(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    for a, (_, want) in zip(st, po.predict_pairs(st, m, nb_max=1)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], ref[k])
        np.testing.assert_allclose(pairs[k], want, rtol=0, atol=1e-9)
        check_marginals(preds[k], pairs[k])
    with pytest.raises(NotImplementedError):
        xt.predict_transitions(tracks, 0.02, p, nb_states=2, nb_max=50,
                               input_LocErr={k: np.full(v.shape[:2] + (1,), 0.02) for k, v in tracks.items()})
    with pytest.raises(NotImplementedError):
        xt.predict_transitions(tracks, {k: np.full(v.shape[:2], 0.02) for k, v in tracks.items()}, p, nb_states=2, nb_max=50)
    with pytest.raises(TypeError):
        xt.predict_transitions(tracks, 0.02, {"D0": 1.0}, nb_states=2)
    with pytest.raises(ValueError):
        xt.predict_transitions(tracks, 0.02, p, nb_states=3)


@pytest.mark.gpu
def test_empirical_transition_matrix_on_simulated_tracks(xt):
    """10^5 simulated tracks annotated at the simulation's parameters: the empirical per-step transition matrix is
    within 10 % (relative) of the model's off-diagonal TrMat.  A sanity bound with a fixed seed, not a parity check:
    fusion makes the posteriors approximate, and the simulation switches at 20 sub-steps per frame."""
    from extrack_b200.simulate import sim_tracks
    from extrack_b200._lmfit_compat import Parameters

    rates = [[0.9, 0.1], [0.1, 0.9]]
    tracks = sim_tracks(100_000, seed=11, max_track_len=30, min_track_len=5, LocErr=0.02, Ds=[0, 0.25], nb_dims=2,
                        initial_fractions=[0.6, 0.4], TrMat=rates, dt=0.02, pBL=0.05, cell_dims=[1, None, None])
    p = Parameters()
    for k, v in dict(D0=1e-5, D1=0.25, LocErr=0.02, F0=0.6, p01=0.1, p10=0.1, pBL=0.05).items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    preds, pairs = xt.predict_transitions(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    expected, emp = xt.transition_summary(preds, pairs)
    TrMat = xt.extract_params(p, 0.02, 2, 1)[3]
    off = ~np.eye(2, dtype=bool)
    rel = np.abs(emp[off] - TrMat[off]) / TrMat[off]
    assert np.all(rel < 0.10), (emp, TrMat)
    np.testing.assert_allclose(emp.sum(1), 1.0, atol=1e-9)
    assert all(np.all((e >= -1e-9) & (e <= int(k) - 1 + 1e-9)) for k, e in expected.items())
