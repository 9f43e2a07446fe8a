"""Posterior samples of whole state paths (forward filtering, backward sampling on the annotation lattice): the sample
oracle's random stream, its exactness against enumeration and its marginal / pair identities (CPU), ``sample_segments``
(CPU), and ``sample_paths`` / ``Engine.predict_samples`` against the sample oracle (GPU).

Every statistical check uses fixed seeds and bounds of at least 5 sigma, so its outcome is deterministic."""
import glob
import os

import numpy as np
import pytest
from scipy import stats

from helpers import engine_params, load_var_case, make_model, random_walk_tracks, var_oracle_inputs
from oracle import extrack_oracle as orc
from oracle import pair_oracle as po
from oracle import sample_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "s*.npz")) if "seglen_" not in f)
NBMAX_CASES = sorted(glob.glob(os.path.join(GOLDEN, "nbmax_*.npz")))
VAR_CASES = sorted(glob.glob(os.path.join(GOLDEN, "var_*.npz")))
# golden cases whose tracks are longer than frame_len (sequences fuse) and that annotate with nb_substeps = 1
FUSED_CASES = [f for f in CASES if os.path.basename(f)[:-4] in ("s2_escalate", "s2_fl6_L30_noBL", "s2_fl8_L20", "s3_3d", "s4")]
_ids = lambda paths: [os.path.basename(p)[:-4] for p in paths]
LOGP_TOL = 1e-10  # GPU vs oracle (FP64, different summation orders)
MARGIN = 1e-9  # a draw whose choices all lie this far from a boundary must match the oracle's exactly
N_GPU = 64  # draws per track in the GPU comparisons


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


def freq_within(count, N, p, nsig):
    """|count - N p| <= nsig sigma + 1 for every entry (sigma of a binomial count; + 1: one count of granularity)."""
    p = np.clip(p, 0.0, 1.0)
    dev = np.abs(count - N * p)
    bound = nsig * np.sqrt(N * p * (1 - p)) + 1.0
    assert np.all(dev <= bound), "largest excess %g counts" % np.max(dev - bound)


# ---------------------------------------------------------------- CPU: the random stream
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0), "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_philox_known_answers(ctr, key, want):
    assert " ".join("%08x" % int(x) for x in so.philox4x32_10(ctr, key)) == want


def test_uniforms_use_the_top_53_bits_of_the_first_two_words():
    seed = 0x0123456789ABCDEF
    x = so.philox4x32_10((5, 9, 3, 8), (seed & 0xFFFFFFFF, seed >> 32))
    want = ((int(x[0]) << 32 | int(x[1])) >> 11) * 2.0**-53
    assert so.uniforms(seed, 5, 9, np.array([3], dtype=np.uint64), 8)[0] == want


# ---------------------------------------------------------------- CPU: the sample oracle
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_sample_oracle_posteriors_equal_predict_states(path):
    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    for i in range(len(C)):
        preds, smp, lp, margin = so.chunk_recursion_sample(C[i : i + 1], m, isBL, 8, 3, i, tb)
        assert np.array_equal(preds, orc.chunk_recursion(C[i : i + 1], m, isBL, 1, None, tb)[2])
        assert smp.shape == (1, 8, C.shape[1]) and smp.dtype == np.int8
        assert np.all(lp <= 1e-12) and np.all(margin > 0)


@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_sample_oracle_with_shared_plans_posteriors_equal_predict_states(path):
    tracks, keys, _, _, _, nb_max, m = nbmax_case(path)
    st = [tracks[k] for k in keys]
    for w, (preds, _, lp, _) in zip(orc.predict_states(st, m, nb_max=nb_max), so.predict_samples(st, m, 4, 1, nb_max=nb_max)):
        assert np.array_equal(preds, w)
        assert np.all(lp <= 1e-12)


@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_sample_oracle_with_peakwise_inputs_posteriors_equal_predict_states(path):
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    for w, (preds, _, lp, _) in zip(orc.predict_states(st, m, 1, sigs, ds_list), so.predict_samples(st, m, 4, 1, 1, sigs, ds_list)):
        assert np.array_equal(preds, w)
        assert np.all(lp <= 1e-12)


@pytest.mark.parametrize("nS,L", [(2, 6), (3, 4), (4, 4)])
@pytest.mark.parametrize("isBL", [0, 1])
def test_sample_oracle_is_exact_without_fusion(nS, L, isBL):
    """Tracks no longer than frame_len: every draw is an exact sample of P(s_0..s_L-1 | track).  2^16 draws per track:
    the count of every full sequence within 5 sigma of the enumerated posterior, a chi-square statistic below its 1e-6
    quantile, and sample_logp equal to the log posterior of the drawn sequence."""
    m = make_model(nS=nS, frame_len=L, threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(3, L, 2, np.random.default_rng(300 + 10 * nS + L), Ds=m.ds**2 / 0.04)
    N = 2**16
    _, smp, lp, _ = so.chunk_recursion_sample(C, m, isBL, N, 11 + isBL)
    labels, logpost = so.enumerate_posterior(C, m, isBL)
    code = lambda x: (x.astype(np.int64) * nS ** np.arange(L)).sum(-1)
    index = np.full(nS**L, -1)
    index[code(labels)] = np.arange(len(labels))
    for t in range(len(C)):
        seq = index[code(smp[t])]
        assert np.all(seq >= 0)
        np.testing.assert_allclose(lp[t], logpost[t][seq], rtol=0, atol=1e-12)
        p = np.exp(logpost[t])
        cnt = np.bincount(seq, minlength=len(labels))
        freq_within(cnt, N, p, 5)
        # chi-square over the sequences expected at least 5 times, the rest pooled into one cell
        e = N * p
        big = e >= 5
        obs = np.append(cnt[big], cnt[~big].sum())
        exp_ = np.append(e[big], e[~big].sum())
        keep = exp_ > 0
        chi2 = np.sum((obs[keep] - exp_[keep]) ** 2 / exp_[keep])
        assert chi2 < stats.chi2.isf(1e-6, keep.sum() - 1)


@pytest.mark.parametrize("path", FUSED_CASES, ids=_ids(FUSED_CASES))
def test_sample_oracle_label_and_pair_frequencies_match_posteriors_with_fusion(path):
    """With fusion the draws are routes of the lattice: label frequencies converge to predict_states' posteriors and
    consecutive-pair frequencies to the two-slice posteriors (within 6 sigma, 4096 draws per track)."""
    C, isBL, m = golden_case(path)
    C = C[:8]
    N = 4096
    tb = orc.HeadTables(m)
    nS = m.nS
    fused = False
    for t in range(len(C)):  # one track per chunk (nb_max = 1)
        preds, smp, _, _ = so.chunk_recursion_sample(C[t : t + 1], m, isBL, N, 5, t, tb)
        _, want_preds, want_pairs = po.chunk_recursion_pairs(C[t : t + 1], m, isBL, tb)
        assert np.array_equal(preds, want_preds)
        lab = smp[0].astype(np.int64)  # [N, L]
        cnt = np.stack([np.bincount(lab[:, k], minlength=nS) for k in range(C.shape[1])])
        freq_within(cnt, N, want_preds[0], 6)
        pair = lab[:, :-1] * nS + lab[:, 1:]
        pcnt = np.stack([np.bincount(pair[:, k], minlength=nS * nS) for k in range(C.shape[1] - 1)]).reshape(-1, nS, nS)
        freq_within(pcnt, N, want_pairs[0], 6)
        fused |= bool(np.any((want_preds[0] > 1e-6) & (want_preds[0] < 1 - 1e-6)))
    assert C.shape[1] > m.frame_len and fused


# ---------------------------------------------------------------- CPU: sample_segments
def test_sample_segments_on_hand_made_draws():
    from extrack_b200.tracking import sample_segments

    samples = {
        "4": np.array([[[0, 0, 1, 1], [1, 0, 1, 1]],  # draw 0: censored 0 x2, censored 1 x2; draw 1: c 1, i 0, c 1 x2
                       [[1, 1, 1, 1], [0, 1, 1, 0]]],  # draw 0: censored 1 x4; draw 1: c 0, i 1 x2, c 0
                      dtype=np.int8),
        "3": np.zeros((0, 2, 3), dtype=np.int8),
    }
    interior, censored = sample_segments(samples, 2)
    assert interior.dtype == censored.dtype == np.int64 and interior.shape == censored.shape == (2, 4, 2)
    want_i = np.zeros((2, 4, 2), dtype=np.int64)
    want_i[1, 0, 0] = 1
    want_i[1, 1, 1] = 1
    want_c = np.zeros((2, 4, 2), dtype=np.int64)
    want_c[0, 1] = [1, 1]
    want_c[0, 3, 1] = 1
    want_c[1, 0] = [2, 1]
    want_c[1, 1, 1] = 1
    assert np.array_equal(interior, want_i) and np.array_equal(censored, want_c)


def test_sample_segments_slice_is_path_segments_of_that_draw():
    from extrack_b200.tracking import path_segments, sample_segments

    rng = np.random.default_rng(4)
    samples = {str(L): rng.integers(0, 3, size=(n, 7, L)).astype(np.int8) for L, n in ((2, 5), (6, 11), (9, 4))}
    samples["5"] = np.zeros((0, 7, 5), dtype=np.int8)
    interior, censored = sample_segments(samples, 3)
    assert interior.shape == (7, 9, 3)
    for d in range(7):
        wi, wc = path_segments({k: v[:, d] for k, v in samples.items()}, 3)
        assert np.array_equal(interior[d], wi) and np.array_equal(censored[d], wc)


def test_path_segments_unchanged():
    """path_segments after the run-length counting moved into a shared helper: the counts of the original code."""
    from extrack_b200.tracking import path_segments

    def original(paths, nb_states):
        items = [np.asarray(a) for a in paths.values()]
        L_max = max((a.shape[1] for a in items if a.ndim == 2), default=0)
        interior = np.zeros((L_max, nb_states), dtype=np.int64)
        censored = np.zeros((L_max, nb_states), dtype=np.int64)
        for a in items:
            if a.size == 0:
                continue
            a = a.astype(np.int64)
            n, L = a.shape
            change = a[:, 1:] != a[:, :-1]
            t_e, k_e = np.nonzero(np.concatenate([change, np.ones((n, 1), dtype=bool)], axis=1))
            _, k_s = np.nonzero(np.concatenate([np.ones((n, 1), dtype=bool), change], axis=1))
            length, state = k_e - k_s + 1, a[t_e, k_e]
            cens = (k_s == 0) | (k_e == L - 1)
            np.add.at(interior, (length[~cens] - 1, state[~cens]), 1)
            np.add.at(censored, (length[cens] - 1, state[cens]), 1)
        return interior, censored

    rng = np.random.default_rng(12)
    paths = {str(L): rng.integers(0, 2, size=(n, L)).astype(np.int8) for L, n in ((2, 9), (5, 30), (12, 17))}
    paths["3"] = np.zeros((0, 3), dtype=np.int8)
    paths["7"] = np.array([[0, 0, 1, 1, 0, 1, 1]], dtype=np.int8)
    for got, want in zip(path_segments(paths, 2), original(paths, 2)):
        assert np.array_equal(got, want)


# ---------------------------------------------------------------- GPU: predict_samples / sample_paths
@pytest.fixture(scope="module")
def xt():
    from extrack_b200 import tracking

    return tracking


def check_samples(smp, lp, want_smp, want_lp, margin):
    """Draws whose oracle margin exceeds MARGIN have the oracle's labels; they are at least 99.9 % of all draws (a
    property of the data); sample_logp within LOGP_TOL."""
    assert smp.dtype == np.int8 and smp.shape == want_smp.shape and lp.shape == want_lp.shape
    clear = margin > MARGIN
    assert clear.mean() >= 0.999, "near-ties in the test data (%d of %d draws)" % ((~clear).sum(), clear.size)
    assert np.array_equal(smp[clear], want_smp[clear])
    np.testing.assert_allclose(lp[clear], want_lp[clear], rtol=0, atol=LOGP_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("path", CASES, ids=_ids(CASES))
def test_engine_samples_match_oracle_on_golden_tracks(path):
    """nb_max = 1 (own plans, NSC 2 / 3 and generic instantiations): 2, 3 and 4 states, 2-D and 3-D, bleaching and
    longest buckets; preds bitwise equal to predict, no draw heavier than the MAP route."""
    from extrack_b200 import _native

    C, isBL, m = golden_case(path)
    tb = orc.HeadTables(m)
    want = [so.chunk_recursion_sample(C[i : i + 1], m, isBL, N_GPU, 17, i, tb) for i in range(len(C))]
    eng = _native.Engine(0)
    try:
        eng.upload([C], [isBL], 2000)
        p = engine_params(m, C.shape[2])
        preds_only = eng.predict(p, m.nS)[0]
        (preds,), (smp,), (lp,) = eng.predict_samples(p, m.nS, N_GPU, 17)
        path_logp = eng.predict_path(p, m.nS)[2][0]
    finally:
        eng.close()
    assert np.array_equal(preds, preds_only)
    check_samples(smp, lp, *(np.concatenate([w[k] for w in want]) for k in (1, 2, 3)))
    assert np.all(lp.max(axis=1) <= path_logp + 1e-12)


@pytest.mark.gpu
def test_engine_samples_three_states_past_the_int8_label_wrap():
    """729 sequences at the last step without fusion (generic and NSC = 3 instantiations): the int8-wrapped labels."""
    from extrack_b200 import _native

    m = make_model(nS=3, frame_len=6, threshold=1e-9, max_nb_states=10**6, min_len=3)
    C = random_walk_tracks(64, 6, 2, np.random.default_rng(70), Ds=m.ds**2 / 0.04)
    for isBL in (0, 1):
        _, want_smp, want_lp, margin = so.chunk_recursion_sample(C, m, isBL, N_GPU, 23)
        eng = _native.Engine(0)
        try:
            eng.upload([C], [isBL], 2000)
            p = engine_params(m, 2)
            preds_only = eng.predict(p, 3)[0]
            (preds,), (smp,), (lp,) = eng.predict_samples(p, 3, N_GPU, 23)
        finally:
            eng.close()
        assert np.array_equal(preds, preds_only)
        check_samples(smp, lp, want_smp, want_lp, margin)


@pytest.mark.gpu
@pytest.mark.parametrize("path", NBMAX_CASES, ids=_ids(NBMAX_CASES))
def test_sample_paths_with_shared_plans_matches_oracle(path, xt):
    """nb_max > 1 (plans shared per chunk, the FOLLOW instantiation)."""
    tracks, keys, params, nS, fl, nb_max, m = nbmax_case(path)
    preds, smp, lp = xt.sample_paths(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max,
                                     n_samples=N_GPU, seed=29)
    ref = xt.predict_Bs(tracks, 0.02, params, cell_dims=[1], nb_states=nS, frame_len=fl, nb_max=nb_max)
    assert set(preds) == set(smp) == set(lp) == set(tracks)
    for k, (_, ws, wl, mar) in zip(keys, so.predict_samples([tracks[k] for k in keys], m, N_GPU, 29, nb_max=nb_max)):
        assert np.array_equal(preds[k], ref[k])
        check_samples(smp[k], lp[k], ws, wl, mar)


@pytest.mark.gpu
@pytest.mark.parametrize("path", VAR_CASES, ids=_ids(VAR_CASES))
def test_sample_paths_with_peakwise_inputs_matches_oracle(path, xt):
    """Peak-wise LocErr (with slope / offset in some cases) and per-track dt, nb_max = 1."""
    st, il, dts, params, _, cfg = load_var_case(path)
    m, sigs, ds_list = var_oracle_inputs(st, il, dts, params, cfg, threshold=0.1, max_nb_states=200, nsub=1)
    tr = {str(a.shape[1]): a for a in st}
    ild = None if il is None else {str(a.shape[1]): x for a, x in zip(st, il)}
    dtd = 0.02 if dts is None else {str(a.shape[1]): x for a, x in zip(st, dts)}
    kw = dict(cell_dims=[1], nb_states=cfg["nS"], frame_len=cfg["fl"], input_LocErr=ild)
    preds, smp, lp = xt.sample_paths(tr, dtd, params, n_samples=N_GPU, seed=31, **kw)
    only = xt.predict_Bs(tr, dtd, params, **kw)
    for a, (_, ws, wl, mar) in zip(st, so.predict_samples(st, m, N_GPU, 31, 1, sigs, ds_list)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], only[k])
        check_samples(smp[k], lp[k], ws, wl, mar)


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
def test_sample_paths_api_buckets_edges_and_errors(xt):
    """L = 2 and 3, bleaching buckets and the longest bucket, an empty bucket, n_samples / seed validation and
    predict_Bs' errors; preds equal predict_Bs, draws match the oracle and never outweigh the MAP route."""
    tracks, p = _api_case()
    preds, smp, lp = xt.sample_paths(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8, n_samples=N_GPU, seed=2**64 - 1)
    assert set(preds) == set(smp) == set(lp) == set(tracks)
    assert preds["9"].shape == (0, 9, 2) and smp["9"].shape == (0, N_GPU, 9) and lp["9"].shape == (0, N_GPU)
    assert smp["9"].dtype == smp["2"].dtype == np.int8
    _, _, path_logp = xt.predict_path(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    ref = xt.predict_Bs(tracks, 0.02, p, cell_dims=[1], nb_states=2, frame_len=8)
    st, _ = xt._sorted_buckets(tracks)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    m = orc.Model(LocErr[0].reshape(-1), ds, Fs, TrMat, pBL, [1], 1, 8, 2, 0.1, 200)
    for a, (_, ws, wl, mar) in zip(st, so.predict_samples(st, m, N_GPU, 2**64 - 1)):
        k = str(a.shape[1])
        assert np.array_equal(preds[k], ref[k])
        check_samples(smp[k], lp[k], ws, wl, mar)
        assert np.all(lp[k].max(axis=1) <= path_logp[k] + 1e-12)
    kw = dict(cell_dims=[1], nb_states=2, frame_len=8)
    for bad in (0, 65536, -1, 2.0, True, "10"):
        with pytest.raises(ValueError):
            xt.sample_paths(tracks, 0.02, p, n_samples=bad, **kw)
    for bad in (-1, 2**64, 1.5, None):
        with pytest.raises(ValueError):
            xt.sample_paths(tracks, 0.02, p, seed=bad, **kw)
    with pytest.raises(NotImplementedError):
        xt.sample_paths(tracks, 0.02, p, nb_states=2, nb_max=50,
                        input_LocErr={k: np.full(v.shape[:2] + (1,), 0.02) for k, v in tracks.items()})
    with pytest.raises(NotImplementedError):
        xt.sample_paths(tracks, {k: np.full(v.shape[:2], 0.02) for k, v in tracks.items()}, p, nb_states=2, nb_max=50)
    with pytest.raises(TypeError):
        xt.sample_paths(tracks, 0.02, {"D0": 1.0}, nb_states=2)
    with pytest.raises(ValueError):
        xt.sample_paths(tracks, 0.02, p, nb_states=3)
    with pytest.raises(ValueError):
        xt.sample_paths(tracks, 0.02, p, nb_states=2, nb_max=0)


@pytest.mark.gpu
def test_engine_samples_reproducible_across_calls_draw_counts_seeds_and_rows():
    """Draw d of a track depends only on (seed, L, row, d): a repeated call, the first k draws of a larger request and
    the second half of a bucket uploaded alone with its row offset give identical draws; another seed does not."""
    from extrack_b200 import _native

    m = make_model(nS=2, frame_len=5, threshold=0.1, max_nb_states=200, min_len=4)
    C = random_walk_tracks(200, 12, 2, np.random.default_rng(41), Ds=m.ds**2 / 0.04)
    p = engine_params(m, 2)
    eng = _native.Engine(0)
    try:
        eng.upload([C], [1], 64)  # several chunks: the row is the track's, not its chunk's
        a = eng.predict_samples(p, 2, 100, 5)
        b = eng.predict_samples(p, 2, 100, 5)
        k7 = eng.predict_samples(p, 2, 7, 5)
        k1 = eng.predict_samples(p, 2, 1, 5)
        other = eng.predict_samples(p, 2, 100, 6)
        eng.upload([C[120:]], [1], 2000)
        half = eng.predict_samples(p, 2, 100, 5, row0=[120])
        with pytest.raises(ValueError):
            eng.predict_samples(p, 2, 0, 5)
    finally:
        eng.close()
    for x, y in zip(a, b):
        assert np.array_equal(x[0], y[0])
    assert np.array_equal(k7[1][0], a[1][0][:, :7]) and np.array_equal(k7[2][0], a[2][0][:, :7])
    assert np.array_equal(k1[1][0], a[1][0][:, :1]) and np.array_equal(k1[2][0], a[2][0][:, :1])
    assert np.array_equal(half[1][0], a[1][0][120:]) and np.array_equal(half[2][0], a[2][0][120:])
    assert np.array_equal(other[0][0], a[0][0])
    assert np.mean(other[1][0] != a[1][0]) > 0.01


@pytest.mark.gpu
def test_engine_samples_identical_after_capacity_retry():
    """A small first capacity makes most tracks run again with more: the draws are those of one run."""
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
            res.append(eng.predict_samples(engine_params(m, 2), 3, 40, 9))
            if cap0:
                assert eng.stats()["k3_launches"] > 1
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        assert np.array_equal(a[0], b[0])


@pytest.mark.gpu
def test_engine_samples_identical_with_and_without_pieces():
    """Large enough for the launch in pieces with the read-back of a piece under the next: same draws as one launch."""
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
            res.append(eng.predict_samples(engine_params(m, 2), 2, 3, 13))
            launches = eng.stats()["k3_launches"]
            assert (launches == 1) if pieces else (launches > 1)
        finally:
            eng.close()
    for a, b in zip(res[0], res[1]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
