"""Segment-length histogram (SURVEY.md §8(f) N2, reference extrack/histograms.py): oracle vs the golden
vectors produced by the unmodified reference (CPU), CUDA engine vs both (GPU, through the C ABI).
Tolerances: LP 1e-9 relative (north star), histogram 1e-9 absolute on weights that sum to ~1 per track,
state histories identical."""
import glob
import os

import numpy as np
import pytest

from oracle import extrack_oracle as orc
from oracle import seglen_oracle as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SEG_CASES = sorted(f for f in glob.glob(os.path.join(GOLDEN, "seglen_*.npz")) if "len_hist" not in f)
IDS = [os.path.basename(p)[:-4] for p in SEG_CASES]


def seg_model(z):
    return orc.Model(z["loc_err"], z["ds"], z["Fs"], z["TrMat"], float(z["pBL"]), list(z["cell_dims"]), 1, 6, int(z["min_l"]), 0.2,
                     int(z["max_nb_states"]))


def test_golden_cases_exist():
    assert len(SEG_CASES) >= 8 and os.path.isfile(os.path.join(GOLDEN, "seglen_len_hist.npz"))


@pytest.mark.parametrize("path", SEG_CASES, ids=IDS)
def test_oracle_reproduces_reference_golden(path):
    z = np.load(path)
    LP, hist, H = so.segment_len_chunk(z["C"], seg_model(z), int(z["isBL"]), int(z["max_nb_states"]), int(z["min_l"]),
                                       want_histories=True)
    np.testing.assert_allclose(LP, z["ref_LP"], rtol=1e-12)
    np.testing.assert_array_equal(H, z["ref_Bs"])
    np.testing.assert_allclose(hist, z["ref_hist"], atol=1e-12)


def test_oracle_len_hist_matches_reference_golden():
    z = np.load(os.path.join(GOLDEN, "seglen_len_hist.npz"))
    from extrack_b200 import tracking as xt

    params = xt.generate_params(nb_states=2, LocErr_type=1, nb_dims=2, LocErr_bounds=[0.005, 0.1], D_max=10,
                                Fractions_bounds=[0.001, 0.99], estimated_LocErr=[0.02], estimated_Ds=[1e-5, 0.25],
                                estimated_Fs=[0.6, 0.4], estimated_transition_rates=0.1)
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, 0.02, 2, 1)
    m = orc.Model(np.asarray(LocErr).reshape(-1), ds, Fs, TrMat, pBL, [1.0], 1, 6, 3, 0.2, 64)
    tracks = [z["C" + str(k)] for k in z["keys"]]
    got = so.len_hist(tracks, m, 64)
    np.testing.assert_allclose(got, z["ref_hist"], atol=1e-10)


# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", SEG_CASES, ids=IDS)
def test_gpu_P_segment_len_matches_reference_golden(path):
    from extrack_b200 import histograms as xh

    z = np.load(path)
    LP, Bs, hist = xh.P_segment_len(z["C"], z["loc_err"][None, None], z["ds"], z["Fs"], z["TrMat"], min_l=int(z["min_l"]),
                                    pBL=float(z["pBL"]), isBL=int(z["isBL"]), cell_dims=list(z["cell_dims"]), nb_substeps=1,
                                    max_nb_states=int(z["max_nb_states"]))
    assert LP.shape == z["ref_LP"].shape and Bs.shape == z["ref_Bs"].shape and hist.shape == z["ref_hist"].shape
    np.testing.assert_allclose(LP, z["ref_LP"], rtol=1e-9)
    np.testing.assert_array_equal(Bs, z["ref_Bs"])
    np.testing.assert_allclose(hist, z["ref_hist"], atol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [dict(nS=2, L=30, d=2, mx=500, isBL=1, nT=50, min_l=10),
                                 dict(nS=3, L=15, d=2, mx=500, isBL=0, nT=23, min_l=5),
                                 dict(nS=2, L=25, d=3, mx=200, isBL=1, nT=50, min_l=3, le=(0.02, 0.025, 0.04))])
def test_gpu_segment_len_vs_oracle_seeded(cfg):
    """Default-sized pruning (max_nb_states 500: 1000 / 1500 live sequences per track) against the oracle: histories per
    track identical unless the oracle finds a near-tie of the sort keys there (test_seglen_edges.check_chunk)."""
    import sys
    sys.path.insert(0, GOLDEN)
    from helpers import random_walk_tracks
    from make_golden_seglen import model
    from test_seglen_edges import check_chunk, oracle_chunk
    from extrack_b200 import histograms as xh

    m = model(cfg["nS"], cfg.get("le", (0.02,)))
    C = random_walk_tracks(cfg["nT"], cfg["L"], cfg["d"], np.random.default_rng(5), Ds=m.ds**2 / 0.04)
    LP, Bs, hist = xh.P_segment_len(C, np.asarray(m.loc_err)[None, None], m.ds, m.Fs, m.TrMat, min_l=cfg["min_l"], pBL=m.pBL,
                                    isBL=cfg["isBL"], cell_dims=[1.0], nb_substeps=1, max_nb_states=cfg["mx"])
    assert check_chunk(LP, Bs, hist, oracle_chunk(C, m, cfg["isBL"], cfg["mx"], cfg["min_l"]), str(cfg)) <= 0.05 * cfg["nT"]
    # size-independent properties: every track contributes weight <= number of segments; rows beyond L-1 empty
    assert hist.shape == (cfg["L"] - 1, cfg["nS"]) and (hist >= 0).all()


@pytest.mark.gpu
def test_gpu_len_hist_matches_reference_golden_and_errors():
    from extrack_b200 import histograms as xh
    from extrack_b200 import tracking as xt

    z = np.load(os.path.join(GOLDEN, "seglen_len_hist.npz"))
    vals = dict(zip([str(n) for n in z["names"]], z["values"]))
    params = xt.generate_params(nb_states=2, LocErr_type=1, nb_dims=2, LocErr_bounds=[0.005, 0.1], D_max=10,
                                Fractions_bounds=[0.001, 0.99], estimated_LocErr=[0.02], estimated_Ds=[1e-5, 0.25],
                                estimated_Fs=[0.6, 0.4], estimated_transition_rates=0.1)
    for k in params:
        assert abs(float(params[k].value) - vals[k]) <= 1e-15 * max(1.0, abs(vals[k])), k
    tracks = {str(k): z["C" + str(k)] for k in z["keys"]}
    tm = {}
    got = xh.len_hist(tracks, params, 0.02, cell_dims=[1.0], nb_states=2, max_nb_states=64, workers=1, nb_substeps=1, _timing=tm)
    assert got.shape == z["ref_hist"].shape and tm["kernel_ms"] > 0
    np.testing.assert_allclose(got, z["ref_hist"], atol=1e-9)
    with pytest.raises(NotImplementedError):
        xh.len_hist(tracks, params, 0.02, cell_dims=[1.0], nb_states=2, nb_substeps=2)
    with pytest.raises(NotImplementedError):
        xh.len_hist(tracks, params, 0.02, cell_dims=[1.0], nb_states=2, input_LocErr={k: v for k, v in tracks.items()})
    with pytest.raises(ValueError):  # 3 * 20000 live sequences per track do not fit in shared memory
        xh.len_hist(tracks, params, 0.02, cell_dims=[1.0], nb_states=2, max_nb_states=20000)
