#!/usr/bin/env python3
"""Cost of standard errors along the frozen grouping plan, config-2 shape (BASELINE.json: sim_FOV 2-state 2-D tracks of
10-30 localisations, frame_len 8, threshold 0.2, max_nb_states 120), one GPU.

In one process, on tracks uploaded once:
  * ms per frozen evaluation (``Engine.eval_frozen``, one parameter set) against ms per verified evaluation
    (``Engine.sum_logp`` along the resident plan with every decision re-checked), alternating the two;
  * the ``score_outer`` call time for the 7 free parameters of the default 2-state model (14 replays + k_score_gram),
    and k_score_gram's own kernel time from torch.profiler in a separate pass;
  * the wall time of ``tracking.param_uncertainty`` (upload and plan evaluation included) and its evaluation count;
  * the card's name and power limit.  Prints one JSON line.

    python tools/bench_uncertainty.py [--tracks 1000000] [--reps 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from extrack_b200 import _native  # noqa: E402
from extrack_b200 import tracking as xt  # noqa: E402
from extrack_b200._lmfit_compat import Parameters  # noqa: E402
from extrack_b200.simulate import sim_tracks  # noqa: E402

SIM = dict(max_track_len=30, min_track_len=10, LocErr=0.02, Ds=[0, 0.25], nb_dims=2, initial_fractions=[0.6, 0.4],
           TrMat=[[0.9, 0.1], [0.1, 0.9]], dt=0.02, pBL=0.05, cell_dims=[1, None, None])
KW = dict(cell_dims=[1], nb_states=2, frame_len=8, threshold=0.2, max_nb_states=120)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # (the measurement stands; the record says why the limit is missing)
        info["power_limit"] = f"unavailable: {e}"
    return info


def params(scale=1.0):
    p = Parameters()
    for k, v, lo, hi in (("LocErr", 0.02, 0.005, 0.1), ("D0", 1e-3, 0, 1), ("D1", 0.25, 0, 3), ("F0", 0.6, 0.001, 0.999),
                         ("p01", 0.1, 1e-4, 1), ("p10", 0.1, 1e-4, 1), ("pBL", 0.05, 1e-4, 1)):
        p.add(k, value=v * scale if k in ("D1", "LocErr") else v, min=lo, max=hi)
    p.add("F1", expr="1-F0")
    return p


def tables(p, st):
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    return xt.build_tables(LocErr, ds, Fs, TrMat, pBL, KW["cell_dims"], 1, KW["frame_len"], st[0].shape[1], KW["threshold"],
                           KW["max_nb_states"], 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_uncertainty: no CUDA device (this measurement runs on the GPU only)")
    tracks = sim_tracks(a.tracks, seed=99, device="cuda:0", **SIM)
    st, _ = xt._sorted_buckets(tracks)
    n = sum(x.shape[0] for x in st)
    p0 = tables(params(), st)
    ps = [tables(params(1 + 1e-4 * (k + 1)), st) for k in range(7)]
    pm = [tables(params(1 - 1e-4 * (k + 1)), st) for k in range(7)]
    inv = np.full(7, 1.0 / 2e-4)

    eng = _native.Engine(0)
    eng.upload(st, [0 if x.shape[1] == st[-1].shape[1] else 1 for x in st], xt.MAX_TRACKS_PER_CHUNK)
    eng.sum_logp(p0)
    eng.sum_logp(ps[0])  # verified evaluations from here on (same plan: the perturbation changes no decision)
    eng.eval_frozen([ps[0]])
    eng.score_outer(ps, pm, inv)
    t_ver, t_fro, t_sc = [], [], []
    for r in range(a.reps):
        for k in range(4):
            q = ps[k % 7]
            t = time.perf_counter()
            eng.sum_logp(q)
            t_ver.append(time.perf_counter() - t)
            t = time.perf_counter()
            eng.eval_frozen([q])
            t_fro.append(time.perf_counter() - t)
        t = time.perf_counter()
        eng.score_outer(ps, pm, inv)
        t_sc.append(time.perf_counter() - t)
    st_ = eng.stats()
    ref = eng.sum_logp(p0)
    same = bool(eng.eval_frozen([p0])[0] == ref)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            eng.score_outer(ps, pm, inv)
        torch.cuda.synchronize()
    k_ms = [e.device_time_total / 1e3 / e.count for e in prof.key_averages() if "k_score_gram" in e.key]
    eng.close()

    xt.param_uncertainty({k: v for k, v in tracks.items()}, 0.02, params(), **KW)  # warm-up
    w_u = []
    for _ in range(2):
        t = time.perf_counter()
        u = xt.param_uncertainty(tracks, 0.02, params(), **KW)
        w_u.append(time.perf_counter() - t)

    med = lambda v: float(np.median(v))
    out = {"bench": "standard errors along the frozen plan, config-2 shape (2 states, 2-D, L 10-30, fl 8, th 0.2)",
           **gpu_info(), "tracks": n, "reps": a.reps,
           "ms_verified_eval": 1e3 * med(t_ver), "ms_frozen_eval": 1e3 * med(t_fro), "frozen_over_verified": med(t_fro) / med(t_ver),
           "ms_all": {"verified": [1e3 * x for x in t_ver], "frozen": [1e3 * x for x in t_fro]},
           "last_verified_eval_stats": {k: st_[k] for k in ("plan_verified", "replanned", "pipelined")},
           "ms_score_outer_7dirs": 1e3 * med(t_sc), "ms_k_score_gram": k_ms[0] if k_ms else None,
           "frozen_sum_bitwise_equal_sum_logp": same,
           "ms_param_uncertainty": 1e3 * med(w_u), "param_uncertainty_evaluations": u.n_evaluations,
           "stderr": {k: v for k, v in u.stderr.items()}, "newton_decrement": u.newton_decrement}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
