#!/usr/bin/env python3
"""Cost of the posterior samples: sample_paths at n_samples = 1, 10 and 100 against predict_Bs on the config-4 shape
(BASELINE.json: 2-state 2-D tracks of 10-30 localisations, frame_len 8, threshold 0.1, max_nb_states 200, nb_max 1),
one GPU.

In one process, alternating the calls so that all see the same machine state:
  * engine level (tracks uploaded once): kernel time (the engine's CUDA-event ``ms_predict``) and call time including
    the read-back, for ``Engine.predict`` and ``Engine.predict_samples`` at every n_samples;
  * API level: wall time of ``tracking.predict_Bs`` and ``tracking.sample_paths`` (upload included).
It also checks that every call returns the same posteriors bit for bit, and records the GPU name and power limit.
Prints one JSON line.

    python tools/bench_samples.py [--tracks 1000000] [--reps 3]
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
KW = dict(cell_dims=[1], nb_states=2, frame_len=8, threshold=0.1, max_nb_states=200)
COUNTS = (1, 10, 100)


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")][:2]
    except Exception as e:  # (the measurement stands; the record says why the limit is missing)
        info["power_limit"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_samples: no CUDA device (this measurement runs on the GPU only)")
    tracks = sim_tracks(a.tracks, seed=99, device="cuda:0", **SIM)
    st, _ = xt._sorted_buckets(tracks)
    p = Parameters()
    for k, v in dict(LocErr=0.02, D0=1e-5, D1=0.25, F0=0.6, p01=0.1, p10=0.1, pBL=0.05).items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(p, 0.02, 2, 1)
    tab = xt.build_tables(LocErr, ds, Fs, TrMat, pBL, [1], 1, KW["frame_len"], st[0].shape[1], KW["threshold"],
                          KW["max_nb_states"], 2)
    locs = sum(x.shape[0] * x.shape[1] for x in st)
    n = sum(x.shape[0] for x in st)

    eng = _native.Engine(0)
    eng.upload(st, [0 if x.shape[1] == st[-1].shape[1] else 1 for x in st], xt.MAX_TRACKS_PER_CHUNK)
    eng.predict(tab, 2)  # warm-up of both instantiations and of the host allocations
    eng.predict_samples(tab, 2, COUNTS[0], 0)
    k_b, w_b = [], []
    k_s = {c: [] for c in COUNTS}
    w_s = {c: [] for c in COUNTS}
    same = True
    for _ in range(a.reps):
        t = time.perf_counter()
        pb = eng.predict(tab, 2)
        w_b.append(time.perf_counter() - t)
        k_b.append(eng.stats()["ms_predict"])
        for c in COUNTS:
            t = time.perf_counter()
            pr, smp, lps = eng.predict_samples(tab, 2, c, 0)
            w_s[c].append(time.perf_counter() - t)
            k_s[c].append(eng.stats()["ms_predict"])
            same = same and all(np.array_equal(x, y) for x, y in zip(pb, pr))
            del pr, smp, lps
    eng.close()
    del pb

    xt.predict_Bs(tracks, 0.02, p, **KW)
    xt.sample_paths(tracks, 0.02, p, n_samples=COUNTS[0], **KW)
    a_b = []
    a_s = {c: [] for c in COUNTS}
    for _ in range(a.reps):
        t = time.perf_counter()
        ref = xt.predict_Bs(tracks, 0.02, p, **KW)
        a_b.append(time.perf_counter() - t)
        for c in COUNTS:
            t = time.perf_counter()
            preds, smp, lp = xt.sample_paths(tracks, 0.02, p, n_samples=c, **KW)
            a_s[c].append(time.perf_counter() - t)
            same = same and all(np.array_equal(ref[k], preds[k]) for k in ref)
            del preds, smp, lp

    med = lambda v: float(np.median(v))
    out = {"bench": "posterior samples vs predict_Bs, config-4 shape (2 states, 2-D, L 10-30, fl 8, th 0.1, nb_max 1)",
           **gpu_info(), "tracks": n, "localisations": locs, "reps": a.reps, "n_samples": list(COUNTS),
           "kernel_ms_predict_Bs": med(k_b), "kernel_ms_samples": {c: med(k_s[c]) for c in COUNTS},
           "kernel_ratio": {c: med(k_s[c]) / med(k_b) for c in COUNTS},
           "kernel_ms_all": {"predict_Bs": k_b, **{f"samples_{c}": k_s[c] for c in COUNTS}},
           "engine_call_ms_predict_Bs": 1e3 * med(w_b), "engine_call_ms_samples": {c: 1e3 * med(w_s[c]) for c in COUNTS},
           "api_ms_predict_Bs": 1e3 * med(a_b), "api_ms_sample_paths": {c: 1e3 * med(a_s[c]) for c in COUNTS},
           "d2h_bytes_predict_Bs": locs * 2 * 8, "d2h_bytes_samples": {c: locs * 2 * 8 + c * (locs + n * 8) for c in COUNTS},
           "preds_bitwise_equal": bool(same)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
