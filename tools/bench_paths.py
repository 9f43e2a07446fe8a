#!/usr/bin/env python3
"""Cost of the MAP state paths: predict_path against predict_Bs on the config-4 shape (BASELINE.json: 2-state 2-D
tracks of 10-30 localisations, frame_len 8, threshold 0.1, max_nb_states 200, nb_max 1), one GPU.

In one process, alternating the two calls so that both see the same machine state:
  * engine level (tracks uploaded once): kernel time (the engine's CUDA-event ``ms_predict``) and call time including
    the read-back, for ``Engine.predict`` and ``Engine.predict_path``;
  * API level: wall time of ``tracking.predict_Bs`` and ``tracking.predict_path`` (upload included).
It also checks that both calls return the same posteriors bit for bit, and records the GPU name and power limit, the
spread of path_logp and the switch counts of the MAP paths and of the frame-wise argmax.  Prints one JSON line.

    python tools/bench_paths.py [--tracks 1000000] [--reps 3]
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
        raise SystemExit("bench_paths: no CUDA device (this measurement runs on the GPU only)")
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
    eng.predict_path(tab, 2)
    k_b, k_p, w_b, w_p = [], [], [], []
    for _ in range(a.reps):
        t = time.perf_counter()
        pb = eng.predict(tab, 2)
        w_b.append(time.perf_counter() - t)
        k_b.append(eng.stats()["ms_predict"])
        t = time.perf_counter()
        pr, paths, logps = eng.predict_path(tab, 2)
        w_p.append(time.perf_counter() - t)
        k_p.append(eng.stats()["ms_predict"])
    same = all(np.array_equal(x, y) for x, y in zip(pb, pr))
    eng.close()
    del pb, pr, paths, logps

    xt.predict_Bs(tracks, 0.02, p, **KW)
    xt.predict_path(tracks, 0.02, p, **KW)
    a_b, a_p = [], []
    for _ in range(a.reps):
        t = time.perf_counter()
        xt.predict_Bs(tracks, 0.02, p, **KW)
        a_b.append(time.perf_counter() - t)
        t = time.perf_counter()
        preds, paths, logp = xt.predict_path(tracks, 0.02, p, **KW)
        a_p.append(time.perf_counter() - t)
    lp = np.concatenate(list(logp.values()))
    switches = lambda d: int(sum(np.sum(x[:, 1:] != x[:, :-1]) for x in d.values()))
    interior, censored = xt.path_segments(paths, 2)

    med = lambda v: float(np.median(v))
    out = {"bench": "MAP state paths vs predict_Bs, config-4 shape (2 states, 2-D, L 10-30, fl 8, th 0.1, nb_max 1)",
           **gpu_info(), "tracks": n, "localisations": locs, "reps": a.reps,
           "kernel_ms_predict_Bs": med(k_b), "kernel_ms_path": med(k_p), "kernel_ratio": med(k_p) / med(k_b),
           "kernel_ms_all": {"predict_Bs": k_b, "path": k_p},
           "engine_call_ms_predict_Bs": 1e3 * med(w_b), "engine_call_ms_path": 1e3 * med(w_p),
           "api_ms_predict_Bs": 1e3 * med(a_b), "api_ms_predict_path": 1e3 * med(a_p),
           "d2h_bytes_predict_Bs": locs * 2 * 8, "d2h_bytes_path": locs * 2 * 8 + locs + n * 8,
           "preds_bitwise_equal": bool(same),
           "path_logp_quantiles": np.quantile(lp, [0.01, 0.1, 0.5, 0.9, 1.0]).tolist(),
           "switches_map": switches(paths), "switches_argmax": switches({k: np.argmax(v, -1) for k, v in preds.items()}),
           "segments_interior": int(interior.sum()), "segments_censored": int(censored.sum())}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
