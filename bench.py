#!/usr/bin/env python3
"""Benchmark of the track-likelihood hot path (BASELINE.json metric: track-steps/s of one -log L
evaluation, 2-state 2-D, frame_len = 8, sim_FOV synthetic tracks of length 10-30).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--tracks T] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one objective evaluation over the resident data set (plan kernels, replay kernels,
device reduction; plus one 8-byte all-reduce when N > 1).  Plan and replay are launched per group of
length buckets on several streams (the latency-bound plan kernel of one group overlaps the replay
of another); the per-kernel times behind `roofline` come from a few extra evaluations in the
two-phase mode (one plan launch, one replay launch) after the timed region.  N = 1 workload: BASELINE.json configs[1]
(10^6 tracks on one B200).  For N > 1 every rank holds its own 10^6-track field of view
(weak scaling); ranks evaluate their chunks independently and the partial log-likelihoods are
summed with one NCCL all-reduce per step.  Prints ONE JSON line (rank 0).

Besides the headline the line carries: `strong` (the SAME 10^6 tracks split over the N ranks by
`shard_chunks` — the split the north star names — with per-evaluation time, per-rank plan / replay times and the
efficiency against one GPU), `api` (one evaluation through the Python objective `cum_Proba_Cs` with parameters that
change every call, as BFGS does) and `secondary` (BASELINE configs 3, 5 and 4 at bounded sizes, sharded over the N
ranks through the API).

--impl reference times the CPU path instead: the numpy oracle port of the reference algorithm
(the reference is pure Python and does not travel to the GPU box) on all host cores, on a bounded
sample of the same workload.

--dump-outputs DIR writes what the timed path returned in its last timed step to DIR/sum_logp.npy (float64, shape
[1]: the log-likelihood summed over the data set, after the all-reduce when N > 1).  The data set is generated from
fixed seeds and the parameter table of a step depends only on its index, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SIM_KW = dict(max_track_len=30, min_track_len=10, LocErr=0.02, Ds=[0, 0.25], nb_dims=2, initial_fractions=[0.6, 0.4],
              TrMat=[[0.9, 0.1], [0.1, 0.9]], dt=0.02, pBL=0.05, cell_dims=[1, None, None])
EVAL = dict(D0=1e-5, D1=0.25, LocErr=0.02, F0=0.6, p01=0.1, p10=0.1, pBL=0.05)
FRAME_LEN, THRESHOLD, MAX_NB_STATES, DT, CELL = 8, 0.2, 120, 0.02, [1]
METRIC = "track-steps/sec of -logL eval (2-state, frame_len=8)"
UNIT = "track-steps/s"


def eval_params():
    from extrack_b200._lmfit_compat import Parameters

    p = Parameters()
    for k, v in EVAL.items():
        p.add(k, value=v)
    p.add("F1", expr="1-F0")
    return p


def param_variants(min_len, n=8):
    """Parameter tables of consecutive objective calls the way BFGS makes them: the base point, then one parameter at a
    time moved by 1.5e-8 relative (scipy's finite-difference step).  Every timed step uses the next table, so no two
    consecutive evaluations see the same numbers."""
    from extrack_b200 import tracking as xt

    out = []
    names = [None, "D1", "LocErr", "F0", "p01", "p10", "pBL", "D0"]
    for i in range(n):
        params = eval_params()
        k = names[i % len(names)]
        if k is not None:
            params[k].value = EVAL[k] * (1.0 + 1.5e-8 * (1 + i // len(names)))
        LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, DT, 2, 1)
        out.append(xt.build_tables(LocErr, ds, Fs, TrMat, pBL, CELL, 1, FRAME_LEN, min_len, THRESHOLD, MAX_NB_STATES, 2))
    return out


def oracle_model(min_len):
    import numpy as np

    from extrack_b200 import tracking as xt
    from oracle import extrack_oracle as orc

    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(eval_params(), DT, 2, 1)
    return orc.Model(np.asarray(LocErr[0]).reshape(-1), ds, Fs, TrMat, pBL, CELL, 1, FRAME_LEN, min_len, THRESHOLD, MAX_NB_STATES)


def cpu_leg(npz_path):
    """Runs in a fresh, CUDA-free subprocess (the oracle forks a worker pool): evaluate the sample
    stored in `npz_path` with the numpy oracle port on all host cores; print one JSON line."""
    import numpy as np

    from oracle import extrack_oracle as orc

    z = np.load(npz_path)
    st = [z[k] for k in sorted(z.files, key=int)]
    cores = len(os.sched_getaffinity(0))
    model = oracle_model(st[0].shape[1])
    orc.neg_log_likelihood(st[:1], model, workers=1)  # warm-up: lazy scipy.stats import
    t = time.perf_counter()
    val = orc.neg_log_likelihood(st, model, workers=cores)
    secs = time.perf_counter() - t
    print(json.dumps({"value": orc.track_steps(st) / secs, "neglogl": val, "secs": secs, "cores": cores,
                      "tracks": int(sum(len(a) for a in st))}))


def cpu_baseline(st):
    """cpu_baseline leg: the oracle port on a bounded sample, in a subprocess."""
    import tempfile

    import numpy as np

    path = os.path.join(tempfile.mkdtemp(), "sample.npz")
    np.savez(path, **{str(a.shape[1]): a for a in st})
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-leg", path], capture_output=True, text=True, timeout=1200)
    os.remove(path)
    if out.returncode != 0:
        raise RuntimeError("cpu_baseline leg failed: " + out.stderr[-2000:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def dump_outputs(path, sum_logp):
    """--dump-outputs: the result of the last timed step as `path`/sum_logp.npy."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "sum_logp.npy"), np.array([sum_logp], dtype=np.float64))


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons of this rank's GPU, sampled during the timed region.  Through NVML in-process (one
    handle, a few microseconds per sample); spawning `nvidia-smi` every 100 ms - the fallback when NVML cannot be loaded -
    initialises the driver's management layer for all GPUs of the box at every call and was seen to stretch the timed
    steps of an 8-GPU run by tenths of a millisecond."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []
        self.nvml = self.handle = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(index)
            bdf = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(bdf.encode())
            self.nvml = pynvml
        except Exception:
            self.nvml = self.handle = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            pw = float("nan")
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        flag = lambda bit: "Active" if (r & bit) else "Not Active"  # noqa: E731
        return [str(sm), str(mx), f"{pw:.1f}", flag(n.nvmlClocksEventReasonHwSlowdown), flag(n.nvmlClocksEventReasonHwThermalSlowdown),
                flag(n.nvmlClocksEventReasonSwThermalSlowdown), flag(n.nvmlClocksEventReasonSwPowerCap)]

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.rows.append(self._sample_nvml())
                    time.sleep(0.02)
                    continue
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                if self.nvml is not None:  # NVML query failed: fall back to the command-line tool
                    self.nvml = None
            time.sleep(0.1)

    def summary(self):
        import statistics

        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "via": "nvml" if self.handle is not None and self.nvml is not None else "nvidia-smi"}


def _bind_to_gpu_numa_node(local):
    """Restrict this rank to the CPUs of the NUMA node its GPU hangs off, so that the pinned host buffers of the e2e leg
    are first touched (= placed) next to the GPU.  Returns (previous affinity, description); a no-op when sysfs has no answer."""
    import torch

    try:
        pr = torch.cuda.get_device_properties(local)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None, {"node": None, "why": "sysfs reports no NUMA node for " + bdf}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        prev = os.sched_getaffinity(0)
        cpus &= prev
        if not cpus:
            return None, {"node": node, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, cpus)
        return prev, {"node": node, "cpus": len(cpus)}
    except Exception as e:  # noqa: BLE001 - placement is an optimisation, never a failure
        return None, {"node": None, "why": f"{type(e).__name__}: {e}"}


def _dist_max(x, local, world):
    """max over ranks of a scalar (device-timed milliseconds)."""
    import torch

    t = torch.tensor([float(x)], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        import torch.distributed as dist

        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _time_sharded(ts, p, steps, local, world):
    """Per-evaluation device time (max over ranks) of a TrackSet sharded over the process group: K evaluations, each
    followed by the 8-byte all-reduce, bracketed by barrier + synchronize; plus this rank's two-phase kernel times."""
    import torch

    buf = torch.zeros(1, dtype=torch.float64, device=f"cuda:{local}")
    stream = torch.cuda.current_stream().cuda_stream
    eng = ts.engine

    plist = p if isinstance(p, (list, tuple)) else [p]
    p = plist[0]
    count = [0]

    def step():
        if ts.n_local_chunks:
            eng.sum_logp_async(plist[count[0] % len(plist)], buf.data_ptr(), stream)
            count[0] += 1
        else:
            buf.zero_()
        if world > 1:
            import torch.distributed as dist

            dist.all_reduce(buf)

    def barrier():
        if world > 1:
            import torch.distributed as dist

            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(3):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    ms = _dist_max(e0.elapsed_time(e1) / steps, local, world)
    total = float(buf.item())
    plan = replay = 0.0
    if ts.n_local_chunks:
        eng.set_option("pipeline", 0)
        for i in range(5):
            eng.sum_logp(p)
            if i >= 2:
                s = eng.stats()
                plan += s["ms_plan"] / 3
                replay += s["ms_replay"] / 3
        eng.set_option("pipeline", 1)
    return ms, total, _dist_max(plan, local, world), _dist_max(replay, local, world)


def strong_block(st0, p, steps, local, rank, world, ms_one_gpu):
    """The SAME data set split over the ranks by `shard_chunks` (whole chunks, longest-processing-time-first on
    nT*(L-1); reference unit: the chunk list of tracking.py:1030-1044): per-evaluation time and the efficiency
    against one GPU holding all chunks (`ms_one_gpu`, measured on rank 0 in this run)."""
    from extrack_b200 import tracking as xt

    ts = xt.TrackSet(st0, device=local)  # rank / world size from the initialised process group
    ms, total, plan, replay = _time_sharded(ts, p, steps, local, world)
    chunks = ts.n_local_chunks
    steps_local = ts.engine.stats()["track_steps"] if chunks else 0
    ts.close()
    all_steps = sum((a.shape[1] - 1) * a.shape[0] for a in st0)
    return {"what": "the same 10^6-track data set (seed 0) split over the N ranks by shard_chunks; one 8-byte all-reduce per evaluation",
            "n_gpus": world, "tracks": int(sum(len(a) for a in st0)), "track_steps": int(all_steps), "ms_per_eval": ms,
            "value": all_steps / (ms * 1e-3), "unit": UNIT, "ms_per_eval_one_gpu": ms_one_gpu,
            "efficiency_vs_one_gpu": ms_one_gpu / (world * ms), "target_efficiency_at_8": 0.85,
            "rank0": {"chunks": int(chunks), "track_steps": int(steps_local)},
            "kernel_ms_max_over_ranks": {"plan": plan, "replay_and_reduce": replay}, "sum_logp": total}


def in_process_block(st0, pvar, steps, rank, world, ms_one_gpu):
    """Strong scaling of the same data set with ONE Python process driving the N GPUs through TrackSet(devices=...)
    (xt_multi_*: per-device worker threads, per-chunk sums added in global chunk order, no collective)."""
    import torch.distributed as dist

    from extrack_b200 import _native
    from extrack_b200 import tracking as xt

    store = dist.distributed_c10d._get_default_store()
    out = None
    if rank == 0:
        try:
            if _native.device_count() < world:
                raise RuntimeError("fewer visible devices than ranks")
            ts = xt.TrackSet(st0, devices=list(range(world)), rank=0, world_size=1)
            for p in pvar * 2:
                ts.sum_logp(p)
            n = max(steps, len(pvar))
            t = time.perf_counter()
            for i in range(n):
                v = ts.sum_logp(pvar[i % len(pvar)])
            ms = (time.perf_counter() - t) / n * 1e3
            st_ = ts.engine.stats()
            load = ts.engine.device_load()
            all_steps = sum((a.shape[1] - 1) * a.shape[0] for a in st0)
            out = {"what": "one process, N GPUs: TrackSet(devices=range(N)).sum_logp, wall clock per call incl. the read-back",
                   "n_gpus": world, "ms_per_eval": ms, "value": all_steps / (ms * 1e-3), "unit": UNIT,
                   "efficiency_vs_one_gpu": ms_one_gpu / (world * ms), "chunks_per_device": [c for _, c, _ in load],
                   "plan_verified": int(st_["plan_verified"]), "sum_logp_last": v}
            ts.close()
        except Exception as e:  # noqa: BLE001 - reported in the line, the other ranks must be released
            out = {"error": repr(e)}
        store.set("xt_in_process_done", "1")
    else:
        store.wait(["xt_in_process_done"])
    return out


def api_block(ts, st, n_calls=60):
    """One evaluation through the Python objective `extrack_b200.tracking.cum_Proba_Cs` (parameter extraction, the
    field-of-view table with its 1000-point ndtr, the ctypes call, the read-back) on the resident data set, with
    parameters that change at every call the way BFGS finite differences do."""
    import contextlib
    import io

    from extrack_b200 import tracking as xt

    params = eval_params()
    base = dict(EVAL)
    names = ["D1", "LocErr", "F0", "p01", "p10", "pBL", "D0"]
    sink = io.StringIO()
    with contextlib.redirect_stdout(sink):
        for i in range(5):
            xt.cum_Proba_Cs(params, st, DT, CELL, None, 2, 1, FRAME_LEN, 0, 1, 1, THRESHOLD, MAX_NB_STATES, _trackset=ts)
        t = time.perf_counter()
        for i in range(n_calls):
            k = names[i % len(names)]
            params[k].value = base[k] * (1.0 + 1.5e-8 * (1 + i // len(names)))
            v = xt.cum_Proba_Cs(params, st, DT, CELL, None, 2, 1, FRAME_LEN, 0, 1, 1, THRESHOLD, MAX_NB_STATES, _trackset=ts)
            params[k].value = base[k]
        wall = (time.perf_counter() - t) / n_calls
    return {"api_eval_ms": wall * 1e3, "calls": n_calls, "neglogl_last": v,
            "what": "wall time per extrack_b200.tracking.cum_Proba_Cs call on the resident config-2 data set, one parameter "
                    "perturbed by 1.5e-8 relative per call (finite-difference pattern of BFGS)"}


SECONDARY = {
    "3": dict(name="configs[2]: 3-state 2D, nb_substeps=2, frame_len=6, max_nb_states=500", tracks=200_000,
              sim=dict(max_track_len=30, min_track_len=10, LocErr=0.02, Ds=[0, 0.04, 0.25], nb_dims=2,
                       initial_fractions=[0.33, 0.33, 0.34], TrMat=[[0.9, 0.1, 0.0], [0.05, 0.91, 0.04], [0.01, 0.06, 0.93]],
                       dt=0.02, pBL=0.05, cell_dims=[1, None, None]),
              ev=dict(nb_substeps=2, frame_len=6, threshold=0.2, max_nb_states=500)),
    "5": dict(name="configs[4]: 3-state 3D long tracks (100-200), frame_len=10", tracks=20_000,
              sim=dict(max_track_len=200, min_track_len=100, LocErr=0.02, Ds=[0, 0.05, 0.25], nb_dims=3,
                       initial_fractions=[0.3, 0.3, 0.4], TrMat=[[0.9, 0.05, 0.05], [0.05, 0.9, 0.05], [0.05, 0.05, 0.9]],
                       dt=0.02, pBL=0.002, cell_dims=[10, None, None]),
              ev=dict(nb_substeps=1, frame_len=10, threshold=0.2, max_nb_states=120)),
}


def _params_for(sim):
    from extrack_b200._lmfit_compat import Parameters

    p = Parameters()
    p.add("LocErr", value=sim["LocErr"])
    nS = len(sim["Ds"])
    for i, D in enumerate(sim["Ds"]):
        p.add(f"D{i}", value=max(D, 1e-5))
    for i, F in enumerate(sim["initial_fractions"][:-1]):
        p.add(f"F{i}", value=F)
    p.add(f"F{nS-1}", expr="1-" + "-".join(f"F{i}" for i in range(nS - 1)))
    for i in range(nS):
        for j in range(nS):
            if i != j:
                p.add(f"p{i}{j}", value=max(sim["TrMat"][i][j], 1e-4))
    p.add("pBL", value=sim["pBL"])
    return p


def secondary_block(local, rank, world, scale=1.0):
    """BASELINE configs 3, 5 (likelihood) and 4 (predict_Bs) at bounded sizes, sharded over the ranks through the API
    (TrackSet under the process group / predict_Bs(gather=False)); every rank generates the same data set."""
    import torch

    from extrack_b200 import tracking as xt
    from extrack_b200.simulate import sim_tracks

    out = {}
    for key, cfg in SECONDARY.items():
        sim, ev = cfg["sim"], cfg["ev"]
        tracks = sim_tracks(int(cfg["tracks"] * scale), seed=4242, device=f"cuda:{local}", **sim)
        st, _ = xt._sorted_buckets(tracks)
        nS = len(sim["Ds"])
        LocErr, ds, Fs, TrMat, pBL = xt.extract_params(_params_for(sim), sim["dt"], nS, ev["nb_substeps"])
        p = xt.build_tables(LocErr, ds, Fs, TrMat, pBL, [sim["cell_dims"][0]], ev["nb_substeps"], ev["frame_len"], st[0].shape[1],
                            ev["threshold"], ev["max_nb_states"], st[0].shape[2])
        ts = xt.TrackSet(st, device=local)
        ms, total, plan, replay = _time_sharded(ts, p, 5, local, world)
        stats = ts.engine.stats() if ts.n_local_chunks else {"max_nB_in": 0}
        ts.close()
        steps = sum((a.shape[1] - 1) * a.shape[0] for a in st)
        out["config_" + key] = {"workload": cfg["name"], "tracks": int(sum(len(a) for a in st)), "track_steps": int(steps),
                                "n_gpus": world, "ms_per_eval": ms, "track_steps_per_s": steps / (ms * 1e-3),
                                "kernel_ms_max_over_ranks": {"plan": plan, "replay_and_reduce": replay},
                                "max_live_sequences_rank0": int(stats["max_nB_in"]), "sum_logp": total}
        del tracks, st
        torch.cuda.empty_cache()
    # config 4: state annotation, every rank annotates its slice of every bucket (no collective on the data path)
    n4 = int(1_000_000 * scale)
    tracks = sim_tracks(n4, seed=99, device=f"cuda:{local}", **SIM_KW)
    params = eval_params()
    xt.predict_Bs({k: v[:64] for k, v in tracks.items()}, DT, params, cell_dims=CELL, nb_states=2, frame_len=FRAME_LEN, gather=False)
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()
    t = time.perf_counter()
    pred = xt.predict_Bs(tracks, DT, params, cell_dims=CELL, nb_states=2, frame_len=FRAME_LEN, gather=False)
    torch.cuda.synchronize()
    wall = _dist_max(time.perf_counter() - t, local, world)
    locs = sum(int(k) * len(v) for k, v in tracks.items())
    out["config_4"] = {"workload": "configs[3]: predict_Bs, 2-state, frame_len=8, threshold 0.1, max_nb_states 200, nb_max=1",
                       "tracks": n4, "localisations": int(locs), "n_gpus": world, "s_per_call_incl_upload_and_readback": wall,
                       "localisations_per_s": locs / wall,
                       "rows_annotated_rank0": int(sum(len(v) for v in pred.values()))}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    n = args.ref_tracks
    # build the sample once, then time K steps (each step = one objective evaluation of the sample)
    from extrack_b200 import tracking as xt
    from extrack_b200.simulate import sim_tracks
    from oracle import extrack_oracle as orc

    tracks = sim_tracks(n, seed=10_000, device="cpu", **SIM_KW)
    st, _ = xt._sorted_buckets(tracks)
    model = oracle_model(st[0].shape[1])
    steps_per_eval = orc.track_steps(st)
    for _ in range(args.warmup):
        orc.neg_log_likelihood(st, model, workers=cores)
    t = time.perf_counter()
    for _ in range(args.steps):
        val = orc.neg_log_likelihood(st, model, workers=cores)
    dt = time.perf_counter() - t
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, -val)
    v = steps_per_eval * args.steps / dt
    sample = f"{n} sim_FOV tracks ({steps_per_eval} track-steps, whole 2000-track chunks) per step, numpy oracle port, fork pool"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: sim_FOV synthetic 2-state 2D, 10^6 tracks length 10-30, frame_len=8, one -logL evaluation",
                   "sample": f"{n} tracks of the same generator per step (the metric is throughput-normalised: the CPU path needs "
                             f"~{1e6 / n * 1e-3 * (1e3 * dt / args.steps):.0f} s per evaluation of the full 10^6 tracks)",
                   "tracks_per_step": n, "neglogl": val},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--tracks", type=int, default=1_000_000, help="tracks per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-tracks", type=int, default=100_000)
    ap.add_argument("--cpu-tracks", type=int, default=200_000, help="sample size of the cpu_baseline leg")
    ap.add_argument("--cpu-leg", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the strong / api / secondary blocks (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step to DIR/sum_logp.npy (rank 0)")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.cpu_leg:
        return cpu_leg(args.cpu_leg)
    if args.impl == "reference":
        return run_reference(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    import numpy as np
    import torch

    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from extrack_b200 import _native
    from extrack_b200 import tracking as xt
    from extrack_b200.simulate import sim_tracks

    # ---- synthetic data: generated on this rank's GPU (seed differs per rank), config 2 ----
    t0 = time.perf_counter()
    tracks = sim_tracks(args.tracks, seed=1000 * rank, device=f"cuda:{local}", **SIM_KW)
    st, _ = xt._sorted_buckets(tracks)
    gen_s = time.perf_counter() - t0
    torch.cuda.empty_cache()
    params = eval_params()
    LocErr, ds, Fs, TrMat, pBL = xt.extract_params(params, DT, 2, 1)
    p = xt.build_tables(LocErr, ds, Fs, TrMat, pBL, CELL, 1, FRAME_LEN, st[0].shape[1], THRESHOLD, MAX_NB_STATES, 2)

    ts = xt.TrackSet(st, rank=0, world_size=1, device=local)  # every rank owns its whole field of view
    eng = ts.engine
    if os.environ.get("XT_BENCH_TWO_PHASE"):  # profiling aid: one plan launch + one replay launch per evaluation
        eng.set_option("pipeline", 0)
    buf = torch.zeros(1, dtype=torch.float64, device=f"cuda:{local}")
    stream = torch.cuda.current_stream().cuda_stream

    pvar = param_variants(st[0].shape[1])  # pvar[0] = p; the others differ by one BFGS finite-difference step each
    nstep = [0]
    served = {"verified": 0, "chunks_planned_again": 0, "planned_from_scratch": 0}

    # N > 1: one 8-byte all-reduce per step on torch's current stream, right behind the evaluation that produced the
    # partial sum (the engine orders its streams after that stream, so step i + 1 starts when the collective of step i
    # is done).  An asynchronous variant (collective on NCCL's own stream, two alternating result buffers) was measured:
    # 0.97 of N x one GPU at N = 2, but at N = 8 the collective's kernels compete with the next replay for SM slots on
    # all eight ranks and the step time rose from 1.76 to 2.17 ms (profiles/r12/bench_n8_async_allreduce.json).
    def step():
        eng.sum_logp_async(pvar[nstep[0] % len(pvar)], buf.data_ptr(), stream)
        nstep[0] += 1
        if world > 1:
            dist.all_reduce(buf)

    def drain():
        pass

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    launches = 0
    for _ in range(args.steps):
        step()
        s = eng.stats()
        launches += s["k1_launches"] + s["k2_launches"]
        served["verified" if s["plan_verified"] else "planned_from_scratch"] += 1
        served["chunks_planned_again"] += s["replanned"]
    drain()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    last = float(buf.item()) if args.dump_outputs else None  # result of the last timed step (buf is reused below)
    eng.sum_logp_async(p, buf.data_ptr(), stream)  # (untimed) the base parameters again: `sum_logp` of the line
    if world > 1:
        dist.all_reduce(buf)
    torch.cuda.synchronize()
    total = float(buf.item())
    stats = eng.stats()
    total_local = eng.sum_logp(p)  # this rank's own sum (== total on one GPU)
    # per-kernel device times (CUDA events recorded by the engine on its own stream around the
    # single plan launch and the single replay launch of the two-phase mode)
    eng.set_option("pipeline", 0)
    ms_plan = ms_replay = 0.0
    ksteps = max(3, min(20, args.steps))
    for i in range(ksteps + 2):
        eng.sum_logp(p)
        if i >= 2:
            s = eng.stats()
            ms_plan += s["ms_plan"]
            ms_replay += s["ms_replay"]
    ms_plan /= ksteps
    ms_replay /= ksteps
    eng.set_option("pipeline", 1)
    # ---- optional FP32 replay (north star: FP32 path within 1e-4 relative): same data, same plan kernel ----
    eng.set_option("fp32_replay", 1)
    for _ in range(3):
        step32 = eng.sum_logp(p)
    f32_used = eng.stats()["fp32"]
    fsteps = max(3, min(50, args.steps))
    torch.cuda.synchronize()
    fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fe0.record()
    for _ in range(fsteps):
        eng.sum_logp_async(p, buf.data_ptr(), stream)
    fe1.record()
    torch.cuda.synchronize()
    f32_ms = fe0.elapsed_time(fe1) / fsteps
    eng.set_option("pipeline", 0)
    f32_replay = 0.0
    for i in range(5):
        eng.sum_logp(p)
        if i >= 2:
            f32_replay += eng.stats()["ms_replay"] / 3
    eng.set_option("pipeline", 1)
    eng.set_option("fp32_replay", 0)
    sampler.stop_flag = True
    tms = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{local}")
    tsteps = torch.tensor([float(stats["track_steps"])], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsteps)
    ms = float(tms.item())
    all_steps = float(tsteps.item())
    value = all_steps * args.steps / (ms * 1e-3)

    # ---- e2e: public API with HOST buffers: upload (pinned H2D + device repack) + evaluate + read back ----
    h2d = int(sum(a.nbytes for a in st))
    prev_aff, numa = _bind_to_gpu_numa_node(local)
    pinned = []
    for a in st:
        b = _native.pinned_empty(a.shape)
        b[...] = a
        pinned.append(b)
    if prev_aff is not None:
        os.sched_setaffinity(0, prev_aff)
    bl = [0 if a.shape[1] == st[-1].shape[1] else 1 for a in st]
    e2e_eng = _native.Engine(local)
    for _ in range(2):  # warm-up: allocations, first (two-phase) evaluation
        e2e_eng.sum_logp_host(pinned, bl, xt.MAX_TRACKS_PER_CHUNK, p)
    barrier()
    t = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_val = e2e_eng.sum_logp_host(pinned, bl, xt.MAX_TRACKS_PER_CHUNK, p)
        if world > 1:
            b2 = torch.tensor([e2e_val], dtype=torch.float64, device=f"cuda:{local}")
            dist.all_reduce(b2)
            e2e_val = float(b2.item())
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t) / args.e2e_steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{local}")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = all_steps / float(te.item())
    e2e_eng.close()

    # ---- strong scaling of the headline data set, API-level evaluation cost, other BASELINE configs ----
    strong = api = secondary = None
    if not args.no_secondary:
        ksteps2 = max(5, min(50, args.steps))
        # one GPU holding every chunk of the seed-0 data set: that is rank 0's own (weak-scaling) data set
        ms_one = _time_sharded(ts, pvar, ksteps2, local, 1)[0] if rank == 0 else 0.0
        ms_one = _dist_max(ms_one, local, world)
        if world > 1:
            st0 = st if rank == 0 else xt._sorted_buckets(sim_tracks(args.tracks, seed=0, device=f"cuda:{local}", **SIM_KW))[0]
            torch.cuda.empty_cache()
            strong = strong_block(st0, pvar, ksteps2, local, rank, world, ms_one)
            # the same split driven by ONE process (xt_multi_*: what a notebook / GUI caller of param_fitting gets with
            # workers = N): rank 0 drives all N GPUs while the other ranks wait on the store (no GPU work, no collective)
            strong["in_process"] = in_process_block(st0, pvar, ksteps2, rank, world, ms_one)
            del st0
        else:
            strong = {"what": "one GPU: the strong-scaling split is the headline itself", "n_gpus": 1, "tracks": int(stats["n_tracks"]),
                      "track_steps": int(stats["track_steps"]), "ms_per_eval": ms_one, "value": stats["track_steps"] / (ms_one * 1e-3),
                      "unit": UNIT, "ms_per_eval_one_gpu": ms_one, "efficiency_vs_one_gpu": 1.0, "target_efficiency_at_8": 0.85,
                      "kernel_ms_max_over_ranks": {"plan": ms_plan, "replay_and_reduce": ms_replay}}
        if rank == 0:
            api = api_block(ts, st)
            api["resident_ms_per_eval"] = ms_one
            api["host_tail_ms"] = api["api_eval_ms"] - ms_one
        secondary = secondary_block(local, rank, world)

    if rank == 0:
        peak = eng.fp64_peak_tflops()
        # algorithmic flops of the replay kernel (SURVEY.md §8d): F = nB_in*(25+9d) + nG*(3+d) per track-step
        d = 2
        flops = stats["seq_updates"] * (25 + 9 * d) + stats["seq_groups"] * (3 + d)
        replay_ms = ms_replay
        achieved = flops / (replay_ms * 1e-3) / 1e12
        alg_bytes = sum(a.size for a in st) * 8 + stats["n_tracks"] * 8
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # ---- cpu_baseline: oracle port on a bounded sample of the same generator, in a CUDA-free
        #      subprocess; the engine is evaluated on the same sample as a parity check ----
        cpu, parity = None, None
        if world == 1 and not args.no_cpu:
            sample = sim_tracks(args.cpu_tracks, seed=777_000, device=f"cuda:{local}", **SIM_KW)
            st_c, _ = xt._sorted_buckets(sample)
            r = cpu_baseline(st_c)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                   "sample": f"{r['tracks']} sim_FOV tracks of the same generator/config (seed 777000), one evaluation = "
                             f"{r['secs']:.1f} s on {r['cores']} processes (numpy oracle port of the reference algorithm, fork pool)"}
            tsc = xt.TrackSet(st_c, rank=0, world_size=1, device=local)
            pc = xt.build_tables(LocErr, ds, Fs, TrMat, pBL, CELL, 1, FRAME_LEN, st_c[0].shape[1], THRESHOLD, MAX_NB_STATES, 2)
            parity = abs(-tsc.sum_logp(pc) - r["neglogl"]) / abs(r["neglogl"])
            tsc.close()
        traffic = None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "k2_traffic.json")))
            if int(tj.get("tracks", -1)) == int(stats["n_tracks"]):
                traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "configs[1]: sim_FOV synthetic 2-state 2D, 10^6 tracks length 10-30, frame_len=8, one -logL evaluation",
                       "tracks_per_gpu": int(stats["n_tracks"]), "track_steps_per_gpu": int(stats["track_steps"]),
                       "chunks_per_gpu": int(stats["n_chunks"]), "max_live_sequences": int(stats["max_nB_in"]),
                       "l2_policy": f"inputs larger than L2 ({alg_bytes/1e6:.0f} MB of localisations per GPU vs 126 MB L2)",
                       "sum_logp": total, "generator_seconds": round(gen_s, 1),
                       "collective": ("none (one GPU)" if world == 1 else
                                      "one 8-byte NCCL all-reduce of the partial sums per step on the evaluation's stream")},
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                    "what": "xt_sum_logp_host per step: pinned host buffers -> device + repack, overlapped per length "
                            "bucket with the plan / replay kernels, result read back",
                    "parity_rel_diff_vs_resident": abs(e2e_val - total) / abs(total), "pinned_host_numa": numa},
            "gpu_launches": int(launches),
            "plan": {"steps_verified": served["verified"], "steps_planned_from_scratch": served["planned_from_scratch"],
                     "chunks_planned_again": served["chunks_planned_again"],
                     "what": "every timed step evaluates other parameters than the step before (one parameter moved by 1.5e-8 relative, "
                             "the finite-difference pattern of BFGS).  `verified`: the evaluation ran along the resident plan while the "
                             "plan kernel re-evaluated every floating-point decision behind it (k1_plan<VERIFY>, concurrent with the "
                             "replay); a chunk with a changed decision is planned and replayed again inside the step.  "
                             "kernel_ms / roofline are the construction-mode kernels (one plan launch, one replay launch)"},
            "seq_updates_per_s": float(stats["seq_updates"]) * world * args.steps / (ms * 1e-3),  # SURVEY 8(d): sum of nT * nB_in per step

            "kernel_ms": {"plan": ms_plan, "replay_and_reduce": replay_ms,
                          "what": "two-phase mode (one plan launch, one replay launch), measured after the timed region"},
            "roofline": {"bound": "fp64", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": traffic, "kernel": "k2_replay_fused",
                         "peak_source": "FP64 FMA microbenchmark measured live on this GPU (xt_fp64_peak_tflops); MEASURED_PEAKS.json has no FP64 figure",
                         "algorithmic_flops_per_launch": flops,
                         "hbm": {"algorithmic_bytes": alg_bytes, "achieved_gbs": alg_bytes / (replay_ms * 1e-3) / 1e9,
                                 "peak_gbs": peaks.get("hbm_gbs")}},
            "fp32_path": {"value": stats["track_steps"] / (f32_ms * 1e-3), "unit": UNIT, "ms_per_step": f32_ms,
                          "replay_and_reduce_ms": f32_replay, "kernel_used": bool(f32_used),
                          "rel_diff_vs_fp64": abs(step32 - total_local) / abs(total_local), "stated_tolerance": 1e-4,
                          "what": "same evaluation on this rank with xt_set_option('fp32_replay', 1): FP64 plan kernel, FP32 replay "
                                  "kernel k2_replay_f32 (not the headline: `value`, `e2e` and `roofline` are FP64)"},
            "cpu_baseline": cpu,
            "parity_rel_err_vs_oracle_on_cpu_sample": parity,
            "strong": strong,
            "api": api,
            "secondary": secondary,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
    ts.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
