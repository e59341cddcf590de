"""Throughput of a group of stations advanced together (rfinv_pt_group_run) against the same stations run one after another.

Stations: the sample configuration (sample_syn/params.in: 20 ranks x 5 chains, 2 traces x 101 samples, bookkeeping on), each
with its own I_SEED and its own noise on the observed traces; N_BURN = 0 so that the timed iterations record the bookkeeping
every N_CORR-th iteration as a run after its burn-in does.  P = 1, 2, 4, ..., 64, and one mixed group: one station of the
bench's target shape with 1024 chains (64 ranks x 16, nfft 1024, k_max 30, 3 traces x 512 samples) beside 15 sample stations.

Per P, after a warm-up (which captures every graph), alternately: every station runs `--iters` iterations alone, back to back
(rfinv_pt_run, synchronous), then the group runs the same number (rfinv_pt_group_run, synchronous).  Host wall clock around the
calls, median of `--reps`.  Reported: station-iterations/s of both and the speedup of the group.

The whole measurement runs twice: with the process's defaults and in a child process with CUDA_DEVICE_MAX_CONNECTIONS=32 (the
number of hardware queues graph branches are spread over; 8 by default).  A torch.profiler trace of group iterations at
P = 16 gives the GPU's busy time and how many kernels overlap on average.

    python tools/group_time.py [--out FILE] [--trace-dir DIR]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
from rf_inv_b200 import workloads
from rf_inv_b200.pt import ParallelTempering, PtGroup

PS = [1, 2, 4, 8, 16, 32, 64]


def attach_obs(cfg, seed):
    """bench.py's observations (oracle forward of the data-generating model + noise, float32) with noise seed `seed`."""
    import oracle_c
    tm = workloads.true_model(cfg)
    cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp))
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    _, rft, _ = oracle_c.eval_batch(cfg, tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"])
    noise = np.random.default_rng(seed).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))
    cfg.obs = (rft[0, :, :cfg.nsmp] + noise).astype(np.float32).astype(np.float64)
    return cfg


def station(i, shape="sample"):
    """(cfg, nproc) of station i."""
    cfg = workloads.make_config(shape)
    cfg.nburn, cfg.niter, cfg.ncorr = 0, 8000, 10
    cfg.iseed = 12345678 + 1000 * i
    if shape == "sample":
        return attach_obs(cfg, 100 + i), 20
    return attach_obs(cfg, 100 + i), 1024 // cfg.nchains


def measure(stations, iters, reps, warm=100):
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in stations]
    try:
        with PtGroup(pts) as g:
            for pt in pts:
                pt.run(warm)
            g.run(warm)
            solo, group = [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                for pt in pts:
                    pt.run(iters)
                solo.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                g.run(iters)
                group.append(time.perf_counter() - t0)
    finally:
        for pt in pts:
            pt.close()
    p = len(stations)
    ts, tg = float(np.median(solo)), float(np.median(group))
    return dict(stations=p, chains=int(sum(c.nchains * n for c, n in stations)), iterations=iters,
                solo_ms_per_iteration=round(ts * 1e3 / iters, 4), group_ms_per_iteration=round(tg * 1e3 / iters, 4),
                solo_station_iters_per_s=round(p * iters / ts, 1), group_station_iters_per_s=round(p * iters / tg, 1),
                speedup=round(ts / tg, 3), solo_s=[round(x, 4) for x in solo], group_s=[round(x, 4) for x in group])


def profile_group(stations, trace_dir, iters=20):
    """Kernel activity of `iters` group iterations from torch.profiler: wall time, GPU busy time (union of the kernels'
    intervals), summed kernel time (their average overlap is sum / busy) and the longest kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in stations]
    try:
        with PtGroup(pts) as g:
            g.run(50)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                t0 = time.perf_counter()
                g.run(iters)
                wall = time.perf_counter() - t0
    finally:
        for pt in pts:
            pt.close()
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    iv = sorted((e.time_range.start, e.time_range.end) for e in kern)
    busy, cur_s, cur_e = 0.0, None, None
    for s, e in iv:
        if cur_e is None or s > cur_e:
            if cur_e is not None:
                busy += cur_e - cur_s
            cur_s, cur_e = s, e
        else:
            cur_e = max(cur_e, e)
    if cur_e is not None:
        busy += cur_e - cur_s
    total = sum(e - s for s, e in iv)
    span = (iv[-1][1] - iv[0][0]) if iv else 0.0
    by_name = {}
    for e in kern:
        n = re.sub(r"^void\s+", "", e.name).replace("(anonymous namespace)::", "")
        n = re.split(r"[<(]", n, 1)[0] or n
        d = by_name.setdefault(n, [0, 0.0])
        d[0] += 1
        d[1] += e.time_range.end - e.time_range.start
    if trace_dir:
        os.makedirs(trace_dir, exist_ok=True)
        prof.export_chrome_trace(os.path.join(trace_dir, f"group_p{len(stations)}.pt.trace.json"))
    return dict(stations=len(stations), iterations=iters, wall_ms_per_iteration=round(wall * 1e3 / iters, 4),
                kernel_span_ms_per_iteration=round(span / 1e3 / iters, 4),
                gpu_busy_ms_per_iteration=round(busy / 1e3 / iters, 4),
                kernel_ms_per_iteration=round(total / 1e3 / iters, 4),
                mean_kernels_in_flight=round(total / busy, 3) if busy else 0.0,
                kernels_per_iteration=round(len(kern) / iters, 1),
                kernels={n: dict(count_per_iteration=round(c / iters, 1), us_per_launch=round(t / c, 2))
                         for n, (c, t) in sorted(by_name.items(), key=lambda kv: -kv[1][1])})


def run_all(iters, reps, trace_dir):
    all_st = [station(i) for i in range(max(PS))]
    rows = [measure(all_st[:p], iters, reps) for p in PS]
    mixed = measure([station(999, "target")] + all_st[:15], iters, reps)
    prof = profile_group(all_st[:16], trace_dir)
    return dict(rows=rows, mixed_target_1024_plus_15_sample=mixed, profile_p16=prof)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--trace-dir", default=None, help="write the torch.profiler traces here")
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:                                           # one setting, in this process's environment
        print(json.dumps(run_all(a.iters, a.reps, a.trace_dir)), flush=True)
        return
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(gpu=gpu[0] if gpu else "unknown",
               timing=f"host wall clock around synchronous calls, median of {a.reps}; {a.iters} iterations per station "
                      "and repetition")
    for name, extra in (("default", {}), ("cuda_device_max_connections_32", {"CUDA_DEVICE_MAX_CONNECTIONS": "32"})):
        env = {k: v for k, v in os.environ.items() if k != "CUDA_DEVICE_MAX_CONNECTIONS"}
        env.update(extra)
        td = os.path.join(a.trace_dir, name) if a.trace_dir else None
        cmd = [sys.executable, os.path.abspath(__file__), "--child", "--iters", str(a.iters), "--reps", str(a.reps)]
        if td:
            cmd += ["--trace-dir", td]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stderr)
            raise SystemExit(f"{name}: exit code {r.returncode}")
        res[name] = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
