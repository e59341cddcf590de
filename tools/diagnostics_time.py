"""Cost and findings of the convergence diagnostics (rfinv_pt_set_diagnostics, DESIGN.md 7f).

Shapes, as in tools/rank_swap_time.py: the sample configuration (20 ranks x 5 chains, ncool 1, N_BURN 3000, N_ITER 8000,
N_CORR 10) and the bench's PT shape (1024 ranks x 16 chains = 16 384 chains, ncool 1, N_CORR 10), both with bench.py's
observations.

Cost: for modes 0 and 1, one handle with the diagnostics off and one with them on (four depth bins), both warmed up, with
N_BURN 0 so that every N_CORR-th iteration records; then off and on alternately run `--iters` iterations (rfinv_pt_run,
synchronous).  Host wall clock around the calls, median of `--reps`: milliseconds per iteration.  Then the time of one
rfinv_pt_get_diagnostics call (statistics kernels, rows, summary and trips to preallocated host arrays) at 1024 ranks x 800
samples, median of `--reps` calls after one untimed call; and of ParallelTempering.diagnostics() (the same plus the Python
arrays).

Findings, mode 0 / mode 1 / mode 1 with the ladder and the width tuning: the sample configuration over N_BURN + N_ITER and
the bench shape over N_BURN 1024 + N_ITER 2000, in one rfinv_pt_run each.  Reported: the tempered share, round trips per rank
per 1000 iterations during and after the burn-in, and R-hat, ESS and median IAT of k and logL.

    python tools/diagnostics_time.py [--out FILE]
"""
import argparse
import ctypes as C
import copy
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
from rank_swap_time import gpu_name, shape
from rf_inv_b200 import capi
from rf_inv_b200.pt import ParallelTempering


def make(cfg, nproc, mode, diag, tune=False):
    pt = ParallelTempering(cfg, nproc)
    pt.set_rank_swaps(mode)
    if tune:
        pt.set_ladder_tuning(1)
        pt.set_step_tuning(1)
    if diag:
        pt.set_diagnostics(1, [15, 25, 50, 75])
    return pt


def cost(name, iters, reps, warm=100):
    cfg, nproc = shape(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter = 0, warm + iters * reps * 2 + 10
    out = dict(chains=nproc * cfg.nchains, iterations=iters, ncorr=cfg.ncorr)
    for mode in (0, 1):
        pts = {d: make(cfg, nproc, mode, d) for d in (0, 1)}
        t = {0: [], 1: []}
        try:
            for pt in pts.values():
                pt.run(warm)
            for _ in range(reps):
                for d in (0, 1):
                    t0 = time.perf_counter()
                    pts[d].run(iters)
                    t[d].append(time.perf_counter() - t0)
        finally:
            for pt in pts.values():
                pt.close()
        ms = {d: 1e3 * float(np.median(t[d])) / iters for d in (0, 1)}
        out[f"mode{mode}"] = dict(off_ms_per_iteration=round(ms[0], 4), on_ms_per_iteration=round(ms[1], 4),
                                  overhead_percent=round(100.0 * (ms[1] / ms[0] - 1.0), 2),
                                  off_s=[round(x, 4) for x in t[0]], on_s=[round(x, 4) for x in t[1]])
    return out


def getter_time(reps):
    cfg, nproc = shape("bench")
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter = 0, 800 * cfg.ncorr
    pt = make(cfg, nproc, 1, 1)
    try:
        pt.run(cfg.niter)
        dg = pt.diagnostics()   # (untimed: the first call raises the kernel's shared-memory limit)
        G, nq = dg["n_ranks"], len(dg["names"])
        rows, summary, trips = np.zeros((G, nq, 9)), np.zeros((nq, 4)), np.zeros((G, 2), np.int64)
        ns, nr, nqq = C.c_int64(0), C.c_int32(0), C.c_int32(0)
        tc, tp = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            capi.check(pt._lib.rfinv_pt_get_diagnostics(pt.ev.handle, C.byref(ns), C.byref(nr), C.byref(nqq),
                                                        rows.ctypes.data_as(capi.dp), summary.ctypes.data_as(capi.dp),
                                                        trips.ctypes.data_as(capi.i64p)))
            tc.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            pt.diagnostics()
            tp.append(time.perf_counter() - t0)
        return dict(ranks=G, samples=dg["n_samples"], quantities=nq, c_getter_ms=round(1e3 * float(np.median(tc)), 3),
                    c_getter_ms_all=[round(1e3 * x, 3) for x in tc], python_ms=round(1e3 * float(np.median(tp)), 3),
                    python_ms_all=[round(1e3 * x, 3) for x in tp])
    finally:
        pt.close()


def findings(name, setting):
    cfg, nproc = shape(name)
    cfg = copy.deepcopy(cfg)
    if name == "bench":
        cfg.nburn, cfg.niter = 1024, 2000
    mode, tune = {"mode0": (0, False), "mode1": (1, False), "mode1_tuned": (1, True)}[setting]
    pt = make(cfg, nproc, mode, 1, tune)
    try:
        pt.run(cfg.nburn + cfg.niter)
        dg = pt.diagnostics()
    finally:
        pt.close()
    trips = dg["trips"].sum(axis=0)
    q = {n: i for i, n in enumerate(dg["names"])}
    per = lambda x, n: round(1000.0 * float(x) / nproc / n, 4) if n else None
    return dict(setting=setting, ranks=dg["n_ranks"], samples_per_rank=dg["n_samples"], nburn=cfg.nburn, niter=cfg.niter,
                tempered_share=round(float(dg["tempered_share"][0]), 5),
                trips_per_rank_per_1000_burn_in=per(trips[0], cfg.nburn), trips_per_rank_per_1000_after=per(trips[1], cfg.niter),
                **{f"{n}_{k}": round(float(dg[key][q[n]]), 4) for n in ("k", "logL")
                   for k, key in (("rhat", "rhat"), ("ess", "ess_total"), ("tau_median", "tau_median"))})


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "diagnostics_time.json"))
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    res = dict(gpu=gpu_name(), timing="host wall clock around synchronous rfinv_pt_run calls, median of the repetitions; "
                                      "diagnostics off and on alternate")
    res["cost"] = {n: cost(n, a.iters, a.reps) for n in ("sample", "bench")}
    print(json.dumps(res["cost"]), flush=True)
    res["get_diagnostics"] = getter_time(a.reps)
    print(json.dumps(res["get_diagnostics"]), flush=True)
    res["findings"] = {n: [findings(n, s) for s in ("mode0", "mode1", "mode1_tuned")] for n in ("sample", "bench")}
    res["gpu_after"] = gpu_name()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
