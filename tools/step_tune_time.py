"""Cost and effect of the random-walk width tuning during the burn-in (rfinv_pt_set_step_tuning, DESIGN.md 7e), against the
rank sweep alone (mode 1).

Shapes, as in tools/ladder_tune_time.py: the sample configuration (20 ranks x 5 chains, ncool 1; its N_BURN 3000 passes the
tuning points 64 .. 2048) and the bench's PT shape (1024 ranks x 16 chains, here with N_BURN 1024: tuning points 64 .. 1024),
both with bench.py's observations.

Cost: one handle per setting, both warmed up; then mode 1 and mode 1 + width tuning alternately run `--iters` iterations
(rfinv_pt_run, synchronous), once from iteration 100 on (the tuning points of that window included) and once after the burn-in.
Host wall clock around the calls, median of `--reps`: milliseconds per iteration.

Mixing, three settings -- mode 1, the width tuning alone, the width and the ladder tuning: the burn-in, then `--sample-iters`
sampling iterations, one iteration per call so that the temperatures can be read after each.  Over the sampling phase only:
  * the acceptance of every (level, move type) -- z, dVs, dVp, sigma -- over all ranks, a proposal counted at the level its
    chain held at the end of the iteration before (logs of flags and types);
  * swaps into the cold level per rank per 1000 iterations (the chain at level 0 of a rank changes);
  * the integrated autocorrelation time of k and logL at the cold level (Sokal's window, c = 5), sampled every N_CORR
    iterations, median and mean over the ranks, in samples;
  * with the width tuning, the final widths' mean over the ranks per level and type, relative to params.in.

    python tools/step_tune_time.py [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
from ladder_tune_time import shape
from rank_swap_time import gpu_name, iat
from rf_inv_b200 import capi
from rf_inv_b200.pt import ParallelTempering

TYPES = ("z", "dvs", "dvp", "sig")


def make(cfg, nproc, steps, ladder=0):
    pt = ParallelTempering(cfg, nproc)
    pt.set_rank_swaps(1)
    pt.set_ladder_tuning(ladder)
    pt.set_step_tuning(steps)
    return pt


def cost(name, iters, reps, warm=100):
    cfg, nproc = shape(name, 0)
    pts = {t: make(cfg, nproc, t) for t in (0, 1)}
    out = dict(chains=nproc * cfg.nchains, iterations=iters, nburn=cfg.nburn)
    try:
        for pt in pts.values():
            pt.run(warm)
        for phase in ("from_iteration_100", "after_burn_in"):
            if phase == "after_burn_in":
                for pt in pts.values():
                    pt.run(max(cfg.nburn - pt.iterations_done, 0))
            start = pts[0].iterations_done
            t = {0: [], 1: []}
            for _ in range(reps):
                for m in (0, 1):
                    t0 = time.perf_counter()
                    pts[m].run(iters)
                    t[m].append(time.perf_counter() - t0)
            ms = {m: 1e3 * float(np.median(t[m])) / iters for m in (0, 1)}
            points = [e for e in (64 * 2 ** j for j in range(20)) if start < e <= min(start + reps * iters, cfg.nburn)]
            out[phase] = dict(first_iteration=start, tuning_points_inside=points, mode1_ms_per_iteration=round(ms[0], 4),
                              tuned_ms_per_iteration=round(ms[1], 4), overhead_percent=round(100.0 * (ms[1] / ms[0] - 1.0), 2),
                              mode1_s=[round(x, 4) for x in t[0]], tuned_s=[round(x, 4) for x in t[1]])
        return out
    finally:
        for pt in pts.values():
            pt.close()


def mixing(name, steps, ladder, sample_iters):
    cfg, nproc = shape(name, sample_iters)
    nch, Cl = cfg.nchains, nproc * cfg.nchains
    pt = make(cfg, nproc, steps, ladder)
    lib, h = pt._lib, pt.ev.handle
    temps, logl, k = np.empty(Cl), np.empty(Cl), np.empty(Cl, dtype=np.int32)
    nul = C.cast(None, capi.dp)
    idx = np.arange(nch)
    it_z, it_dvs = 3, 4
    it_dvp = 5 if cfg.vp_mode == 1 else -1
    it_sig = pt.ntype if any(cfg.sig_max[t] - cfg.sig_min[t] > float(np.float32(1.0e-5)) for t in range(cfg.ntrc)) else -1
    n_prop, n_acc = np.zeros((nch, 4), np.int64), np.zeros((nch, 4), np.int64)
    try:
        pt.run(cfg.nburn)
        pt.set_logging(sample_iters)

        def levels():   # [nproc][nch]: chain of each level
            t = temps.reshape(nproc, nch)
            return np.lexsort((np.broadcast_to(idx, t.shape), t), axis=1)

        def level_of(at):
            lvl = np.empty((nproc, nch), np.int64)
            np.put_along_axis(lvl, at, np.broadcast_to(idx, at.shape), axis=1)
            return lvl.reshape(Cl)

        capi.check(lib.rfinv_pt_get_state(h, C.cast(None, capi.i32p), nul, nul, nul, nul, nul, temps.ctypes.data_as(capi.dp)))
        at = levels()
        lvl = level_of(at)
        cur = at[:, 0].copy()
        moves = 0
        ks, lls = [], []
        lvl_hist = np.empty((sample_iters, Cl), np.int16)   # each chain's level before iteration i
        for i in range(1, sample_iters + 1):
            lvl_hist[i - 1] = lvl
            pt.run(1)
            if i % cfg.ncorr == 0:
                capi.check(lib.rfinv_pt_get_state(h, k.ctypes.data_as(capi.i32p), nul, nul, nul, nul,
                                                  logl.ctypes.data_as(capi.dp), temps.ctypes.data_as(capi.dp)))
            else:
                capi.check(lib.rfinv_pt_get_state(h, C.cast(None, capi.i32p), nul, nul, nul, nul, nul, temps.ctypes.data_as(capi.dp)))
            at = levels()
            lvl = level_of(at)
            nxt = at[:, 0]
            moves += int(np.sum(nxt != cur))
            cur = nxt.copy()
            if i % cfg.ncorr == 0:
                sel = np.arange(nproc) * nch + cur
                ks.append(k[sel].copy()); lls.append(logl[sel].copy())
        st = pt.step_tuning()
        flags, itypes, _ = pt.log(sample_iters)
        for tau, it in enumerate((it_z, it_dvs, it_dvp, it_sig)):
            sel = itypes == it
            n_prop[:, tau] = np.bincount(lvl_hist[sel], minlength=nch)
            n_acc[:, tau] = np.bincount(lvl_hist[sel & (flags == 1)], minlength=nch)
    finally:
        pt.close()
    ks, lls = np.array(ks), np.array(lls)
    tk = np.array([iat(ks[:, r]) for r in range(nproc)])
    tl = np.array([iat(lls[:, r]) for r in range(nproc)])
    acc = np.where(n_prop > 0, n_acc / np.maximum(n_prop, 1), np.nan)
    dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])
    out = dict(step_tuning=bool(steps), ladder_tuning=bool(ladder), tuning_points=st["n_points"], chains=Cl, nburn=cfg.nburn,
               sampling_iterations=sample_iters, samples_per_rank=len(ks),
               acceptance_by_level={TYPES[t]: [None if np.isnan(a) else round(float(a), 4) for a in acc[:, t]] for t in range(4)},
               cold_level_swaps_per_rank_per_1000_iterations=round(1000.0 * moves / nproc / sample_iters, 3),
               iat_k_median=round(float(np.nanmedian(tk)), 2), iat_k_mean=round(float(np.nanmean(tk)), 2),
               iat_logl_median=round(float(np.nanmedian(tl)), 2), iat_logl_mean=round(float(np.nanmean(tl)), 2))
    if steps:
        rel = st["widths"].mean(axis=0) / dev
        out["mean_width_over_params_in"] = {TYPES[t]: [round(float(x), 4) for x in rel[:, t]] for t in range(4)}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "step_tune.json"))
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample-iters", type=int, default=8000, help="sampling iterations of the sample shape (its N_ITER)")
    ap.add_argument("--bench-sample-iters", type=int, default=2000)
    a = ap.parse_args()
    res = dict(gpu=gpu_name(), timing="host wall clock around synchronous rfinv_pt_run calls, median of the repetitions; "
                                      "mode 1 and mode 1 + width tuning alternate")
    res["cost"] = {n: cost(n, a.iters, a.reps) for n in ("sample", "bench")}
    print(json.dumps(res["cost"]), flush=True)
    settings = ((0, 0), (1, 0), (1, 1))   # (width tuning, ladder tuning)
    res["mixing"] = {"sample": [mixing("sample", s, l, a.sample_iters) for s, l in settings],
                     "bench": [mixing("bench", s, l, a.bench_sample_iters) for s, l in settings]}
    res["gpu_after"] = gpu_name()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
