"""Cost and effect of the even/odd swaps inside every virtual rank (rfinv_pt_set_rank_swaps, DESIGN.md 7c).

Shapes: the sample configuration (sample_syn/params.in: 20 ranks x 5 chains, ncool 1) and the bench's PT shape (target
configuration, 1024 ranks x 16 chains = 16 384 chains, ncool 1), both with bench.py's observations.

Cost: one handle per mode, both warmed up (every graph captured); then mode 0 and mode 1 alternately run `--iters`
iterations (rfinv_pt_run, synchronous).  Host wall clock around the calls, median of `--reps`: milliseconds per iteration.

Mixing, both modes: the sample configuration over its full N_BURN + N_ITER (3000 + 8000) and the bench shape over 2000
iterations, one iteration per call so that the temperatures can be read after each.  Reported:
  * per-level acceptance of the rank sweep (mode 1) and the acceptance of the global swap (both modes, from its log);
  * swaps into the cold level per rank per 1000 iterations: how often the chain at level 0 of a rank -- its chain of lowest
    (temperature, chain index) -- changes from one iteration to the next.  In mode 0 only the global swap can do that;
  * the integrated autocorrelation time (Sokal's window, c = 5) of k and logL at the cold level of each rank, sampled every
    N_CORR iterations, following the level and not a chain index; median and mean over the ranks, in samples.

    python tools/rank_swap_time.py [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np
from group_time import attach_obs
from rf_inv_b200 import capi, workloads
from rf_inv_b200.pt import ParallelTempering


def shape(name):
    """(cfg, nproc) of a shape."""
    cfg = workloads.make_config("sample" if name == "sample" else "target")
    if name == "sample":
        return attach_obs(cfg, 100), 20
    cfg.nburn, cfg.niter, cfg.ncorr = 0, 2000, 10
    return attach_obs(cfg, 100), 16384 // cfg.nchains


def cost(name, iters, reps, warm=100):
    cfg, nproc = shape(name)
    pts = {m: ParallelTempering(cfg, nproc) for m in (0, 1)}
    try:
        pts[1].set_rank_swaps(1)
        for pt in pts.values():
            pt.run(warm)
        t = {0: [], 1: []}
        for _ in range(reps):
            for m in (0, 1):
                t0 = time.perf_counter()
                pts[m].run(iters)
                t[m].append(time.perf_counter() - t0)
        ms = {m: 1e3 * float(np.median(t[m])) / iters for m in (0, 1)}
        return dict(chains=nproc * cfg.nchains, iterations=iters, mode0_ms_per_iteration=round(ms[0], 4),
                    mode1_ms_per_iteration=round(ms[1], 4), overhead_percent=round(100.0 * (ms[1] / ms[0] - 1.0), 2),
                    mode0_s=[round(x, 4) for x in t[0]], mode1_s=[round(x, 4) for x in t[1]])
    finally:
        for pt in pts.values():
            pt.close()


def iat(x, c=5.0):
    """Integrated autocorrelation time of a series (Sokal's automatic window): 1 + 2 sum rho(t) up to the first M >= c tau."""
    x = np.asarray(x, dtype=np.float64) - np.mean(x)
    n = len(x)
    if n < 4 or not np.any(x):
        return float("nan")
    f = np.fft.rfft(x, 2 * n)
    acf = np.fft.irfft(f * np.conj(f))[:n]
    acf /= acf[0]
    tau = 1.0
    for m in range(1, n):
        tau += 2.0 * acf[m]
        if m >= c * tau:
            break
    return float(tau)


def mixing(name, mode, n_iter):
    cfg, nproc = shape(name)
    nch, Cl = cfg.nchains, nproc * cfg.nchains
    pt = ParallelTempering(cfg, nproc)
    lib, h = pt._lib, pt.ev.handle
    temps, logl, k = np.empty(Cl), np.empty(Cl), np.empty(Cl, dtype=np.int32)
    nul = C.cast(None, capi.dp)
    try:
        pt.set_rank_swaps(mode)
        pt.set_logging(n_iter)
        idx = np.arange(nch)

        def cold_chain():   # per rank: the chain of lowest (temperature, chain index)
            t = temps.reshape(nproc, nch)
            return np.lexsort((np.broadcast_to(idx, t.shape), t), axis=1)[:, 0]

        capi.check(lib.rfinv_pt_get_state(h, C.cast(None, capi.i32p), nul, nul, nul, nul, nul, temps.ctypes.data_as(capi.dp)))
        cur = cold_chain()
        moves = 0
        ks, lls = [], []
        for i in range(1, n_iter + 1):
            pt.run(1)
            if i % cfg.ncorr == 0:
                capi.check(lib.rfinv_pt_get_state(h, k.ctypes.data_as(capi.i32p), nul, nul, nul, nul,
                                                  logl.ctypes.data_as(capi.dp), temps.ctypes.data_as(capi.dp)))
            else:
                capi.check(lib.rfinv_pt_get_state(h, C.cast(None, capi.i32p), nul, nul, nul, nul, nul, temps.ctypes.data_as(capi.dp)))
            nxt = cold_chain()
            moves += int(np.sum(nxt != cur))
            cur = nxt
            if i % cfg.ncorr == 0:
                sel = np.arange(nproc) * nch + cur
                ks.append(k[sel].copy()); lls.append(logl[sel].copy())
        _, _, swaps = pt.log(n_iter)
        rs = pt.rank_swaps()
    finally:
        pt.close()
    ks, lls = np.array(ks), np.array(lls)
    tk = np.array([iat(ks[:, r]) for r in range(nproc)])
    tl = np.array([iat(lls[:, r]) for r in range(nproc)])
    out = dict(mode=mode, chains=Cl, iterations=n_iter, samples_per_rank=len(ks),
               global_swap_acceptance=round(float(swaps[:, 2].mean()), 4),
               cold_level_swaps_per_rank_per_1000_iterations=round(1000.0 * moves / nproc / n_iter, 3),
               iat_k_median=round(float(np.nanmedian(tk)), 2), iat_k_mean=round(float(np.nanmean(tk)), 2),
               iat_logl_median=round(float(np.nanmedian(tl)), 2), iat_logl_mean=round(float(np.nanmean(tl)), 2))
    if mode == 1:
        out["level_acceptance"] = [round(float(a) / float(p), 4) if p else None for a, p in zip(rs["n_acc"], rs["n_prop"])]
    return out


def gpu_name():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        return q
    except Exception as e:   # the figure is still worth keeping; say that the card was not read
        return f"not read ({e})"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rank_swap_time.json"))
    ap.add_argument("--iters", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--mixing-bench-iters", type=int, default=2000)
    a = ap.parse_args()
    res = dict(gpu=gpu_name(), timing="host wall clock around synchronous rfinv_pt_run calls, median of the repetitions; "
                                      "mode 0 and mode 1 alternate")
    res["cost"] = {n: cost(n, a.iters, a.reps) for n in ("sample", "bench")}
    print(json.dumps(res["cost"]), flush=True)
    cfg, _ = shape("sample")
    res["mixing"] = {"sample": [mixing("sample", m, cfg.nburn + cfg.niter) for m in (0, 1)],
                     "bench": [mixing("bench", m, a.mixing_bench_iters) for m in (0, 1)]}
    res["gpu_after"] = gpu_name()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f)
        f.write("\n")
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
