"""Save time, restore time and file size of a parallel-tempering checkpoint (rfinv_pt_save / rfinv_pt_restore), against the
time of one iteration, at two shapes:

  sample  sample_syn/params.in: 20 ranks x 5 chains, 2 traces x 101 samples, bookkeeping on, saved after the full
          N_BURN + N_ITER = 11 000 iterations (all_models holds every recorded model)
  pt      the PT shape of bench.py: 16 384 chains (1 024 ranks x 16), nfft 1024, k_max 30, 3 traces x 512 samples

Times are host wall clock around the call, which synchronises the device before it returns; the file goes to a temporary
directory (local disk of the machine).  Each is the median of a few repetitions.  Prints one JSON line; --out FILE also
writes it there.

    python tools/checkpoint_time.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np
from rf_inv_b200 import workloads
from rf_inv_b200.pt import ParallelTempering


def attach_obs(cfg):
    """bench.py's observations: oracle forward of the data-generating model + noise, rounded to float32."""
    import oracle_c
    tm = workloads.true_model(cfg)
    cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp))
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    _, rft, _ = oracle_c.eval_batch(cfg, tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"])
    cfg.obs = (rft[0, :, :cfg.nsmp] + np.random.default_rng(7).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))).astype(np.float32).astype(np.float64)
    return cfg


def measure(cfg, nproc, n_run, n_timed, tmp, reps=3):
    pt = ParallelTempering(cfg, nproc)
    pt.run(n_run - n_timed)
    t0 = time.perf_counter()
    pt.run(n_timed)                                  # (rfinv_pt_run synchronises before it returns)
    iter_ms = (time.perf_counter() - t0) * 1e3 / n_timed
    path = os.path.join(tmp, "ck")
    save = []
    for _ in range(reps):
        t0 = time.perf_counter()
        pt.save(path)
        save.append(time.perf_counter() - t0)
    pt.close()
    restore = []
    for _ in range(reps):
        q = ParallelTempering(cfg, nproc)
        t0 = time.perf_counter()
        q.restore(path)
        q.ev.synchronize()
        restore.append(time.perf_counter() - t0)
        q.close()
    size = os.path.getsize(path)
    os.remove(path)
    every = max(cfg.ncorr, 1) * 100                  # run.py's default --checkpoint-every: one progress step
    save_ms = float(np.median(save)) * 1e3
    return dict(chains=nproc * cfg.nchains, virtual_ranks=nproc, ntrc=cfg.ntrc, nsmp=cfg.nsmp, nfft=cfg.nfft, k_max=cfg.k_max,
                bookkeeping=cfg.niter > 0, iterations_before_save=n_run, file_bytes=size, file_mb=round(size / 1e6, 2),
                save_ms=round(save_ms, 2), restore_ms=round(float(np.median(restore)) * 1e3, 2),
                save_gb_per_s=round(size / (save_ms * 1e-3) / 1e9, 2), iteration_ms=round(iter_ms, 4),
                default_checkpoint_every=every,
                save_cost_vs_iterations_between_saves=round(save_ms / (iter_ms * every), 5))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(gpu=gpu[0] if gpu else "unknown", timing="host wall clock around the call (synchronised), median of 3")
    with tempfile.TemporaryDirectory() as tmp:
        cfg = attach_obs(workloads.make_config("sample"))
        res["sample"] = measure(cfg, 20, cfg.nburn + cfg.niter, 1000, tmp)
        cfg = attach_obs(workloads.make_config("target"))
        res["pt"] = measure(cfg, 16384 // cfg.nchains, 220, 200, tmp)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
