"""Checkpoint / resume of the distributed parallel-tempering run (launch under torchrun, one process per GPU): every process
runs N1 iterations of rfinv_pt_run_distributed, saves its own virtual ranks and closes; new handles join a new communicator,
restore and run N2 more.  The result must equal an uninterrupted distributed run of N1 + N2 in the same job: each process's
logs, state, counters, likelihood history, histograms and recorded models before rfinv_pt_reduce_outputs, and the job-wide
outputs on process 0 after it.  A file of process 0 restored into a handle that owns process 1's ranks must be refused.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \\
        tools/checkpoint_check.py DIR

DIR receives the checkpoint files (one per process).  Prints one JSON line on process 0; exit code 0 when identical.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist
from rf_inv_b200 import capi, workloads
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering

N1, N2 = 130, 170


def config(world, local_rank):
    cfg = workloads.make_config("sample")
    cfg.nburn, cfg.niter = 100, 200                  # ncorr 10: the split falls inside recording, off an ncorr multiple
    cfg.nbin_z, cfg.nbin_vs, cfg.nbin_vp, cfg.nbin_vpvs, cfg.nbin_sig, cfg.nbin_amp = 50, 25, 25, 20, 10, 40
    cfg.amp_min, cfg.amp_max = -0.6, 0.6
    cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp)); cfg.r_inv = workloads.lapack_r_inv(cfg)
    tm = workloads.true_model(cfg)
    with Evaluator(cfg, device=local_rank) as ev:
        _, rft, _ = ev.calc_likelihood(tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"], want_rft=True)
    cfg.obs = (rft[0, :, :cfg.nsmp] + np.random.default_rng(7).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))).astype(np.float32).astype(np.float64)
    return cfg, 4 * world


def outputs(pt, n_log, rank):
    """Local results before reduce_outputs, then (process 0) the job-wide ones after it."""
    flags, itypes, swaps = pt.log(n_log)
    cnt = pt.counters()
    local = dict(flags=flags, itypes=itypes, swaps=swaps, nprop=cnt["nprop"], naccept=cnt["naccept"],
                 lhist=cnt["likelihood_hist"], n_eval=np.int64(cnt["n_eval"]), it=np.int64(pt.iterations_done), **pt.state())
    local.update({"hist_" + k: np.asarray(v) for k, v in pt.hist().items()})
    local["vp_model"], local["vs_model"] = pt.models()
    pt.reduce_outputs()
    job = {}
    if rank == 0:
        cnt = pt.counters()
        job = dict(nprop=cnt["nprop"], naccept=cnt["naccept"], lhist=cnt["likelihood_hist"])
        job.update({"hist_" + k: np.asarray(v) for k, v in pt.hist().items()})
        job["vp_model"], job["vs_model"] = pt.models()
    return local, job


def main():
    out_dir = sys.argv[1]
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("gloo")                  # carries the library's communicator ids only
    cfg, nproc = config(world, local_rank)
    path = os.path.join(out_dir, f"ck.{rank}-of-{world}")
    say = lambda m: print(f"[rank {rank}] {m}", file=sys.stderr, flush=True)

    ref = ParallelTempering(cfg, nproc, device=local_rank, world=world, rank=rank)
    ref.set_logging(N1 + N2)
    ref.run_distributed(N1 + N2, dist, torch)
    exchange = ref.exchange_mode
    ref_local, ref_job = outputs(ref, N1 + N2, rank)
    ref.close()
    say(f"uninterrupted run done ({exchange})")

    a = ParallelTempering(cfg, nproc, device=local_rank, world=world, rank=rank)
    a.run_distributed(N1, dist, torch)
    a.save(path)
    a.close()
    b = ParallelTempering(cfg, nproc, device=local_rank, world=world, rank=rank)
    b.init_comm(dist, torch)
    b.restore(path)
    b.set_logging(N2)
    b.run_distributed(N2, dist, torch)
    got_local, got_job = outputs(b, N2, rank)
    b.close()
    say("resumed run done")

    # the profile means are added with double-precision atomics (their last bits follow the arrival order of the CTAs, also
    # between two uninterrupted runs): 1e-12 like tools/dist_check.py; everything else bit for bit
    same = lambda k, a, b: np.allclose(a, b, rtol=1e-12, atol=0) if k.endswith("_mean") else np.array_equal(a, b)
    failed = []
    for k, v in ref_local.items():
        want = v[N1:] if k in ("flags", "itypes", "swaps") else v
        if not same(k, got_local[k], want):
            failed.append("local_" + k)
    for k, v in ref_job.items():
        if not same(k, got_job[k], v):
            failed.append("job_" + k)

    dist.barrier()                                   # every file is complete
    refused = True
    if rank == 1:                                    # process 0's file into a handle that owns process 1's ranks
        c = ParallelTempering(cfg, nproc, device=local_rank, world=world, rank=rank)
        try:
            c.restore(os.path.join(out_dir, f"ck.0-of-{world}"))
            refused = False
        except capi.RfinvError as e:
            refused = e.status == capi.RFINV_ERR_ARG
        c.close()
    if failed:
        say("FAILED: " + ", ".join(failed))
    res = [None] * world
    dist.all_gather_object(res, dict(ok=not failed, refused=refused, failed=failed))
    if rank == 0:
        print(json.dumps(dict(identical=all(r["ok"] for r in res), cross_restore_refused=all(r["refused"] for r in res),
                              failed=[f for r in res for f in r["failed"]], exchange=exchange, world=world,
                              virtual_ranks=nproc, n1=N1, n2=N2, nmod=int(got_job["hist_nmod"]))), flush=True)
    ok = all(r["ok"] and r["refused"] for r in res)
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
