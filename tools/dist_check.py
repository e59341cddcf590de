"""Identity of the distributed parallel-tempering run on the real NCCL path (launch under torchrun, one process per GPU):
the accept / reject flags, proposal types, swap decisions, final state and job-wide bookkeeping of N processes driving
rfinv_pt_run_distributed (in-library ncclAllGather, CUDA graph) equal those of ONE process holding every virtual rank.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/dist_check.py

--rank-swaps runs both sides with the even/odd sweep inside every virtual rank (set_rank_swaps(1)) and also compares its
job-wide counters.  --tune-ladder adds the ladder tuning during the burn-in (set_ladder_tuning(1), implies --rank-swaps), with
burn-ins and run lengths that pass two or three tuning points, and also compares the number of tuning points passed.
--tune-steps adds the width tuning during the burn-in (set_step_tuning(1), implies --rank-swaps) with the same run lengths, and
also compares each process's widths and width counters with its rows of the single-process run.
"""
import faulthandler, hashlib, json, os, signal, sys
faulthandler.register(signal.SIGTERM, all_threads=True, chain=False)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist
from rf_inv_b200 import workloads
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering


def identity_check(cfg, nproc_total, n_iter, world, rank, local_rank, dist, torch, rank_swaps=0, tune_ladder=False,
                   tune_steps=False):
    """Returns (ok, detail) on every process."""
    dev = torch.device("cuda", local_rank)
    # distributed run
    def say(msg):
        print(f"[rank {rank}] {msg}", file=sys.stderr, flush=True)
    pt = ParallelTempering(cfg, nproc_total, device=local_rank, world=world, rank=rank)
    pt.set_logging(n_iter)
    if rank_swaps:
        pt.set_rank_swaps(rank_swaps)
    if tune_ladder:
        pt.set_ladder_tuning(1)
    if tune_steps:
        pt.set_step_tuning(1)
    pt.init_comm(dist, torch)
    say("communicator up")
    pt.run_distributed(n_iter, dist, torch)
    exchange = pt.exchange_mode
    say("distributed run done (exchange: %s)" % exchange)
    flags, itypes, swaps = pt.log(n_iter)
    st = pt.state()
    tuning = pt.ladder_tuning()
    steps = pt.step_tuning() if tune_steps else None
    pt.reduce_outputs()
    say("outputs reduced")
    cnt = pt.counters()
    hist = pt.hist() if cfg.niter > 0 else None
    rsw = pt.rank_swaps() if rank_swaps else None
    say("getters done")
    pt.close()
    say("closed")
    # single-process reference on process 0, broadcast to the others
    if rank == 0:
        ref = ParallelTempering(cfg, nproc_total, device=local_rank)
        ref.set_logging(n_iter)
        if rank_swaps:
            ref.set_rank_swaps(rank_swaps)
        if tune_ladder:
            ref.set_ladder_tuning(1)
        if tune_steps:
            ref.set_step_tuning(1)
        ref.run(n_iter)
        rsteps = ref.step_tuning() if tune_steps else None
        rtuning = ref.ladder_tuning()
        rf, ri, rs = ref.log(n_iter)
        rst = ref.state()
        rcnt = ref.counters()
        rhist = ref.hist() if cfg.niter > 0 else None
        rrsw = ref.rank_swaps() if rank_swaps else None
        ref.close()
        say("reference run done")
        box = [dict(flags=rf, itypes=ri, swaps=rs, state=rst, tuning=rtuning, steps=rsteps)]
    else:
        box = [None]
    dist.broadcast_object_list(box, src=0)
    say("reference broadcast")
    r = box[0]
    n_local = pt.n_local
    sl = slice(rank * n_local, (rank + 1) * n_local)
    parts = dict(flags=np.array_equal(flags, r["flags"][:, sl]), itypes=np.array_equal(itypes, r["itypes"][:, sl]),
                 swaps=np.array_equal(swaps, r["swaps"]))
    for k in ("k", "z", "dvp", "dvs", "sig", "logl", "temps"):
        parts["state_" + k] = np.array_equal(st[k], r["state"][k][sl])
    if tune_ladder:
        parts["ladder_tuning"] = tuning == r["tuning"] and tuning[0] and tuning[1] >= 2
    if tune_steps:
        rsl = slice(pt.rank_begin, pt.rank_begin + pt.rank_count)
        parts["step_tuning"] = (steps["on"] and steps["n_points"] == r["steps"]["n_points"] >= 2
                                and not np.all(r["steps"]["widths"] == r["steps"]["widths"][0, 0])
                                and all(np.array_equal(steps[k], r["steps"][k][rsl]) for k in ("widths", "n_prop", "n_acc")))
    detail = {}
    if rank == 0:
        parts["nprop"] = np.array_equal(cnt["nprop"], rcnt["nprop"]); parts["naccept"] = np.array_equal(cnt["naccept"], rcnt["naccept"])
        # likelihood_hist is a sum over processes of per-process tree sums: equal up to the order of additions
        if rank_swaps:
            parts["rank_swaps"] = (rsw["mode"] == rrsw["mode"] == 1 and np.array_equal(rsw["n_prop"], rrsw["n_prop"])
                                   and np.array_equal(rsw["n_acc"], rrsw["n_acc"]) and int(rrsw["n_acc"].sum()) > 0)
        parts["likelihood_hist"] = bool(np.allclose(cnt["likelihood_hist"], rcnt["likelihood_hist"], rtol=1e-12, atol=0))
        if hist is not None:
            parts["nmod"] = hist["nmod"] == rhist["nmod"]
            for k in ("nk", "nz", "nsig", "namp", "nvpz", "nvsz", "nvpvsz"):
                parts["hist_" + k] = np.array_equal(hist[k], rhist[k])
            for k in ("vp_mean", "vs_mean", "vpvs_mean"):
                parts["hist_" + k] = bool(np.allclose(hist[k], rhist[k], rtol=1e-12))
        detail = dict(flags_sha1=hashlib.sha1(r["flags"].tobytes()).hexdigest()[:16], accepted=int((r["flags"] == 1).sum()),
                      swaps_accepted=int(r["swaps"][:, 2].sum()), nmod=None if hist is None else int(hist["nmod"]),
                      failed=[k for k, v in parts.items() if not v], exchange=exchange)
    ok = all(parts.values())
    if not ok:
        say("FAILED: " + ", ".join(k for k, v in parts.items() if not v))
    t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item()), detail


if __name__ == "__main__":
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    tune_ladder = "--tune-ladder" in sys.argv[1:]
    tune_steps = "--tune-steps" in sys.argv[1:]
    rank_swaps = 1 if "--rank-swaps" in sys.argv[1:] or tune_ladder or tune_steps else 0
    out = {}
    runs = (("sample", 4 * world, 300, dict(nburn=100, niter=200)), ("c4", 8 * world, 120, dict()), ("target", 16 * world, 60, dict()))
    if tune_ladder or tune_steps:   # tuning points 64, 128, 256 / 64, 128, inside and at the end of the burn-in
        runs = (("sample", 4 * world, 300, dict(nburn=280, niter=20)), ("c4", 8 * world, 140, dict(nburn=128)),
                ("target", 16 * world, 130, dict(nburn=200)))
    for name, nproc, iters, kw in runs:
        cfg = workloads.make_config(name)
        for k_, v_ in kw.items():
            setattr(cfg, k_, v_)
        if cfg.niter > 0:
            cfg.nbin_z, cfg.nbin_vs, cfg.nbin_vp, cfg.nbin_vpvs, cfg.nbin_sig, cfg.nbin_amp = 50, 25, 25, 20, 10, 40
            cfg.amp_min, cfg.amp_max = -0.6, 0.6
        cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp)); cfg.r_inv = workloads.lapack_r_inv(cfg)
        tm = workloads.true_model(cfg)
        with Evaluator(cfg, device=local_rank) as ev:
            _, rft, _ = ev.calc_likelihood(tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"], want_rft=True)
        cfg.obs = (rft[0, :, :cfg.nsmp] + np.random.default_rng(7).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))).astype(np.float32).astype(np.float64)
        ok, detail = identity_check(cfg, nproc, iters, world, rank, local_rank, dist, torch, rank_swaps, tune_ladder,
                                    tune_steps)
        out[name] = dict(identical=ok, world=world, virtual_ranks=nproc, iterations=iters, **detail)
    if rank == 0:
        print(json.dumps(out), flush=True)
    dist.destroy_process_group()
    sys.exit(0 if all(v["identical"] for v in out.values()) else 1)
