"""Driver with the reference's command line (src/rf_inv.f90:28-108):  python -m rf_inv_b200.run [params.in] --nproc N

``--nproc`` is the number of MPI ranks the reference would be started with (``mpirun -np N``): N virtual ranks of
N_CHAINS chains each, all resident on the GPU(s).  Under torchrun (one process per GPU) the virtual ranks are split
over the processes and the per-iteration swap exchange is one NCCL all-gather issued by the library itself.  Writes the reference's output files
into OUT_DIR.

``--checkpoint PATH`` saves the complete chain state as the run goes (under torchrun one file per process,
``PATH.<rank>-of-<world>``); ``--resume`` continues from it if it exists, so the same command can be resubmitted after an
interruption, or with a larger N_ITER in params.in.  A resumed run writes exactly the files an uninterrupted run writes.

Several params files (``python -m rf_inv_b200.run a/params.in b/params.in ... --nproc N``), one per station, run side by
side on one GPU as one group (rfinv_pt_group_run): every station writes into its own OUT_DIR exactly the files a run of its
params file alone writes.  The stations must agree on N_BURN, N_ITER and N_CORR and write to different OUT_DIRs.  Station i
(its position on the command line) checkpoints to ``PATH.<i>``.  Under torchrun process r runs the stations i with
i % world == r as its group on its own GPU; the processes do not communicate.

``--rank-swaps`` adds even/odd temperature swaps between neighbouring levels inside every virtual rank (DESIGN.md 7c).  The
reference's files are written as without it, plus OUT_DIR/rank_swaps with the acceptance of each neighbour pair.

``--tune-ladder`` (implies ``--rank-swaps``) also retunes every virtual rank's temperature ladder at the iteration counts 64,
128, 256, ... up to N_BURN towards equal neighbour-swap rejection rates (DESIGN.md 7d); the ladders are fixed after the
burn-in.  It adds OUT_DIR/ladder: one line per virtual rank, its temperatures by level (coldest first) at the end of the run.

``--tune-steps`` (implies ``--rank-swaps``) also tunes the random-walk widths of the moves z, dVs, dVp and sigma of every
virtual rank and level at the same iteration counts towards the acceptance rate ``--step-target`` (default 0.44; DESIGN.md
7e); the widths are fixed after the burn-in.  It adds OUT_DIR/step_widths: one line per virtual rank and level,
``rank level w_z w_dvs w_dvp w_sig acc_z acc_dvs acc_dvp acc_sig`` -- the final widths and the acceptance they produced since
the last tuning point (-1 without proposals)."""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

from . import io as rio
from . import workloads
from .pt import ParallelTempering, PtGroup


def checkpoint_path(path: str, world: int, rank: int) -> str:
    """The file of this process: `path` itself for one process, `path.<rank>-of-<world>` under torchrun."""
    return path if world == 1 else f"{path}.{rank}-of-{world}"


def print_summary(cfg, hist, cnt) -> None:
    """The acceptance summary of src/mcmc_out.f90:99-107."""
    labels = ["Birth proposal", "Death proposal", "Moving interface depth proposal", "Perturbing dVs proposal"]
    if cfg.vp_mode == 1:
        labels.append("Perturbing dVs proposal")  # sic: the reference labels the dVp proposal like this (pt_mcmc.f90:386)
    if any(cfg.sig_mode):
        labels.append("Perturbing sigma proposal")
    print(" --- Summary ---")
    print(f" # of sampled models: {hist['nmod']}")
    for lab, a, n in zip(labels, cnt["naccept"], cnt["nprop"]):
        print(f" # of {lab}: {int(a)} / {int(n)}")


def write_rank_swaps(out_dir: str, rs) -> None:
    """OUT_DIR/rank_swaps: one line per neighbour pair l = 1 .. nchains-1 (levels l-1 and l, level 0 the coldest):
    l, swaps accepted, swaps proposed, acceptance rate."""
    with open(os.path.join(out_dir, "rank_swaps"), "w") as f:
        for l, (a, n) in enumerate(zip(rs["n_acc"], rs["n_prop"]), start=1):
            f.write(f"{l:5d} {int(a):12d} {int(n):12d} {a / n if n else 0.0:12.6f}\n")


def rank_ladders(pt) -> np.ndarray:
    """[local ranks][nchains]: each virtual rank's temperatures sorted by (temperature, chain index), coldest first."""
    t = pt.state()["temps"].reshape(pt.rank_count, pt.cfg.nchains)
    idx = np.arange(pt.cfg.nchains)
    return np.take_along_axis(t, np.lexsort((np.broadcast_to(idx, t.shape), t), axis=1), axis=1)


def write_ladder(out_dir: str, ladders) -> None:
    """OUT_DIR/ladder: one line per virtual rank, its temperatures by level."""
    with open(os.path.join(out_dir, "ladder"), "w") as f:
        for row in ladders:
            f.write(" ".join(f"{t:.17g}" for t in row) + "\n")


def step_rows(pt) -> np.ndarray:
    """[local ranks * nchains][10]: global rank, level, the four widths, the four acceptance rates (-1 without proposals)."""
    st = pt.step_tuning()
    nr, nc = pt.rank_count, pt.cfg.nchains
    acc = np.where(st["n_prop"] > 0, st["n_acc"] / np.maximum(st["n_prop"], 1), -1.0)
    ranks = np.repeat(np.arange(pt.rank_begin, pt.rank_begin + nr), nc)
    levels = np.tile(np.arange(nc), nr)
    return np.column_stack([ranks, levels, st["widths"].reshape(-1, 4), acc.reshape(-1, 4)])


def write_step_widths(out_dir: str, rows) -> None:
    """OUT_DIR/step_widths: one line per virtual rank and level."""
    with open(os.path.join(out_dir, "step_widths"), "w") as f:
        for row in rows:
            f.write(f"{int(row[0]):6d} {int(row[1]):5d} " + " ".join(f"{x:.17g}" for x in row[2:6]) + " "
                    + " ".join(f"{x:.6f}" for x in row[6:]) + "\n")


def print_rank_swaps(rs) -> None:
    print(" --- Swaps between neighbouring temperature levels inside the ranks ---")
    for l, (a, n) in enumerate(zip(rs["n_acc"], rs["n_prop"]), start=1):
        print(f" # of swaps between levels {l - 1} and {l}: {int(a)} / {int(n)} ({a / n if n else 0.0:.4f})")


def run(params_path: str, nproc: int, verbose: bool = True, n_iter: int = None, checkpoint: str = None,
        checkpoint_every: int = None, resume: bool = False, rank_swaps: bool = False, tune_ladder: bool = False,
        tune_steps: bool = False, step_target: float = 0.44):
    """checkpoint: save the state to this path every `checkpoint_every` iterations (rounded up to the progress steps; default:
    every progress step) and at the end.  resume: restore it first if it exists and continue from its iteration count.
    rank_swaps: the even/odd sweep inside every virtual rank (ParallelTempering.set_rank_swaps(1)); adds OUT_DIR/rank_swaps.
    tune_ladder: implies rank_swaps, plus the ladder tuning during the burn-in (set_ladder_tuning(1)); adds OUT_DIR/ladder.
    tune_steps: implies rank_swaps, plus the width tuning during the burn-in towards the acceptance rate step_target
    (set_step_tuning(1, step_target)); adds OUT_DIR/step_widths."""
    rank_swaps = rank_swaps or tune_ladder or tune_steps
    if resume and not checkpoint:
        raise ValueError("resume needs a checkpoint path")
    if checkpoint_every is not None and checkpoint_every < 1:
        raise ValueError("checkpoint_every must be at least 1")
    cfg = rio.load_problem(params_path)
    cfg.r_inv = workloads.lapack_r_inv(cfg)          # init_r_inv: LAPACK dgesvd like the reference
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = torch = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        # torch.distributed only carries the library's communicator id between the processes (gloo: no second NCCL communicator)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")
    if rank == 0:
        os.makedirs(cfg.out_dir, exist_ok=True)
        rio.write_side_copies(params_path, cfg.out_dir, os.path.dirname(os.path.abspath(params_path)))
    pt = ParallelTempering(cfg, nproc, device=local_rank, world=world, rank=rank)
    if rank_swaps:                                        # before a restore: the checkpoint holds the sweep's counters
        pt.set_rank_swaps(1)
    if tune_ladder:
        pt.set_ladder_tuning(1)
    if tune_steps:
        pt.set_step_tuning(1, step_target)
    n_tot = cfg.nburn + cfg.niter if n_iter is None else n_iter
    ck = checkpoint_path(checkpoint, world, rank) if checkpoint else None
    if resume:
        found = [os.path.exists(ck)]
        if world > 1:                                     # every process restores, or none does
            found = [None] * world
            dist.all_gather_object(found, os.path.exists(ck))
        if all(found):
            pt.restore(ck)
            if verbose and rank == 0:
                print(f" Resuming at iteration {pt.iterations_done} from {checkpoint}", flush=True)
        elif any(found):
            raise FileNotFoundError(f"checkpoint files of {checkpoint} exist for some processes only: {found}")
    done = pt.iterations_done
    if done > n_tot:
        raise ValueError(f"the checkpoint is at iteration {done}, beyond the {n_tot} iterations asked for")
    step_len = max(cfg.ncorr, 1) * 100
    every = step_len if checkpoint_every is None else checkpoint_every
    saved = done
    while done < n_tot:                                   # progress line every N_CORR iterations (src/pt_mcmc.f90:489-491)
        step = min(step_len - done % step_len, n_tot - done)   # (a resumed run keeps the progress steps of a fresh one)
        if world == 1:
            pt.run(step)
        else:
            pt.run_distributed(step, dist, torch)
        done += step
        if verbose and rank == 0:
            print(f" Iteration #: {done} / {n_tot}", flush=True)
        if ck and (done - saved >= every or done == n_tot):   # always at the end
            pt.save(ck)
            saved = done
    ladders = rank_ladders(pt) if tune_ladder else None
    if tune_ladder and world > 1:                         # process 0 writes the rows of every process, in rank order
        rows = [None] * world
        dist.all_gather_object(rows, ladders)
        ladders = np.concatenate(rows)
    widths = step_rows(pt) if tune_steps else None
    if tune_steps and world > 1:
        rows = [None] * world
        dist.all_gather_object(rows, widths)
        widths = np.concatenate(rows)
    if world > 1:                                         # the reference's mpi_reduce / mpi_gather (src/mcmc_out.f90:52-93)
        pt.reduce_outputs()                               # ncclReduce / ncclSend+Recv inside the library: process 0 is job-wide now
    hist, cnt = pt.hist(), pt.counters()
    vp_model, vs_model = pt.models()
    rs = pt.rank_swaps() if rank_swaps else None
    lh = cnt["likelihood_hist"]
    if rank == 0:
        if verbose:
            print_summary(cfg, hist, cnt)
            if rs:
                print_rank_swaps(rs)
        rio.write_outputs(cfg, cfg.out_dir, nproc, hist, lh, vp_model, vs_model)
        if rs:
            write_rank_swaps(cfg.out_dir, rs)
        if ladders is not None:
            write_ladder(cfg.out_dir, ladders)
        if widths is not None:
            write_step_widths(cfg.out_dir, widths)
    pt.close()
    if world > 1:
        dist.destroy_process_group()
    return hist, cnt


def station_checkpoint_path(path: str, station: int) -> str:
    """The checkpoint file of station `station` (its position on the command line) of a group run."""
    return f"{path}.{station}"


def load_stations(params_paths):
    """The configurations of the stations of a group run, refused before any GPU work when two stations write to the same
    OUT_DIR or when they differ in N_BURN, N_ITER or N_CORR (a group advances its stations in lock step)."""
    cfgs = [rio.load_problem(p) for p in params_paths]
    seen = {}
    for i, (p, c) in enumerate(zip(params_paths, cfgs)):
        d = os.path.realpath(c.out_dir)
        if d in seen:
            j = seen[d]
            raise ValueError(f"stations {j} ({params_paths[j]}) and {i} ({p}) write to the same OUT_DIR {c.out_dir}")
        seen[d] = i
    for key, name in (("nburn", "N_BURN"), ("niter", "N_ITER"), ("ncorr", "N_CORR")):
        vals = [getattr(c, key) for c in cfgs]
        if len(set(vals)) > 1:
            raise ValueError(f"the stations of a group must have equal {name}: "
                             + ", ".join(f"{p}: {v}" for p, v in zip(params_paths, vals)))
    return cfgs


def run_group(params_paths, nproc: int, verbose: bool = True, n_iter: int = None, checkpoint: str = None,
              checkpoint_every: int = None, resume: bool = False, rank_swaps: bool = False, tune_ladder: bool = False,
              tune_steps: bool = False, step_target: float = 0.44):
    """Several stations (one params file each) as one group on one GPU; arguments as in run().  Under torchrun process r
    takes the stations i with i % world == r.  Returns {station index: (hist, counters)} of this process's stations."""
    rank_swaps = rank_swaps or tune_ladder or tune_steps
    if resume and not checkpoint:
        raise ValueError("resume needs a checkpoint path")
    if checkpoint_every is not None and checkpoint_every < 1:
        raise ValueError("checkpoint_every must be at least 1")
    params_paths = list(params_paths)
    cfgs = load_stations(params_paths)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    mine = [i for i in range(len(params_paths)) if i % world == rank]
    cks = [station_checkpoint_path(checkpoint, i) for i in range(len(params_paths))] if checkpoint else None
    restore = False
    if resume:                                            # every station restores, or none does (all processes see all files)
        found = [os.path.exists(p) for p in cks]
        if any(found) and not all(found):
            raise FileNotFoundError(f"checkpoint files of {checkpoint} exist for some stations only: {found}")
        restore = all(found)
    if not mine:
        return {}
    for i in mine:
        os.makedirs(cfgs[i].out_dir, exist_ok=True)
        rio.write_side_copies(params_paths[i], cfgs[i].out_dir, os.path.dirname(os.path.abspath(params_paths[i])))
        cfgs[i].r_inv = workloads.lapack_r_inv(cfgs[i])
    pts = [ParallelTempering(cfgs[i], nproc, device=local_rank) for i in mine]
    try:
        if rank_swaps:
            for pt in pts:
                pt.set_rank_swaps(1)
                if tune_ladder:
                    pt.set_ladder_tuning(1)
                if tune_steps:
                    pt.set_step_tuning(1, step_target)
        if restore:
            for i, pt in zip(mine, pts):
                pt.restore(cks[i])
            if verbose:
                print(f" Resuming at iteration {pts[0].iterations_done} from {checkpoint}.<station>", flush=True)
        cfg0 = cfgs[mine[0]]
        n_tot = cfg0.nburn + cfg0.niter if n_iter is None else n_iter
        done = pts[0].iterations_done
        if done > n_tot:
            raise ValueError(f"the checkpoints are at iteration {done}, beyond the {n_tot} iterations asked for")
        step_len = max(cfg0.ncorr, 1) * 100
        every = step_len if checkpoint_every is None else checkpoint_every
        saved = done
        with PtGroup(pts) as group:
            while done < n_tot:                           # the progress steps of run()
                step = min(step_len - done % step_len, n_tot - done)
                group.run(step)
                done += step
                if verbose:
                    print(f" Iteration #: {done} / {n_tot}", flush=True)
                if cks and (done - saved >= every or done == n_tot):
                    for i, pt in zip(mine, pts):
                        pt.save(cks[i])
                    saved = done
        out = {}
        for i, pt in zip(mine, pts):
            cfg = cfgs[i]
            hist, cnt = pt.hist(), pt.counters()
            vp_model, vs_model = pt.models()
            if verbose:
                print(f" === {params_paths[i]} ===")
                print_summary(cfg, hist, cnt)
                if rank_swaps:
                    print_rank_swaps(pt.rank_swaps())
            rio.write_outputs(cfg, cfg.out_dir, nproc, hist, cnt["likelihood_hist"], vp_model, vs_model)
            if rank_swaps:
                write_rank_swaps(cfg.out_dir, pt.rank_swaps())
            if tune_ladder:
                write_ladder(cfg.out_dir, rank_ladders(pt))
            if tune_steps:
                write_step_widths(cfg.out_dir, step_rows(pt))
            out[i] = (hist, cnt)
        return out
    finally:
        for pt in pts:
            pt.close()


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("params", nargs="*", default=["params.in"],
                    help="params.in of the run; several files (one per station) run side by side as one group")
    ap.add_argument("--nproc", type=int, default=20, help="number of virtual MPI ranks (mpirun -np of the reference)")
    ap.add_argument("--iters", type=int, default=None, help="override N_BURN + N_ITER (testing)")
    ap.add_argument("--checkpoint", default=None, metavar="PATH",
                    help="save the chain state to PATH (under torchrun: PATH.<rank>-of-<world>; station i of a group: "
                         "PATH.<i>) during and at the end of the run")
    ap.add_argument("--checkpoint-every", type=int, default=None, metavar="N",
                    help="save every N iterations, rounded up to the progress steps (default: every progress step)")
    ap.add_argument("--resume", action="store_true",
                    help="continue from the checkpoint if it exists (a missing file starts a fresh run)")
    ap.add_argument("--rank-swaps", action="store_true",
                    help="also swap temperatures between neighbouring levels inside every virtual rank, even and odd pairs "
                         "in turn (writes OUT_DIR/rank_swaps)")
    ap.add_argument("--tune-ladder", action="store_true",
                    help="with --rank-swaps (implied): retune every rank's temperature ladder during the burn-in towards equal "
                         "swap rejection rates between neighbouring levels (writes OUT_DIR/ladder)")
    ap.add_argument("--tune-steps", action="store_true",
                    help="with --rank-swaps (implied): tune the random-walk widths of every rank's levels during the burn-in "
                         "towards the acceptance rate --step-target (writes OUT_DIR/step_widths)")
    ap.add_argument("--step-target", type=float, default=0.44,
                    help="acceptance rate --tune-steps aims at, in (0, 1) (default 0.44)")
    a = ap.parse_args(argv)
    if a.resume and not a.checkpoint:
        ap.error("--resume needs --checkpoint")
    if not 0.0 < a.step_target < 1.0:
        ap.error("--step-target must lie in (0, 1)")
    if len(a.params) == 1:
        run(a.params[0], a.nproc, n_iter=a.iters, checkpoint=a.checkpoint, checkpoint_every=a.checkpoint_every, resume=a.resume,
            rank_swaps=a.rank_swaps, tune_ladder=a.tune_ladder, tune_steps=a.tune_steps, step_target=a.step_target)
    else:
        run_group(a.params, a.nproc, n_iter=a.iters, checkpoint=a.checkpoint, checkpoint_every=a.checkpoint_every,
                  resume=a.resume, rank_swaps=a.rank_swaps, tune_ladder=a.tune_ladder, tune_steps=a.tune_steps,
                  step_target=a.step_target)


if __name__ == "__main__":
    main()
