"""Driver with the reference's command line (src/rf_inv.f90:28-108):  python -m rf_inv_b200.run [params.in] --nproc N

``--nproc`` is the number of MPI ranks the reference would be started with (``mpirun -np N``): N virtual ranks of
N_CHAINS chains each, all resident on the GPU(s).  Under torchrun (one process per GPU) the virtual ranks are split
over the processes and the per-iteration swap exchange is one NCCL all-gather issued by the library itself.  Writes the reference's output files
into OUT_DIR.

``--checkpoint PATH`` saves the complete chain state as the run goes (under torchrun one file per process,
``PATH.<rank>-of-<world>``); ``--resume`` continues from it if it exists, so the same command can be resubmitted after an
interruption, or with a larger N_ITER in params.in.  A resumed run writes exactly the files an uninterrupted run writes."""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

from . import io as rio
from . import workloads
from .pt import ParallelTempering


def checkpoint_path(path: str, world: int, rank: int) -> str:
    """The file of this process: `path` itself for one process, `path.<rank>-of-<world>` under torchrun."""
    return path if world == 1 else f"{path}.{rank}-of-{world}"


def run(params_path: str, nproc: int, verbose: bool = True, n_iter: int = None, checkpoint: str = None,
        checkpoint_every: int = None, resume: bool = False):
    """checkpoint: save the state to this path every `checkpoint_every` iterations (rounded up to the progress steps; default:
    every progress step) and at the end.  resume: restore it first if it exists and continue from its iteration count."""
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
    if world > 1:                                         # the reference's mpi_reduce / mpi_gather (src/mcmc_out.f90:52-93)
        pt.reduce_outputs()                               # ncclReduce / ncclSend+Recv inside the library: process 0 is job-wide now
    hist, cnt = pt.hist(), pt.counters()
    vp_model, vs_model = pt.models()
    lh = cnt["likelihood_hist"]
    if rank == 0:
        if verbose:                                       # summary, src/mcmc_out.f90:99-107
            labels = ["Birth proposal", "Death proposal", "Moving interface depth proposal", "Perturbing dVs proposal"]
            if cfg.vp_mode == 1:
                labels.append("Perturbing dVs proposal")  # sic: the reference labels the dVp proposal like this (pt_mcmc.f90:386)
            if any(cfg.sig_mode):
                labels.append("Perturbing sigma proposal")
            print(" --- Summary ---")
            print(f" # of sampled models: {hist['nmod']}")
            for lab, a, n in zip(labels, cnt["naccept"], cnt["nprop"]):
                print(f" # of {lab}: {int(a)} / {int(n)}")
        rio.write_outputs(cfg, cfg.out_dir, nproc, hist, lh, vp_model, vs_model)
    pt.close()
    if world > 1:
        dist.destroy_process_group()
    return hist, cnt


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("params", nargs="?", default="params.in")
    ap.add_argument("--nproc", type=int, default=20, help="number of virtual MPI ranks (mpirun -np of the reference)")
    ap.add_argument("--iters", type=int, default=None, help="override N_BURN + N_ITER (testing)")
    ap.add_argument("--checkpoint", default=None, metavar="PATH",
                    help="save the chain state to PATH (under torchrun: PATH.<rank>-of-<world>) during and at the end of the run")
    ap.add_argument("--checkpoint-every", type=int, default=None, metavar="N",
                    help="save every N iterations, rounded up to the progress steps (default: every progress step)")
    ap.add_argument("--resume", action="store_true",
                    help="continue from the checkpoint if it exists (a missing file starts a fresh run)")
    a = ap.parse_args(argv)
    if a.resume and not a.checkpoint:
        ap.error("--resume needs --checkpoint")
    run(a.params, a.nproc, n_iter=a.iters, checkpoint=a.checkpoint, checkpoint_every=a.checkpoint_every, resume=a.resume)


if __name__ == "__main__":
    main()
