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
the last tuning point (-1 without proposals).

``--diagnostics`` records level 0 of every virtual rank (its coldest chain) at every recording iteration and reports whether the
run has converged (DESIGN.md 7f): OUT_DIR/convergence has one line per quantity -- ``name samples ranks R-hat ESS tau_median
tempered_share`` for k, logL, every solved sigma (``sig_<trace>``) and the Vs at each depth of ``--diag-depths KM,KM,...``
(``vs_<km>``).  With the rank swaps it adds OUT_DIR/round_trips: ``rank trips_burn_in trips_after`` per virtual rank.  The
reference's files are written as without it."""
from __future__ import annotations

import argparse
import os
import sys
from collections import namedtuple

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


def depth_bins(cfg, depths):
    """The bookkeeping's depth bins int(z / dbin_z) + 1 of depths in km, the bottom z_max in the last bin nbin_z; a depth
    outside [0, z_max] or inside the sea layer is refused."""
    dbin_z = (cfg.z_max - 0.0) / cfg.nbin_z
    sea = int(cfg.sdep / dbin_z) + 1 if cfg.sdep > 0.0 else 1     # the first bin below the sea layer
    bins = []
    for z in depths:
        if not 0.0 <= z <= cfg.z_max:
            raise ValueError(f"diagnostic depth {z} km is outside [0, Z_MAX = {cfg.z_max}] km")
        b = min(int(z / dbin_z) + 1, cfg.nbin_z)   # (z_max itself, or a depth rounded past the last bin's bottom)
        if b < sea:
            raise ValueError(f"diagnostic depth {z} km lies inside the sea layer (SEA_DEP = {cfg.sdep} km)")
        bins.append(b)
    if len(bins) > 16:
        raise ValueError(f"{len(bins)} diagnostic depths: at most 16")
    return bins


def convergence_rows(diag, depths):
    """[(name, samples, ranks, R-hat, ESS, median tau, tempered share)] with the Vs quantities named by their depths."""
    names = diag["names"]
    nv = len(depths)
    if nv:
        names = names[:-nv] + [f"vs_{z:g}" for z in depths]
    return [(n, diag["n_samples"], diag["n_ranks"], diag["rhat"][q], diag["ess_total"][q], diag["tau_median"][q],
             diag["tempered_share"][q]) for q, n in enumerate(names)]


def write_convergence(out_dir: str, rows) -> None:
    """OUT_DIR/convergence: one line per quantity."""
    with open(os.path.join(out_dir, "convergence"), "w") as f:
        for n, ns, nr, rhat, ess, tau, share in rows:
            f.write(f"{n:12s} {ns:8d} {nr:6d} {rhat:.17g} {ess:.17g} {tau:.17g} {share:.17g}\n")


def write_round_trips(out_dir: str, trips) -> None:
    """OUT_DIR/round_trips: one line per virtual rank: rank, round trips during the burn-in, after it."""
    with open(os.path.join(out_dir, "round_trips"), "w") as f:
        for r, (a, b) in enumerate(trips):
            f.write(f"{r:6d} {int(a):8d} {int(b):8d}\n")


def print_convergence(rows) -> None:
    print(" --- Convergence of the cold level (R-hat, ESS, median IAT, tempered share) ---")
    for n, ns, nr, rhat, ess, tau, share in rows:
        print(f" {n}: R-hat {rhat:.4f}, ESS {ess:.1f} of {ns * nr} samples over {nr} ranks, median IAT {tau:.2f}, "
              f"tempered {share:.4f}")


def print_rank_swaps(rs) -> None:
    print(" --- Swaps between neighbouring temperature levels inside the ranks ---")
    for l, (a, n) in enumerate(zip(rs["n_acc"], rs["n_prop"]), start=1):
        print(f" # of swaps between levels {l - 1} and {l}: {int(a)} / {int(n)} ({a / n if n else 0.0:.4f})")


# the opt-in settings of a run (DESIGN.md 7c-7f), as run() takes them
Settings = namedtuple("Settings", "rank_swaps tune_ladder tune_steps step_target diagnostics diag_depths")


def checked_settings(checkpoint, checkpoint_every, resume, rank_swaps, tune_ladder, tune_steps, step_target, diagnostics,
                     diag_depths) -> Settings:
    """run()'s arguments checked, and the settings with the rank swaps that the tunings imply."""
    if resume and not checkpoint:
        raise ValueError("resume needs a checkpoint path")
    if checkpoint_every is not None and checkpoint_every < 1:
        raise ValueError("checkpoint_every must be at least 1")
    return Settings(rank_swaps or tune_ladder or tune_steps, tune_ladder, tune_steps, step_target, diagnostics,
                    tuple(diag_depths))


def switch_on(pt, opt: Settings, bins) -> None:
    """Switches the settings on, before a restore: the checkpoint holds their state.  bins: depth_bins of opt.diag_depths."""
    if opt.rank_swaps:
        pt.set_rank_swaps(1)
    if opt.tune_ladder:
        pt.set_ladder_tuning(1)
    if opt.tune_steps:
        pt.set_step_tuning(1, opt.step_target)
    if opt.diagnostics:
        pt.set_diagnostics(1, bins)


def iterate(run_step, save, done: int, n_tot: int, ncorr: int, checkpoint_every, verbose: bool) -> None:
    """Runs iterations done .. n_tot by run_step(n) with a progress line every N_CORR iterations (src/pt_mcmc.f90:489-491);
    save(), if given, every `checkpoint_every` iterations (rounded up to the progress steps; default: every step) and at the end."""
    step_len = max(ncorr, 1) * 100
    every = step_len if checkpoint_every is None else checkpoint_every
    saved = done
    while done < n_tot:
        step = min(step_len - done % step_len, n_tot - done)   # (a resumed run keeps the progress steps of a fresh one)
        run_step(step)
        done += step
        if verbose:
            print(f" Iteration #: {done} / {n_tot}", flush=True)
        if save and (done - saved >= every or done == n_tot):   # always at the end
            save()
            saved = done


def report(pt, cfg, nproc: int, opt: Settings, ladders, widths, write: bool, verbose: bool):
    """Reads the results of pt (job-wide on process 0 after reduce_outputs) and, with `write`, prints them (verbose) and writes
    the reference's output files and those of the settings into OUT_DIR.  ladders / widths: the rows of rank_ladders /
    step_rows with the tunings on, else None.  Returns (hist, counters)."""
    hist, cnt = pt.hist(), pt.counters()
    vp_model, vs_model = pt.models()
    rs = pt.rank_swaps() if opt.rank_swaps else None
    diag = pt.diagnostics() if opt.diagnostics else None
    if not write:
        return hist, cnt
    if verbose:
        print_summary(cfg, hist, cnt)
        if rs:
            print_rank_swaps(rs)
    rio.write_outputs(cfg, cfg.out_dir, nproc, hist, cnt["likelihood_hist"], vp_model, vs_model)
    if rs:
        write_rank_swaps(cfg.out_dir, rs)
    if ladders is not None:
        write_ladder(cfg.out_dir, ladders)
    if widths is not None:
        write_step_widths(cfg.out_dir, widths)
    if diag is not None:
        conv = convergence_rows(diag, opt.diag_depths)
        if verbose:
            print_convergence(conv)
        write_convergence(cfg.out_dir, conv)
        if rs:
            write_round_trips(cfg.out_dir, diag["trips"])
    return hist, cnt


def run(params_path: str, nproc: int, verbose: bool = True, n_iter: int = None, checkpoint: str = None,
        checkpoint_every: int = None, resume: bool = False, rank_swaps: bool = False, tune_ladder: bool = False,
        tune_steps: bool = False, step_target: float = 0.44, diagnostics: bool = False, diag_depths=()):
    """checkpoint: save the state to this path every `checkpoint_every` iterations (rounded up to the progress steps; default:
    every progress step) and at the end.  resume: restore it first if it exists and continue from its iteration count.
    rank_swaps: the even/odd sweep inside every virtual rank (ParallelTempering.set_rank_swaps(1)); adds OUT_DIR/rank_swaps.
    tune_ladder: implies rank_swaps, plus the ladder tuning during the burn-in (set_ladder_tuning(1)); adds OUT_DIR/ladder.
    tune_steps: implies rank_swaps, plus the width tuning during the burn-in towards the acceptance rate step_target
    (set_step_tuning(1, step_target)); adds OUT_DIR/step_widths.
    diagnostics: record the cold level and report convergence (set_diagnostics) at the depths diag_depths (km); adds
    OUT_DIR/convergence and, with rank_swaps, OUT_DIR/round_trips."""
    opt = checked_settings(checkpoint, checkpoint_every, resume, rank_swaps, tune_ladder, tune_steps, step_target, diagnostics,
                           diag_depths)
    cfg = rio.load_problem(params_path)
    bins = depth_bins(cfg, opt.diag_depths) if opt.diagnostics else []
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
    switch_on(pt, opt, bins)
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
    iterate(pt.run if world == 1 else lambda n: pt.run_distributed(n, dist, torch), (lambda: pt.save(ck)) if ck else None,
            done, n_tot, cfg.ncorr, checkpoint_every, verbose and rank == 0)

    def gathered(rows):                                   # process 0 writes the rows of every process, in rank order
        if rows is None or world == 1:
            return rows
        parts = [None] * world
        dist.all_gather_object(parts, rows)
        return np.concatenate(parts)
    ladders = gathered(rank_ladders(pt) if opt.tune_ladder else None)
    widths = gathered(step_rows(pt) if opt.tune_steps else None)
    if world > 1:                                         # the reference's mpi_reduce / mpi_gather (src/mcmc_out.f90:52-93)
        pt.reduce_outputs()                               # ncclReduce / ncclSend+Recv inside the library: process 0 is job-wide now
    hist, cnt = report(pt, cfg, nproc, opt, ladders, widths, rank == 0, verbose)
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
              tune_steps: bool = False, step_target: float = 0.44, diagnostics: bool = False, diag_depths=()):
    """Several stations (one params file each) as one group on one GPU; arguments as in run().  Under torchrun process r
    takes the stations i with i % world == r.  Returns {station index: (hist, counters)} of this process's stations."""
    opt = checked_settings(checkpoint, checkpoint_every, resume, rank_swaps, tune_ladder, tune_steps, step_target, diagnostics,
                           diag_depths)
    params_paths = list(params_paths)
    cfgs = load_stations(params_paths)
    bins = [depth_bins(c, opt.diag_depths) if opt.diagnostics else [] for c in cfgs]
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
        for i, pt in zip(mine, pts):
            switch_on(pt, opt, bins[i])
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

        def save():
            for i, pt in zip(mine, pts):
                pt.save(cks[i])
        with PtGroup(pts) as group:
            iterate(group.run, save if cks else None, done, n_tot, cfg0.ncorr, checkpoint_every, verbose)
        out = {}
        for i, pt in zip(mine, pts):
            if verbose:
                print(f" === {params_paths[i]} ===")
            out[i] = report(pt, cfgs[i], nproc, opt, rank_ladders(pt) if opt.tune_ladder else None,
                            step_rows(pt) if opt.tune_steps else None, True, verbose)
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
    ap.add_argument("--diagnostics", action="store_true",
                    help="record the coldest level of every virtual rank and report convergence: R-hat, ESS, median IAT, "
                         "tempered share (writes OUT_DIR/convergence; with --rank-swaps also OUT_DIR/round_trips)")
    ap.add_argument("--diag-depths", default="", metavar="KM,KM,...",
                    help="with --diagnostics: also follow Vs at these depths in km (at most 16, below the sea layer)")
    a = ap.parse_args(argv)
    if a.resume and not a.checkpoint:
        ap.error("--resume needs --checkpoint")
    if not 0.0 < a.step_target < 1.0:
        ap.error("--step-target must lie in (0, 1)")
    try:
        depths = [float(x) for x in a.diag_depths.split(",") if x.strip()]
    except ValueError:
        ap.error("--diag-depths takes depths in km separated by commas")
    if depths and not a.diagnostics:
        ap.error("--diag-depths needs --diagnostics")
    kw = dict(n_iter=a.iters, checkpoint=a.checkpoint, checkpoint_every=a.checkpoint_every, resume=a.resume,
              rank_swaps=a.rank_swaps, tune_ladder=a.tune_ladder, tune_steps=a.tune_steps, step_target=a.step_target,
              diagnostics=a.diagnostics, diag_depths=depths)
    if len(a.params) == 1:
        run(a.params[0], a.nproc, **kw)
    else:
        run_group(a.params, a.nproc, **kw)


if __name__ == "__main__":
    main()
