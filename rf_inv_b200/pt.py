"""Host driver of the device-resident parallel-tempering MCMC (mirror of pt_control, src/pt_mcmc.f90:468-576).

Single GPU: ``ParallelTempering(cfg, nproc).run(n)``.  Several GPUs (one process per GPU, torch.distributed):
virtual ranks are split contiguously over processes; per iteration each process runs ``local_step`` and the
swap tables -- per-chain (temperature, logL) pairs plus the pair-selection draws -- are exchanged with ONE
all-gather (NCCL over NVLink on GPUs); every process then evaluates the same swap decision.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import numpy as np

from . import capi
from .config import RFConfig
from .evaluator import Evaluator, _p


def split_ranks(nproc_total: int, world: int, rank: int):
    """Contiguous, even split of the virtual ranks over processes: (rank_begin, rank_count)."""
    if nproc_total % world != 0:
        raise ValueError(f"nproc_total={nproc_total} must be divisible by the number of processes {world}")
    per = nproc_total // world
    return rank * per, per


class ParallelTempering:
    def __init__(self, cfg: RFConfig, nproc_total: int, device: int = 0, world: int = 1, rank: int = 0,
                 evaluator: Optional[Evaluator] = None):
        self.cfg = cfg
        self.nproc_total = nproc_total
        self.world, self.rank = world, rank
        self.rank_begin, self.rank_count = split_ranks(nproc_total, world, rank)
        self.ev = evaluator or Evaluator(cfg, device=device)
        self._lib = self.ev._lib
        capi.check(self._lib.rfinv_pt_init(self.ev.handle, nproc_total, self.rank_begin, self.rank_count))
        self.n_local = self.rank_count * cfg.nchains
        self.ntype = int(self._lib.rfinv_pt_ntype(self.ev.handle))
        self._gather_buf = None
        self._comm = False

    def close(self):
        self.ev.close()

    # -- single process ---------------------------------------------------------------------------
    def run(self, n_iter: int) -> None:
        if self.world != 1:
            raise RuntimeError("run() is the single-process driver; use run_distributed()")
        capi.check(self._lib.rfinv_pt_run(self.ev.handle, int(n_iter)))

    # -- one process per GPU ----------------------------------------------------------------------
    def swap_table(self):
        ptr, n = C.c_uint64(0), C.c_int32(0)
        capi.check(self._lib.rfinv_pt_swap_table(self.ev.handle, C.byref(ptr), C.byref(n)))
        return ptr.value, n.value

    def init_comm(self, dist=None, torch=None, id_bytes: Optional[bytes] = None) -> None:
        """Joins the library's own NCCL communicator (rfinv_comm_init).  The communicator id is created on process 0 and
        carried to the others by the host -- here through torch.distributed (any backend), or pass `id_bytes`."""
        if self.world == 1 or self._comm:
            return
        n = int(self._lib.rfinv_comm_id_bytes())
        if id_bytes is None:
            buf = (C.c_ubyte * n)()
            if self.rank == 0:
                capi.check(self._lib.rfinv_comm_create_id(buf))
            box = [bytes(buf)]
            dist.broadcast_object_list(box, src=0)
            id_bytes = box[0]
        raw = (C.c_ubyte * n).from_buffer_copy(id_bytes)
        capi.check(self._lib.rfinv_comm_init(self.ev.handle, raw, self.world, self.rank))
        self._comm = True

    def run_distributed(self, n_iter: int, dist=None, torch=None) -> None:
        """pt_control over all processes: local step, ncclAllGather of the swap tables and swap decision, all queued by the
        library on the handle's stream (one CUDA graph launch per iteration).  dist / torch are only needed once, to carry
        the communicator id (init_comm)."""
        self.init_comm(dist, torch)
        capi.check(self._lib.rfinv_pt_run_distributed(self.ev.handle, int(n_iter)))

    @property
    def exchange_mode(self) -> str:
        """How run_distributed moves the swap tables: "peer memory" (stores into IPC-mapped peer buffers from the kernel that
        builds the table), "nccl all-gather", or "none" (single process / not run yet)."""
        return {0: "none", 1: "peer memory", 2: "nccl all-gather"}[int(self._lib.rfinv_pt_exchange_mode(self.ev.handle))]

    def run_distributed_torch(self, n_iter: int, dist, torch) -> None:
        """The same loop with the exchange done by torch.distributed (kept for comparison with the in-library collective).
        The handle must share torch's current stream (set_stream), or the all-gather races with the library's kernels."""
        self.ev.set_stream(torch.cuda.current_stream(torch.device("cuda", self.ev.device)).cuda_stream)
        ptr, n = self.swap_table()
        dev = torch.device("cuda", self.ev.device)
        if self._gather_buf is None:
            self._gather_buf = torch.empty(self.world * n, dtype=torch.float64, device=dev)
        table = _tensor_from_ptr(torch, ptr, n, dev)   # zero-copy view of the library's table
        for _ in range(n_iter):
            capi.check(self._lib.rfinv_pt_local_step(self.ev.handle))
            dist.all_gather_into_tensor(self._gather_buf, table)
            capi.check(self._lib.rfinv_pt_apply_swap(self.ev.handle, self._gather_buf.data_ptr(), self.world))
        self.ev.synchronize()

    def reduce_outputs(self) -> None:
        """output_results' mpi_reduce / mpi_gather (src/mcmc_out.f90:52-93): afterwards process 0's hist() / counters() / models()
        are job-wide.  Collective; call once after the last iteration."""
        capi.check(self._lib.rfinv_pt_reduce_outputs(self.ev.handle))

    # -- checkpoint / resume ----------------------------------------------------------------------
    def save(self, path) -> None:
        """Writes this process's complete PT state to `path` (atomically).  Not between local_step and the swap, and not
        after reduce_outputs()."""
        capi.check(self._lib.rfinv_pt_save(self.ev.handle, os.fsencode(path)))

    def restore(self, path) -> None:
        """Loads a state written by save() into this freshly initialised object (same configuration -- niter may be larger --
        and the same nproc_total / world / rank).  The run continues at the saved iteration, bit-identical to an
        uninterrupted run.  Logging is switched off: call set_logging() again."""
        capi.check(self._lib.rfinv_pt_restore(self.ev.handle, os.fsencode(path)))

    # -- even/odd swaps inside every virtual rank (DESIGN.md 7c) -----------------------------------
    def set_rank_swaps(self, mode: int) -> None:
        """0: the reference's one global swap per iteration (default); 1: also a sweep of swaps between neighbouring
        temperature levels inside every virtual rank, before the global swap.  Between runs; every process the same."""
        capi.check(self._lib.rfinv_pt_set_rank_swaps(self.ev.handle, int(mode)))

    def rank_swaps(self) -> Dict[str, object]:
        """{mode, n_prop, n_acc}: swaps the sweep proposed and accepted per neighbour pair l = 0 .. nchains-2, summed over
        this process's ranks (over the job on process 0 after reduce_outputs() in mode 1)."""
        n = max(self.cfg.nchains - 1, 0)
        mode = C.c_int32(0)
        n_prop = np.zeros(n, dtype=np.int64); n_acc = np.zeros(n, dtype=np.int64)
        capi.check(self._lib.rfinv_pt_get_rank_swaps(self.ev.handle, C.byref(mode), _p(n_prop, capi.i64p), _p(n_acc, capi.i64p)))
        return dict(mode=int(mode.value), n_prop=n_prop, n_acc=n_acc)

    # -- ladder tuning during the burn-in (DESIGN.md 7d) -------------------------------------------------------------
    def set_ladder_tuning(self, on: bool) -> None:
        """On top of set_rank_swaps(1), before the first iteration (and before restore()): at the iteration counts 64, 128,
        256, ... up to N_BURN every virtual rank respaces the temperatures of its levels above the cold ones towards equal
        neighbour-swap rejection rates.  The ladders stay fixed after the burn-in.  Off is allowed between runs;
        set_rank_swaps(0) switches it off too."""
        capi.check(self._lib.rfinv_pt_set_ladder_tuning(self.ev.handle, int(on)))

    def ladder_tuning(self) -> Tuple[bool, int]:
        """(on, number of tuning points passed with the tuning on)."""
        on, n = C.c_int32(0), C.c_int32(0)
        capi.check(self._lib.rfinv_pt_get_ladder_tuning(self.ev.handle, C.byref(on), C.byref(n)))
        return bool(on.value), int(n.value)

    # -- random-walk width tuning during the burn-in (DESIGN.md 7e) ----------------------------------------------------
    def set_step_tuning(self, on: bool, target: float = 0.44) -> None:
        """On top of set_rank_swaps(1), before the first iteration (and before restore()): at the iteration counts 64, 128,
        256, ... up to N_BURN every virtual rank scales the widths of the moves z, dVs, dVp and sigma of each of its levels
        towards the acceptance rate `target`.  The widths stay fixed after the burn-in.  Off is allowed between runs and
        returns the widths to the params.in values; set_rank_swaps(0) switches it off too."""
        capi.check(self._lib.rfinv_pt_set_step_tuning(self.ev.handle, int(on), float(target)))

    def step_tuning(self) -> Dict[str, object]:
        """{on, target, n_points, widths, n_prop, n_acc}: widths [local ranks][nchains][4] the absolute widths of the levels
        in the order z, dVs, dVp, sigma; n_prop / n_acc the same shape, the proposals and acceptances since the last tuning
        point (after the burn-in: those of the final widths)."""
        shape = (self.rank_count, self.cfg.nchains, 4)
        on, n, target = C.c_int32(0), C.c_int32(0), C.c_double(0.0)
        widths = np.zeros(shape); n_prop = np.zeros(shape, np.int64); n_acc = np.zeros(shape, np.int64)
        capi.check(self._lib.rfinv_pt_get_step_tuning(self.ev.handle, C.byref(on), C.byref(target), C.byref(n),
                                                      _p(widths, C.POINTER(C.c_double)), _p(n_prop, capi.i64p), _p(n_acc, capi.i64p)))
        return dict(on=bool(on.value), target=float(target.value), n_points=int(n.value), widths=widths, n_prop=n_prop,
                    n_acc=n_acc)

    # -- results ----------------------------------------------------------------------------------
    def set_logging(self, cap_iters: int) -> None:
        capi.check(self._lib.rfinv_pt_set_logging(self.ev.handle, int(cap_iters)))

    @property
    def iterations_done(self) -> int:
        return int(self._lib.rfinv_pt_iterations_done(self.ev.handle))

    def state(self) -> Dict[str, np.ndarray]:
        cfg, n = self.cfg, self.n_local
        out = dict(k=np.empty(n, dtype=np.int32), z=np.empty((n, cfg.k_max - 1)), dvp=np.empty((n, cfg.k_max)),
                   dvs=np.empty((n, cfg.k_max)), sig=np.empty((n, cfg.ntrc)), logl=np.empty(n), temps=np.empty(n))
        capi.check(self._lib.rfinv_pt_get_state(self.ev.handle, _p(out["k"], capi.i32p), _p(out["z"], capi.dp),
                                                _p(out["dvp"], capi.dp), _p(out["dvs"], capi.dp), _p(out["sig"], capi.dp),
                                                _p(out["logl"], capi.dp), _p(out["temps"], capi.dp)))
        return out

    def counters(self) -> Dict[str, np.ndarray]:
        n_it = self.iterations_done
        nprop = np.zeros(self.ntype, dtype=np.int64); nacc = np.zeros(self.ntype, dtype=np.int64)
        hist = np.zeros(max(n_it, 1)); n_eval = C.c_int64(0)
        capi.check(self._lib.rfinv_pt_get_counters(self.ev.handle, _p(nprop, capi.i64p), _p(nacc, capi.i64p),
                                                   _p(hist, capi.dp), n_it, C.byref(n_eval)))
        return dict(nprop=nprop, naccept=nacc, likelihood_hist=hist[:n_it], n_eval=n_eval.value)

    def hist(self) -> Dict[str, np.ndarray]:
        """Posterior bookkeeping of the local non-tempered chains (src/pt_mcmc.f90:204-286)."""
        c = self.cfg
        o = dict(nk=np.zeros(c.k_max, np.int64), nz=np.zeros(c.nbin_z, np.int64), nsig=np.zeros((c.ntrc, c.nbin_sig), np.int64),
                 namp=np.zeros((c.ntrc, c.nsmp, c.nbin_amp), np.int64), nvpz=np.zeros((c.nbin_vp, c.nbin_z), np.int64),
                 nvsz=np.zeros((c.nbin_vs, c.nbin_z), np.int64), nvpvsz=np.zeros((c.nbin_vpvs, c.nbin_z), np.int64),
                 vp_mean=np.zeros(c.nbin_z), vs_mean=np.zeros(c.nbin_z), vpvs_mean=np.zeros(c.nbin_z))
        nmod = C.c_int64(0)
        capi.check(self._lib.rfinv_pt_get_hist(self.ev.handle, C.byref(nmod), *[_p(o[n], capi.i64p) for n in
                                               ("nk", "nz", "nsig", "namp", "nvpz", "nvsz", "nvpvsz")],
                                               *[_p(o[n], capi.dp) for n in ("vp_mean", "vs_mean", "vpvs_mean")]))
        o["nmod"] = int(nmod.value)
        return o

    def models(self):
        """Recorded models of the local non-tempered chains: (vp_model, vs_model) [n_models][nbin_z] (all_models)."""
        cap = max(1, (self.cfg.niter // max(self.cfg.ncorr, 1)) * self.n_local * self.world)   # job-wide after reduce_outputs()
        vp = np.zeros((cap, self.cfg.nbin_z)); vs = np.zeros((cap, self.cfg.nbin_z))
        n = C.c_int64(0)
        capi.check(self._lib.rfinv_pt_get_models(self.ev.handle, cap, _p(vp, capi.dp), _p(vs, capi.dp), C.byref(n)))
        return vp[:n.value], vs[:n.value]

    def log(self, cap_iters: int):
        flags = np.zeros((cap_iters, self.n_local), dtype=np.int8)
        itypes = np.zeros((cap_iters, self.n_local), dtype=np.int8)
        swaps = np.zeros((cap_iters, 3), dtype=np.int32)
        n = C.c_int32(0)
        capi.check(self._lib.rfinv_pt_get_log(self.ev.handle, _p(flags, capi.i8p), _p(itypes, capi.i8p),
                                              _p(swaps, capi.i32p), C.byref(n)))
        return flags[:n.value], itypes[:n.value], swaps[:n.value]


class PtGroup:
    """Several single-process runs (one per station) advanced together on one GPU: ``PtGroup([pt_a, pt_b, ...]).run(n)``
    leaves every member with the bits ``member.run(n)`` alone would give, in one graph launch per iteration for all of them
    (rfinv_pt_group_run).  The members stay usable on their own between group runs."""

    def __init__(self, pts):
        self._g = None
        self.pts = list(pts)                          # keeps the handles alive as long as the group
        if not self.pts:
            raise ValueError("a group needs at least one ParallelTempering")
        self._lib = self.pts[0]._lib
        handles = (C.c_void_p * len(self.pts))(*[p.ev.handle for p in self.pts])
        g = C.c_void_p()
        capi.check(self._lib.rfinv_pt_group_create(C.cast(handles, C.POINTER(C.c_void_p)), len(self.pts), C.byref(g)))
        self._g = g

    def run(self, n_iter: int) -> None:
        if self._g is None:
            raise RuntimeError("the group is closed")
        capi.check(self._lib.rfinv_pt_group_run(self._g, int(n_iter)))

    def close(self) -> None:
        if self._g is not None:
            self._lib.rfinv_pt_group_destroy(self._g)
            self._g = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def build_table(temps, logl, peeks, pair=(-1, -1)) -> np.ndarray:
    """Host-side layout of one process's swap table (what pt_finish_kernel / pt_propose_kernel write)."""
    return np.concatenate([np.asarray(temps, dtype=np.float64), np.asarray(logl, dtype=np.float64),
                           np.asarray(peeks, dtype=np.float64), np.asarray(pair, dtype=np.float64)])


def decode_swap(gathered: np.ndarray, world: int, n_local: int, ranks_local: int, nchains: int):
    """Host mirror of pt_swap_kernel (judge_pt, src/pt_mcmc.f90:580-595) on the gathered tables; used by the
    CPU (gloo) tests of the exchange protocol and for diagnostics.  Returns (itarget1, itarget2, accepted,
    owner1, local1, owner2, local2)."""
    import math
    tl = 2 * n_local + ranks_local + 2
    tabs = np.asarray(gathered, dtype=np.float64).reshape(world, tl)
    i1, i2 = int(tabs[0, 2 * n_local + ranks_local]), int(tabs[0, 2 * n_local + ranks_local + 1])
    own1, l1 = divmod(i1, n_local)
    own2, l2 = divmod(i2, n_local)
    temp1, temp2 = tabs[own1, l1], tabs[own2, l2]
    e1, e2 = tabs[own1, n_local + l1], tabs[own2, n_local + l2]
    u = tabs[own1, 2 * n_local + l1 // nchains]
    del_s = (e2 - e1) * (1.0 / temp1 - 1.0 / temp2)
    yn = (math.log(u) if u > 0.0 else -math.inf) <= del_s
    return i1, i2, bool(yn), own1, l1, own2, l2


def _tensor_from_ptr(torch, ptr: int, n: int, dev):
    """float64 torch view of `n` doubles of device memory owned by the library (no copy)."""
    class _Holder:
        pass
    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(h, device=dev)
