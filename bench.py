#!/usr/bin/env python
"""bench.py -- forward+likelihood evaluations per second on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload target|c2|c3|c3_buried|c4|c5|sample] [--chains C]
    python bench.py --impl reference ...      # the CPU restatement of the reference algorithm on the host cores
    python bench.py --dump-outputs DIR ...    # also writes the logL of the last timed step as DIR/logl.npy

A step = one pass of the hot path (format_model -> propagator -> filter/FFT -> misfit -> correlated-noise
likelihood) over one batch of `--chains` models per GPU.  `value` is measured with the models resident in HBM
(rfinv_eval_batch_device); `e2e` goes through the C-ABI with HOST buffers, H2D/D2H copies in the timed region:
`e2e.value` with two half-batches in flight (rfinv_eval_batch_begin / _end: the transfers of one hide behind the kernels of
the other), `e2e.sync_value` with one blocking rfinv_eval_batch call per step, `e2e.with_rft_value` with the complete RF
returned.  One process per GPU (torchrun); chains shard across ranks with no data-path collective (weak scaling).
The other workloads BASELINE.json names ride along as sub-keys (`configs`), together with a sustained leg, a layer-count
sweep and the parallel-tempering leg (in-library ncclAllGather per iteration; identity with the single-process run checked).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from rf_inv_b200 import workloads  # noqa: E402

METRIC = "forward+likelihood evals/sec"
UNIT = "evals/s"
# models per GPU and step.  Target shape: 32 768 -- the three kernels of a step are persistent, dynamically scheduled grids whose ramp and
# tail are paid once per launch (measured on one B200: 4096 models 10.25, 8192 11.73, 16 384 12.53, 32 768 12.90, 65 536 13.15 M evals/s;
# DESIGN.md section 6); round 1 and the first half of round 2 quoted 16 384.
DEFAULT_CHAINS = {"target": 32768, "c2": 4096, "c3": 8192, "c3_buried": 8192, "c4": 16384, "c5": 65536, "sample": 4096}
# chains per GPU of the PT-MCMC leg of the primary workload (iterations/s depend on the chain count: kept at round 1's figure)
PT_CHAINS = {"target": 16384}
# totals that BASELINE.json fixes for the whole job (strong scaling: chains per GPU = total / N); the others are per GPU
FIXED_TOTAL = {"c4": 16384, "c5": 65536}
SIDE_CONFIGS = ["sample", "c2", "c3", "c3_buried", "c4", "c5"]


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="target")
    ap.add_argument("--chains", type=int, default=0, help="models per GPU per step")
    ap.add_argument("--cpu-sample", type=int, default=0, help="models in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pt-iters", type=int, default=200, help="timed PT-MCMC iterations (0 = skip the PT leg)")
    ap.add_argument("--no-configs", action="store_true", help="skip the side workloads (configs sub-keys), sustained leg and k sweep")
    ap.add_argument("--sustain-s", type=float, default=2.5, help="seconds of back-to-back steps in the sustained leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step (logL per model, float64) as DIR/logl.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy.  Above DUMP_LIMIT bytes in all, each keeps the same fixed, evenly spaced
    subset of its models, so that two runs with the same arguments still compare entry for entry."""
    stride = -(-sum(a.nbytes for a in arrays.values()) // DUMP_LIMIT)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[::stride])


def workload_desc(cfg, name, chains, k_mean):
    return {"workload": name, "nfft": cfg.nfft, "k_max": cfg.k_max, "ntrc": cfg.ntrc, "nsmp": cfg.nsmp,
            "rays": "common" if cfg.is_ray_common else "distinct", "sea_layer": cfg.sdep > 0,
            "chains_per_gpu": chains, "k_mean": round(float(k_mean), 2),
            "models": "k uniform on [k_min,k_max), interfaces uniform, dVs ~ N(0,0.3): as init_model draws them",
            "l2": "flushed between timed steps (256 MiB write); e2e pipelined and sustained legs: working set of a step "
                  "(misfit rows + layer constants, > 0.4 GB) exceeds L2, no explicit flush"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        sm, reasons, mx, pw = [], set(), None, []
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1]); pw.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        hi = [s for s in sm if s > 0.5 * (max(sm) if sm else 1)]
        return {"sm_mhz": float(np.median(hi)) if hi else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(pw) if pw else None}


def make_inputs(cfg, chains, seed, k_fixed=None):
    return workloads.draw_models(cfg, chains, seed=seed, dvs_scale=0.3, k_fixed=k_fixed)


def attach_obs(cfg):
    """Observed traces = forward of the data-generating model + noise, rounded to float32 like a SAC file.  The forward is
    the C restatement's (oracle/), so the inputs of a run do not depend on the build of the library being measured."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c
    tm = workloads.true_model(cfg)
    cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp))
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    _, rft, _ = oracle_c.eval_batch(cfg, tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"])
    obs = rft[0, :, :cfg.nsmp] + np.random.default_rng(7).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))
    cfg.obs = obs.astype(np.float32).astype(np.float64)
    return cfg


def host_cores():
    """Host threads the CPU arm uses: every core this process may run on (torchrun exports OMP_NUM_THREADS=1 to its
    workers, which must not throttle the CPU baseline)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_sample_size(cfg, models, target_s, cap):
    """Number of models that keep one CPU pass near `target_s` seconds (calibrated on a 64-model probe)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c
    cores = host_cores()
    probe = min(max(4 * cores, 64), cap)
    sub = {k: v[:probe] for k, v in models.items()}
    oracle_c.eval_batch(cfg, sub["k"], sub["z"], sub["dvp"], sub["dvs"], sub["sig"], want_rft=False, nthreads=cores)
    t0 = time.perf_counter()
    oracle_c.eval_batch(cfg, sub["k"], sub["z"], sub["dvp"], sub["dvs"], sub["sig"], want_rft=False, nthreads=cores)
    rate = probe / max(time.perf_counter() - t0, 1e-6)
    return int(min(cap, max(probe, rate * target_s)))


def cpu_arm(cfg, models, n_sample, steps, warmup):
    """Times the C restatement of the reference algorithm (oracle/) on all host cores: evals/s, cores, seconds per pass and
    the logL of the last pass."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c
    cores = host_cores()
    sub = {k: v[:n_sample] for k, v in models.items()}
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ll, _, _ = oracle_c.eval_batch(cfg, sub["k"], sub["z"], sub["dvp"], sub["dvs"], sub["sig"], want_rft=False, nthreads=cores)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return n_sample / float(np.mean(times)), cores, float(np.mean(times)), ll


def run_reference(args):
    """--impl reference: the reference's own CPU algorithm (C restatement; the Fortran/MPI/FFTW/LAPACK original cannot
    be compiled in this image) on the box's host cores, same config/metric.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = workloads.make_config(args.workload)
    chains = args.chains or DEFAULT_CHAINS.get(args.workload, 4096)
    sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers
    cfg = helpers.attach_obs_and_rinv(cfg, noise=0.01)
    cores = host_cores()
    steps, warmup = args.steps, max(1, min(args.warmup, 1))
    models = make_inputs(cfg, min(chains, 16384), seed=100)
    # bounded sample: about 20 s of CPU work over the whole --steps/--warmup run
    n_sample = args.cpu_sample or cpu_sample_size(cfg, models, 20.0 / (steps + warmup), len(models["k"]))
    models = {k: v[:n_sample] for k, v in models.items()}
    k_mean = float(np.mean(models["k"]))
    val, cores, sec, ll = cpu_arm(cfg, models, n_sample, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logl": ll})
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_desc(cfg, args.workload, chains, k_mean),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n_sample} models of the workload per step, OpenMP over models"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Leg:
    """One workload on this rank's GPU: device-resident inputs, pinned host copies, an Evaluator on torch's stream."""

    def __init__(self, torch, Evaluator, capi, cfg, chains, local_rank, seed, k_fixed=None):
        self.torch, self.capi, self.cfg, self.chains = torch, capi, cfg, chains
        self.dev = torch.device("cuda", local_rank)
        self.models = make_inputs(cfg, chains, seed=seed, k_fixed=k_fixed)
        self.k_mean = float(np.mean(self.models["k"]))
        soa = workloads.to_soa(self.models)
        self.d = {k: torch.from_numpy(v).to(self.dev) for k, v in soa.items()}
        self.logl = torch.empty(chains, dtype=torch.float64, device=self.dev)
        self.ev = Evaluator(cfg, device=local_rank)
        self.stream = torch.cuda.current_stream()
        self.ev.set_stream(self.stream.cuda_stream)
        self.lib = capi.load()
        self._pin = None

    def close(self):
        self.ev.close()

    def step_device(self):
        d = self.d
        self.ev.calc_likelihood_device(self.chains, d["k"].data_ptr(), d["z"].data_ptr(), d["dvp"].data_ptr(), d["dvs"].data_ptr(),
                                       d["sig"].data_ptr(), self.logl.data_ptr())

    def time_device(self, steps, warmup, flush):
        """CUDA-event time of every step (no events between the kernels of a step), L2 flushed before each."""
        torch = self.torch
        self.capi.check(self.lib.rfinv_set_timing(self.ev.handle, 0))
        for _ in range(warmup):
            self.step_device()
        torch.cuda.synchronize()
        ms, launches = [], 0
        for _ in range(steps):
            if flush is not None:
                flush.fill_(1)                   # evict L2 between timed steps (outside the per-step events)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(self.stream)
            self.step_device()
            e1.record(self.stream)
            e1.synchronize()
            ms.append(e0.elapsed_time(e1))
            launches += self.ev.last_launch_count
        return ms, launches

    def kernel_split(self, steps, flush):
        """Per-kernel CUDA-event times (events between the kernels: a separate pass, not the one `value` comes from)."""
        self.capi.check(self.lib.rfinv_set_timing(self.ev.handle, 1))
        out = []
        for _ in range(steps):
            if flush is not None:
                flush.fill_(1)
            self.step_device()
            t3 = (C.c_double * 3)()
            self.capi.check(self.lib.rfinv_get_timing(self.ev.handle, t3))
            out.append([t3[0], t3[1]])
        self.capi.check(self.lib.rfinv_set_timing(self.ev.handle, 0))
        return np.mean(np.array(out), axis=0)

    def sustained(self, seconds):
        """Back-to-back steps for `seconds` (no flush: the working set of a step exceeds L2): evals/s and the step count."""
        torch = self.torch
        self.step_device(); torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        n = 0
        t0 = time.perf_counter()
        e0.record(self.stream)
        while time.perf_counter() - t0 < seconds:
            for _ in range(20):
                self.step_device()
            n += 20
            torch.cuda.synchronize()          # keeps the launch queue short; < 1 % of 20 steps
        e1.record(self.stream)
        e1.synchronize()
        return n, e0.elapsed_time(e1)

    def pin(self):
        if self._pin is None:
            torch = self.torch
            self._pin = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory().numpy() for k, v in self.models.items()}
        return self._pin

    def h2d_bytes(self):
        return sum(v.nbytes for k, v in self.pin().items() if not (k == "dvp" and self.cfg.vp_mode == 0))

    def time_e2e_sync(self, steps, flush, want_rft=False):
        p = self.pin()
        for _ in range(2):
            out = self.ev.calc_likelihood(p["k"], p["z"], p["dvp"], p["dvs"], p["sig"], want_rft=want_rft)
        self.torch.cuda.synchronize()
        ts = []
        for _ in range(steps):
            if flush is not None:
                flush.fill_(1)
            self.torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = self.ev.calc_likelihood(p["k"], p["z"], p["dvp"], p["dvs"], p["sig"], want_rft=want_rft)
            ts.append(time.perf_counter() - t0)
        return float(np.sum(ts)), out[0]

    def time_e2e_pipelined(self, steps):
        """Two half-batches in flight (rfinv_eval_batch_begin / _end): a host that keeps two groups of chains going, each
        group re-proposed as soon as its own results are back.  Wall time from the first _begin to the last _end."""
        torch = self.torch
        p = self.pin()
        h = self.chains // 2
        halves = [{k: v[:h] for k, v in p.items()}, {k: v[h:] for k, v in p.items()}]
        outs = [torch.empty(x["k"].shape[0], dtype=torch.float64).pin_memory().numpy() for x in halves]

        def begin(s):
            x = halves[s]
            self.ev.calc_likelihood_begin(s, x["k"], x["z"], x["dvp"], x["dvs"], x["sig"], outs[s])

        for _ in range(2):                     # warm-up: buffers of both slots
            begin(0); begin(1); self.ev.calc_likelihood_end(0); self.ev.calc_likelihood_end(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        begin(0); begin(1)
        for _ in range(steps - 1):
            self.ev.calc_likelihood_end(0); begin(0)
            self.ev.calc_likelihood_end(1); begin(1)
        self.ev.calc_likelihood_end(0); self.ev.calc_likelihood_end(1)
        return time.perf_counter() - t0, np.concatenate(outs)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from rf_inv_b200 import capi
    from rf_inv_b200.evaluator import Evaluator

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; rf_inv_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL announces its version on stdout when the communicator is created (NCCL_DEBUG=VERSION in this image); rank 0's
        # stdout must carry the one JSON line and nothing else, so stdout points at stderr until the run is over
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
        torch.cuda.synchronize()
    dev = torch.device("cuda", local_rank)
    lib = capi.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ================= primary workload =================
    cfg = attach_obs(workloads.make_config(args.workload))
    chains = args.chains or (FIXED_TOTAL[args.workload] // world if args.workload in FIXED_TOTAL else DEFAULT_CHAINS.get(args.workload, 4096))
    leg = Leg(torch, Evaluator, capi, cfg, chains, local_rank, seed=100 + rank)
    steps, warmup = args.steps, max(args.warmup, 3)

    # ---- device-resident arm (value) ----
    leg.time_device(0, warmup, None)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    t_wall0 = time.perf_counter()
    step_ms, launches = leg.time_device(steps, 0, flush)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    total_ms = allmax(float(np.sum(step_ms)))
    value = world * chains * steps / (total_ms * 1e-3)
    out_logl = None
    if args.dump_outputs:
        # the logL every step writes into leg.logl, as the last timed step left it (the passes below write it again)
        out_logl = leg.logl
        if world > 1:
            out_logl = torch.empty(world * chains, dtype=torch.float64, device=dev)
            dist.all_gather_into_tensor(out_logl, leg.logl)
        out_logl = out_logl.cpu().numpy()
    km = leg.kernel_split(5, flush)          # [prep + forward, quadratic form + logL] ms, separate pass

    # ---- end-to-end arms: host buffers through the C-ABI calls a Fortran host would make ----
    barrier()
    sync_total, ll_host = leg.time_e2e_sync(steps, flush)
    sync_total = allmax(sync_total)
    assert np.array_equal(ll_host, leg.logl.cpu().numpy()), "host and device entry points disagree"
    barrier()
    pipe_total, ll_pipe = leg.time_e2e_pipelined(steps)
    pipe_total = allmax(pipe_total)
    assert np.array_equal(ll_pipe, ll_host), "asynchronous and synchronous entry points disagree"
    e2e = {"value": world * chains * steps / pipe_total, "unit": UNIT, "h2d_bytes_per_step": int(leg.h2d_bytes()),
           "d2h_bytes_per_step": int(8 * chains),
           "how": "two half-batches in flight through rfinv_eval_batch_begin/_end (pinned host arrays, logL back per half); "
                  "wall time from the first _begin to the last _end of `steps` full batches",
           "sync_value": world * chains * steps / sync_total,
           "sync_how": "one blocking rfinv_eval_batch per step (upload in 4 pieces overlapped with prep_kernel), logL only"}
    if not args.no_configs:
        barrier()
        rft_total, _ = leg.time_e2e_sync(3, flush, want_rft=True)
        rft_total = allmax(rft_total)
        e2e["with_rft_value"] = world * chains * 3 / rft_total
        e2e["with_rft_d2h_bytes_per_step"] = int(8 * chains * (1 + cfg.ntrc * cfg.nfft))
        e2e["with_rft_how"] = "blocking rfinv_eval_batch returning the reference's prop_rft(nfft, ntrc) of every model as well"

    # ---- sustained leg: seconds of back-to-back steps, with its own clock record ----
    sustained = None
    k_sweep = None
    if not args.no_configs:
        barrier()
        s2 = ClockSampler(local_rank); s2.start(); time.sleep(0.2)
        n_s, ms_s = leg.sustained(args.sustain_s)
        c2 = s2.stop()
        ms_s = allmax(ms_s)
        sustained = {"value": allsum(n_s * chains) / (ms_s * 1e-3), "unit": UNIT, "steps": n_s, "seconds": ms_s * 1e-3,
                     "ms_per_step": ms_s / n_s, "clocks": c2}
        # ---- layer-count sweep on the same shape: every model with k = 15 / k = 29 interfaces ----
        k_sweep = {}
        for kf in (15, 29):
            lk = Leg(torch, Evaluator, capi, cfg, chains, local_rank, seed=300 + rank, k_fixed=kf)
            lk.time_device(0, 3, None)
            ms_k, _ = lk.time_device(10, 0, flush)
            tk = allmax(float(np.sum(ms_k)))
            fl = workloads.flops_per_eval(cfg, float(kf))
            k_sweep[f"k{kf}"] = {"value": world * chains * 10 / (tk * 1e-3), "unit": UNIT, "ms_per_step": tk / 10,
                                 "algorithmic_flop_per_eval_dense_quadform": fl["total"]}
            lk.close()

    # ---- PT-MCMC leg: iterations/s of pt_control with every chain on device (second half of BASELINE.json's metric) ----
    pt_info = None
    if args.pt_iters > 0:
        from rf_inv_b200.pt import ParallelTempering
        nch = cfg.nchains
        pt_chains = min(chains, PT_CHAINS.get(args.workload, chains)) if not args.chains else chains
        nproc_total = world * max(1, pt_chains // nch)
        pt = ParallelTempering(cfg, nproc_total, device=local_rank, world=world, rank=rank)
        pt.ev.set_stream(leg.stream.cuda_stream)
        if world > 1:
            pt.init_comm(dist, torch)

        def pt_iters(n):
            if world == 1:
                pt.run(n)
            else:
                pt.run_distributed(n)

        pt_iters(5)
        pt_exchange = pt.exchange_mode
        barrier()
        n_eval0 = pt.counters()["n_eval"]
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(leg.stream)
        pt_iters(args.pt_iters)
        e1.record(leg.stream)
        e1.synchronize()
        pt_ms = allmax(e0.elapsed_time(e1))
        n_eval = allsum(pt.counters()["n_eval"] - n_eval0)
        k_pt = float(np.mean(pt.state()["k"]))
        pt_info = {"iters_per_s": args.pt_iters / (pt_ms * 1e-3), "chain_steps_per_s": world * pt.n_local * args.pt_iters / (pt_ms * 1e-3),
                   "forward_evals_per_s": n_eval / (pt_ms * 1e-3), "iters": args.pt_iters, "chains_total": world * pt.n_local,
                   "virtual_ranks": nproc_total, "chains_per_rank": nch, "k_mean_after": round(k_pt, 2),
                   "launch": "one CUDA graph launch per iteration (rfinv_pt_run / rfinv_pt_run_distributed)",
                   "exchange": "none (single process)" if world == 1 else (
                       "peer memory: the pair and the (T, logL, next-uniform) table go into every process's buffers (CUDA IPC over NVLink) from "
                       "a side branch of the iteration's graph; the swap is applied one iteration later -- no collective call, no waiting"
                       if pt_exchange == "peer memory" else
                       "one ncclAllGather of the (T, logL, next-uniform) tables per iteration, issued by the library inside the iteration's graph")}
        pt.close()
        if not args.no_configs:
            # the same loop with chains as deep as the evaluation batch: a dVs prior of 0.3 km/s lets init_model keep models with
            # many interfaces (the configured prior of 2 km/s rejects them: k stays near 2.5 above)
            import copy
            dcfg = copy.copy(cfg)
            dcfg.dvs_prior = 0.3
            ptd = ParallelTempering(dcfg, nproc_total, device=local_rank, world=world, rank=rank)
            ptd.ev.set_stream(leg.stream.cuda_stream)
            if world > 1:
                ptd.init_comm(dist, torch)
            run_d = (lambda n: ptd.run(n)) if world == 1 else (lambda n: ptd.run_distributed(n))
            run_d(5)
            barrier()
            n0 = ptd.counters()["n_eval"]
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(leg.stream); run_d(100); e1.record(leg.stream); e1.synchronize()
            ms_d = allmax(e0.elapsed_time(e1))
            pt_info["deep_chains"] = {"iters_per_s": 100 / (ms_d * 1e-3), "forward_evals_per_s": allsum(ptd.counters()["n_eval"] - n0) / (ms_d * 1e-3),
                                      "k_mean_after": round(float(np.mean(ptd.state()["k"])), 2), "dvs_prior": 0.3, "iters": 100}
            ptd.close()
        if world > 1:
            # identity of the distributed run on the real NCCL path: 100 iterations, accept flags / proposal types / swaps /
            # final state of N processes == one process holding every virtual rank
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            from dist_check import identity_check
            icfg = workloads.make_config(args.workload)
            icfg.obs, icfg.r_inv = cfg.obs, cfg.r_inv
            ok, detail = identity_check(icfg, 4 * world, 100, world, rank, local_rank, dist, torch)
            pt_info["identity"] = bool(ok)
            pt_info["identity_detail"] = dict(detail, iterations=100, virtual_ranks=4 * world)

    # ================= the other named workloads, as sub-keys =================
    configs = {}
    if not args.no_configs:
        for name in SIDE_CONFIGS:
            if name == args.workload:
                continue
            c = attach_obs(workloads.make_config(name))
            fixed = name in FIXED_TOTAL
            n_c = FIXED_TOTAL[name] // world if fixed else DEFAULT_CHAINS[name]
            lc = Leg(torch, Evaluator, capi, c, n_c, local_rank, seed=500 + rank)
            st_c = 5
            lc.time_device(0, 3, None)
            barrier()
            ms_c, _ = lc.time_device(st_c, 0, flush)
            t_dev = allmax(float(np.sum(ms_c)))
            barrier()
            t_sync, _ = lc.time_e2e_sync(st_c, flush)
            t_sync = allmax(t_sync)
            barrier()
            t_pipe, _ = lc.time_e2e_pipelined(st_c)
            t_pipe = allmax(t_pipe)
            entry = {"value": world * n_c * st_c / (t_dev * 1e-3), "e2e_value": world * n_c * st_c / t_pipe,
                     "e2e_sync_value": world * n_c * st_c / t_sync, "unit": UNIT, "ms_per_step": t_dev / st_c, "steps": st_c,
                     "chains_per_gpu": n_c, "chains_total": world * n_c, "scaling": "strong" if fixed else "weak",
                     "k_mean": round(lc.k_mean, 2), "nfft": c.nfft, "ntrc": c.ntrc, "k_max": c.k_max}
            lc.close()
            if args.pt_iters > 0 and name != "c2":          # c2 has one chain per rank: nothing to temper
                from rf_inv_b200.pt import ParallelTempering
                n_it = 100
                nproc_total = world * max(1, n_c // c.nchains)
                ptc = ParallelTempering(c, nproc_total, device=local_rank, world=world, rank=rank)
                ptc.ev.set_stream(leg.stream.cuda_stream)
                if world > 1:
                    ptc.init_comm(dist, torch)
                run_c = (lambda n: ptc.run(n)) if world == 1 else (lambda n: ptc.run_distributed(n))
                run_c(5)
                barrier()
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(leg.stream); run_c(n_it); e1.record(leg.stream); e1.synchronize()
                ms_pt = allmax(e0.elapsed_time(e1))
                entry["pt_iters_per_s"] = n_it / (ms_pt * 1e-3)
                entry["pt_chain_steps_per_s"] = world * ptc.n_local * n_it / (ms_pt * 1e-3)
                entry["pt_k_mean_after"] = round(float(np.mean(ptc.state()["k"])), 2)
                ptc.close()
            configs[name] = entry

    if world > 1:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if rank == 0:
        # ---- roofline of the dominant kernel (forward_kernel): algorithmic fp64 flop / CUDA-event time ----
        dfma, dmma = C.c_double(0), C.c_double(0)
        capi.check(lib.rfinv_measure_fp64_peak(local_rank, C.byref(dfma), C.byref(dmma)))
        peak = max(dfma.value, dmma.value)
        k_mean = leg.k_mean
        fl = workloads.flops_per_eval(cfg, k_mean)
        # the quadratic form as the library evaluates it (chosen at rfinv_create): S^2 + 3S dense, 2 S r + 2 r factor form,
        # S r + S + 2 r split form (sums / differences of mirrored samples against the two half-length factors)
        form = leg.ev.quadform_form()
        S = cfg.nsmp
        fl["quadform_dense_form"] = fl["quadform"]
        fl["quadform"] = float(sum((S * r + S + 2 * r) if sp else ((2 * S * r + 2 * r) if r > 0 else (S * S + 3 * S)) for r, rs, sp in form))
        fl["quadform_form"] = [{"rank": r, "rank_sym": rs, "split": bool(sp)} for r, rs, sp in form]
        fl["total"] = fl["propagator"] + fl["fft"] + fl["quadform"]
        fwd_flop = (fl["propagator"] + fl["fft"]) * chains
        achieved = fwd_flop / (km[0] * 1e-3) * 1e-12
        qf_achieved = fl["quadform"] * chains / (km[1] * 1e-3) * 1e-12
        whole = fl["total"] * chains * steps / (float(np.sum(step_ms)) * 1e-3) * 1e-12
        # share of the FP64 pipe's issue slots the forward path fills (an FP64 instruction holds the pipe for the time of
        # one FMA whether or not it is one): instructions x 2 flop-slots / time / peak
        slot_frac = fl["forward_fp64_instructions"] * 2.0 * chains / (km[0] * 1e-3) * 1e-12 / peak
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "forward_kernel_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            if tj.get("workload") == args.workload and tj.get("chains") == chains:
                traffic = tj.get("dram_bytes_per_launch")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_desc(cfg, args.workload, chains, k_mean),
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "fp64", "kernel": "forward_kernel", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "fp64_issue_slot_frac": slot_frac,
                         "note": "FP64-pipe bound (arithmetic intensity > 100 flop/B, DRAM < 5% of peak): `achieved` = algorithmic "
                                 "flop of prep_kernel + forward_kernel / their CUDA-event time (a pass of its own with events between "
                                 "the kernels); `traffic` = ncu dram bytes of one forward_kernel launch at this shape "
                                 "(profiles/forward_kernel_traffic.json)",
                         "peak_source": "measured live: rfinv_measure_fp64_peak (max of DFMA %.1f / DMMA %.1f TFLOP/s); "
                                        "MEASURED_PEAKS.json has no FP64 figure" % (dfma.value, dmma.value),
                         "flop_per_eval": fl, "kernel_ms": {"forward": float(km[0]), "quadform": float(km[1])},
                         "quadform_tflops": qf_achieved, "whole_step_tflops": whole, "whole_step_frac": whole / peak},
            "wall_s_timed_region": t_wall,
            "pt": pt_info,
            "sustained": sustained,
            "k_sweep": k_sweep,
            "configs": configs,
        }
        if world == 1 and not args.no_cpu_baseline:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            n_sample = args.cpu_sample or cpu_sample_size(cfg, leg.models, 5.0, chains)   # ~15 s of CPU work in 3 passes
            val, cores, sec, _ = cpu_arm(cfg, leg.models, min(n_sample, chains), 2, 1)
            line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"first {min(n_sample, chains)} models of the same batch, {sec:.2f} s per pass, "
                                              "C restatement of the reference algorithm (OpenMP over models)"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"logl": out_logl})
        print(json.dumps(line), flush=True)
    leg.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
