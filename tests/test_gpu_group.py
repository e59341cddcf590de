"""Several PT runs advanced together on one GPU (rfinv_pt_group_*, rf_inv_b200.pt.PtGroup, the multi-station driver): after
a group run every member holds exactly the bits a solo rfinv_pt_run of the same length gives -- chain state, counters,
evaluations, likelihood history, histograms, recorded models and the per-iteration logs; the profile means agree to 1e-12
(fp64 atomics, as in tests/test_gpu_checkpoint.py)."""
import copy
import ctypes as C
import filecmp
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import helpers
from rf_inv_b200 import capi
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering, PtGroup
from test_gpu_checkpoint import assert_identical, snapshot, variant_config
from test_group_driver import station_dirs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = ["sample_bookkeeping", "sigma_solved_vp_solved", "laplace_prior_joint_PS", "transform_length_250",
            "single_chain_per_rank"]
N = 90
OUTPUT_FILES = ["params.in.copy", "all_models", "likelihood", "num_interface.ppd", "syn_trace.ppd", "interface_depth.ppd",
                "sigma.ppd", "vs_z.ppd", "vp_z.ppd", "vpvs_z.ppd", "vs_z.mean", "vp_z.mean", "vpvs_z.mean"]


def member_config(name):
    """The checkpoint tests' variant with the iteration counts every member of a group shares."""
    cfg, nproc, _, _ = variant_config(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter, cfg.ncorr = 30, 60, 4
    return cfg, nproc


def solo(cfg, nproc, n):
    pt = ParallelTempering(cfg, nproc)
    try:
        pt.set_logging(n)
        pt.run(n)
        return snapshot(pt), pt.log(n)
    finally:
        pt.close()


@pytest.fixture(scope="module")
def members():
    """(cfg, nproc, solo snapshot after N, solo logs of N) of the five variants: several nfft, k_max, ntrc and nchains."""
    out = []
    for name in VARIANTS:
        cfg, nproc = member_config(name)
        ref, logs = solo(cfg, nproc, N)
        out.append((cfg, nproc, ref, logs))
    return out


def open_members(members, logging=N):
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc, _, _ in members]
    for pt in pts:
        if logging:
            pt.set_logging(logging)
    return pts


def check(pts, members, log_from=None):
    """Every member equals its solo run of N iterations; its logs cover iterations log_from[i]..N."""
    for i, (pt, (_, _, ref, ref_logs)) in enumerate(zip(pts, members)):
        assert pt.iterations_done == N
        assert_identical(snapshot(pt), ref)
        start = 0 if log_from is None else log_from[i]
        for mine, whole in zip(pt.log(N), ref_logs):
            assert np.array_equal(mine, whole[start:]), i


def close_all(pts):
    for pt in pts:
        pt.close()


def test_group_equals_solo_runs(members):
    ref0 = members[0][2]
    assert ref0["hist_nmod"] > 0 and len(ref0["vp_model"]) == ref0["hist_nmod"]
    pts = open_members(members)
    try:
        with PtGroup(pts) as g:
            g.run(17)
            g.run(N - 17)
        check(pts, members)
    finally:
        close_all(pts)


def test_member_order_does_not_matter(members):
    rev = members[::-1]
    pts = open_members(rev)
    try:
        with PtGroup(pts) as g:
            g.run(N)
        check(pts, rev)
    finally:
        close_all(pts)


def test_group_and_solo_runs_mix(members):
    pts = open_members(members)
    try:
        with PtGroup(pts) as g:
            g.run(20)
            pts[0].set_logging(N - 20)               # drops member 0's graphs (new log buffers)
            pts[0].run(10)
            with pytest.raises(capi.RfinvError) as e:
                g.run(5)
            assert e.value.status == capi.RFINV_ERR_STATE and "member 1" in str(e.value), str(e.value)
            assert all(pt.iterations_done == 20 for pt in pts[1:])
            for pt in pts[1:]:
                pt.run(10)
            g.run(N - 30)
        check(pts, members, log_from=[20] + [0] * (len(pts) - 1))
    finally:
        close_all(pts)


def test_group_checkpoint_and_resume(members, tmp_path):
    pts = open_members(members, logging=0)
    try:
        with PtGroup(pts) as g:
            g.run(40)
        for i, pt in enumerate(pts):
            pt.save(str(tmp_path / f"ck.{i}"))
    finally:
        close_all(pts)
    pts = open_members(members, logging=0)
    try:
        for i, pt in enumerate(pts):
            pt.restore(str(tmp_path / f"ck.{i}"))
            pt.set_logging(N - 40)
        with PtGroup(pts) as g:
            g.run(N - 40)
        check(pts, members, log_from=[40] * len(pts))
    finally:
        close_all(pts)


def test_shared_memory_limits_of_differently_shaped_members():
    """Two members of one nfft whose kernels need different amounts of shared memory (k_max 30 and 8): whichever handle sets
    its launch up last must not lower the limit below what the other's captured graph launches with."""
    cfgs = []
    for k_max, seed in ((30, 11), (8, 12)):
        c = helpers.small_config(k_max=k_max, nchains=4, ncool=1, t_high=8.0, iseed=seed)
        c.nburn, c.niter, c.ncorr = 10, 40, 4
        cfgs.append(helpers.attach_obs_and_rinv(c, noise=0.01))
    big, small = (ParallelTempering(c, 4) for c in cfgs)
    try:
        big.run(10)          # captures the large member's graph
        small.run(20)        # sets the small member's launches up
        big.run(10)          # replays the large member's graph
        with PtGroup([big, small]) as g:
            g.run(30)
        got = [snapshot(big), snapshot(small)]
    finally:
        big.close(); small.close()
    for c, mine in zip(cfgs, got):
        ref, _ = solo(c, 4, 50)
        assert_identical(mine, ref)


def test_group_refusals(members):
    lib = capi.load()
    cfg, nproc, _, _ = members[0]
    cfg4, nproc4, _, _ = members[4]

    def create(handles):
        arr = (C.c_void_p * len(handles))(*handles)
        g = C.c_void_p()
        st = lib.rfinv_pt_group_create(C.cast(arr, C.POINTER(C.c_void_p)), len(handles), C.byref(g))
        if st == capi.RFINV_OK:
            lib.rfinv_pt_group_destroy(g)
        return st, lib.rfinv_last_error().decode()

    a, b = ParallelTempering(cfg, nproc), ParallelTempering(cfg4, nproc4)
    try:
        ha, hb = a.ev.handle.value, b.ev.handle.value
        assert create([ha, hb])[0] == capi.RFINV_OK
        st, msg = create([ha, None])
        assert st == capi.RFINV_ERR_ARG and "member 1" in msg, msg
        st, msg = create([ha, hb, ha])
        assert st == capi.RFINV_ERR_ARG and "member 2" in msg, msg
        with Evaluator(cfg) as ev:                                      # no rfinv_pt_init
            st, msg = create([ha, ev.handle.value])
            assert st == capi.RFINV_ERR_STATE and "member 1" in msg, msg
        half = ParallelTempering(cfg, nproc, world=2, rank=0)          # a distributed layout
        try:
            st, msg = create([ha, hb, half.ev.handle.value])
            assert st == capi.RFINV_ERR_STATE and "member 2" in msg, msg
        finally:
            half.close()
        if int(lib.rfinv_device_count()) >= 2:
            other = ParallelTempering(cfg4, nproc4, device=1)
            try:
                st, msg = create([ha, other.ev.handle.value])
                assert st == capi.RFINV_ERR_ARG and "member 1" in msg and "device" in msg, msg
            finally:
                other.close()

        def refused_run(pts, idx, word):
            with PtGroup(pts) as g:
                with pytest.raises(capi.RfinvError) as e:
                    g.run(3)
            assert e.value.status == capi.RFINV_ERR_STATE, str(e.value)
            assert f"member {idx}" in str(e.value) and word in str(e.value), str(e.value)
            assert all(pt.iterations_done == pts[0].iterations_done or pt is pts[idx] for pt in pts)

        for name, value in (("nburn", 31), ("ncorr", 5)):
            c = copy.deepcopy(cfg4); setattr(c, name, value)
            odd = ParallelTempering(c, nproc4)
            try:
                refused_run([a, b, odd], 2, "ncorr")
            finally:
                odd.close()
        a.run(1)
        refused_run([b, a], 1, "iterations done")
        b.run(1)
        capi.check(lib.rfinv_pt_local_step(b.ev.handle))                # half an iteration
        refused_run([a, b], 1, "local_step")
        ptr, _ = b.swap_table()
        capi.check(lib.rfinv_pt_apply_swap(b.ev.handle, ptr, 1))       # b's iteration is complete again
        a.run(1)
        with PtGroup([a, b]) as g:
            g.run(2)
        b.reduce_outputs()
        refused_run([a, b], 1, "reduce_outputs")
    finally:
        a.close(); b.close()


_NO_GRAPH_SCRIPT = r"""
import sys
sys.path[:0] = [{tests!r}, {root!r}, {oracle!r}]
from test_gpu_checkpoint import assert_identical, snapshot
from test_gpu_group import member_config
from rf_inv_b200.pt import ParallelTempering, PtGroup
ms = [member_config(n) for n in ("sample_bookkeeping", "transform_length_250", "single_chain_per_rank")]
refs = []
for cfg, nproc in ms:
    pt = ParallelTempering(cfg, nproc); pt.run(45); refs.append(snapshot(pt)); pt.close()
pts = [ParallelTempering(cfg, nproc) for cfg, nproc in ms]
with PtGroup(pts) as g:
    g.run(20); g.run(25)
for pt, ref in zip(pts, refs):
    assert_identical(snapshot(pt), ref)
    pt.close()
print("GROUP_NO_GRAPH_OK")
"""


def test_group_without_graphs_equals_solo_runs():
    env = dict(os.environ, RFINV_PT_GRAPH="0")
    script = _NO_GRAPH_SCRIPT.format(tests=os.path.join(ROOT, "tests"), root=ROOT, oracle=os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "GROUP_NO_GRAPH_OK" in r.stdout, r.stderr[-3000:]


def _solo_outputs(paths, tmp_path):
    """Each station run alone (rf_inv_b200.run.run) in a copy of its directory: the output directories."""
    from rf_inv_b200 import run as rrun
    outs = []
    for i, p in enumerate(paths):
        d = tmp_path / f"solo{i}"
        shutil.copytree(os.path.dirname(p), d)
        rrun.run(str(d / "params.in"), nproc=4, verbose=False)
        outs.append(d / "rslt")
    return outs


def _assert_same_files(paths, solo_outs):
    for p, ref in zip(paths, solo_outs):
        got = os.path.join(os.path.dirname(p), "rslt")
        for n in OUTPUT_FILES:
            assert filecmp.cmp(os.path.join(got, n), ref / n, shallow=False), (p, n)
        assert os.path.getsize(ref / "all_models") > 0


@pytest.fixture(scope="module")
def stations(tmp_path_factory):
    base = tmp_path_factory.mktemp("stations")
    paths = station_dirs(base / "src", 4, noise=0.01)
    return paths, _solo_outputs(paths, base)


def _copy_stations(paths, dst):
    out = []
    for p in paths:
        d = dst / os.path.basename(os.path.dirname(p))
        shutil.copytree(os.path.dirname(p), d)
        out.append(str(d / "params.in"))
    return out


def test_driver_group_writes_the_files_of_solo_runs(stations, tmp_path):
    from rf_inv_b200 import run as rrun
    paths, solo_outs = stations
    mine = _copy_stations(paths[:3], tmp_path)
    rrun.main(mine + ["--nproc", "4"])
    _assert_same_files(mine, solo_outs[:3])


def test_driver_group_checkpoint_resume_writes_the_files_of_solo_runs(stations, tmp_path):
    from rf_inv_b200 import run as rrun
    paths, solo_outs = stations
    mine = _copy_stations(paths[:3], tmp_path)
    ck = str(tmp_path / "state.ck")
    # a missing checkpoint starts a fresh run; the second call continues the first (N_BURN + N_ITER = 160)
    rrun.run_group(mine, 4, verbose=False, n_iter=70, checkpoint=ck, resume=True)
    assert all(os.path.exists(f"{ck}.{i}") for i in range(3))
    rrun.run_group(mine, 4, verbose=False, checkpoint=ck, resume=True)
    _assert_same_files(mine, solo_outs[:3])
    # the files of another order do not fit: the configuration fingerprints refuse the restore
    with pytest.raises(capi.RfinvError):
        rrun.run_group([mine[1], mine[0], mine[2]], 4, verbose=False, checkpoint=ck, resume=True)


def test_driver_group_under_torchrun_on_two_gpus(stations, tmp_path):
    if int(capi.load().rfinv_device_count()) < 2:
        pytest.skip("needs two GPUs")
    paths, solo_outs = stations
    mine = _copy_stations(paths, tmp_path)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", "-m", "rf_inv_b200.run"] + mine + ["--nproc", "4"]
    r = subprocess.run(cmd, env=dict(os.environ, MASTER_ADDR="127.0.0.1"), capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    _assert_same_files(mine, solo_outs)
