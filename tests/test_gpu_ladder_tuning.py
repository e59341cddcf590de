"""Ladder tuning during the burn-in (rfinv_pt_set_ladder_tuning, DESIGN.md 7d) on the GPU: tuned runs reproduce the C reference
(tests/ladder_oracle.c) across several tuning points, and keep the identity guarantees of plain launches, split runs,
checkpoints, groups and two processes; the driver writes OUT_DIR/ladder."""
import copy
import filecmp
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import ladder_oracle as lo
from rf_inv_b200 import capi, workloads
from rf_inv_b200 import io as rio
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering, PtGroup
from test_gpu_checkpoint import assert_identical, snapshot, variant_config
from test_gpu_group import OUTPUT_FILES, member_config
from test_gpu_pt import check as check_against_oracle
from test_gpu_rank_swaps import VARIANTS, oracle_variant
from test_group_driver import set_param, station_dirs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def tuned_variant(name, nburn=300):
    """test_gpu_rank_swaps.py's variant with a burn-in holding the tuning points 64, 128 and 256, run through them."""
    cfg, nproc, _ = oracle_variant(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn = nburn
    return cfg, nproc, nburn


def _levels(temps, nchains):
    """Per rank, the chains by level: (temperature, chain index) order."""
    t = temps.reshape(-1, nchains)
    return np.lexsort((np.broadcast_to(np.arange(nchains), t.shape), t), axis=1)


def gpu_run(cfg, nproc, plan):
    """plan: [(mode, tune, iterations), ...] on one handle with logs of the whole run."""
    n = sum(k for _, _, k in plan)
    pt = ParallelTempering(cfg, nproc)
    try:
        pt.set_logging(n)
        st0 = pt.state()
        for mode, tune, k in plan:
            pt.set_rank_swaps(mode)
            if tune or pt.ladder_tuning()[0]:
                pt.set_ladder_tuning(tune)
            pt.run(k)
        flags, itypes, swaps = pt.log(n)
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=pt.state(), cnt=pt.counters(), rs=pt.rank_swaps(),
                    lt=pt.ladder_tuning())
    finally:
        pt.close()


def oracle_run(cfg, nproc, plan):
    orc = lo.LadderOraclePT(cfg, nproc)
    try:
        st0 = orc.state()
        logs = []
        for mode, tune, k in plan:
            orc.set_rank_swaps(mode)
            if tune or orc.tune:
                orc.set_ladder_tuning(tune)
            logs.append(orc.run(k))
        n = sum(k for _, _, k in plan)
        flags, itypes, swaps = (np.concatenate([l[i] for l in logs]) for i in range(3))
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=orc.state(), cnt=orc.counters(n), n_eval=orc.n_eval,
                    rs=orc.rank_swaps(), lt=orc.ladder_tuning())
    finally:
        orc.close()


def check(g, o, cfg):
    # decisions, counters and sweep counters exact; the state to 1e-12 and logL to 1e-9 (the initial temperatures are exp()
    # of the same draws on the device and in libm, so the tuned ladders agree to rounding)
    check_against_oracle(g, o, cfg)
    for key in ("mode", "n_prop", "n_acc"):
        assert np.array_equal(g["rs"][key], o["rs"][key]), key
    assert g["lt"] == o["lt"]
    assert np.array_equal(_levels(g["st"]["temps"], cfg.nchains), _levels(o["st"]["temps"], cfg.nchains))
    cold = 1.0 + lo.COLD_EPS
    assert np.array_equal(g["st"]["temps"] <= cold, o["st"]["temps"] <= cold)


@pytest.mark.parametrize("variant", VARIANTS)
def test_tuned_run_matches_oracle(variant):
    cfg, nproc, n = tuned_variant(variant)
    g = gpu_run(cfg, nproc, [(1, 1, n)])
    check(g, oracle_run(cfg, nproc, [(1, 1, n)]), cfg)
    assert g["lt"] == (True, 3)
    if cfg.nchains >= 3:            # the ladders moved: the multiset of temperatures is no longer the initial one
        assert not np.allclose(np.sort(g["st"]["temps"]), np.sort(g["st0"]["temps"]), rtol=1e-9)


def test_rank_swaps_off_switches_tuning_off_and_matches_oracle():
    cfg, nproc, _ = tuned_variant("sigma_solved_vp_solved")
    plan = [(1, 1, 100), (0, 0, 60), (1, 0, 100)]     # tuned through 64, then the reference, then the sweep without tuning
    g = gpu_run(cfg, nproc, plan)
    assert g["lt"] == (False, 1)
    check(g, oracle_run(cfg, nproc, plan), cfg)


def test_short_burn_in_equals_mode1():
    cfg, nproc, _ = tuned_variant("laplace_prior_joint_PS", nburn=63)
    a, b = gpu_run(cfg, nproc, [(1, 1, 150)]), gpu_run(cfg, nproc, [(1, 0, 150)])
    for key in ("flags", "itypes", "swaps"):
        assert np.array_equal(a[key], b[key]), key
    for key in a["st"]:
        assert np.array_equal(a["st"][key], b["st"][key]), key
    assert a["lt"] == (True, 0)


# ---- launch paths ----
def _cfg(name, nburn, niter=60, ncorr=4):
    cfg, nproc, _, _ = variant_config(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter, cfg.ncorr = nburn, niter, ncorr
    return cfg, nproc


def _snap(pt):
    out = snapshot(pt)
    rs = pt.rank_swaps()
    on, n_points = pt.ladder_tuning()
    out.update(rs_n_prop=rs["n_prop"], rs_n_acc=rs["n_acc"], lt_on=np.int64(on), lt_points=np.int64(n_points))
    return out


def _tuned(cfg, nproc):
    pt = ParallelTempering(cfg, nproc)
    pt.set_rank_swaps(1)
    pt.set_ladder_tuning(1)
    return pt


def fingerprint(name, nburn, n):
    """sha1 over logs, state, counters and sweep counters of a tuned run (bookkeeping on after nburn)."""
    import hashlib
    cfg, nproc = _cfg(name, nburn)
    pt = _tuned(cfg, nproc)
    pt.set_logging(n)
    pt.run(n)
    snap = _snap(pt)
    h = hashlib.sha1()
    for k in sorted(snap):
        if not k.endswith("_mean"):
            h.update(np.ascontiguousarray(snap[k]).tobytes())
    for a in pt.log(n):
        h.update(a.tobytes())
    pt.close()
    return h.hexdigest()


_NO_GRAPH_SCRIPT = r"""
import sys
sys.path[:0] = [{tests!r}, {root!r}, {oracle!r}]
from test_gpu_ladder_tuning import fingerprint
print("FP", fingerprint("sample_bookkeeping", 140, 200), fingerprint("laplace_prior_joint_PS", 130, 140))
"""


def test_plain_launches_equal_graph_replay():
    script = _NO_GRAPH_SCRIPT.format(tests=os.path.join(ROOT, "tests"), root=ROOT, oracle=os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, RFINV_PT_GRAPH="0"), capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("FP ")][-1].split()
    assert line[1:] == [fingerprint("sample_bookkeeping", 140, 200), fingerprint("laplace_prior_joint_PS", 130, 140)]


def test_runs_split_around_tuning_points():
    cfg, nproc = _cfg("sigma_solved_vp_solved", 300)
    n = 300
    ref = _tuned(cfg, nproc)
    ref.run(n)
    want = _snap(ref)
    ref.close()
    assert want["lt_points"] == 3
    for cut in (63, 64, 65, 127, 128, 129, 255, 256, 257):
        pt = _tuned(cfg, nproc)
        pt.run(cut)
        pt.run(n - cut)
        assert_identical(_snap(pt), want)
        pt.close()


def test_split_driver_matches_single_process():
    """local_step / swap_table / apply_swap with two handles on one GPU equals rfinv_pt_run with one handle, tuned."""
    import torch
    from rf_inv_b200.pt import _tensor_from_ptr
    cfg, nproc = _cfg("sigma_solved_vp_solved", 200)
    n_iter = 140
    one = _tuned(cfg, nproc)
    one.run(n_iter)
    st1, lt1 = one.state(), one.ladder_tuning()
    one.close()
    parts = [ParallelTempering(cfg, nproc, world=2, rank=r) for r in range(2)]
    for p in parts:
        p.set_rank_swaps(1)
        p.set_ladder_tuning(1)
    lib = parts[0]._lib
    dev = torch.device("cuda:0")
    tabs = [_tensor_from_ptr(torch, *p.swap_table(), dev) for p in parts]
    for _ in range(n_iter):
        for p in parts:
            capi.check(lib.rfinv_pt_local_step(p.ev.handle))
        for p in parts:
            p.ev.synchronize()
        gathered = torch.cat(tabs).contiguous()
        for p in parts:
            capi.check(lib.rfinv_pt_apply_swap(p.ev.handle, gathered.data_ptr(), 2))
        for p in parts:
            p.ev.synchronize()
    st2 = [p.state() for p in parts]
    for key in ("k", "z", "dvs", "logl", "temps"):
        assert np.array_equal(np.concatenate([s[key] for s in st2]), st1[key]), key
    assert lt1 == (True, 2) and all(p.ladder_tuning() == lt1 for p in parts)
    for p in parts:
        p.close()


# ---- checkpoints ----
def test_resume_across_tuning_points(tmp_path):
    cfg, nproc = _cfg("sample_bookkeeping", 140, niter=40)
    n = 180
    ref = _tuned(cfg, nproc)
    ref.run(n)
    want = _snap(ref)
    ref.close()
    for n1 in (63, 64, 100, 127, 128, 150):
        path = str(tmp_path / f"ck{n1}")
        a = _tuned(cfg, nproc)
        a.run(n1)
        a.save(path)
        a.close()
        b = _tuned(cfg, nproc)
        b.restore(path)
        assert b.ladder_tuning() == (True, sum(1 for e in (64, 128) if e <= n1))
        b.save(str(tmp_path / f"again{n1}"))
        assert filecmp.cmp(path, tmp_path / f"again{n1}", shallow=False)
        b.run(n - n1)
        assert_identical(_snap(b), want)
        b.close()


def test_checkpoint_tuning_must_match(tmp_path):
    cfg, nproc = _cfg("laplace_prior_joint_PS", 130)
    for tune in (1, 0):
        pt = ParallelTempering(cfg, nproc)
        pt.set_rank_swaps(1)
        pt.set_ladder_tuning(tune)
        pt.run(70)
        pt.save(str(tmp_path / f"f{tune}"))
        pt.close()
    assert os.path.getsize(tmp_path / "f1") > os.path.getsize(tmp_path / "f0")
    for file_tune in (1, 0):             # in either direction
        pt = ParallelTempering(cfg, nproc)
        try:
            pt.set_rank_swaps(1)
            pt.set_ladder_tuning(1 - file_tune)
            with pytest.raises(capi.RfinvError) as e:
                pt.restore(str(tmp_path / f"f{file_tune}"))
            assert e.value.status == capi.RFINV_ERR_ARG and "ladder tuning" in str(e.value), str(e.value)
            assert pt.iterations_done == 0
        finally:
            pt.close()


def test_set_ladder_tuning_refusals():
    cfg, nproc = _cfg("laplace_prior_joint_PS", 130)
    with Evaluator(cfg) as ev:                       # no rfinv_pt_init
        assert ev._lib.rfinv_pt_set_ladder_tuning(ev.handle, 1) == capi.RFINV_ERR_STATE
    pt = ParallelTempering(cfg, nproc)
    try:
        for bad in (-1, 2):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_ladder_tuning(bad)
            assert e.value.status == capi.RFINV_ERR_ARG
        with pytest.raises(capi.RfinvError) as e:     # rank swaps in mode 0
            pt.set_ladder_tuning(1)
        assert e.value.status == capi.RFINV_ERR_STATE
        pt.set_rank_swaps(1)
        pt.set_ladder_tuning(1)
        pt.set_ladder_tuning(0)                        # off and on again before any iteration
        pt.set_ladder_tuning(1)
        capi.check(pt._lib.rfinv_pt_local_step(pt.ev.handle))
        for v in (0, 1):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_ladder_tuning(v)
            assert e.value.status == capi.RFINV_ERR_STATE
        ptr, _ = pt.swap_table()
        capi.check(pt._lib.rfinv_pt_apply_swap(pt.ev.handle, ptr, 1))
        pt.run(70)
        assert pt.ladder_tuning() == (True, 1)
        pt.set_ladder_tuning(0)                        # off between runs
        assert pt.ladder_tuning() == (False, 1)
        with pytest.raises(capi.RfinvError) as e:      # not on again after iterations
            pt.set_ladder_tuning(1)
        assert e.value.status == capi.RFINV_ERR_STATE
        pt.reduce_outputs()
        with pytest.raises(capi.RfinvError) as e:
            pt.set_ladder_tuning(0)
        assert e.value.status == capi.RFINV_ERR_STATE
    finally:
        pt.close()


# ---- groups ----
def test_group_with_tuned_and_untuned_members_equals_solo_runs():
    ms = [member_config("sample_bookkeeping"), member_config("sigma_solved_vp_solved"), member_config("laplace_prior_joint_PS")]
    ms = [(copy.deepcopy(cfg), nproc) for cfg, nproc in ms]
    for cfg, _ in ms:
        cfg.nburn, cfg.niter, cfg.ncorr = 140, 30, 4
    tunes = [1, 0, 1]
    refs = []
    for (cfg, nproc), tune in zip(ms, tunes):
        pt = ParallelTempering(cfg, nproc)
        pt.set_rank_swaps(1)
        pt.set_ladder_tuning(tune)
        pt.run(170)
        refs.append(_snap(pt))
        pt.close()
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in ms]
    try:
        for pt, tune in zip(pts, tunes):
            pt.set_rank_swaps(1)
            pt.set_ladder_tuning(tune)
        with PtGroup(pts) as g:
            g.run(64)
            g.run(106)
        for pt, ref in zip(pts, refs):
            assert_identical(_snap(pt), ref)
    finally:
        for pt in pts:
            pt.close()


# ---- two processes ----
@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_processes_reproduce_the_single_process_run(exchange):
    if int(capi.load().rfinv_device_count()) < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, RFINV_PT_EXCHANGE=exchange, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29571" if exchange == "peer" else "29572", os.path.join(ROOT, "tools", "dist_check.py"), "--tune-ladder"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    for name, res in out.items():
        assert res["identical"], (name, res)


# ---- the driver ----
def test_driver_writes_ladder(tmp_path, capsys):
    from rf_inv_b200 import run as rrun
    paths = station_dirs(tmp_path / "src", 2, noise=0.01)
    for p in paths:
        set_param(p, "N_BURN", 130)                    # tuning points 64 and 128
    d_rs, d_tl = tmp_path / "rs", tmp_path / "tl"
    shutil.copytree(os.path.dirname(paths[0]), d_rs)
    shutil.copytree(os.path.dirname(paths[0]), d_tl)
    rrun.main([str(d_rs / "params.in"), "--nproc", "4", "--rank-swaps"])
    capsys.readouterr()
    rrun.main([str(d_tl / "params.in"), "--nproc", "4", "--tune-ladder"])
    out = capsys.readouterr().out
    rs_files, tl_files = set(os.listdir(d_rs / "rslt")), set(os.listdir(d_tl / "rslt"))
    assert tl_files == rs_files | {"ladder"} and "levels 0 and 1" in out
    # the files of the API run with the tuning
    cfg = rio.load_problem(str(d_tl / "params.in"))
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    pt = _tuned(cfg, 4)
    pt.run(cfg.nburn + cfg.niter)
    hist, cnt = pt.hist(), pt.counters()
    vp, vs = pt.models()
    ladders = rrun.rank_ladders(pt)
    pt.close()
    rio.write_outputs(cfg, str(tmp_path / "api"), 4, hist, cnt["likelihood_hist"], vp, vs)
    for n in OUTPUT_FILES:
        if n != "params.in.copy":
            assert filecmp.cmp(d_tl / "rslt" / n, tmp_path / "api" / n, shallow=False), n
    table = np.loadtxt(d_tl / "rslt" / "ladder", ndmin=2)
    assert table.shape == (4, cfg.nchains) and np.array_equal(table, ladders)
    assert np.all(np.diff(table, axis=1) >= 0) and int(np.sum(table <= 1.0 + lo.COLD_EPS)) == 4   # one cold chain per rank in all
    # a checkpointed run resumed half way writes the same files
    d_ck = tmp_path / "ck"
    shutil.copytree(os.path.dirname(paths[0]), d_ck)
    ck = str(d_ck / "state.ck")
    rrun.run(str(d_ck / "params.in"), nproc=4, verbose=False, n_iter=100, checkpoint=ck, resume=True, tune_ladder=True)
    rrun.run(str(d_ck / "params.in"), nproc=4, verbose=False, checkpoint=ck, resume=True, tune_ladder=True)
    for n in OUTPUT_FILES + ["rank_swaps", "ladder"]:
        if n != "params.in.copy":
            assert filecmp.cmp(d_ck / "rslt" / n, d_tl / "rslt" / n, shallow=False), n
    # two stations as a group: the files of the solo runs
    solo_dirs = []
    for i, p in enumerate(paths):
        d = tmp_path / f"solo{i}"
        shutil.copytree(os.path.dirname(p), d)
        rrun.run(str(d / "params.in"), nproc=4, verbose=False, tune_ladder=True)
        solo_dirs.append(d / "rslt")
    grp = []
    for i, p in enumerate(paths):
        d = tmp_path / "group" / f"station{i}"
        shutil.copytree(os.path.dirname(p), d)
        grp.append(str(d / "params.in"))
    rrun.main(grp + ["--nproc", "4", "--tune-ladder"])
    for p, ref in zip(grp, solo_dirs):
        for n in OUTPUT_FILES + ["rank_swaps", "ladder"]:
            assert filecmp.cmp(os.path.join(os.path.dirname(p), "rslt", n), ref / n, shallow=False), (p, n)
