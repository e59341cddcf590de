"""Random-walk width tuning during the burn-in (rfinv_pt_set_step_tuning, DESIGN.md 7e) on the GPU: tuned runs reproduce the C
reference (tests/step_oracle.c) across several tuning points, with and without the ladder tuning, and keep the identity
guarantees of plain launches, split runs, checkpoints, groups and two processes; the driver writes OUT_DIR/step_widths."""
import copy
import filecmp
import hashlib
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import step_oracle as so
from rf_inv_b200 import capi, workloads
from rf_inv_b200 import io as rio
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering, PtGroup
from test_gpu_checkpoint import assert_identical, snapshot, variant_config
from test_gpu_group import OUTPUT_FILES, member_config
from test_gpu_ladder_tuning import check as check_ladder
from test_gpu_rank_swaps import VARIANTS, oracle_variant
from test_group_driver import set_param, station_dirs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TUNED_VARIANTS = [v for v in VARIANTS if v != "single_chain_per_rank"]   # (no levels with one chain per rank)


def tuned_variant(name):
    """test_gpu_rank_swaps.py's variant with a burn-in holding the tuning points 64 ... 256 (the sample: 64 ... 512)."""
    cfg, nproc, _ = oracle_variant(name)
    cfg = copy.deepcopy(cfg)
    n = 520 if name == "sample" else 300
    cfg.nburn = n
    return cfg, nproc, n


def _apply(obj, mode, ladder, steps, target=0.44):
    obj.set_rank_swaps(mode)
    if ladder or obj.ladder_tuning()[0]:
        obj.set_ladder_tuning(ladder)
    if steps or obj.step_tuning()["on"]:
        obj.set_step_tuning(steps, target)


def gpu_run(cfg, nproc, plan):
    """plan: [(mode, ladder tuning, step tuning, iterations), ...] on one handle with logs of the whole run."""
    n = sum(p[-1] for p in plan)
    pt = ParallelTempering(cfg, nproc)
    try:
        pt.set_logging(n)
        st0 = pt.state()
        for mode, ladder, steps, k in plan:
            _apply(pt, mode, ladder, steps)
            pt.run(k)
        flags, itypes, swaps = pt.log(n)
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=pt.state(), cnt=pt.counters(), rs=pt.rank_swaps(),
                    lt=pt.ladder_tuning(), steps=pt.step_tuning())
    finally:
        pt.close()


def oracle_run(cfg, nproc, plan):
    orc = so.StepOraclePT(cfg, nproc)
    try:
        st0 = orc.state()
        logs = []
        for mode, ladder, steps, k in plan:
            _apply(orc, mode, ladder, steps)
            logs.append(orc.run(k))
        n = sum(p[-1] for p in plan)
        flags, itypes, swaps = (np.concatenate([l[i] for l in logs]) for i in range(3))
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=orc.state(), cnt=orc.counters(n), n_eval=orc.n_eval,
                    rs=orc.rank_swaps(), lt=orc.ladder_tuning(), steps=orc.step_tuning())
    finally:
        orc.close()


def check(g, o, cfg):
    # test_gpu_ladder_tuning's check (decisions, counters, sweep counters and ladder tuning exact; state to 1e-12, logL to 1e-9),
    # and the width tuning exact: setting, tuning points, widths and counters
    check_ladder(g, o, cfg)
    gs, os_ = g["steps"], o["steps"]
    assert (gs["on"], gs["n_points"]) == (os_["on"], os_["n_points"])
    for key in ("widths", "n_prop", "n_acc"):
        assert gs[key].tobytes() == os_[key].tobytes(), key


@pytest.mark.parametrize("ladder", [0, 1])
@pytest.mark.parametrize("variant", TUNED_VARIANTS)
def test_tuned_run_matches_oracle(variant, ladder):
    cfg, nproc, n = tuned_variant(variant)
    g = gpu_run(cfg, nproc, [(1, ladder, 1, n)])
    check(g, oracle_run(cfg, nproc, [(1, ladder, 1, n)]), cfg)
    assert g["steps"]["n_points"] == (4 if variant == "sample" else 3)
    dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])
    assert not np.array_equal(g["steps"]["widths"], np.broadcast_to(dev, g["steps"]["widths"].shape))   # a scale moved


def test_rank_swaps_off_switches_step_tuning_off_and_matches_oracle():
    cfg, nproc, _ = tuned_variant("sigma_solved_vp_solved")
    plan = [(1, 0, 1, 100), (0, 0, 0, 60), (1, 0, 0, 100)]   # tuned through 64, then the reference, then the sweep alone
    g = gpu_run(cfg, nproc, plan)
    assert not g["steps"]["on"] and g["steps"]["n_points"] == 1
    dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])
    assert np.array_equal(g["steps"]["widths"], np.broadcast_to(dev, g["steps"]["widths"].shape))   # back to params.in
    check(g, oracle_run(cfg, nproc, plan), cfg)


def test_short_burn_in_equals_mode1():
    cfg, nproc, _ = tuned_variant("laplace_prior_joint_PS")
    cfg.nburn = 63
    a, b = gpu_run(cfg, nproc, [(1, 0, 1, 150)]), gpu_run(cfg, nproc, [(1, 0, 0, 150)])
    for key in ("flags", "itypes", "swaps"):
        assert np.array_equal(a[key], b[key]), key
    for key in a["st"]:
        assert np.array_equal(a["st"][key], b["st"][key]), key
    assert a["steps"]["on"] and a["steps"]["n_points"] == 0


# ---- launch paths ----
def _cfg(name, nburn, niter=60, ncorr=4):
    cfg, nproc, _, _ = variant_config(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter, cfg.ncorr = nburn, niter, ncorr
    return cfg, nproc


def _snap(pt):
    out = snapshot(pt)
    rs, st = pt.rank_swaps(), pt.step_tuning()
    out.update(rs_n_prop=rs["n_prop"], rs_n_acc=rs["n_acc"], lt_on=np.int64(pt.ladder_tuning()[0]),
               st_on=np.int64(st["on"]), st_points=np.int64(st["n_points"]), st_widths=st["widths"], st_n_prop=st["n_prop"],
               st_n_acc=st["n_acc"])
    return out


def _tuned(cfg, nproc, ladder=0, target=0.44):
    pt = ParallelTempering(cfg, nproc)
    pt.set_rank_swaps(1)
    if ladder:
        pt.set_ladder_tuning(1)
    pt.set_step_tuning(1, target)
    return pt


def fingerprint(name, nburn, n):
    """sha1 over logs, state, counters, sweep counters and the width tuning of a tuned run (bookkeeping on after nburn)."""
    cfg, nproc = _cfg(name, nburn)
    pt = _tuned(cfg, nproc, ladder=1)
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
from test_gpu_step_tuning import fingerprint
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
    assert want["st_points"] == 3
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
    st1, s1 = one.state(), one.step_tuning()
    one.close()
    parts = [ParallelTempering(cfg, nproc, world=2, rank=r) for r in range(2)]
    for p in parts:
        p.set_rank_swaps(1)
        p.set_step_tuning(1)
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
    s2 = [p.step_tuning() for p in parts]
    assert s1["n_points"] == 2 and all(s["n_points"] == 2 for s in s2)
    for key in ("widths", "n_prop", "n_acc"):
        assert np.array_equal(np.concatenate([s[key] for s in s2]), s1[key]), key
    for p in parts:
        p.close()


# ---- checkpoints ----
def test_resume_across_tuning_points(tmp_path):
    cfg, nproc = _cfg("sample_bookkeeping", 140, niter=40)
    n = 180
    ref = _tuned(cfg, nproc, ladder=1, target=0.3)
    ref.run(n)
    want = _snap(ref)
    ref.close()
    for n1 in (63, 64, 100, 127, 128, 150):
        path = str(tmp_path / f"ck{n1}")
        a = _tuned(cfg, nproc, ladder=1, target=0.3)
        a.run(n1)
        a.save(path)
        a.close()
        b = _tuned(cfg, nproc, ladder=1, target=0.3)
        b.restore(path)
        assert b.step_tuning()["n_points"] == sum(1 for e in (64, 128) if e <= n1)
        b.save(str(tmp_path / f"again{n1}"))
        assert filecmp.cmp(path, tmp_path / f"again{n1}", shallow=False)
        b.run(n - n1)
        assert_identical(_snap(b), want)
        b.close()


def test_checkpoint_setting_and_target_must_match(tmp_path):
    cfg, nproc = _cfg("laplace_prior_joint_PS", 130)
    for steps in (1, 0):
        pt = ParallelTempering(cfg, nproc)
        pt.set_rank_swaps(1)
        pt.set_step_tuning(steps)
        pt.run(70)
        pt.save(str(tmp_path / f"f{steps}"))
        pt.close()
    assert os.path.getsize(tmp_path / "f1") > os.path.getsize(tmp_path / "f0")
    for file_steps, handle_steps, target in ((1, 0, 0.44), (0, 1, 0.44), (1, 1, 0.3)):   # either direction, another target
        pt = ParallelTempering(cfg, nproc)
        try:
            pt.set_rank_swaps(1)
            pt.set_step_tuning(handle_steps, target)
            with pytest.raises(capi.RfinvError) as e:
                pt.restore(str(tmp_path / f"f{file_steps}"))
            assert e.value.status == capi.RFINV_ERR_ARG and "step tuning" in str(e.value), str(e.value)
            assert pt.iterations_done == 0
        finally:
            pt.close()


def test_set_step_tuning_refusals():
    cfg, nproc = _cfg("laplace_prior_joint_PS", 130)
    with Evaluator(cfg) as ev:                       # no rfinv_pt_init
        assert ev._lib.rfinv_pt_set_step_tuning(ev.handle, 1, 0.44) == capi.RFINV_ERR_STATE
    one = copy.deepcopy(cfg)
    one.nchains, one.ncool = 1, 1
    pt = ParallelTempering(one, nproc)
    try:
        pt.set_rank_swaps(1)
        with pytest.raises(capi.RfinvError) as e:     # nchains < 2
            pt.set_step_tuning(1)
        assert e.value.status == capi.RFINV_ERR_ARG
    finally:
        pt.close()
    pt = ParallelTempering(cfg, nproc)
    try:
        for bad, target in ((-1, 0.44), (2, 0.44), (1, 0.0), (1, 1.0), (1, -0.5), (1, float("nan"))):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_step_tuning(bad, target)
            assert e.value.status == capi.RFINV_ERR_ARG, (bad, target)
        with pytest.raises(capi.RfinvError) as e:     # rank swaps in mode 0
            pt.set_step_tuning(1)
        assert e.value.status == capi.RFINV_ERR_STATE
        pt.set_rank_swaps(1)
        pt.set_step_tuning(1, 0.5)
        pt.set_step_tuning(0)                          # off and on again before any iteration
        pt.set_step_tuning(1, 0.44)
        assert pt.step_tuning()["target"] == 0.44
        capi.check(pt._lib.rfinv_pt_local_step(pt.ev.handle))
        for v in (0, 1):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_step_tuning(v)
            assert e.value.status == capi.RFINV_ERR_STATE
        ptr, _ = pt.swap_table()
        capi.check(pt._lib.rfinv_pt_apply_swap(pt.ev.handle, ptr, 1))
        pt.run(70)
        st = pt.step_tuning()
        assert st["on"] and st["n_points"] == 1
        pt.set_step_tuning(0)                          # off between runs: the params.in widths
        st = pt.step_tuning()
        assert not st["on"] and st["n_points"] == 1
        dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])
        assert np.array_equal(st["widths"], np.broadcast_to(dev, st["widths"].shape))
        with pytest.raises(capi.RfinvError) as e:      # not on again after iterations
            pt.set_step_tuning(1)
        assert e.value.status == capi.RFINV_ERR_STATE
        pt.reduce_outputs()
        with pytest.raises(capi.RfinvError) as e:
            pt.set_step_tuning(0)
        assert e.value.status == capi.RFINV_ERR_STATE
    finally:
        pt.close()


def test_switching_off_between_runs_matches_oracle():
    cfg, nproc, _ = tuned_variant("laplace_prior_joint_PS")
    plan = [(1, 1, 1, 130), (1, 1, 0, 70)]             # tuned through 64 and 128, then the params.in widths
    check(gpu_run(cfg, nproc, plan), oracle_run(cfg, nproc, plan), cfg)


# ---- groups ----
def test_group_with_tuned_and_untuned_members_equals_solo_runs():
    ms = [member_config("sample_bookkeeping"), member_config("sigma_solved_vp_solved"), member_config("laplace_prior_joint_PS")]
    ms = [(copy.deepcopy(cfg), nproc) for cfg, nproc in ms]
    for cfg, _ in ms:
        cfg.nburn, cfg.niter, cfg.ncorr = 140, 30, 4
    settings = [(1, 0), (0, 1), (1, 1)]                # (step tuning, ladder tuning)
    refs = []
    for (cfg, nproc), (steps, ladder) in zip(ms, settings):
        pt = ParallelTempering(cfg, nproc)
        pt.set_rank_swaps(1)
        pt.set_ladder_tuning(ladder)
        pt.set_step_tuning(steps)
        pt.run(170)
        refs.append(_snap(pt))
        pt.close()
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in ms]
    try:
        for pt, (steps, ladder) in zip(pts, settings):
            pt.set_rank_swaps(1)
            pt.set_ladder_tuning(ladder)
            pt.set_step_tuning(steps)
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
           "--master-port", "29573" if exchange == "peer" else "29574", os.path.join(ROOT, "tools", "dist_check.py"), "--tune-steps"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    for name, res in out.items():
        assert res["identical"], (name, res)


# ---- the driver ----
def test_driver_writes_step_widths(tmp_path, capsys):
    from rf_inv_b200 import run as rrun
    paths = station_dirs(tmp_path / "src", 2, noise=0.01)
    for p in paths:
        set_param(p, "N_BURN", 130)                    # tuning points 64 and 128
    d_rs, d_st = tmp_path / "rs", tmp_path / "st"
    shutil.copytree(os.path.dirname(paths[0]), d_rs)
    shutil.copytree(os.path.dirname(paths[0]), d_st)
    rrun.main([str(d_rs / "params.in"), "--nproc", "4", "--rank-swaps"])
    rrun.main([str(d_st / "params.in"), "--nproc", "4", "--tune-steps", "--step-target", "0.3"])
    capsys.readouterr()
    assert set(os.listdir(d_st / "rslt")) == set(os.listdir(d_rs / "rslt")) | {"step_widths"}
    # the files of the API run with the tuning
    cfg = rio.load_problem(str(d_st / "params.in"))
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    pt = _tuned(cfg, 4, target=0.3)
    pt.run(cfg.nburn + cfg.niter)
    hist, cnt = pt.hist(), pt.counters()
    vp, vs = pt.models()
    rows = rrun.step_rows(pt)
    st = pt.step_tuning()
    pt.close()
    rio.write_outputs(cfg, str(tmp_path / "api"), 4, hist, cnt["likelihood_hist"], vp, vs)
    for n in OUTPUT_FILES:
        if n != "params.in.copy":
            assert filecmp.cmp(d_st / "rslt" / n, tmp_path / "api" / n, shallow=False), n
    table = np.loadtxt(d_st / "rslt" / "step_widths", ndmin=2)
    assert table.shape == (4 * cfg.nchains, 10)
    assert np.array_equal(table[:, :2], rows[:, :2]) and np.array_equal(table[:, 2:6], st["widths"].reshape(-1, 4))
    assert np.allclose(table[:, 6:], rows[:, 6:], atol=1e-6, rtol=0)
    # a checkpointed run resumed half way writes the same files
    d_ck = tmp_path / "ck"
    shutil.copytree(os.path.dirname(paths[0]), d_ck)
    ck = str(d_ck / "state.ck")
    rrun.run(str(d_ck / "params.in"), nproc=4, verbose=False, n_iter=100, checkpoint=ck, resume=True, tune_steps=True, step_target=0.3)
    rrun.run(str(d_ck / "params.in"), nproc=4, verbose=False, checkpoint=ck, resume=True, tune_steps=True, step_target=0.3)
    for n in OUTPUT_FILES + ["rank_swaps", "step_widths"]:
        if n != "params.in.copy":
            assert filecmp.cmp(d_ck / "rslt" / n, d_st / "rslt" / n, shallow=False), n
    # two stations as a group: the files of the solo runs
    solo_dirs = []
    for i, p in enumerate(paths):
        d = tmp_path / f"solo{i}"
        shutil.copytree(os.path.dirname(p), d)
        rrun.run(str(d / "params.in"), nproc=4, verbose=False, tune_steps=True, tune_ladder=True)
        solo_dirs.append(d / "rslt")
    grp = []
    for i, p in enumerate(paths):
        d = tmp_path / "group" / f"station{i}"
        shutil.copytree(os.path.dirname(p), d)
        grp.append(str(d / "params.in"))
    rrun.main(grp + ["--nproc", "4", "--tune-steps", "--tune-ladder"])
    for p, ref in zip(grp, solo_dirs):
        for n in OUTPUT_FILES + ["rank_swaps", "ladder", "step_widths"]:
            assert filecmp.cmp(os.path.join(os.path.dirname(p), "rslt", n), ref / n, shallow=False), (p, n)
