"""Even/odd temperature swaps inside every virtual rank (rfinv_pt_set_rank_swaps, DESIGN.md 7c) on the GPU: mode 1 reproduces
the C restatement with the sweep (tests/rank_swap_oracle.c) exactly on every path an iteration can take -- the captured graph, plain launches, the split driver,
checkpoints, groups, two processes -- and the driver writes the reference's files plus OUT_DIR/rank_swaps."""
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

import helpers
import rank_swap_oracle as rso
from rf_inv_b200 import capi, workloads
from rf_inv_b200 import io as rio
from rf_inv_b200.pt import ParallelTempering, PtGroup
from test_gpu_checkpoint import assert_identical, snapshot, variant_config
from test_gpu_group import OUTPUT_FILES, member_config
from test_gpu_pt import check as check_against_oracle
from test_group_driver import station_dirs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = ["sample", "sigma_solved_vp_solved", "laplace_prior_joint_PS", "single_chain_per_rank", "transform_length_250",
            "transform_length_375_odd"]


def oracle_variant(name):
    """(cfg, nproc, n_iter): tests/test_gpu_pt.py's sample run and proposal variants."""
    if name == "sample":
        return helpers.attach_obs_and_rinv(workloads.make_config("sample"), noise=0.01), 20, 200
    if name == "sigma_solved_vp_solved":
        cfg = helpers.small_config(sdep=2.0, vp_mode=1, rayps=[0.06, 0.06], a_gus=[2.5, 4.0], nfft=128, nsmp=64,
                                   sig_min=[0.005, 0.01], sig_max=[0.05, 0.01], nchains=4, ncool=2, t_high=10.0, iseed=777)
        nproc, n_iter = 6, 120
    elif name == "laplace_prior_joint_PS":
        cfg = helpers.small_config(prior_mode=1, dvs_prior=0.3, dvp_prior=0.1, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.10],
                                   nfft=128, nsmp=64, nchains=3, ncool=1, t_high=5.0, iseed=4242)
        nproc, n_iter = 5, 120
    elif name.startswith("transform_length"):
        n = 250 if name.endswith("250") else 375
        cfg = helpers.small_config(sdep=1.0, nfft=n, nsmp=101, nchains=4, ncool=1, t_high=8.0, iseed=31337)
        nproc, n_iter = 5, 80
    else:
        cfg = helpers.small_config(nfft=64, nsmp=40, nchains=1, ncool=1, iseed=99)
        nproc, n_iter = 8, 60
    return helpers.attach_obs_and_rinv(cfg, noise=0.01), nproc, n_iter


def gpu_run(cfg, nproc, plan):
    """plan: [(mode, iterations), ...] on one handle with logs of the whole run."""
    n = sum(k for _, k in plan)
    pt = ParallelTempering(cfg, nproc)
    try:
        pt.set_logging(n)
        st0 = pt.state()
        for mode, k in plan:
            pt.set_rank_swaps(mode)
            pt.run(k)
        flags, itypes, swaps = pt.log(n)
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=pt.state(), cnt=pt.counters(), rs=pt.rank_swaps())
    finally:
        pt.close()


def oracle_run(cfg, nproc, plan):
    orc = rso.RankSwapOraclePT(cfg, nproc)
    try:
        st0 = orc.state()
        logs = []
        for mode, k in plan:
            orc.set_rank_swaps(mode)
            logs.append(orc.run(k))
        n = sum(k for _, k in plan)
        flags, itypes, swaps = (np.concatenate([l[i] for l in logs]) for i in range(3))
        return dict(flags=flags, itypes=itypes, swaps=swaps, st0=st0, st=orc.state(), cnt=orc.counters(n), n_eval=orc.n_eval,
                    rs=orc.rank_swaps())
    finally:
        orc.close()


def temperature_ranks(st0, st):
    """Each chain's final temperature as its rank among the initial temperatures (equal values: equal ranks)."""
    ranks = np.searchsorted(np.sort(st0["temps"]), st["temps"])
    assert np.array_equal(np.sort(st0["temps"])[ranks], st["temps"])     # swaps only exchange values
    return ranks


def check(g, o, cfg):
    check_against_oracle(g, o, cfg)
    # The initial temperatures are exp() of the same draws, on the device and in libm: they agree to rounding, not bit for
    # bit.  Which of them every chain holds at the end is exact.
    assert np.array_equal(temperature_ranks(g["st0"], g["st"]), temperature_ranks(o["st0"], o["st"]))
    for key in ("mode", "n_prop", "n_acc"):
        assert np.array_equal(g["rs"][key], o["rs"][key]), key


@pytest.mark.parametrize("variant", VARIANTS)
def test_mode1_matches_oracle(variant):
    cfg, nproc, n_iter = oracle_variant(variant)
    g = gpu_run(cfg, nproc, [(1, n_iter)])
    check(g, oracle_run(cfg, nproc, [(1, n_iter)]), cfg)
    if cfg.nchains >= 2:
        assert g["rs"]["n_acc"].sum() > 0
        assert np.array_equal(np.sort(g["st"]["temps"]), np.sort(g["st0"]["temps"]))
    else:                                   # nothing to pair: the reference's run in either mode
        ref = gpu_run(cfg, nproc, [(0, n_iter)])
        for key in ("flags", "itypes", "swaps"):
            assert np.array_equal(g[key], ref[key]), key
        for key in g["st"]:
            assert np.array_equal(g["st"][key], ref["st"][key]), key


def test_mode_switched_between_runs_matches_oracle():
    cfg, nproc, _ = oracle_variant("sigma_solved_vp_solved")
    plan = [(1, 50), (0, 50)]
    g = gpu_run(cfg, nproc, plan)
    check(g, oracle_run(cfg, nproc, plan), cfg)


def fingerprint(name, n):
    """sha1 over logs, state, counters and rank-swap counters of a mode-1 run of a checkpoint variant (bookkeeping on)."""
    cfg, nproc, _, _ = variant_config(name)
    pt = ParallelTempering(cfg, nproc)
    pt.set_logging(n)
    pt.set_rank_swaps(1)
    pt.run(n)
    snap = snapshot(pt)
    h = hashlib.sha1()
    for k in sorted(snap):
        if not k.endswith("_mean"):
            h.update(np.ascontiguousarray(snap[k]).tobytes())
    for a in pt.log(n):
        h.update(a.tobytes())
    rs = pt.rank_swaps()
    h.update(rs["n_prop"].tobytes()); h.update(rs["n_acc"].tobytes())
    pt.close()
    return h.hexdigest()


_NO_GRAPH_SCRIPT = r"""
import sys
sys.path[:0] = [{tests!r}, {root!r}, {oracle!r}]
from test_gpu_rank_swaps import fingerprint
print("FP", fingerprint("sample_bookkeeping", 70), fingerprint("laplace_prior_joint_PS", 60))
"""


def test_plain_launches_equal_graph_replay():
    script = _NO_GRAPH_SCRIPT.format(tests=os.path.join(ROOT, "tests"), root=ROOT, oracle=os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, RFINV_PT_GRAPH="0"), capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("FP ")][-1].split()
    assert line[1:] == [fingerprint("sample_bookkeeping", 70), fingerprint("laplace_prior_joint_PS", 60)]


def test_split_driver_matches_single_process():
    """local_step / swap_table / apply_swap with two handles on one GPU equals rfinv_pt_run with one handle in mode 1."""
    import torch
    from rf_inv_b200.pt import _tensor_from_ptr
    cfg = helpers.attach_obs_and_rinv(helpers.small_config(sdep=2.0, nfft=128, nsmp=64, nchains=5, ncool=1, t_high=8.0), noise=0.01)
    nproc, n_iter = 4, 60
    one = ParallelTempering(cfg, nproc)
    one.set_logging(n_iter)
    one.set_rank_swaps(1)
    one.run(n_iter)
    f1, t1, s1 = one.log(n_iter)
    st1, rs1 = one.state(), one.rank_swaps()
    one.close()
    parts = [ParallelTempering(cfg, nproc, world=2, rank=r) for r in range(2)]
    for p in parts:
        p.set_logging(n_iter)
        p.set_rank_swaps(1)
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
    logs = [p.log(n_iter) for p in parts]
    assert np.array_equal(np.concatenate([l[0] for l in logs], axis=1), f1)
    assert np.array_equal(np.concatenate([l[1] for l in logs], axis=1), t1)
    assert np.array_equal(logs[0][2], s1) and np.array_equal(logs[1][2], s1)
    st2 = [p.state() for p in parts]
    for key in ("k", "z", "dvs", "logl", "temps"):
        assert np.array_equal(np.concatenate([s[key] for s in st2]), st1[key]), key
    rs2 = [p.rank_swaps() for p in parts]
    assert np.array_equal(rs2[0]["n_prop"] + rs2[1]["n_prop"], rs1["n_prop"])
    assert np.array_equal(rs2[0]["n_acc"] + rs2[1]["n_acc"], rs1["n_acc"]) and rs1["n_acc"].sum() > 0
    for p in parts:
        p.close()


# ---- checkpoints ----
def _snap(pt):
    out = snapshot(pt)
    rs = pt.rank_swaps()
    out.update(rs_mode=np.int64(rs["mode"]), rs_n_prop=rs["n_prop"], rs_n_acc=rs["n_acc"])
    return out


@pytest.mark.parametrize("variant", ["sample_bookkeeping", "sigma_solved_vp_solved"])
def test_resume_equals_uninterrupted_run(variant, tmp_path):
    cfg, nproc, splits, n = variant_config(variant)
    ref = ParallelTempering(cfg, nproc)
    ref.set_rank_swaps(1)
    ref.run(n)
    want = _snap(ref)
    ref.close()
    for n1 in splits:
        path = str(tmp_path / f"ck{n1}")
        a = ParallelTempering(cfg, nproc)
        a.set_rank_swaps(1)
        a.run(n1)
        a.save(path)
        a.close()
        b = ParallelTempering(cfg, nproc)
        b.set_rank_swaps(1)
        b.restore(path)
        b.run(n - n1)
        assert_identical(_snap(b), want)
        b.close()


def test_save_restore_save_is_byte_identical_and_modes_must_match(tmp_path):
    cfg, nproc, _, _ = variant_config("sample_bookkeeping")
    for mode in (1, 0):
        a = ParallelTempering(cfg, nproc)
        a.set_rank_swaps(mode)
        a.run(47)
        a.save(str(tmp_path / f"one{mode}"))
        a.close()
        b = ParallelTempering(cfg, nproc)
        b.set_rank_swaps(mode)
        b.restore(str(tmp_path / f"one{mode}"))
        b.save(str(tmp_path / f"two{mode}"))
        b.close()
        assert filecmp.cmp(tmp_path / f"one{mode}", tmp_path / f"two{mode}", shallow=False)
    assert os.path.getsize(tmp_path / "one1") > os.path.getsize(tmp_path / "one0")
    for file_mode in (1, 0):             # a file restores only into a handle of its mode, in either direction
        pt = ParallelTempering(cfg, nproc)
        try:
            pt.set_rank_swaps(1 - file_mode)
            with pytest.raises(capi.RfinvError) as e:
                pt.restore(str(tmp_path / f"one{file_mode}"))
            assert e.value.status == capi.RFINV_ERR_ARG and "rank swaps" in str(e.value), str(e.value)
            assert pt.iterations_done == 0
        finally:
            pt.close()


def test_set_rank_swaps_refusals():
    cfg, nproc, _, _ = variant_config("laplace_prior_joint_PS")
    pt = ParallelTempering(cfg, nproc)
    try:
        for bad in (-1, 2):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_rank_swaps(bad)
            assert e.value.status == capi.RFINV_ERR_ARG
        capi.check(pt._lib.rfinv_pt_local_step(pt.ev.handle))
        with pytest.raises(capi.RfinvError) as e:
            pt.set_rank_swaps(1)
        assert e.value.status == capi.RFINV_ERR_STATE
        ptr, _ = pt.swap_table()
        capi.check(pt._lib.rfinv_pt_apply_swap(pt.ev.handle, ptr, 1))
        pt.set_rank_swaps(1)
        pt.reduce_outputs()
        with pytest.raises(capi.RfinvError) as e:
            pt.set_rank_swaps(0)
        assert e.value.status == capi.RFINV_ERR_STATE
        assert pt.rank_swaps()["mode"] == 1
    finally:
        pt.close()


# ---- groups ----
def _solo(cfg, nproc, plan):
    pt = ParallelTempering(cfg, nproc)
    try:
        for mode, k in plan:
            pt.set_rank_swaps(mode)
            pt.run(k)
        return _snap(pt)
    finally:
        pt.close()


def test_group_with_mixed_and_toggled_modes_equals_solo_runs():
    ms = [member_config("sample_bookkeeping"), member_config("sigma_solved_vp_solved")]
    plans = [[(1, 40), (0, 50)], [(0, 40), (1, 50)]]
    refs = [_solo(cfg, nproc, plan) for (cfg, nproc), plan in zip(ms, plans)]
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in ms]
    try:
        with PtGroup(pts) as g:
            for step in range(2):
                for pt, plan in zip(pts, plans):
                    pt.set_rank_swaps(plan[step][0])
                g.run(plans[0][step][1] - (13 if step == 0 else 0))
                if step == 0:
                    g.run(13)
        for pt, ref in zip(pts, refs):
            assert_identical(_snap(pt), ref)
    finally:
        for pt in pts:
            pt.close()


# ---- two processes ----
def _gpus():
    return int(capi.load().rfinv_device_count())


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_processes_reproduce_the_single_process_run(exchange):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, RFINV_PT_EXCHANGE=exchange, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29561" if exchange == "peer" else "29562", os.path.join(ROOT, "tools", "dist_check.py"), "--rank-swaps"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    for name, res in out.items():
        assert res["identical"], (name, res)


# ---- the driver ----
def _api_outputs(params, out_dir):
    """What a mode-1 run of `params` through the Python API writes with rio.write_outputs."""
    cfg = rio.load_problem(params)
    cfg.r_inv = workloads.lapack_r_inv(cfg)
    pt = ParallelTempering(cfg, 4)
    pt.set_rank_swaps(1)
    pt.run(cfg.nburn + cfg.niter)
    hist, cnt = pt.hist(), pt.counters()
    vp, vs = pt.models()
    rs = pt.rank_swaps()
    pt.close()
    os.makedirs(out_dir)
    rio.write_outputs(cfg, str(out_dir), 4, hist, cnt["likelihood_hist"], vp, vs)
    return rs


def test_driver_writes_reference_files_plus_rank_swaps(tmp_path, capsys):
    from rf_inv_b200 import run as rrun
    paths = station_dirs(tmp_path / "src", 2, noise=0.01)
    # single station: the flag adds OUT_DIR/rank_swaps, the other files are those of the API run in mode 1
    d_plain, d_flag = tmp_path / "plain", tmp_path / "flag"
    shutil.copytree(os.path.dirname(paths[0]), d_plain)
    shutil.copytree(os.path.dirname(paths[0]), d_flag)
    rrun.main([str(d_plain / "params.in"), "--nproc", "4"])
    out_plain = capsys.readouterr().out
    rrun.main([str(d_flag / "params.in"), "--nproc", "4", "--rank-swaps"])
    out_flag = capsys.readouterr().out
    plain, flag = set(os.listdir(d_plain / "rslt")), set(os.listdir(d_flag / "rslt"))
    assert set(OUTPUT_FILES) <= plain and "rank_swaps" not in plain and flag == plain | {"rank_swaps"}
    assert "levels" not in out_plain and "levels 0 and 1" in out_flag
    rs = _api_outputs(str(d_flag / "params.in"), tmp_path / "api")
    for n in OUTPUT_FILES:
        if n != "params.in.copy":
            assert filecmp.cmp(d_flag / "rslt" / n, tmp_path / "api" / n, shallow=False), n
    table = np.loadtxt(d_flag / "rslt" / "rank_swaps", ndmin=2)
    cfg = rio.load_problem(str(d_flag / "params.in"))
    assert table.shape == (cfg.nchains - 1, 4)
    assert np.array_equal(table[:, 0], np.arange(1, cfg.nchains))
    assert np.array_equal(table[:, 1], rs["n_acc"]) and np.array_equal(table[:, 2], rs["n_prop"])
    # two stations as a group with the flag: the files of the solo runs with the flag
    solo_dirs = []
    for i, p in enumerate(paths):
        d = tmp_path / f"solo{i}"
        shutil.copytree(os.path.dirname(p), d)
        rrun.run(str(d / "params.in"), nproc=4, verbose=False, rank_swaps=True)
        solo_dirs.append(d / "rslt")
    grp = []
    for i, p in enumerate(paths):
        d = tmp_path / "group" / f"station{i}"
        shutil.copytree(os.path.dirname(p), d)
        grp.append(str(d / "params.in"))
    rrun.main(grp + ["--nproc", "4", "--rank-swaps"])
    for p, ref in zip(grp, solo_dirs):
        for n in OUTPUT_FILES + ["rank_swaps"]:
            assert filecmp.cmp(os.path.join(os.path.dirname(p), "rslt", n), ref / n, shallow=False), (p, n)
