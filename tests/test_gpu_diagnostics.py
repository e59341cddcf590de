"""Convergence diagnostics (rfinv_pt_set_diagnostics, DESIGN.md 7f) on the GPU: the cold-level trace equals the numpy
selection of every rank's level 0, the round trips equal numpy's count over the per-iteration temperatures, the statistics
equal tests/diag_oracle.py on the returned trace, and the run itself is unchanged; checkpoints, groups, plain launches and the
driver keep their identity guarantees."""
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

import diag_oracle as dgo
from rf_inv_b200 import capi
from rf_inv_b200.pt import ParallelTempering, PtGroup
from test_gpu_checkpoint import assert_identical, snapshot
from test_gpu_group import OUTPUT_FILES
from test_gpu_rank_swaps import oracle_variant
from test_group_driver import set_param, station_dirs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VARIANTS = ["sample", "sigma_solved_vp_solved", "laplace_prior_joint_PS", "transform_length_250"]


def diag_config(name, nburn=20, niter=80, ncorr=2):
    cfg, nproc, _ = oracle_variant(name)
    cfg = copy.deepcopy(cfg)
    cfg.nburn, cfg.niter, cfg.ncorr = nburn, niter, ncorr
    return cfg, nproc


def bins_of(cfg):
    """Depth bins at the surface (the sea layer where there is one), in the middle and at the bottom."""
    return [1, 3, cfg.nbin_z // 2, cfg.nbin_z]


def setup(pt, mode=0, ladder=0, steps=0, bins=None, diag=1):
    pt.set_rank_swaps(mode)
    if ladder:
        pt.set_ladder_tuning(1)
    if steps:
        pt.set_step_tuning(1)
    if diag:
        pt.set_diagnostics(1, bins_of(pt.cfg) if bins is None else bins)


def stepwise(cfg, nproc, n, **kw):
    """One iteration per call: the temperatures at acceptance of every iteration (those after the previous one), the state
    after it and the models recorded by it."""
    pt = ParallelTempering(cfg, nproc)
    try:
        setup(pt, **kw)
        rec = []
        for it in range(1, n + 1):
            temps = pt.state()["temps"]
            nmod = pt.hist()["nmod"]
            pt.run(1)
            st = pt.state()
            vp, vs = pt.models()
            rec.append(dict(it=it, temps=temps, st=st, nmod=nmod, vs_model=vs))
        return rec, pt.cold_trace(), pt.diagnostics()
    finally:
        pt.close()


def check_trace(cfg, nproc, rec, tr):
    nch = cfg.nchains
    bins = tr["vs_bins"]
    sig_t = [t for t, m in enumerate(cfg.sig_mode) if m]
    smp = 0
    for r in rec:
        it = r["it"]
        if not (it > cfg.nburn and it % cfg.ncorr == 0):
            continue
        lv = dgo.cold_levels(r["temps"], nch)
        st = r["st"]
        ch = np.arange(nproc) * nch + lv
        row = tr["trace"][smp]
        assert np.array_equal(row[:, 0], st["k"][ch].astype(np.float64))
        assert row[:, 1].tobytes() == st["logl"][ch].tobytes()
        for j, t in enumerate(sig_t):
            assert row[:, 2 + j].tobytes() == st["sig"][ch, t].tobytes()
        assert tr["t0"][smp].tobytes() == r["temps"][ch].tobytes()
        cold = r["temps"] <= dgo.COLD
        for g, c in enumerate(ch):
            vs = row[g, 2 + len(sig_t):]
            if cold[c]:   # the chain's row of all_models, bit for bit
                model = r["vs_model"][r["nmod"] + int(np.sum(cold[:c]))]
                assert vs.tobytes() == model[bins - 1].tobytes()
            else:
                k = int(st["k"][c])
                want = dgo.recorded_vs(cfg, k, st["z"][c], st["dvp"][c], st["dvs"][c], bins)
                assert np.allclose(vs, want, rtol=1e-12, atol=0), (vs, want)
        smp += 1
    assert len(tr["trace"]) == smp > 0


def check_stats(tr, dg, trips_want):
    n = len(tr["trace"])
    rows = dgo.rows(tr["trace"], tr["t0"])
    got = np.stack([dg[k] for k in ("mean", "var", "tau", "ess", "mean_1", "var_1", "mean_2", "var_2")], axis=-1)
    assert np.array_equal(np.isnan(got), np.isnan(rows[:, :, :8]))
    assert np.allclose(got, rows[:, :, :8], rtol=1e-10, atol=0, equal_nan=True)
    assert np.array_equal(dg["tempered"], rows[:, 0, 8].astype(np.int64))
    s = dgo.summary(rows, n)
    got = np.stack([dg["rhat"], dg["ess_total"], dg["tau_median"], dg["tempered_share"]], axis=-1)
    assert np.array_equal(np.isnan(got), np.isnan(s))
    assert np.allclose(got, s, rtol=1e-10, atol=0, equal_nan=True)
    assert dg["n_samples"] == n
    assert np.array_equal(dg["trips"], trips_want)


def numpy_trips(cfg, rec, sweeping=lambda it: True):
    its = [r["it"] for r in rec if sweeping(r["it"])]
    temps = [r["temps"] for r in rec if sweeping(r["it"])]
    return dgo.round_trips(np.array(temps), cfg.nchains, its, cfg.nburn)[0]


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("variant", VARIANTS)
def test_trace_trips_and_statistics_match_numpy(variant, mode):
    cfg, nproc = diag_config(variant)
    rec, tr, dg = stepwise(cfg, nproc, cfg.nburn + cfg.niter, mode=mode)
    check_trace(cfg, nproc, rec, tr)
    want = numpy_trips(cfg, rec) if mode == 1 else np.zeros((nproc, 2), np.int64)
    check_stats(tr, dg, want)
    if mode == 1 and variant == "sample":
        assert dg["trips"].sum() > 0
    assert np.isfinite(dg["rhat"][:2]).all()   # k and logL (a bin inside the sea layer is constant: R-hat NaN)


@pytest.mark.parametrize("ladder,steps", [(1, 0), (0, 1), (1, 1)])
def test_round_trips_with_tunings(ladder, steps):
    cfg, nproc = diag_config("sample", nburn=130, niter=40, ncorr=2)   # tuning points 64 and 128
    rec, tr, dg = stepwise(cfg, nproc, cfg.nburn + cfg.niter, mode=1, ladder=ladder, steps=steps)
    check_trace(cfg, nproc, rec, tr)
    check_stats(tr, dg, numpy_trips(cfg, rec))


def _full(cfg, nproc, n, diag, **kw):
    pt = ParallelTempering(cfg, nproc)
    try:
        setup(pt, diag=diag, **kw)
        pt.set_logging(n)
        pt.run(n)
        out = snapshot(pt)
        out.update({"log_" + str(i): a for i, a in enumerate(pt.log(n))})
        rs = pt.rank_swaps()
        out.update(rs_n_prop=rs["n_prop"], rs_n_acc=rs["n_acc"])
        if kw.get("steps"):
            out.update({"st_" + k: np.asarray(v) for k, v in pt.step_tuning().items()})
        return out
    finally:
        pt.close()


@pytest.mark.parametrize("mode,ladder,steps", [(0, 0, 0), (1, 0, 0), (1, 1, 1)])
def test_the_run_is_unchanged(mode, ladder, steps):
    cfg, nproc = diag_config("sample", nburn=130, niter=60, ncorr=2)
    on = _full(cfg, nproc, 190, 1, mode=mode, ladder=ladder, steps=steps)
    off = _full(cfg, nproc, 190, 0, mode=mode, ladder=ladder, steps=steps)
    assert_identical(on, off)


def _diag_bytes(pt):
    tr, dg = pt.cold_trace(), pt.diagnostics()
    parts = [tr["trace"], tr["t0"], dg["trips"]] + [dg[k] for k in ("mean", "var", "tau", "ess", "rhat", "ess_total", "tau_median",
                                                                      "tempered_share")]
    return b"".join(np.ascontiguousarray(p).tobytes() for p in parts)


def test_resume_equals_uninterrupted_and_refusals(tmp_path):
    cfg, nproc = diag_config("sigma_solved_vp_solved", nburn=30, niter=80, ncorr=3)
    n1, n = 57, 110
    ref = ParallelTempering(cfg, nproc)
    setup(ref, mode=1)
    ref.run(n)
    want, want_snap = _diag_bytes(ref), snapshot(ref)
    ref.close()
    path = str(tmp_path / "a.ck")
    a = ParallelTempering(cfg, nproc)
    setup(a, mode=1)
    a.run(n1)
    a.save(path)
    a.close()
    b = ParallelTempering(cfg, nproc)
    setup(b, mode=1)
    b.restore(path)
    b.run(n - n1)
    assert _diag_bytes(b) == want
    assert_identical(snapshot(b), want_snap)
    b.close()
    for diag, bins in ((0, None), (1, [2, 5])):   # the setting and the bins must match the file's
        c = ParallelTempering(cfg, nproc)
        try:
            setup(c, mode=1, diag=diag, bins=bins)
            with pytest.raises(capi.RfinvError) as e:
                c.restore(path)
            assert e.value.status == capi.RFINV_ERR_ARG and "diagnostic" in str(e.value)
        finally:
            c.close()
    # a file written without them keeps the sections of a library without them: a handle with them refuses it
    path0 = str(tmp_path / "off.ck")
    d = ParallelTempering(cfg, nproc)
    setup(d, mode=1, diag=0)
    d.run(n1)
    d.save(path0)
    d.close()
    e_ = ParallelTempering(cfg, nproc)
    try:
        setup(e_, mode=1)
        with pytest.raises(capi.RfinvError) as e:
            e_.restore(path0)
        assert e.value.status == capi.RFINV_ERR_ARG
    finally:
        e_.close()


def test_refusals():
    cfg, nproc = diag_config("laplace_prior_joint_PS")
    pt = ParallelTempering(cfg, nproc)
    try:
        with pytest.raises(capi.RfinvError) as e:
            pt.diagnostics()
        assert e.value.status == capi.RFINV_ERR_STATE
        for bins in ([0], [cfg.nbin_z + 1], list(range(1, 18))):
            with pytest.raises(capi.RfinvError) as e:
                pt.set_diagnostics(1, bins)
            assert e.value.status == capi.RFINV_ERR_ARG
        with pytest.raises(capi.RfinvError) as e:
            pt.set_diagnostics(2)
        assert e.value.status == capi.RFINV_ERR_ARG
        pt.set_diagnostics(1, [1, 2])
        pt.run(3)
        with pytest.raises(capi.RfinvError) as e:
            pt.set_diagnostics(0)
        assert e.value.status == capi.RFINV_ERR_STATE
    finally:
        pt.close()
    cfg.niter = 0                                    # no bookkeeping: nothing to record with
    pt = ParallelTempering(cfg, nproc)
    try:
        with pytest.raises(capi.RfinvError) as e:
            pt.set_diagnostics(1)
        assert e.value.status == capi.RFINV_ERR_STATE and "bookkeeping" in str(e.value)
    finally:
        pt.close()


def test_group_member_equals_solo():
    ms = [diag_config("sample", 30, 60, 4), diag_config("sigma_solved_vp_solved", 30, 60, 4)]
    kws = [dict(mode=1), dict(mode=0, diag=0)]
    solo = []
    for (cfg, nproc), kw in zip(ms, kws):
        pt = ParallelTempering(cfg, nproc)
        setup(pt, **kw)
        pt.run(90)
        solo.append((snapshot(pt), _diag_bytes(pt) if kw.get("diag", 1) else None))
        pt.close()
    pts = [ParallelTempering(cfg, nproc) for cfg, nproc in ms]
    try:
        for pt, kw in zip(pts, kws):
            setup(pt, **kw)
        with PtGroup(pts) as g:
            g.run(50)
            g.run(40)
        for pt, (snap, db), kw in zip(pts, solo, kws):
            assert_identical(snapshot(pt), snap)
            if db is not None:
                assert _diag_bytes(pt) == db
    finally:
        for pt in pts:
            pt.close()


_NO_GRAPH_SCRIPT = r"""
import sys
sys.path[:0] = [{tests!r}, {root!r}, {oracle!r}]
import hashlib
from test_gpu_diagnostics import diag_config, setup, _diag_bytes
from rf_inv_b200.pt import ParallelTempering
cfg, nproc = diag_config("sample", 30, 60, 4)
pt = ParallelTempering(cfg, nproc)
setup(pt, mode=1)
pt.run(90)
print(hashlib.sha1(_diag_bytes(pt)).hexdigest())
pt.close()
"""


def test_plain_launches_equal_graph_replay():
    script = _NO_GRAPH_SCRIPT.format(tests=os.path.join(ROOT, "tests"), root=ROOT, oracle=os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, RFINV_PT_GRAPH="0"), capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    cfg, nproc = diag_config("sample", 30, 60, 4)
    pt = ParallelTempering(cfg, nproc)
    setup(pt, mode=1)
    pt.run(90)
    want = hashlib.sha1(_diag_bytes(pt)).hexdigest()
    pt.close()
    assert r.stdout.strip().splitlines()[-1] == want


def test_driver_writes_convergence_and_round_trips(tmp_path, capsys):
    from rf_inv_b200 import run as rrun
    paths = station_dirs(tmp_path / "src", 2, noise=0.01)
    for p in paths:
        set_param(p, "N_BURN", 40)
        set_param(p, "N_ITER", 160)
    d_rs, d_dg = tmp_path / "rs", tmp_path / "dg"
    shutil.copytree(os.path.dirname(paths[0]), d_rs)
    shutil.copytree(os.path.dirname(paths[0]), d_dg)
    rrun.main([str(d_rs / "params.in"), "--nproc", "4", "--rank-swaps"])
    rrun.main([str(d_dg / "params.in"), "--nproc", "4", "--rank-swaps", "--diagnostics", "--diag-depths", "5,12.5"])
    out = capsys.readouterr().out
    assert "R-hat" in out
    assert set(os.listdir(d_dg / "rslt")) == set(os.listdir(d_rs / "rslt")) | {"convergence", "round_trips"}
    for n in OUTPUT_FILES + ["rank_swaps"]:
        if n != "params.in.copy":
            assert filecmp.cmp(d_dg / "rslt" / n, d_rs / "rslt" / n, shallow=False), n
    lines = [l.split() for l in open(d_dg / "rslt" / "convergence")]
    names = [l[0] for l in lines]
    assert names[:2] == ["k", "logL"] and names[-2:] == ["vs_5", "vs_12.5"]
    assert all(int(l[1]) > 0 and int(l[2]) == 4 for l in lines)
    trips = np.loadtxt(d_dg / "rslt" / "round_trips", ndmin=2)
    assert trips.shape == (4, 3)
    # refused depths: above the surface, below Z_MAX, inside the sea layer (SEA_DEP 2 km); Z_MAX itself is the last bin
    assert rrun.depth_bins(rrun.rio.load_problem(str(d_dg / "params.in")), [20.0]) == [100]
    for bad in ("-1", "1e6", "1.0"):
        with pytest.raises(ValueError):
            rrun.main([str(d_dg / "params.in"), "--nproc", "4", "--diagnostics", "--diag-depths", bad])
    # two stations as a group: every station's files are those of its solo run
    solo = []
    for i, p in enumerate(paths):
        d = tmp_path / f"solo{i}"
        shutil.copytree(os.path.dirname(p), d)
        rrun.run(str(d / "params.in"), nproc=4, verbose=False, rank_swaps=True, diagnostics=True, diag_depths=[5.0])
        solo.append(d / "rslt")
    grp = []
    for i, p in enumerate(paths):
        d = tmp_path / f"grp{i}"
        shutil.copytree(os.path.dirname(p), d)
        grp.append(d)
    rrun.run_group([str(d / "params.in") for d in grp], nproc=4, verbose=False, rank_swaps=True, diagnostics=True,
                   diag_depths=[5.0])
    for d, s in zip(grp, solo):
        for n in OUTPUT_FILES + ["rank_swaps", "convergence", "round_trips"]:
            if n != "params.in.copy":
                assert filecmp.cmp(d / "rslt" / n, s / n, shallow=False), n


def test_split_driver_matches_single_process():
    """local_step / swap_table / apply_swap with two handles on one GPU: every handle's trace, round trips and per-rank rows
    are its ranks' share of those of rfinv_pt_run with one handle."""
    import torch
    from rf_inv_b200.pt import _tensor_from_ptr
    cfg, nproc = diag_config("sample", 20, 80, 2)
    n_iter = 100
    one = ParallelTempering(cfg, nproc)
    setup(one, mode=1)
    one.run(n_iter)
    tr1, dg1 = one.cold_trace(), one.diagnostics()
    one.close()
    parts = [ParallelTempering(cfg, nproc, world=2, rank=r) for r in range(2)]
    try:
        for p in parts:
            setup(p, mode=1)
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
        trs, dgs = [p.cold_trace() for p in parts], [p.diagnostics() for p in parts]
    finally:
        for p in parts:
            p.close()
    assert np.array_equal(np.concatenate([t["trace"] for t in trs], axis=1), tr1["trace"])
    assert np.array_equal(np.concatenate([t["t0"] for t in trs], axis=1), tr1["t0"])
    assert dg1["trips"].sum() > 0
    for key in ("trips", "mean", "var", "tau", "ess", "mean_1", "var_1", "mean_2", "var_2", "tempered"):
        assert np.concatenate([d[key] for d in dgs]).tobytes() == np.asarray(dg1[key]).tobytes(), key


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_processes_reproduce_the_single_process_run(exchange):
    """tools/dist_check.py --rank-swaps --diagnostics: every process's trace is its share of the single-process trace, and
    process 0's job-wide rows, summary and round trips after reduce_outputs equal those of one process, bit for bit."""
    if int(capi.load().rfinv_device_count()) < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, RFINV_PT_EXCHANGE=exchange, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29575" if exchange == "peer" else "29576", os.path.join(ROOT, "tools", "dist_check.py"),
           "--rank-swaps", "--diagnostics"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    for name, res in out.items():
        assert res["identical"], (name, res)


_LAUNCH_SCRIPT = r"""
import sys
sys.path[:0] = [{tests!r}, {root!r}, {oracle!r}]
import json
import re
import torch
from torch.profiler import ProfilerActivity, profile
from test_gpu_diagnostics import diag_config, setup
from rf_inv_b200.pt import ParallelTempering
torch.cuda.init()
cfg, nproc = diag_config("sample", 10, 40, 4)
out = {{}}
for mode in (0, 1):
    for diag in (0, 1):
        pt = ParallelTempering(cfg, nproc)
        setup(pt, mode=mode, diag=diag)
        pt.run(2)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            pt.run(40)
            pt.ev.synchronize()
        names = {{}}
        for e in prof.events():
            m = re.search(r"[a-z_]+_kernel", e.name) if e.device_type.name == "CUDA" else None
            if m:
                names[m.group(0)] = names.get(m.group(0), 0) + 1
        out[f"{{mode}}{{diag}}"] = names
        pt.close()
print(json.dumps(out))
"""


def test_launches_are_unchanged_with_the_diagnostics_off():
    """Plain launches (RFINV_PT_GRAPH=0), counted by the profiler over iterations 3 .. 42 (8 of them record): with the
    diagnostics on, the launch sequence gains exactly one pt_trace_kernel per recording iteration and nothing else; with them
    off no diagnostics kernel runs."""
    script = _LAUNCH_SCRIPT.format(tests=os.path.join(ROOT, "tests"), root=ROOT, oracle=os.path.join(ROOT, "oracle"))
    r = subprocess.run([sys.executable, "-c", script], env=dict(os.environ, RFINV_PT_GRAPH="0"), capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    for mode in (0, 1):
        off, on = out[f"{mode}0"], out[f"{mode}1"]
        assert off and not any(k.startswith("pt_trace") or k.startswith("pt_diag") for k in off), off
        assert sum(off.values()) >= 3 * 40
        recording = sum(1 for it in range(3, 43) if it > 10 and it % 4 == 0)
        extra = {k: on.get(k, 0) - off.get(k, 0) for k in set(on) | set(off)}
        assert {k: v for k, v in extra.items() if v} == {"pt_trace_kernel": recording}, extra
