"""Checkpoint and resume of parallel-tempering runs (rfinv_pt_save / rfinv_pt_restore): run(N1); save; restore into a new
handle; run(N2) must give exactly the bits of run(N1 + N2) -- chain state, counters, evaluations, likelihood history,
histograms, means, recorded models and the per-iteration logs.  "Identical" is np.array_equal, no tolerance -- except for
the profile means (vp_mean, vs_mean, vpvs_mean): pt_record_kernel adds them with double-precision atomics from one CTA per
chain, so their last bits depend on the order the CTAs arrive in, also between two uninterrupted runs.  They are compared
to 1e-12 like in tests/test_gpu_pt.py."""
import copy
import filecmp
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import helpers
from rf_inv_b200 import capi, workloads
from rf_inv_b200.evaluator import Evaluator
from rf_inv_b200.pt import ParallelTempering

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def variant_config(name):
    """(cfg, nproc, [N1 splits], N) -- the variants tests/test_gpu_pt.py runs against the oracle."""
    if name == "sample_bookkeeping":     # recording on: one split inside the burn-in, one inside recording off an ncorr multiple
        cfg = workloads.make_config("sample")
        cfg.nburn, cfg.niter, cfg.ncorr = 30, 60, 4
        return helpers.attach_obs_and_rinv(cfg, noise=0.01), 20, [17, 47], 90
    if name == "sigma_solved_vp_solved":
        cfg = helpers.small_config(sdep=2.0, vp_mode=1, rayps=[0.06, 0.06], a_gus=[2.5, 4.0], nfft=128, nsmp=64,
                                   sig_min=[0.005, 0.01], sig_max=[0.05, 0.01], nchains=4, ncool=2, t_high=10.0, iseed=777)
        nproc, splits, n = 6, [53], 120
    elif name == "laplace_prior_joint_PS":
        cfg = helpers.small_config(prior_mode=1, dvs_prior=0.3, dvp_prior=0.1, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.10],
                                   nfft=128, nsmp=64, nchains=3, ncool=1, t_high=5.0, iseed=4242)
        nproc, splits, n = 5, [61], 120
    elif name == "transform_length_250":
        cfg = helpers.small_config(sdep=1.0, nfft=250, nsmp=101, nchains=4, ncool=1, t_high=8.0, iseed=31337)
        nproc, splits, n = 5, [37], 80
    else:                                # single_chain_per_rank
        cfg = helpers.small_config(nfft=64, nsmp=40, nchains=1, ncool=1, iseed=99)
        nproc, splits, n = 8, [29], 60
    return helpers.attach_obs_and_rinv(cfg, noise=0.01), nproc, splits, n


def snapshot(pt):
    out = dict(pt.state())
    cnt = pt.counters()
    out.update(nprop=cnt["nprop"], naccept=cnt["naccept"], likelihood_hist=cnt["likelihood_hist"],
               n_eval=np.int64(cnt["n_eval"]), it=np.int64(pt.iterations_done))
    if pt.cfg.niter > 0:
        out.update({"hist_" + k: np.asarray(v) for k, v in pt.hist().items()})
        out["vp_model"], out["vs_model"] = pt.models()
    return out


MEANS = ("hist_vp_mean", "hist_vs_mean", "hist_vpvs_mean")


def assert_identical(a, b):
    assert a.keys() == b.keys()
    for k in a:
        if k in MEANS:
            assert np.allclose(a[k], b[k], rtol=1e-12, atol=0), k
        else:
            assert np.array_equal(a[k], b[k]), k


def uninterrupted(cfg, nproc, n):
    pt = ParallelTempering(cfg, nproc)
    pt.set_logging(n)
    pt.run(n)
    out, logs = snapshot(pt), pt.log(n)
    pt.close()
    return out, logs


def split_run(cfg, nproc, n1, n2, path, cfg2=None):
    a = ParallelTempering(cfg, nproc)
    a.run(n1)
    a.save(path)
    a.close()
    b = ParallelTempering(cfg2 or cfg, nproc)
    b.restore(path)
    assert b.iterations_done == n1
    b.set_logging(n2)
    b.run(n2)
    out, logs = snapshot(b), b.log(n2)
    b.close()
    return out, logs


@pytest.mark.parametrize("variant", ["sample_bookkeeping", "sigma_solved_vp_solved", "laplace_prior_joint_PS",
                                     "transform_length_250", "single_chain_per_rank"])
def test_resume_equals_uninterrupted_run(variant, tmp_path):
    cfg, nproc, splits, n = variant_config(variant)
    ref, ref_logs = uninterrupted(cfg, nproc, n)
    if cfg.niter > 0:
        assert ref["hist_nmod"] > 0 and len(ref["vp_model"]) == ref["hist_nmod"]
    for n1 in splits:
        got, logs = split_run(cfg, nproc, n1, n - n1, str(tmp_path / f"ck{n1}"))
        assert_identical(got, ref)
        for mine, whole in zip(logs, ref_logs):
            assert np.array_equal(mine, whole[n1:]), n1


def test_save_restore_save_is_byte_identical(tmp_path):
    cfg, nproc, _, _ = variant_config("sample_bookkeeping")
    a = ParallelTempering(cfg, nproc)
    a.run(47)
    a.save(str(tmp_path / "one"))
    a.close()
    b = ParallelTempering(cfg, nproc)
    b.restore(str(tmp_path / "one"))
    b.save(str(tmp_path / "two"))
    b.close()
    assert filecmp.cmp(tmp_path / "one", tmp_path / "two", shallow=False)
    assert not os.path.exists(tmp_path / "one.tmp")


def test_niter_may_grow(tmp_path):
    """A run of N_ITER = N saved at its end continues under N_ITER = 2N exactly like a run that had 2N from the start."""
    cfg, nproc, _, _ = variant_config("sample_bookkeeping")
    cfg.nburn, cfg.niter, cfg.ncorr = 20, 40, 4
    big = copy.deepcopy(cfg)
    big.niter = 80
    ref, ref_logs = uninterrupted(big, nproc, 100)
    got, logs = split_run(cfg, nproc, 60, 40, str(tmp_path / "ck"), cfg2=big)
    assert_identical(got, ref)
    assert got["hist_nmod"] == (80 // 4) * nproc * cfg.ncool and len(got["vp_model"]) == got["hist_nmod"]
    for mine, whole in zip(logs, ref_logs):
        assert np.array_equal(mine, whole[60:])


@pytest.fixture(scope="module")
def saved(tmp_path_factory):
    """A checkpoint of the sample configuration (bookkeeping on) after 25 iterations."""
    cfg, nproc, _, _ = variant_config("sample_bookkeeping")
    path = str(tmp_path_factory.mktemp("ck") / "ck")
    pt = ParallelTempering(cfg, nproc)
    pt.run(25)
    pt.save(path)
    st = pt.state()
    pt.close()
    return cfg, nproc, path, st


def refused(cfg, nproc, path, status, words, **kw):
    pt = ParallelTempering(cfg, nproc, **kw)
    try:
        with pytest.raises(capi.RfinvError) as e:
            pt.restore(path)
        assert e.value.status == status, str(e.value)
        for w in words:
            assert w in str(e.value), (w, str(e.value))
        assert pt.iterations_done == 0
    finally:
        pt.close()


def test_restore_refuses_what_does_not_fit(saved, tmp_path):
    cfg, nproc, path, _ = saved
    c = copy.deepcopy(cfg); c.obs = cfg.obs.copy(); c.obs[1, 17] += 1e-3
    refused(c, nproc, path, capi.RFINV_ERR_ARG, ["observed traces"])
    c = copy.deepcopy(cfg); c.a_gus = [4.0, 3.0]
    refused(c, nproc, path, capi.RFINV_ERR_ARG, ["a_gus"])
    refused(cfg, nproc * 2, path, capi.RFINV_ERR_ARG, ["virtual ranks"])
    refused(cfg, nproc, path, capi.RFINV_ERR_ARG, ["virtual ranks"], world=2, rank=0)
    c = copy.deepcopy(cfg); c.nchains = 4
    refused(c, nproc, path, capi.RFINV_ERR_ARG, ["nchains"])
    c = copy.deepcopy(cfg); c.niter = cfg.niter - 4
    refused(c, nproc, path, capi.RFINV_ERR_ARG, ["niter"])
    data = open(path, "rb").read()
    (tmp_path / "short").write_bytes(data[: len(data) // 2])
    refused(cfg, nproc, str(tmp_path / "short"), capi.RFINV_ERR_IO, ["short"])
    flipped = bytearray(data); flipped[136 + 32 + 100] ^= 0x10      # a word of the first section (mt): header 136 B, section 32 B
    (tmp_path / "flipped").write_bytes(bytes(flipped))
    refused(cfg, nproc, str(tmp_path / "flipped"), capi.RFINV_ERR_IO, ["checksum"])
    refused(cfg, nproc, str(tmp_path / "missing"), capi.RFINV_ERR_IO, ["No such file"])


def test_save_and_restore_refuse_out_of_order_calls(saved, tmp_path):
    cfg, nproc, path, _ = saved
    lib = capi.load()
    with Evaluator(cfg) as ev:                                   # no rfinv_pt_init
        assert lib.rfinv_pt_restore(ev.handle, path.encode()) == capi.RFINV_ERR_STATE
        assert lib.rfinv_pt_save(ev.handle, str(tmp_path / "x").encode()) == capi.RFINV_ERR_STATE
    pt = ParallelTempering(cfg, nproc)
    try:
        pt.run(1)                                                # an iteration has run
        with pytest.raises(capi.RfinvError) as e:
            pt.restore(path)
        assert e.value.status == capi.RFINV_ERR_STATE
        capi.check(lib.rfinv_pt_local_step(pt.ev.handle))       # half an iteration
        with pytest.raises(capi.RfinvError) as e:
            pt.save(str(tmp_path / "mid"))
        assert e.value.status == capi.RFINV_ERR_STATE and "local_step" in str(e.value)
        ptr, _ = pt.swap_table()
        capi.check(lib.rfinv_pt_apply_swap(pt.ev.handle, ptr, 1))
        pt.save(str(tmp_path / "whole"))                         # the iteration is complete again
        pt.reduce_outputs()
        with pytest.raises(capi.RfinvError) as e:
            pt.save(str(tmp_path / "reduced"))
        assert e.value.status == capi.RFINV_ERR_STATE and "reduce_outputs" in str(e.value)
    finally:
        pt.close()
    assert not os.path.exists(tmp_path / "mid") and not os.path.exists(tmp_path / "reduced")


def test_restored_state_is_consistent(saved):
    """The likelihood of the restored models, evaluated afresh, is the restored logL."""
    cfg, nproc, path, st_saved = saved
    pt = ParallelTempering(cfg, nproc)
    pt.restore(path)
    st = pt.state()
    pt.close()
    for k in st:
        assert np.array_equal(st[k], st_saved[k]), k
    with Evaluator(cfg) as ev:
        ll = ev.calc_likelihood(st["k"], st["z"], st["dvp"], st["dvs"], st["sig"])
    ll = ll[0] if isinstance(ll, tuple) else ll
    assert helpers.logl_err(cfg, ll, st["logl"], st["sig"]) < 1e-12


def _problem_dir(d, cfg):
    """The problem directory of tests/test_gpu_pt.py::test_run_driver_writes_reference_output_set."""
    from rf_inv_b200 import io as rio
    (d / "data").mkdir(parents=True); (d / "model").mkdir()
    for t in range(2):
        rio.write_sac(str(d / "data" / f"s{t + 1}.trc"), cfg.obs[t], cfg.delta, 0.0)
    with open(d / "model" / "ref.velmod", "w") as f:
        for i in range(61):
            f.write(f"{0.5 * i} 5.00 2.89\n")
    vals = ["'./rslt'", 40, 120, 10, 5, 1, 15.0, 12345678, 2, 0.06, 0.08, 4.0, 4.0, 1, 1, 256, "'data/s1.trc'", "'data/s2.trc'",
            "0.0 5.0", 0, 2.0, '"model/ref.velmod"', 0, "1 10", "0.0 20.0", 0.05, 2, 2.0, 0.2, "0.01 0.01", "0.01 0.01", 0.02, 0.02,
            0.02, 0.002, 100, 50, 50, 100, 50, 100, "-0.8 0.8", "0.1 8.6", "0.001 5.0", "0.0 5.0"]
    (d / "params.in").write_text("# test problem in the reference's params.in format\n" + "\n".join(str(v) for v in vals) + "\n")


def test_run_driver_resume_writes_identical_output_files(tmp_path):
    from rf_inv_b200 import run as rrun
    cfg = helpers.attach_obs_and_rinv(workloads.make_config("sample"), noise=0.01)
    a, b = tmp_path / "resumed", tmp_path / "fresh"
    _problem_dir(a, cfg)
    shutil.copytree(a, b)
    ck = str(a / "state.ck")
    # a missing checkpoint starts a fresh run; the second call continues the first (N_BURN + N_ITER = 160)
    rrun.run(str(a / "params.in"), nproc=4, verbose=False, n_iter=70, checkpoint=ck, resume=True)
    assert os.path.exists(ck)
    rrun.run(str(a / "params.in"), nproc=4, verbose=False, checkpoint=ck, resume=True)
    rrun.run(str(b / "params.in"), nproc=4, verbose=False)
    names = ["params.in.copy", "all_models", "likelihood", "num_interface.ppd", "syn_trace.ppd", "interface_depth.ppd",
             "sigma.ppd", "vs_z.ppd", "vp_z.ppd", "vpvs_z.ppd", "vs_z.mean", "vp_z.mean", "vpvs_z.mean"]
    for n in names:
        assert filecmp.cmp(a / "rslt" / n, b / "rslt" / n, shallow=False), n
    assert os.path.getsize(b / "rslt" / "all_models") > 0


def _gpus():
    return int(capi.load().rfinv_device_count())


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
def test_two_processes_resume_equals_uninterrupted_run(exchange, tmp_path):
    if _gpus() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ, RFINV_PT_EXCHANGE=exchange, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541" if exchange == "peer" else "29542", os.path.join(ROOT, "tools", "checkpoint_check.py"),
           str(tmp_path)]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads([line for line in r.stdout.splitlines() if line.startswith("{")][-1])
    assert out["identical"], out
    assert out["cross_restore_refused"], out
    assert out["exchange"] == ("peer memory" if exchange == "peer" else "nccl all-gather")
