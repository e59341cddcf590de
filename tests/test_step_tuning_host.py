"""The random-walk width tuning of the C reference (tests/step_oracle.c, DESIGN.md 7e), without a GPU: one rank against a
Python restatement of the rule, the copied chain step against the restatement's, runs without tuning against lo_pt_run, and
the invariants of tuned runs."""
import numpy as np
import pytest

import helpers
import ladder_oracle as lo
import oracle_c
import step_oracle as so


def py_tune(scale, n_prop, n_acc, proposed, target):
    """The rule in Python floats, each operation rounded on its own like the C reference."""
    s = np.array(scale, dtype=np.float64)
    for (l, t), P in np.ndenumerate(np.asarray(n_prop)):
        if proposed[t] and P >= so.MIN_PROPOSALS:
            f = min(max((float(n_acc[l][t]) / float(P)) / target, 0.5), 2.0)
            s[l, t] = min(max(s[l, t] * f, so.SCALE_MIN), so.SCALE_MAX)
    return s


def check_rank(scale, n_prop, n_acc, proposed, target=0.44):
    s, p, a = so.tune_rank(scale, n_prop, n_acc, proposed, target)
    assert s.tobytes() == py_tune(scale, n_prop, n_acc, proposed, target).tobytes()
    assert not p.any() and not a.any()                       # the counters restart, whatever happened
    return s


def test_tune_rank_rule():
    rng = np.random.default_rng(3)
    for target in (0.44, 0.23, 0.7):
        n_prop = rng.integers(0, 80, (6, 4))
        n_acc = (n_prop * rng.uniform(0, 1, (6, 4))).astype(np.int64)
        scale = np.exp(rng.uniform(-3, 3, (6, 4)))
        check_rank(scale, n_prop, n_acc, [1, 1, 1, 1], target)
    # by hand: below 16 proposals kept; acceptance = target kept; factor 1/2 and 2 at the clamps
    s = check_rank(np.ones((1, 4)), [[15, 25, 32, 32]], [[15, 11, 0, 32]], [1, 1, 1, 1], 0.44)
    assert s.tolist() == [[1.0, 1.0, 0.5, 2.0]]
    s = check_rank(np.ones((1, 4)), [[32, 32, 32, 32]], [[16, 8, 4, 20]], [1, 1, 1, 1], 0.5)
    assert s.tolist() == [[1.0, 0.5, 0.5, 1.25]]


def test_tune_rank_scale_clamps_and_absent_types():
    s = check_rank([[2.0 ** -8 * 1.5, 2.0 ** 8 / 1.5, 3.0, 3.0]], [[64] * 4], [[0, 64, 64, 64]], [1, 1, 0, 0])
    assert s.tolist() == [[2.0 ** -8, 2.0 ** 8, 3.0, 3.0]]   # the lower and upper clamp; dVp and sigma not proposed


def _config(**kw):
    d = dict(nfft=64, nsmp=40, nchains=6, ncool=1, t_high=20.0, iseed=1618)
    d.update(kw)
    return helpers.attach_obs_and_rinv(helpers.small_config(**d), noise=0.01)


def test_copied_step_with_scale_one_is_mcmc_step():
    cfg, cfg_b = _config(), _config()   # one config each: RFConfig.to_c keeps only its latest buffers alive
    dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])
    a, b = oracle_c.OraclePT(cfg, 2), oracle_c.OraclePT(cfg_b, 2)
    try:
        t = oracle_c.i32p
        for i in range(200):
            r, ic = i % 2, (i * 5) % cfg.nchains
            ta, tb = np.zeros(1, np.int32), np.zeros(1, np.int32)
            fa = so.lib().so_step(a._h, r, ic, dev.ctypes.data_as(oracle_c.dp), 0, ta.ctypes.data_as(t))
            fb = so.lib().so_step(b._h, r, ic, (dev * 1.0).ctypes.data_as(oracle_c.dp), 1, tb.ctypes.data_as(t))
            assert (fa, ta[0]) == (fb, tb[0])
        sa, sb = a.state(), b.state()
        for key in sa:
            assert sa[key].tobytes() == sb[key].tobytes(), key
    finally:
        a.close(); b.close()


def _run(cfg, nproc, n, steps, tune=0, ladder_cls=False):
    orc = lo.LadderOraclePT(cfg, nproc) if ladder_cls else so.StepOraclePT(cfg, nproc)
    try:
        orc.set_rank_swaps(1)
        if tune:
            orc.set_ladder_tuning(1)
        if steps:
            orc.set_step_tuning(1)
        logs = orc.run(n)
        return logs, orc.state(), orc.counters(n), orc.rank_swaps(), orc.ladder_tuning()
    finally:
        orc.close()


@pytest.mark.parametrize("nburn,n", [(300, 150), (40, 120)])
def test_untuned_and_short_burn_in_equal_lo_pt_run(nburn, n):
    """steps off (any burn-in), or on with nburn < 64: lo_pt_run byte for byte, with and without the ladder tuning."""
    cfg = _config(nchains=4)
    cfg.nburn, cfg.niter = nburn, 200
    for tune in (0, 1):
        want = _run(cfg, 3, n, 0, tune, ladder_cls=True)
        for steps in ((0, 1) if nburn < 64 else (0,)):
            got = _run(cfg, 3, n, steps, tune)
            for x, y in zip(got[0], want[0]):
                assert x.tobytes() == y.tobytes()
            for key in want[1]:
                assert got[1][key].tobytes() == want[1][key].tobytes(), key
            for key in ("nprop", "naccept", "likelihood_hist"):
                assert got[2][key].tobytes() == want[2][key].tobytes(), key
            for key in ("n_prop", "n_acc"):
                assert got[3][key].tobytes() == want[3][key].tobytes(), key
            assert got[4] == want[4]


def _levels(temps, nc):
    t = temps.reshape(-1, nc)
    order = np.lexsort((np.broadcast_to(np.arange(nc), t.shape), t), axis=1)
    lvl = np.empty_like(order)
    np.put_along_axis(lvl, order, np.arange(nc)[None, :].repeat(t.shape[0], 0), axis=1)
    return lvl.ravel()


@pytest.mark.parametrize("tune", [0, 1])
def test_tuned_run_invariants(tune):
    cfg = _config()
    cfg.nburn, cfg.niter = 300, 60
    nproc, nc = 4, cfg.nchains
    points = lo.tuning_points(cfg.nburn)
    orc = so.StepOraclePT(cfg, nproc)
    try:
        orc.set_rank_swaps(1)
        if tune:
            orc.set_ladder_tuning(1)
        orc.set_step_tuning(1, 0.44)
        t0 = orc.state()["temps"]
        assert np.array_equal(orc.lvl, _levels(t0, nc))
        n_cold = int(np.sum(t0 <= 1.0 + lo.COLD_EPS))
        prev_scale, prev_swap = orc.scale.copy(), None
        for done in range(1, cfg.nburn + cfg.niter + 1):
            _, _, swaps = orc.run(1)
            t = orc.state()["temps"]
            # lvl: the post-sweep levels, i.e. those of the temperatures before this iteration's global swap
            before = t.copy()
            if swaps[0, 2]:
                before[swaps[0, 0]], before[swaps[0, 1]] = before[swaps[0, 1]], before[swaps[0, 0]]
            assert np.array_equal(orc.lvl, _levels(before, nc)), done
            # the chains under the pair rule are exactly the previous iteration's global pair
            want = np.zeros(orc.G, np.int8)
            if prev_swap is not None:
                want[prev_swap[:2]] = 1
            assert np.array_equal(orc.pairlog[0], want), done
            prev_swap = swaps[0].copy()
            assert tuple(orc.pair) == tuple(swaps[0, :2])
            assert int(np.sum(t <= 1.0 + lo.COLD_EPS)) == n_cold   # the job's T = 1 chains
            if done not in points:                                  # scales move only at the tuning points
                assert np.array_equal(orc.scale, prev_scale), done
            else:
                assert not orc.st_nprop.any() and not orc.st_nacc.any()
            prev_scale = orc.scale.copy()
        st = orc.step_tuning()
        assert st["n_points"] == len(points) and st["on"]
        assert not np.all(orc.scale == 1.0)
        assert np.all((orc.scale >= so.SCALE_MIN) & (orc.scale <= so.SCALE_MAX))
        # counters since the last point: one proposal per chain and iteration at most, acceptances <= proposals
        assert orc.st_nprop.sum() <= (cfg.nburn + cfg.niter - points[-1]) * orc.G
        assert np.all(orc.st_nacc <= orc.st_nprop)
    finally:
        orc.close()


def test_scales_at_a_tuning_point_are_so_tune_rank_of_the_round():
    """At e = 128 every rank's scales are so_tune_rank of the counts of [64, 128): those of the same run with nburn = 127, which
    passes 64 alike but not 128."""
    cfg = _config()
    cfg.nburn, cfg.niter = 140, 10
    nproc = 3
    sig = any(cfg.sig_max[t] - cfg.sig_min[t] > float(np.float32(1.0e-5)) for t in range(cfg.ntrc))
    proposed = [1, 1, int(cfg.vp_mode == 1), int(sig)]
    runs = []
    for nburn in (140, 127):
        cfg.nburn = nburn
        orc = so.StepOraclePT(cfg, nproc)
        try:
            orc.set_rank_swaps(1)
            orc.set_step_tuning(1, 0.3)
            orc.run(127, log=False)
            before = orc.scale.copy()
            orc.run(1, log=False)
            runs.append((before, orc.scale.copy(), orc.st_nprop.copy(), orc.st_nacc.copy(), orc.step_tuning()["n_points"]))
        finally:
            orc.close()
    (before, tuned, _, _, n2), (before_b, kept, nprop, nacc, n1) = runs
    assert (n2, n1) == (2, 1) and before.tobytes() == before_b.tobytes() and kept.tobytes() == before.tobytes()
    assert nprop.sum() > 0 and not np.array_equal(tuned, before)
    for r in range(nproc):
        assert tuned[r].tobytes() == check_rank(before[r], nprop[r], nacc[r], proposed, 0.3).tobytes(), r
