"""The ladder tuning of the C reference (tests/ladder_oracle.c, DESIGN.md 7d), without a GPU: one rank against a Python
restatement of the contract and hand-computed ladders, the floor, the guard, the anchors, and the invariants of tuned runs."""
import numpy as np
import pytest

import helpers
import ladder_oracle as lo
import rank_swap_oracle as rso

FLOOR = 2.0 ** -10


def py_tune(temps, acc, base, e):
    """The contract step by step in Python floats (each operation rounded on its own, like the C reference)."""
    t = [float(x) for x in temps]
    n = len(t)
    at = sorted(range(n), key=lambda a: (t[a], a))
    c = sum(1 for x in t if x <= 1.0 + lo.COLD_EPS)
    a0, h = max(c - 1, 0), n - 1
    K = h - a0
    if K >= 2:
        s = 0 if e == 64 else e // 2
        P = float((e - s) // 2)
        lam = [0.0]
        for m in range(K):
            rho = 1.0 - float(acc[a0 + m] - base[a0 + m]) / P
            lam.append(lam[-1] + max(rho, FLOOR))
        beta = [1.0 / t[at[a0 + m]] for m in range(K + 1)]
        tn = [t[at[a0]]] + [0.0] * (K - 1) + [t[at[h]]]
        for k in range(1, K):
            x = (lam[K] * float(k)) / float(K)
            m = next((j for j in range(K) if x < lam[j + 1]), K - 1)
            f = (x - lam[m]) / (lam[m + 1] - lam[m])
            tn[k] = 1.0 / (beta[m] + (f * (beta[m + 1] - beta[m])))
        if all(tn[k] > tn[k - 1] for k in range(1, K + 1)) and all(x > 1.0 + lo.COLD_EPS for x in tn[1:K]):
            for k in range(1, K):
                t[at[a0 + k]] = tn[k]
    return np.array(t)


def check_rank(temps, acc, base, e):
    t, b, _ = lo.tune_rank(temps, acc, base, e)
    assert t.tobytes() == py_tune(temps, acc, base, e).tobytes()
    assert np.array_equal(b, acc)                                 # the snapshot, whatever happened
    return t


def test_known_ladder():
    # rejection 0.5, 0.25, 0.25 over the round of e = 64 (32 proposals per pair): barrier 0, 0.5, 0.75, 1; the new levels sit
    # at 1/3 and 2/3 of it -- beta 1 - (2/3)(1/2) = 2/3 and 1/2 - (2/3)(1/4) = 1/3
    t = check_rank([1.0, 2.0, 4.0, 8.0], [16, 24, 24], [0, 0, 0], 64)
    assert np.allclose(t, [1.0, 1.5, 3.0, 8.0], rtol=1e-14, atol=0)
    # the same rates in a later round: e = 256, s = 128, 64 proposals per pair, counted from the snapshot
    t = check_rank([8.0, 1.0, 4.0, 2.0], [100 + 32, 7 + 48, 50 + 48], [100, 7, 50], 256)
    assert np.allclose(t, [8.0, 1.0, 3.0, 1.5], rtol=1e-14, atol=0)


def test_equal_rates_leave_the_ladder():
    rng = np.random.default_rng(5)
    for n in (3, 5, 16):
        temps = np.concatenate([[1.0], np.sort(np.exp(rng.uniform(0.05, 1.0, n - 1) * np.log(30.0)))])
        rng.shuffle(temps)
        for q in (0, 7, 20, 32):
            t = check_rank(temps, [q] * (n - 1), [0] * (n - 1), 64)
            assert np.allclose(t, temps, rtol=1e-12, atol=0), (n, q)


def test_floor():
    # every pair always accepted: every rejection is the floor, all equal -- the ladder stays
    temps = [1.0, 1.7, 2.9, 5.0, 9.0]
    t = check_rank(temps, [32] * 4, [0] * 4, 64)
    assert np.allclose(t, temps, rtol=1e-12, atol=0)
    # one floored pair among rejections 0.5: barrier 0, 2^-10, 0.5 + 2^-10, 1 + 2^-10
    t = check_rank([1.0, 2.0, 4.0, 8.0], [32, 16, 16], [0, 0, 0], 64)
    L = 1.0 + FLOOR
    b1 = 0.5 - (L / 3 - FLOOR) / 0.5 * 0.25
    b2 = 0.25 - (2 * L / 3 - 0.5 - FLOOR) / 0.5 * 0.125
    assert np.allclose(t, [1.0, 1 / b1, 1 / b2, 8.0], rtol=1e-13, atol=0)


def test_guard():
    # a retuned level would fall to the cold test's threshold: the rank keeps its ladder
    temps = [1.0, 1.0 + 2e-6, 1.0 + 4e-6, 8.0]
    t, b, changed = lo.tune_rank(temps, [0, 32, 32], [0, 0, 0], 64)
    assert not changed and t.tobytes() == np.array(temps).tobytes() and np.array_equal(b, [0, 32, 32])
    assert t.tobytes() == py_tune(temps, [0, 32, 32], [0, 0, 0], 64).tobytes()
    # two equal temperatures above the cold level: the new ladder would not be strictly increasing
    temps = [1.0, 2.0, 2.0, 2.0, 6.0]
    t, _, changed = lo.tune_rank(temps, [10, 10, 10, 10], [0] * 4, 64)
    assert not changed and t.tobytes() == np.array(temps).tobytes()


@pytest.mark.parametrize("temps", [[1.0, 3.0], [1.0, 1.0, 5.0], [1.0, 1.0, 1.0, 2.0]])
def test_fewer_than_two_free_levels(temps):
    """K < 2: the rank is left alone, its snapshot still taken."""
    n = len(temps)
    acc = list(range(3, 3 + n - 1))
    t, b, changed = lo.tune_rank(temps, acc, [0] * (n - 1), 64)
    assert not changed and t.tobytes() == np.array(temps).tobytes() and np.array_equal(b, acc)


@pytest.mark.parametrize("n_cold", [0, 1, 2])
def test_anchors_and_cold_chains(n_cold):
    rng = np.random.default_rng(11 + n_cold)
    n = 7
    hot = np.sort(np.exp(rng.uniform(0.02, 1.0, n - n_cold) * np.log(50.0)))
    temps = np.concatenate([np.ones(n_cold), hot])
    perm = rng.permutation(n)
    temps = temps[perm]
    acc = rng.integers(0, 33, n - 1)
    t = check_rank(temps, acc, np.zeros(n - 1, np.int64), 64)
    order, new_order = np.lexsort((np.arange(n), temps)), np.lexsort((np.arange(n), t))
    assert np.array_equal(order, new_order)                          # level order preserved
    a0 = max(n_cold - 1, 0)
    assert np.array_equal(t[order[:a0 + 1]], temps[order[:a0 + 1]])  # cold chains and the anchor
    assert t[order[-1]] == temps[order[-1]]                          # the hottest level
    assert int(np.sum(t <= 1.0 + lo.COLD_EPS)) == n_cold
    assert not np.array_equal(t, temps)


def _config(**kw):
    d = dict(nfft=64, nsmp=40, nchains=6, ncool=1, t_high=20.0, iseed=1618)
    d.update(kw)
    cfg = helpers.attach_obs_and_rinv(helpers.small_config(**d), noise=0.01)
    return cfg


def _undo_swap(temps, swap):
    """The temperatures before the global swap of an iteration, from its log entry (itarget1, itarget2, accepted)."""
    t = temps.copy()
    if swap[2]:
        t[swap[0]], t[swap[1]] = t[swap[1]], t[swap[0]]
    return t


def _tuned_run_to(cfg, nproc, n, tune_last=True):
    """A tuned run of n iterations, the last one with the tuning switched on or off: (temps after the run, temps before the
    last global swap, rows and base before the last iteration, ladder_tuning())."""
    orc = lo.LadderOraclePT(cfg, nproc)
    try:
        orc.set_rank_swaps(1)
        orc.set_ladder_tuning(1)
        orc.run(n - 1, log=False)
        base = orc.base.copy()
        orc.set_ladder_tuning(tune_last)
        _, _, swaps = orc.run(1)
        t = orc.state()["temps"]
        return t, _undo_swap(t, swaps[0]), orc.rows.copy(), base, orc.ladder_tuning()
    finally:
        orc.close()


def test_tuned_run_at_the_tuning_points():
    """At every tuning point each rank's ladder is lo_tune_rank of the ladder the sweep left: anchors and level order kept."""
    cfg = _config()
    cfg.nburn, cfg.niter = 300, 100
    nproc, nc = 4, cfg.nchains
    assert lo.tuning_points(cfg.nburn) == [64, 128, 256]
    moved = 0
    for e in lo.tuning_points(cfg.nburn):
        _, tuned, rows, base, (_, n_points) = _tuned_run_to(cfg, nproc, e, True)
        _, plain, rows_p, _, _ = _tuned_run_to(cfg, nproc, e, False)
        assert n_points == lo.tuning_points(cfg.nburn).index(e) + 1
        assert np.array_equal(rows, rows_p)
        for r in range(nproc):
            sl, rl = slice(r * nc, (r + 1) * nc), slice(r * (nc - 1), (r + 1) * (nc - 1))
            want, _, _ = lo.tune_rank(plain[sl], rows[rl], base[rl], e)
            assert want.tobytes() == tuned[sl].tobytes(), (e, r)
            order = np.lexsort((np.arange(nc), plain[sl]))
            assert np.array_equal(order, np.lexsort((np.arange(nc), tuned[sl])))
            c = int(np.sum(plain[sl] <= 1.0 + lo.COLD_EPS))
            keep = np.concatenate([order[:max(c - 1, 0) + 1], order[-1:]])
            assert np.array_equal(tuned[sl][keep], plain[sl][keep])
            moved += int(not np.array_equal(tuned[sl], plain[sl]))
    assert moved >= nproc


def test_tuned_run_invariants():
    cfg = _config()
    cfg.nburn, cfg.niter = 300, 100
    nproc = 4
    points = lo.tuning_points(cfg.nburn)
    orc = lo.LadderOraclePT(cfg, nproc)
    try:
        orc.set_rank_swaps(1)
        orc.set_ladder_tuning(1)
        t0 = orc.state()["temps"]
        n_cold = int(np.sum(t0 <= 1.0 + lo.COLD_EPS))
        assert n_cold == nproc * cfg.ncool
        prev, frozen = t0, None
        for done in range(1, cfg.nburn + cfg.niter + 1):
            orc.run(1, log=False)
            t = orc.state()["temps"]
            assert int(np.sum(t <= 1.0 + lo.COLD_EPS)) == n_cold   # the job's T = 1 chains
            if done not in points:                                  # swaps only exchange values
                assert np.array_equal(np.sort(t), np.sort(prev)), done
            if done >= points[-1]:                                  # after the last point the ladders stay
                frozen = np.sort(t) if frozen is None else frozen
                assert np.array_equal(np.sort(t), frozen)
            prev = t
        assert orc.ladder_tuning() == (True, len(points))
        assert not np.array_equal(np.sort(prev), np.sort(t0))
    finally:
        orc.close()


def test_tuned_equals_mode1_before_the_first_point_and_with_short_burn_in():
    """nburn < 64 has no tuning point: a tuned run is the mode-1 run byte for byte; so is any run up to iteration 63."""
    for nburn, n_iter in ((40, 120), (500, 63)):
        cfg = _config(nchains=4)
        cfg.nburn, cfg.niter = nburn, 200
        nproc = 3
        out = []
        for tune in (0, 1):
            orc = lo.LadderOraclePT(cfg, nproc) if tune else rso.RankSwapOraclePT(cfg, nproc)
            orc.set_rank_swaps(1)
            if tune:
                orc.set_ladder_tuning(1)
            logs = orc.run(n_iter)
            out.append((logs, orc.state(), orc.counters(n_iter), orc.rank_swaps()))
            if tune:
                assert orc.ladder_tuning() == (True, 0)
            orc.close()                     # before the next handle: RFConfig.to_c keeps only its latest buffers alive
        (la, sa, ca, ra), (lb, sb, cb, rb) = out
        for x, y in zip(la, lb):
            assert x.tobytes() == y.tobytes()
        for key in sa:
            assert sa[key].tobytes() == sb[key].tobytes(), key
        for key in ("nprop", "naccept", "likelihood_hist"):
            assert ca[key].tobytes() == cb[key].tobytes(), key
        for key in ("n_prop", "n_acc"):
            assert ra[key].tobytes() == rb[key].tobytes(), key
