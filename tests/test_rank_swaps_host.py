"""The rank sweep on top of the C restatement (tests/rank_swap_oracle.c, DESIGN.md 7c), without a GPU: its Philox4x64-10
against numpy's, the invariants of a mode-1 run, and mode 0 as the restatement's own run."""
import numpy as np
import pytest

import helpers
import oracle_c
import rank_swap_oracle as rso


def _minus_one(counter):
    """counter - 1 over the 256-bit counter (word 0 least significant), with borrow: numpy's Philox increments before it
    generates."""
    v = sum(int(w) << (64 * i) for i, w in enumerate(counter))
    v = (v - 1) % (1 << 256)
    return np.array([(v >> (64 * i)) & ((1 << 64) - 1) for i in range(4)], dtype=np.uint64)


def test_philox_matches_numpy():
    rng = np.random.default_rng(2026)
    counters = [rng.integers(0, 2**64, size=4, dtype=np.uint64) for _ in range(64)]
    counters += [np.array(c, dtype=np.uint64) for c in ([0, 0, 0, 0], [0, 1, 0, 0], [0, 0, 0, 1], [0, 0, 1, 5],
                                                         [2**64 - 1, 0, 0, 0], [1, 2**64 - 1, 2**64 - 1, 2**64 - 1])]
    for i, ctr in enumerate(counters):
        key = rng.integers(0, 2**64, size=2, dtype=np.uint64) if i % 2 else np.array([12345678, 0], dtype=np.uint64)
        want = np.random.Philox(counter=_minus_one(ctr), key=key).random_raw(4)
        assert np.array_equal(rso.philox4x64(ctr, key), want), (ctr, key)


def _config(**kw):
    d = dict(nfft=64, nsmp=40, nchains=5, ncool=2, t_high=8.0, iseed=2718)
    d.update(kw)
    return helpers.attach_obs_and_rinv(helpers.small_config(**d), noise=0.01)


def test_mode1_invariants():
    cfg = _config()
    nproc, chunk, n_chunks = 3, 15, 3
    orc = rso.RankSwapOraclePT(cfg, nproc)
    orc.set_rank_swaps(1)
    t0 = orc.state()["temps"]
    n_cold = int(np.sum(t0 == 1.0))
    assert n_cold == nproc * cfg.ncool
    for c in range(n_chunks):
        orc.run(chunk, log=False)
        t = orc.state()["temps"]
        assert np.array_equal(np.sort(t), np.sort(t0))          # swaps only exchange values
        assert int(np.sum(t == 1.0)) == n_cold
        rs = orc.rank_swaps()
        n_it = (c + 1) * chunk
        for l in range(cfg.nchains - 1):
            assert rs["n_prop"][l] == nproc * sum(1 for i in range(n_it) if i % 2 == l % 2), l
        assert (rs["n_acc"] <= rs["n_prop"]).all()
    assert rs["mode"] == 1 and rs["n_acc"].sum() > 0
    assert not np.array_equal(orc.state()["temps"], t0)


def test_mode0_is_the_reference():
    cfg = _config(nchains=4, ncool=1)
    nproc, n_iter = 3, 30
    runs = []
    for told in (False, True):             # the restatement itself, and the run with the sweep told mode 0
        orc = rso.RankSwapOraclePT(cfg, nproc) if told else oracle_c.OraclePT(cfg, nproc)
        if told:
            orc.set_rank_swaps(0)
        logs = orc.run(n_iter)
        runs.append((logs, orc.state(), orc.counters(n_iter)))
        if told:
            rb = orc.rank_swaps()
        orc.close()                        # before the next handle: RFConfig.to_c keeps only its latest buffers alive
    (la, sa, ca), (lb, sb, cb) = runs
    for x, y in zip(la, lb):
        assert x.tobytes() == y.tobytes()
    for key in sa:
        assert sa[key].tobytes() == sb[key].tobytes(), key
    for key in ("nprop", "naccept", "likelihood_hist"):
        assert ca[key].tobytes() == cb[key].tobytes(), key
    assert rb["mode"] == 0 and not rb["n_prop"].any() and not rb["n_acc"].any()


@pytest.mark.parametrize("nchains", [1, 2])
def test_mode1_small_ranks(nchains):
    """One chain per rank: nothing to pair, the run is the reference's.  Two: level pair 0 on even iterations only."""
    cfg = _config(nchains=nchains, ncool=1)
    nproc, n_iter = 2, 11
    # one handle at a time: RFConfig.to_c keeps only the buffers of its latest call alive
    a = oracle_c.OraclePT(cfg, nproc)
    la, ta = a.run(n_iter), a.state()["temps"]
    a.close()
    b = rso.RankSwapOraclePT(cfg, nproc)
    b.set_rank_swaps(1)
    lb = b.run(n_iter)
    rs = b.rank_swaps()
    if nchains == 1:
        assert all(x.tobytes() == y.tobytes() for x, y in zip(la, lb))
        assert ta.tobytes() == b.state()["temps"].tobytes()
        assert rs["n_prop"].size == 0
    else:
        assert rs["n_prop"].tolist() == [nproc * 6]
