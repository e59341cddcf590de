"""CPU checks of the numpy reference of the convergence diagnostics (tests/diag_oracle.py, DESIGN.md 7f): tau against the
measurement tools' FFT estimator and AR(1) theory, split-R-hat on iid and shifted chains, the round-trip counter on
hand-written level sequences."""
import os
import sys

import numpy as np
import pytest

import diag_oracle as dgo

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))


def test_tau_equals_the_tools_estimator_on_random_series():
    from rank_swap_time import iat as tool_iat
    rng = np.random.default_rng(7)
    for n in (4, 5, 17, 200, 801):
        for _ in range(5):
            x = np.cumsum(rng.normal(size=n)) * rng.uniform(0.1, 10) + rng.normal(size=n)
            assert dgo.iat(x) == pytest.approx(tool_iat(x), rel=1e-10)
    assert np.isnan(dgo.iat([1.0, 2.0, 3.0])) and np.isnan(dgo.iat(np.full(50, 0.1)))


@pytest.mark.parametrize("rho", [0.0, 0.5, 0.9])
def test_tau_recovers_ar1(rho):
    rng = np.random.default_rng(11)
    n = 400_000
    e = rng.normal(size=n)
    x = np.empty(n)
    x[0] = e[0] / np.sqrt(1 - rho * rho)
    for i in range(1, n):
        x[i] = rho * x[i - 1] + e[i]
    want = (1 + rho) / (1 - rho)
    assert dgo.iat(x) == pytest.approx(want, rel=0.05)


def test_split_rhat_iid_and_shifted():
    rng = np.random.default_rng(3)
    n, G = 400, 64
    trace = rng.normal(size=(n, G, 1))
    t0 = np.ones((n, G))
    s = dgo.summary(dgo.rows(trace, t0), n)
    assert abs(s[0, 0] - 1.0) < 0.01
    assert s[0, 1] == pytest.approx(n * G, rel=0.15)
    assert s[0, 3] == 0.0
    trace[:, :8, 0] += 3.0
    t0[:n // 4, 0] = 2.0
    s = dgo.summary(dgo.rows(trace, t0), n)
    assert s[0, 0] > 1.1
    assert s[0, 3] == pytest.approx((n // 4) / (n * G))


def test_nan_rules():
    r = dgo.row_stats([1.0, 2.0, 3.0])
    assert np.isnan(r[2]) and np.isnan(r[3]) and np.isnan(r[5]) and np.isnan(r[7])   # n < 4, h = 1
    s = dgo.summary(dgo.rows(np.ones((10, 3, 1)), np.ones((10, 3))), 10)
    assert np.isnan(s[0, 0]) and s[0, 1] == 0.0 and np.isnan(s[0, 2])            # W = 0; no finite tau


def _temps_of_levels(seq, nchains, temps):
    """One rank: per iteration, the chain at each level -> the temperatures each chain holds."""
    out = []
    for order in seq:
        t = np.empty(nchains)
        t[list(order)] = temps
        out.append(t)
    return np.array(out)


def test_round_trips_hand_written():
    # n = 2: chain 0 at the bottom, top, bottom, top, bottom -> 2 trips; chain 1 the mirror -> 1 trip (it starts at the top)
    seq = [(0, 1), (1, 0), (0, 1), (1, 0), (0, 1)]
    lt = _temps_of_levels(seq, 2, [1.0, 3.0])
    trips, st = dgo.round_trips(lt, 2, [1, 2, 3, 4, 5], nburn=3)
    assert trips.tolist() == [[1, 2]]
    assert st.tolist() == [1, 2]
    # ncool > 1 ties: two chains at T = 1, the lower index is level 0; a chain in the middle never reaches the top
    seq = [(0, 1, 2, 3), (2, 1, 0, 3), (1, 0, 3, 2), (2, 0, 1, 3), (1, 2, 3, 0), (0, 2, 1, 3)]
    temps = [1.0, 1.0, 2.0, 4.0]
    lt = _temps_of_levels(seq, 4, temps)
    # the tie rule: chains at equal temperature are ordered by index
    for row, order in zip(lt, seq):
        lo = dgo.level_order(row)
        assert lo[0] == min(order[0], order[1])
    levels = [dgo.level_order(row) for row in lt]
    trips, _ = dgo.round_trips(lt, 4, range(1, 7), nburn=0)
    # by hand from `levels`
    st, want = [0] * 4, 0
    for lv in levels:
        if st[lv[0]] == 2:
            want += 1
        st[lv[0]] = 1
        if st[lv[-1]] == 1:
            st[lv[-1]] = 2
    assert trips.tolist() == [[0, want]]
    # split calls continue the states
    a, sa = dgo.round_trips(lt[:3], 4, range(1, 4), nburn=0)
    b, _ = dgo.round_trips(lt[3:], 4, range(4, 7), nburn=0, states=sa)
    assert (a + b).tolist() == trips.tolist()
    # one chain per rank: no levels, no trips
    assert dgo.round_trips(np.ones((3, 5)), 1, [1, 2, 3], 0)[0].sum() == 0
