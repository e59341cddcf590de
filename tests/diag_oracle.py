"""numpy reference of the convergence diagnostics (rfinv_pt_set_diagnostics / rfinv_pt_get_diagnostics, DESIGN.md 7f).

Everything here restates the contract in include/rfinv_b200.h directly, with plain loops where the order matters:
  * level 0 of a rank: its chain of lowest (temperature, local chain index);
  * the per-rank row of a series: mean (sums shifted by the first sample), variance (n - 1), tau (Sokal's window, c = 5, autocovariance sums taken directly),
    ESS = n / tau, the halves' means and variances, tempered samples;
  * across ranks: split-R-hat (BDA3) over the 2G half-chains, ESS over the ranks with finite tau, median tau, tempered share;
  * round trips of every chain between level 0 and level nchains - 1, counted per rank during / after the burn-in.
"""
from __future__ import annotations

import numpy as np

COLD = 1.0 + float(np.float32(1.0e-6))   # the bookkeeping's cold test: T <= 1 + (double)1e-6f


def level_order(temps_rank) -> np.ndarray:
    """Chain index at each level of one rank: its chains sorted by (temperature, chain index)."""
    t = np.asarray(temps_rank)
    return np.lexsort((np.arange(len(t)), t))


def cold_levels(temps, nchains) -> np.ndarray:
    """[G] local chain index (within the rank) of level 0 of every rank."""
    t = np.asarray(temps).reshape(-1, nchains)
    return np.array([level_order(row)[0] for row in t], dtype=np.int64)


def iat(x, c: float = 5.0) -> float:
    """tau = 1 + 2 sum rho(t), stopped at the first m >= c tau; rho(t) = sum_i d_i d_{i+t} / sum_i d_i^2, d = x - mean.
    NaN for fewer than four samples or a constant series."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    if n < 4 or np.all(x == x[0]):
        return float("nan")
    d = x - (x[0] + float(np.sum(x - x[0])) / n)
    s0 = float(np.dot(d, d))
    tau = 1.0
    for m in range(1, n):
        tau += 2.0 * (float(np.dot(d[:n - m], d[m:])) / s0)
        if m >= c * tau:
            break
    return tau


def _mean_var(x):
    n = len(x)
    if n == 0:
        return float("nan"), float("nan")
    m = x[0] + float(np.sum(x - x[0])) / n          # shifted by the first element, as on the device
    return m, float(np.sum((x - m) ** 2) / (n - 1)) if n > 1 else float("nan")


def row_stats(x) -> np.ndarray:
    """mean, var, tau, ess, mean_1, var_1, mean_2, var_2 of one series."""
    x = np.asarray(x, dtype=np.float64)
    n, h = len(x), len(x) // 2
    mean, var = _mean_var(x)
    m1, v1 = _mean_var(x[:h])
    m2, v2 = _mean_var(x[n - h:])
    tau = iat(x)
    return np.array([mean, var, tau, n / tau, m1, v1, m2, v2])


def rows(trace, t0) -> np.ndarray:
    """trace [n][G][nq], t0 [n][G] -> [G][nq][9] (the ninth column: tempered samples of the rank)."""
    trace, t0 = np.asarray(trace), np.asarray(t0)
    n, G, nq = trace.shape
    out = np.zeros((G, nq, 9))
    for r in range(G):
        tempered = float(np.sum(t0[:, r] > COLD))
        for q in range(nq):
            out[r, q, :8] = row_stats(trace[:, r, q])
            out[r, q, 8] = tempered
    return out


def summary(rows_, n) -> np.ndarray:
    """[nq][4]: split-R-hat, ESS, median tau, tempered share from the per-rank rows of n samples each."""
    G, nq, _ = rows_.shape
    h = n // 2
    out = np.zeros((nq, 4))
    for q in range(nq):
        r = rows_[:, q, :]
        means = np.concatenate([r[:, 4], r[:, 6]])
        varis = np.concatenate([r[:, 5], r[:, 7]])
        W = float(np.mean(varis))
        B_h = float(np.var(means, ddof=1)) if len(means) > 1 else float("nan")
        out[q, 0] = np.sqrt(((h - 1) / h * W + B_h) / W) if h >= 2 and W != 0.0 else float("nan")
        fin = np.isfinite(r[:, 2])
        out[q, 1] = float(np.sum(r[fin, 3]))
        out[q, 2] = float(np.median(r[fin, 2])) if fin.any() else float("nan")
        out[q, 3] = float(np.sum(rows_[:, 0, 8]) / (G * n)) if n > 0 else float("nan")
    return out


def round_trips(level_temps, nchains, iterations, nburn, states=None):
    """Round trips from the temperatures at acceptance of the sweep iterations.
    level_temps: [iterations][Cl] the temperatures each chain held at acceptance of iteration it (1-based, in `iterations`).
    Returns (trips [G][2], states [Cl]); `states` continues a previous call."""
    level_temps = np.asarray(level_temps)
    Cl = level_temps.shape[1]
    G = Cl // nchains
    st = np.zeros(Cl, np.int8) if states is None else states.copy()
    trips = np.zeros((G, 2), np.int64)
    if nchains < 2:
        return trips, st
    for temps, it in zip(level_temps, iterations):
        phase = 0 if it <= nburn else 1
        for r in range(G):
            order = level_order(temps[r * nchains:(r + 1) * nchains])
            bottom, top = r * nchains + order[0], r * nchains + order[-1]
            if st[bottom] == 2:
                trips[r, phase] += 1
            st[bottom] = 1
            if st[top] == 1:
                st[top] = 2
    return trips, st


def recorded_vs(cfg, k, z, dvp, dvs, bins):
    """The Vs the bookkeeping assigns to each 1-based depth bin for one model: format_model's layers cover the bins
    int(depth at the top / dbin_z) + 1 onwards; the sea layer (beta <= 0) records vs_min."""
    import oracle_c
    nlay, _, beta, _, h, _ = oracle_c.format_model(cfg, int(k), z, dvp, dvs)
    dbin_z = (cfg.z_max - 0.0) / cfg.nbin_z
    iz1, top = [], 0.0
    for l in range(nlay):
        iz1.append(int(top / dbin_z) + 1)
        top = top + h[l]
    iz1.append(cfg.nbin_z + 1)
    out = []
    for b in bins:
        l = 0
        while l + 1 < nlay and b >= iz1[l + 1]:
            l += 1
        out.append(float("nan") if b < iz1[l] else (beta[l] if beta[l] > 0.0 else cfg.vs_min))
    return np.array(out)
