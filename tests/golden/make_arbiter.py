"""Generates tests/golden/arbiter_vectors.npz: extended-precision (mpmath, 160 bit) values of rft / phi / logL for a set of
models per variant, from oracle/arbiter_mp.py.  Pure CPU, ~10 minutes; the fixture is committed because the CPU test
suite has to run in minutes (it re-derives a few entries live as a check that script and fixture belong together).

    python tests/golden/make_arbiter.py            # all variants
    python tests/golden/make_arbiter.py land_P     # one variant, printed only
"""
import os, sys, time
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import helpers, oracle_c, arbiter_mp
import rfinv_oracle as pyo
from rf_inv_b200 import workloads

# small shapes in the style of sample_syn (nfft = 256): one entry per code path of calc_seis / calc_rf
SMALL = {
    "land_P": dict(), "sea_P": dict(sdep=2.0), "land_S": dict(ipha=[-1, -1], rayps=[0.10, 0.12]),
    "sea_S_deconv": dict(sdep=1.0, ipha=[-1, -1], deconv_mode=1), "P_deconv": dict(deconv_mode=1),
    "common": dict(rayps=[0.06, 0.06], a_gus=[2.0, 4.0]),
    "three_traces_mixed": dict(ntrc=3, rayps=[0.05, 0.06, 0.11], a_gus=[2.0, 4.0, 8.0], ipha=[1, 1, -1],
                               sig_min=[0.01, 0.02, 0.03], sig_max=[0.01, 0.02, 0.03], sdep=1.5),
}
N_SMALL = 32          # models kept per small variant: the first 32 of a 64-model draw (keeps the fixture below 1 MB)


def variant_config(name):
    if name == "c4":        # joint P + S at nfft = 1024 (BASELINE.json config 4)
        cfg = workloads.make_config("c4")
        return helpers.attach_obs_and_rinv(cfg, noise=0.01)
    return helpers.attach_obs_and_rinv(helpers.small_config(**SMALL[name]), noise=0.01)


def variant_models(name, cfg):
    if name != "c4":
        return {k: v[:N_SMALL] for k, v in workloads.draw_models(cfg, 64, seed=3, dvs_scale=0.3).items()}
    # the worst-conditioned S traces of a 2048-model sample (max|rx| / maxval(rx) > 1e3) plus ordinary models
    m = workloads.draw_models(cfg, 2048, seed=21, dvs_scale=0.3)
    _, _, _, cond = oracle_c.eval_batch(cfg, m["k"], m["z"], m["dvp"], m["dvs"], m["sig"], want_cond=True)
    worst = np.argsort(-cond.max(axis=1))[:12]
    rest = np.setdiff1d(np.arange(2048), worst)[:12]
    sel = np.concatenate([worst, rest])
    return {k: v[sel] for k, v in m.items()}


def run(name):
    cfg = variant_config(name)
    pc = helpers.py_config(cfg)
    flt = pyo.init_filter(pc)
    r_inv = np.ascontiguousarray(np.transpose(cfg.r_inv, (2, 1, 0)))       # [t][j][i] -> r_inv(i, j, t)
    m = variant_models(name, cfg)
    n = m["k"].shape[0]
    out = dict(rft=np.zeros((n, cfg.ntrc, cfg.nsmp)), phi=np.zeros((n, cfg.ntrc)), logl=np.zeros(n), cond=np.zeros((n, cfg.ntrc)),
               npre=np.zeros((n, cfg.ntrc), dtype=np.int64))
    t0 = time.time()
    for i in range(n):
        r = arbiter_mp.evaluate(pc, flt, r_inv, m["k"][i], m["z"][i], m["dvp"][i], m["dvs"][i], m["sig"][i])
        for key in out:
            out[key][i] = r[key][:, :cfg.nsmp] if key == "rft" else r[key]      # the samples the likelihood reads (1:nsmp)
        if i % 8 == 7:
            print(f"  {name}: {i + 1}/{n} models, {time.time() - t0:.0f} s", flush=True)
    ll_o, rft_o, _ = oracle_c.eval_batch(cfg, m["k"], m["z"], m["dvp"], m["dvs"], m["sig"])
    scale = np.max(np.abs(out["rft"]), axis=-1, keepdims=True)
    print(f"{name}: C oracle vs arbiter: rft {np.max(np.abs(rft_o[:, :, :cfg.nsmp] - out['rft']) / scale):.2e} (relative to the trace maximum), "
          f"logL {helpers.logl_err(cfg, ll_o, out['logl'], m['sig']):.2e}, max cond {out['cond'].max():.3g}")
    res = {f"{name}/{k}": v for k, v in m.items()}
    res.update({f"{name}/mp_{k}": v for k, v in out.items()})
    res[f"{name}/obs"] = cfg.obs
    return res


if __name__ == "__main__":
    names = sys.argv[1:] or list(SMALL) + ["c4"]
    path = os.path.join(HERE, "arbiter_vectors.npz")
    data = dict(np.load(path)) if os.path.exists(path) and sys.argv[1:] else {}
    for nm in names:
        data.update(run(nm))
    np.savez_compressed(path, **data)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")
