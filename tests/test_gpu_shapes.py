"""The evaluation kernels at the shapes the C-ABI accepts but the parity suite never reaches: every forward_kernel
instantiation, layer stacks past one warp (k_max 64), many traces (up to RFINV_MAX_TRC = 16), window lengths at the edges
of quadform_kernel's 64-wide tiles and batch sizes at the edges of its 64-wide chain tiles.

Each case evaluates up to 64 models on the GPU and on the C oracle.  Bars (as in test_gpu_parity.py): validity flags
equal, traces within 1e-9 of the trace maximum, logL within 1e-9 of the terms it is summed from.  S traces under
deconv_mode 0 are normalised by a ripple of the vertical trace on some models; there any two fp64 evaluations agree to
eps * cond only, so the traces are held to 1e-9 where cond <= 1e3 and to 1e-12 * cond elsewhere, and logL to 1e-9 on
the models whose traces are all well conditioned.

expected_variants() restates the host dispatch (band_limits in capi.cu, launch_forward_group in forward.cu); a CPU
test checks it against the tables in forward.cu and that every reachable instantiation has a case here, and the GPU
cases check the restatement through the launch count.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import helpers
import oracle_c
from rf_inv_b200 import workloads
from rf_inv_b200.evaluator import Evaluator

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FORWARD_CU = os.path.join(ROOT, "rf_inv_b200", "csrc", "forward.cu")
RTOL = 1e-9

# ---- restatement of the host dispatch ------------------------------------------------------------------------------

ALLOWED_JB = (1, 2, 3, 4, 6, 8)          # capi.cu:64, the bin-group counts forward_kernel is instantiated for


def bins_per_thread(nfft_p2):             # rfinv_forward_bins_per_thread, forward.cu:1679-1684
    return 1 if nfft_p2 <= 64 else 2 if nfft_p2 <= 256 else 4 if nfft_p2 <= 2048 else 8


def nfft_p2(nfft):                        # rfinv_create, capi.cu:445
    n = 64
    while n < nfft:
        n *= 2
    return n


def forward_threads(nfft):                # rfinv_forward_threads, rfinv_common.cuh:173
    p2 = nfft_p2(nfft)
    return (p2 // 2) // bins_per_thread(p2)


# FWD(J, BMAX, MINB) per thread count: (largest JB it takes, J, BMAX, MINB), first match wins (forward.cu:1640-1651)
def fwd_table(minb3=4):
    return {32: [(1, 1, 32, 8), (99, 2, 32, 8)],
            64: [(2, 2, 64, 6), (99, 4, 64, 6)],
            128: [(2, 2, 128, 6), (3, 3, 128, minb3), (99, 4, 128, 4)],
            256: [(3, 3, 256, 2), (4, 4, 256, 2), (6, 6, 256, 1), (99, 8, 256, 1)]}


FWDG_TABLE = {32: (2, 32, 8), 64: (4, 64, 6), 128: (4, 128, 4), 256: (4, 256, 2)}   # forward.cu:1671-1674


def variant(nthr, jb, buried, general, minb3=4):
    """(J, BMAX, MINB, MIXED, BURIED, GEN) that launch_forward_group / rfinv_launch_forward_group_general launch for one
    band-limit group of JB bin groups (forward.cu:1631-1676)."""
    if general:                                                  # FWDG: MIXED always, forward.cu:1666-1670
        j, b, mb = FWDG_TABLE[nthr]
        return (j, b, mb, True, buried, True)
    for lim, j, b, mb in fwd_table(minb3)[nthr]:
        if jb <= lim:
            # FWD: buried -> <.., true, true>; else MIXED = (J != JB), forward.cu:1634-1639
            return (j, b, mb, True, True, False) if buried else (j, b, mb, j != jb, False, False)
    raise AssertionError("unreachable")


def band_groups(cfg):
    """jbins per trace, band_limits() of capi.cu:61-87 on the filter of build_filter() (capi.cu:42-54)."""
    p2 = nfft_p2(cfg.nfft)
    jfull = bins_per_thread(p2)
    nthr = (p2 // 2) // jfull
    nh = cfg.nfft // 2 + 1
    out = []
    for t in range(cfg.ntrc):
        g = jfull
        if cfg.deconv_mode == 0:                     # the water-level deconvolution keeps the full band (capi.cu:68)
            fac = cfg.nfft * cfg.a_gus[t] * cfg.delta / np.sqrt(np.pi)
            om = np.arange(nh) * 2.0 * np.pi * (1.0 / (cfg.delta * cfg.nfft))
            q = om / (2.0 * cfg.a_gus[t])
            f = np.exp(-(q * q)) / fac
            total = float(sum(f))                    # in index order, like the C++ loop
            for cand in range(jfull - 1, 0, -1):
                if float(sum(f[cand * nthr:])) <= total * 2.220446049250313e-16:
                    g = cand
                else:
                    break
        out.append(min(a for a in ALLOWED_JB if g <= a <= jfull) if any(g <= a <= jfull for a in ALLOWED_JB) else jfull)
    if cfg.is_ray_common:                             # capi.cu:86
        out = [max(out)] * cfg.ntrc
    return out


def expected_variants(cfg, minb3=4):
    """One (J, BMAX, MINB, MIXED, BURIED, GEN) per forward_kernel launch, widest band-limit group first
    (rfinv_launch_forward, forward.cu:1741-1750; common ray: one launch at the widest group)."""
    jb = band_groups(cfg)
    groups = [max(jb)] if cfg.is_ray_common else sorted(set(jb), reverse=True)
    nthr = forward_threads(cfg.nfft)
    general = nfft_p2(cfg.nfft) != cfg.nfft
    return [variant(nthr, g, cfg.bdep > 0.0, general, minb3) for g in groups]


def reachable_variants():
    """Every instantiation some configuration launches: all thread counts, every allowed JB up to the full band,
    station at the surface or buried, powers of two and (nfft <= 2048) any other length."""
    out = set()
    for p2 in (64, 128, 256, 512, 1024, 2048, 4096):
        jfull = bins_per_thread(p2)
        nthr = (p2 // 2) // jfull
        for buried in (False, True):
            for general in ((False, True) if 128 <= p2 <= 2048 else (False,)):
                for jb in ALLOWED_JB:
                    if jb <= jfull:
                        out.add(variant(nthr, jb, buried, general))
    return out


# prep_kernel's split of a model's rays over CTAs (rfinv_launch_prep, forward.cu:1704-1708); sizes in doubles of
# PrepBasis / PrepSerial / PrepShared / RayConst (forward.cu:89-103, 228-247)
PB, PS, PSH, RC = 16, 16, 8, 36


def prep_split(k_max, ntr_eff):
    model = ((3 * k_max + 1) & ~1) + (k_max + 2) * PSH + 8
    ray = (k_max + 1) * PB + k_max * PS + RC + 8
    n_groups = 1
    while 8 * (model + -(-ntr_eff // n_groups) * ray) > 96 * 1024 and n_groups < ntr_eff:
        n_groups += 1
    rays = -(-ntr_eff // n_groups)
    return rays, -(-ntr_eff // rays)


# ---- cases -----------------------------------------------------------------------------------------------------------

P4096 = dict(nfft=4096, nsmp=64)
DEEP = dict(k_max=64, z_max=60.0)
# a_gus -> band-limit group at nfft 4096: 0.5 -> 1, 1.0 -> 2, 1.5 -> 3, 2.4 -> 4, 3.0 -> 6, 8.0 -> 8 (2.0 -> 3, 2.2 .. 2.5 -> 4)
WIDTHS_4096 = [0.5, 1.0, 1.5, 2.4, 3.0, 8.0]


def _traces(n, a_gus, s_every=0, ray0=0.04, ray1=0.11):
    rays = list(np.round(np.linspace(ray0, ray1, n), 4))
    ipha = [-1 if s_every and t % s_every == s_every - 1 else 1 for t in range(n)]
    return dict(ntrc=n, rayps=rays, a_gus=[a_gus[t % len(a_gus)] for t in range(n)], ipha=ipha,
                sig_min=[0.01] * n, sig_max=[0.01] * n)


# name -> (small_config keywords, model keywords).  k_fixed: every model has that many interfaces.
CASES = {
    # one or more forward_kernel instantiations per case (mixed Gaussian widths: one launch per band-limit group)
    "n64": (dict(nfft=64, nsmp=40), {}),
    "n64_buried": (dict(nfft=64, nsmp=40, bdep=1.0), {}),
    "n128_widths": (dict(nfft=128, nsmp=64, **_traces(2, [2.0, 4.0])), {}),
    "n128_buried_widths": (dict(nfft=128, nsmp=64, bdep=2.0, sdep=1.0, **_traces(2, [2.0, 4.0])), {}),
    "n256_widths": (dict(nfft=256, nsmp=64, **_traces(2, [2.0, 4.0], s_every=2)), {}),
    "n256_buried": (dict(nfft=256, nsmp=64, bdep=3.0), {}),
    "n512_widths": (dict(nfft=512, nsmp=64, **_traces(4, [2.0, 2.8, 3.2, 8.0])), {}),
    "n512_buried_widths": (dict(nfft=512, nsmp=64, bdep=2.0, **_traces(2, [2.8, 8.0])), {}),
    "n1024_widths": (dict(nfft=1024, nsmp=64, **_traces(4, [1.0, 2.0, 3.0, 8.0])), {}),
    "n1024_buried_widths": (dict(nfft=1024, nsmp=64, bdep=4.0, **_traces(3, [2.0, 3.0, 8.0], s_every=3)), {}),
    "n2048_widths": (dict(nfft=2048, nsmp=64, **_traces(4, [1.0, 2.0, 3.0, 8.0])), {}),
    "n2048_buried_widths": (dict(nfft=2048, nsmp=64, bdep=2.5, sdep=1.0, **_traces(2, [1.0, 8.0])), {}),
    "n4096_deconv": (dict(P4096, deconv_mode=1), {}),
    # 1 and 3 bin groups of 256 threads end inside a leg of the pruned first FFT stage (n/8 = 512 bins)
    "n4096_narrow": (dict(P4096, a_gus=[0.5, 1.5]), {}),
    "n4096_buried_widths": (dict(P4096, bdep=5.0, **_traces(4, [1.5, 2.4, 3.0, 8.0])), {}),
    # Bluestein lengths: 32, 64, 128 and 256 threads, station at the surface and buried
    "n100": (dict(nfft=100, nsmp=64), {}),
    "n100_buried": (dict(nfft=100, nsmp=64, bdep=1.0, sdep=1.0), {}),
    "n375_S": (dict(nfft=375, nsmp=64, ipha=[1, -1], rayps=[0.06, 0.11]), {}),
    "n375_buried": (dict(nfft=375, nsmp=64, bdep=2.0), {}),
    "n600_widths": (dict(nfft=600, nsmp=64, **_traces(2, [2.0, 4.0])), {}),
    "n600_buried_deconv": (dict(nfft=600, nsmp=64, bdep=3.0, deconv_mode=1), {}),
    "n1500": (dict(nfft=1500, nsmp=64), {}),
    "n1500_buried": (dict(nfft=1500, nsmp=64, bdep=6.0, sdep=1.5), {}),
    # deep stacks: 31 .. 63 interfaces, the 32-lane slots of prep_kernel
    "deep_land_k31": (dict(DEEP, nsmp=64, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=31)),
    "deep_land_k32": (dict(DEEP, nsmp=64, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=32)),
    "deep_land_k33": (dict(DEEP, nsmp=64, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=33)),
    "deep_land_k63": (dict(DEEP, nsmp=64, vp_mode=1, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=63)),
    "deep_sea_deconv_k63": (dict(DEEP, nsmp=64, sdep=2.0, deconv_mode=1, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=63)),
    "deep_buried_k33": (dict(DEEP, nsmp=64, bdep=58.5, vp_mode=1), dict(k_fixed=33)),
    "deep_buried_k63": (dict(DEEP, nsmp=64, bdep=45.0, ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=63)),
    # sea floor + buried station + 63 interfaces = 66 layers; nfft 4096 and a buried station: forward_kernel's largest
    # shared-memory configuration (~227 KB)
    "deep_sea_buried_k63_n4096": (dict(DEEP, **P4096, sdep=2.0, bdep=30.0, a_gus=[8.0, 8.0], vp_mode=1,
                                       ipha=[1, -1], rayps=[0.06, 0.11]), dict(k_fixed=63)),
    "deep_sea_buried_deconv_k63_n4096": (dict(DEEP, **P4096, sdep=2.0, bdep=31.0, deconv_mode=1), dict(k_fixed=63)),
    # many traces: several warps of prep_kernel's phase C; spread over several prep CTAs at k_max 64
    "trc7": (dict(nsmp=64, **_traces(7, [4.0], s_every=3)), {}),
    "trc12": (dict(nsmp=64, sdep=1.5, **_traces(12, [4.0, 2.5], s_every=4)), {}),
    "trc16": (dict(nsmp=64, **_traces(16, [4.0, 3.0], s_every=2)), {}),
    "trc16_deep": (dict(DEEP, nsmp=64, **_traces(16, [4.0], s_every=4)), dict(k_fixed=63)),
    "trc13_deep_buried": (dict(DEEP, nsmp=64, bdep=20.0, **_traces(13, [4.0], s_every=5)), {}),
    "trc16_common_ray": (dict(nsmp=64, ntrc=16, rayps=[0.06] * 16, ipha=[1] * 16, a_gus=[2.0, 4.0] * 8,
                              sig_min=[0.01] * 16, sig_max=[0.01] * 16), {}),
    "trc16_n4096_widths": (dict(P4096, **_traces(16, WIDTHS_4096, s_every=8)), {}),
}
# RFINV_FWD_MINB3=5 swaps in <3, 128, 5>: run in a subprocess (the switch is read once per process)
MINB3_CASES = {
    "n1024_minb3": (dict(nfft=1024, nsmp=64, a_gus=[3.0, 3.0]), {}),
    "n1024_minb3_buried": (dict(nfft=1024, nsmp=64, bdep=2.0, a_gus=[3.0, 3.0]), {}),
}


def case_config(name):
    kw, _ = {**CASES, **MINB3_CASES}[name]
    return helpers.small_config(**kw)


def deep_models(cfg, n, seed, k_fixed=None):
    """n valid models of up to k_max - 1 interfaces by construction: interfaces a random partition of the column below a
    1.2 km top layer with every layer thicker than h_min, handed over unsorted (the kernels sort them)."""
    rng = np.random.default_rng(seed)
    km = cfg.k_max
    k = np.full(n, k_fixed, dtype=np.int32) if k_fixed else rng.integers(1, km, n).astype(np.int32)
    z = np.zeros((n, km - 1)); dvp = np.zeros((n, km)); dvs = np.zeros((n, km))
    top, floor = cfg.sdep + 1.2, cfg.z_max - 1.0
    for i in range(n):
        while True:
            kk = int(k[i])
            gaps = 0.08 + rng.dirichlet(np.ones(kk)) * (floor - top - 0.08 * kk)
            z[i, :kk] = rng.permutation(top + np.cumsum(gaps) - gaps[0])
            dvs[i, :kk] = rng.normal(0.0, 0.3, kk); dvs[i, km - 1] = rng.normal(0.0, 0.3)
            if cfg.vp_mode == 1:
                dvp[i, :kk] = rng.normal(0.0, 0.1, kk); dvp[i, km - 1] = rng.normal(0.0, 0.1)
            if workloads.models_valid(cfg, k[i:i + 1], z[i:i + 1], dvp[i:i + 1], dvs[i:i + 1])[0]:
                break
    sig = np.tile(np.asarray(cfg.sig_min, dtype=np.float64), (n, 1))
    return dict(k=k, z=z, dvp=dvp, dvs=dvs, sig=sig)


def case_models(cfg, mkw, n=64, seed=3):
    if cfg.k_max > 30:
        return deep_models(cfg, n, seed, **mkw)
    return workloads.draw_models(cfg, n, seed=seed, dvs_scale=0.3)


def attach_obs(cfg, r_inv=None):
    """Observed traces from the oracle (as helpers.attach_obs_and_rinv), R^-1 given or the reference's (gesvd)."""
    tm = workloads.true_model(cfg)
    cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp))
    cfg.r_inv = np.zeros((cfg.ntrc, cfg.nsmp, cfg.nsmp))
    _, rft, _ = oracle_c.eval_batch(cfg, tm["k"], tm["z"], tm["dvp"], tm["dvs"], tm["sig"])
    obs = rft[0, :, :cfg.nsmp] + np.random.default_rng(7).normal(0.0, 0.01, (cfg.ntrc, cfg.nsmp))
    cfg.obs = obs.astype(np.float32).astype(np.float64)
    cfg.r_inv = helpers.scipy_r_inv(cfg) if r_inv is None else r_inv
    return cfg


def build_case(name, seed=3):
    kw, mkw = {**CASES, **MINB3_CASES}[name]
    cfg = attach_obs(helpers.small_config(**kw))
    return cfg, case_models(cfg, mkw, seed=seed)


def run_gpu(cfg, m):
    with Evaluator(cfg) as ev:
        ll, rft, val = ev.calc_likelihood(m["k"], m["z"], m["dvp"], m["dvs"], m["sig"], want_rft=True, want_valid=True)
        return ll, rft, val, ev.last_launch_count, ev.quadform_form()


def assert_matches_oracle(cfg, m, ll_g, rft_g, val_g):
    ll_o, rft_o, val_o, cond = oracle_c.eval_batch(cfg, m["k"], m["z"], m["dvp"], m["dvs"], m["sig"], want_cond=True)
    assert np.array_equal(val_g, val_o)
    err = np.max(np.abs(rft_g - rft_o), axis=-1) / np.max(np.abs(rft_o), axis=-1)
    well = cond <= 1.0e3
    assert (err <= np.where(well, RTOL, 1e-12 * cond)).all(), (float(np.max(err[well], initial=0.0)), float(np.max(err / cond)))
    ok = well.all(axis=1)
    assert ok.sum() >= len(ok) // 2
    assert helpers.logl_err(cfg, ll_g[ok], ll_o[ok], m["sig"][ok]) < RTOL
    return ll_o


# ---- 1. dispatch restatement and coverage (CPU) ---------------------------------------------------------------------

def _forward_cu_tables():
    src = open(FORWARD_CU).read()
    a = src.index("int launch_forward_group(")
    body = src[a:src.index("#undef FWD\n", a)]
    fwd = {tuple(int(x) for x in t) for t in re.findall(r"\bFWD\((\d+), (\d+), (\d+)\)", body)}
    b = src.index("int rfinv_launch_forward_group_general(const DevConfig& cfg, const ModelBatch& mb, const EvalOutputs& out, const double* lc,\n                                       const double* rc, int* counter, int nthr, cudaStream_t stream, int sel_n,\n                                       unsigned long long sel_packed) {")
    bodyg = src[b:src.index("#undef FWDG", b)]
    fwdg = {tuple(int(x) for x in t) for t in re.findall(r"\bFWDG\((\d+), (\d+), (\d+)\)", bodyg)}
    allowed = re.search(r"const int allowed\[6\] = \{([0-9, ]+)\};", open(os.path.join(ROOT, "rf_inv_b200", "csrc", "capi.cu")).read())
    return fwd, fwdg, tuple(int(x) for x in allowed.group(1).split(","))


def test_dispatch_restatement_matches_forward_cu_and_every_reachable_variant_has_a_case():
    fwd, fwdg, allowed = _forward_cu_tables()
    assert allowed == ALLOWED_JB
    restated = {(j, b, mb) for rows in (fwd_table(4)[32], fwd_table(4)[64], fwd_table(4)[128], fwd_table(4)[256], fwd_table(5)[128])
                for _, j, b, mb in rows}
    assert restated == fwd, "forward.cu's FWD table changed: update fwd_table() and add a case for each new variant"
    assert set(FWDG_TABLE.values()) == fwdg, "forward.cu's FWDG table changed: update FWDG_TABLE and add cases"
    covered = set()
    for name in CASES:
        covered.update(expected_variants(case_config(name)))
    minb3 = set()
    for name in MINB3_CASES:
        minb3.update(expected_variants(case_config(name), minb3=5))
    reach = reachable_variants()
    missing = sorted(reach - covered)
    assert not missing, f"instantiations no case launches: {missing}"
    assert len(reach) == 34
    assert minb3 == {(3, 128, 5, False, False, False), (3, 128, 5, True, True, False)}
    # the widths named in the cases hit the band-limit groups they are meant to
    assert band_groups(helpers.small_config(**P4096, **_traces(6, WIDTHS_4096))) == [1, 2, 3, 4, 6, 8]
    assert len(set(band_groups(case_config("trc16_n4096_widths")))) == 6
    # prep_kernel: more than PREP_RAYS_PER_PASS = 6 rays in one CTA, and a model spread over CTAs with a short last group
    assert prep_split(10, 16) == (16, 1) and prep_split(10, 7) == (7, 1)
    assert prep_split(64, 16) == (4, 4) and prep_split(64, 13) == (5, 3)


# ---- 2. one case per instantiation, 3. deep stacks, 4. many traces --------------------------------------------------

@gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_case_matches_oracle(name):
    cfg, m = build_case(name)
    ll, rft, val, launches, _ = run_gpu(cfg, m)
    assert launches == 3 + len(expected_variants(cfg))      # prep, sig layout, one forward_kernel per group, quadform
    assert_matches_oracle(cfg, m, ll, rft, val)


def _subprocess(tmp_path, names, env, extra=""):
    script = r'''
import sys, numpy as np
sys.path[:0] = [%r, %r, %r]
import test_gpu_shapes as T
out = {}
for name in sys.argv[2:]:
    cfg, m = T.build_case(name) if name in T.CASES or name in T.MINB3_CASES else T.window_case(name)
    ll, rft, val, launches, form = T.run_gpu(cfg, m)
    out[name + "/ll"] = ll; out[name + "/rft"] = rft; out[name + "/val"] = val
    out[name + "/launches"] = np.array(launches); out[name + "/form"] = np.array(form)
np.savez(sys.argv[1], **out)
''' % (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"))
    path = str(tmp_path / "out.npz")
    subprocess.run([sys.executable, "-c", script, path, *names], check=True, env=dict(os.environ, **env))
    return np.load(path)


@gpu
def test_minb3_variant_matches_oracle(tmp_path):
    res = _subprocess(tmp_path, sorted(MINB3_CASES), {"RFINV_FWD_MINB3": "5"})
    for name in sorted(MINB3_CASES):
        cfg, m = build_case(name)
        assert expected_variants(cfg, minb3=5)[0][:3] == (3, 128, 5)
        assert int(res[name + "/launches"]) == 3 + len(expected_variants(cfg, minb3=5))
        assert_matches_oracle(cfg, m, res[name + "/ll"], res[name + "/rft"], res[name + "/val"].astype(bool))


@gpu
def test_format_model_bit_exact_at_63_interfaces_incl_invalid_models():
    cfg = attach_obs(helpers.small_config(**DEEP, nsmp=64, sdep=2.0, vp_mode=1))
    m = deep_models(cfg, 120, seed=5, k_fixed=63)
    m["z"][:30, 40] = m["z"][:30, 41] + 0.01      # a layer thinner than h_min
    m["z"][30:50, 7] = 1.0                        # an interface above the sea floor
    m["dvs"][50:70, 45] -= 3.5                    # a velocity out of bounds
    with Evaluator(cfg) as ev:
        nlay, alpha, beta, rho, h, ok = ev.format_model(m["k"], m["z"], m["dvp"], m["dvs"])
    n_bad = 0
    for i in range(len(m["k"])):
        o = oracle_c.format_model(cfg, int(m["k"][i]), m["z"][i], m["dvp"][i], m["dvs"][i])
        assert o[0] == nlay[i] == 65 and o[5] == ok[i]
        n = o[0]
        assert np.array_equal(o[1], alpha[i, :n]) and np.array_equal(o[2], beta[i, :n])
        assert np.array_equal(o[3], rho[i, :n]) and np.array_equal(o[4], h[i, :n])
        n_bad += not o[5]
    assert n_bad == 70


@gpu
def test_cuda_against_the_arbiter_at_63_interfaces():
    """Three k = 63 land models (two P traces, nfft 256), evaluated live by the mpmath arbiter: CUDA within 1e-9 of the
    exact value of the reference's formulas, and no worse than the C oracle plus 1e-12 of the conditioning."""
    import arbiter_mp
    import rfinv_oracle as pyo
    import test_arbiter as ta
    cfg = attach_obs(helpers.small_config(**DEEP, nsmp=64))
    m = deep_models(cfg, 3, seed=21, k_fixed=63)
    pc = helpers.py_config(cfg)
    flt = pyo.init_filter(pc)
    rinv = np.ascontiguousarray(np.transpose(cfg.r_inv, (2, 1, 0)))
    ref = [arbiter_mp.evaluate(pc, flt, rinv, m["k"][i], m["z"][i], m["dvp"][i], m["dvs"][i], m["sig"][i]) for i in range(3)]
    mp_ = dict(rft=np.stack([r["rft"][:, :cfg.nsmp] for r in ref]), logl=np.array([r["logl"] for r in ref]),
               cond=np.stack([r["cond"] for r in ref]))
    ll_o, rft_o, _ = oracle_c.eval_batch(cfg, m["k"], m["z"], m["dvp"], m["dvs"], m["sig"])
    ll_g, rft_g, _, _, _ = run_gpu(cfg, m)
    eg_rft, eg_ll = ta.errors_vs_arbiter(cfg, m, mp_, rft_g, ll_g)
    eo_rft, eo_ll = ta.errors_vs_arbiter(cfg, m, mp_, rft_o, ll_o)
    c = np.maximum(mp_["cond"], 1.0)
    cm = c.max(axis=1)
    assert (eg_rft[c <= 1e3] <= RTOL).all() and (eg_ll[cm <= 1e3] <= RTOL).all()
    assert (eg_rft <= eo_rft + 1e-12 * c).all() and (eg_ll <= eo_ll + 1e-11 * cm).all()


# ---- 5. window and batch edges ----------------------------------------------------------------------------------------

def _psd(rng, S, rank, neg=False):
    q, _ = np.linalg.qr(rng.normal(size=(S, S)))
    lam = np.zeros(S)
    lam[:rank] = rng.uniform(10.0, 100.0, rank)
    if neg:
        lam[0] = -20.0                              # indefinite: neither factor form applies
    return (q * lam) @ q.T


def window_r_inv(cfg, form, seed=4):
    """R^-1 that makes quadform_kernel take `form` (capi.cu:522-604): the reference's Toeplitz matrix (split), a random
    low-rank positive semi-definite matrix without the mirror symmetry (factor), a random indefinite one (dense)."""
    if form == "split":
        return helpers.scipy_r_inv(cfg)
    rng = np.random.default_rng(seed)
    S = cfg.nsmp
    return np.stack([_psd(rng, S, max(1, S // 3), neg=form == "dense") for _ in range(cfg.ntrc)])


def gauss_toeplitz(S, width):
    """Symmetric Toeplitz positive semi-definite matrix exp(-((i-j)/width)^2): commutes with the exchange matrix."""
    d = np.arange(S, dtype=np.float64)
    col = 50.0 * np.exp(-(d / width) ** 2)
    return col[np.abs(d[:, None] - d[None, :]).astype(np.int64)]


WINDOWS = [(S, f) for S in (1, 2, 63, 64, 65, 127, 129) for f in ("dense", "factor", "split") if not (S == 1 and f == "factor")]


def window_case(name):
    """nsmp 4095 / 4096 at nfft 4096 (the full 64 column tiles of the dense form), R^-1 a Toeplitz Gaussian."""
    S = int(name.split("_")[1])
    cfg = helpers.small_config(nfft=4096, nsmp=S, ntrc=2 if S == 4096 else 1, a_gus=[4.0, 4.0][:2 if S == 4096 else 1],
                               rayps=[0.06, 0.08][:2 if S == 4096 else 1], ipha=[1, 1][:2 if S == 4096 else 1],
                               sig_min=[0.01, 0.01][:2 if S == 4096 else 1], sig_max=[0.01, 0.01][:2 if S == 4096 else 1])
    cfg = attach_obs(cfg, r_inv=np.stack([gauss_toeplitz(S, 6.0 + 3.0 * t) for t in range(cfg.ntrc)]))
    return cfg, workloads.draw_models(cfg, 32, seed=6, dvs_scale=0.3)


@gpu
@pytest.mark.parametrize("nsmp,form", WINDOWS)
def test_window_edges_in_every_quadratic_form(nsmp, form):
    cfg = helpers.small_config(nsmp=nsmp, **_traces(2, [4.0, 2.5]))
    cfg = attach_obs(cfg)
    cfg.r_inv = window_r_inv(cfg, form)
    m = workloads.draw_models(cfg, 64, seed=nsmp, dvs_scale=0.3)
    ll, rft, val, launches, qf = run_gpu(cfg, m)
    assert launches == 3 + len(expected_variants(cfg))
    for rank, _, split in qf:
        assert ("split" if split else "factor" if rank > 0 else "dense") == form, qf
    assert_matches_oracle(cfg, m, ll, rft, val)


@gpu
def test_windows_of_4095_and_4096_samples_dense_form(tmp_path):
    """The dense form over all 64 column tiles (RFINV_QF_DENSE=1; the factor forms' eigen-decomposition at create is
    O(nsmp^3) on the host), against the oracle's dense m^T R^-1 m."""
    names = ["win_4095", "win_4096"]
    res = _subprocess(tmp_path, names, {"RFINV_QF_DENSE": "1"})
    for name in names:
        cfg, m = window_case(name)
        assert (res[name + "/form"][:, 0] == 0).all()
        assert_matches_oracle(cfg, m, res[name + "/ll"], res[name + "/rft"], res[name + "/val"].astype(bool))


@gpu
def test_batch_sizes_at_the_chain_tile_edges_deep_16_traces():
    cfg = attach_obs(case_config("trc16_deep"))
    m = deep_models(cfg, 65, seed=9)
    ll_o, rft_o, val_o, cond = oracle_c.eval_batch(cfg, m["k"], m["z"], m["dvp"], m["dvs"], m["sig"], want_cond=True)
    ok = (cond <= 1e3).all(axis=1)
    with Evaluator(cfg) as ev:
        runs = {}
        for C in (1, 63, 64, 65):
            ll, rft, val = ev.calc_likelihood(m["k"][:C], m["z"][:C], m["dvp"][:C], m["dvs"][:C], m["sig"][:C],
                                              want_rft=True, want_valid=True)
            assert np.array_equal(val, val_o[:C])
            err = np.max(np.abs(rft - rft_o[:C]), axis=-1) / np.max(np.abs(rft_o[:C]), axis=-1)
            assert (err <= np.maximum(RTOL * (cond[:C] <= 1e3), 1e-12 * cond[:C])).all()
            assert helpers.logl_err(cfg, ll[ok[:C]], ll_o[:C][ok[:C]], m["sig"][:C][ok[:C]]) < RTOL
            runs[C] = ll
    for C in (1, 63, 64):                          # a model's logL does not depend on the batch around it
        assert np.array_equal(runs[C], runs[65][:C])


@gpu
def test_large_host_batch_at_64_layers_matches_small_batches():
    """8192 + 77 models at k_max 64 and 4 traces go up in pieces (prep_kernel per piece); bit for bit what batches of
    1500 give, and the oracle on a subsample."""
    cfg = attach_obs(helpers.small_config(**DEEP, nsmp=64, **_traces(4, [4.0, 2.5], s_every=4)))
    n = 8192 + 77
    m = deep_models(cfg, n, seed=17)
    with Evaluator(cfg) as ev:
        ll_big, _, val_big = ev.calc_likelihood(m["k"], m["z"], m["dvp"], m["dvs"], m["sig"], want_valid=True)
        assert ev.last_launch_count == 4 + 1 + len(expected_variants(cfg)) + 1     # 4 prep pieces, sig, forward, quadform
        parts = [ev.calc_likelihood(m["k"][s:s + 1500], m["z"][s:s + 1500], m["dvp"][s:s + 1500], m["dvs"][s:s + 1500],
                                    m["sig"][s:s + 1500], want_valid=True) for s in range(0, n, 1500)]
    assert np.array_equal(ll_big, np.concatenate([p[0] for p in parts]))
    assert np.array_equal(val_big, np.concatenate([p[2] for p in parts])) and val_big.all()
    sub = np.arange(0, n, 257)
    ms = {k: v[sub] for k, v in m.items()}
    ll_o, _, val_o, cond = oracle_c.eval_batch(cfg, ms["k"], ms["z"], ms["dvp"], ms["dvs"], ms["sig"], want_rft=False, want_cond=True)
    ok = (cond <= 1e3).all(axis=1)
    assert np.array_equal(val_big[sub], val_o)
    assert helpers.logl_err(cfg, ll_big[sub][ok], ll_o[ok], ms["sig"][ok]) < RTOL
