"""Generates tests/golden/sample_syn.npz and oracle_vectors.npz (needs the reference's source tree and scipy):

    python tests/golden/make_golden.py <reference>/sample_syn

1. sample_syn.npz   -- the reference's own fixtures, extracted verbatim from its sample_syn directory:
                       the two SAC traces (float32 samples + header words), true/true.velmod, model/sample.velmod
                       and the values of params.in.  These PIN the forward path (land, P, deconv_mode 0).
2. oracle_vectors.npz -- outputs of the numpy restatement (oracle/rfinv_oracle.py) for variants the reference
                       ships no fixture for (sea layer, S phase, deconvolution, common rays, likelihood).  They are
                       regression vectors for the oracle itself ("parity unpinned"), not reference outputs.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]


def read_sac(path):
    raw = np.fromfile(path, dtype="<f4")
    ints = raw.view("<i4")
    npts = int(ints[79])
    return dict(delta=raw[0], b=raw[5], e=raw[6], npts=npts, data=raw[158:158 + npts].copy())


def read_params(path):
    vals = []
    for line in open(path):
        s = line.strip()
        if not s or s.startswith("#"):
            continue
        vals.append(s)
    return vals


def main(sample_syn):
    s1 = read_sac(os.path.join(sample_syn, "data/sample_1.trc"))
    s2 = read_sac(os.path.join(sample_syn, "data/sample_2.trc"))
    true_vm = np.loadtxt(os.path.join(sample_syn, "true/true.velmod"), comments="#")
    ref_vm = np.loadtxt(os.path.join(sample_syn, "model/sample.velmod"))
    params = read_params(os.path.join(sample_syn, "params.in"))
    np.savez(os.path.join(HERE, "sample_syn.npz"),
             trc1=s1["data"], trc2=s2["data"], delta=np.float32(s1["delta"]), b=np.float32(s1["b"]), npts=s1["npts"],
             true_velmod=true_vm, ref_velmod=ref_vm, params=np.array(params))

    import helpers
    import rfinv_oracle as pyo
    from rf_inv_b200 import workloads
    out = {}
    cases = {
        "land_P": dict(), "sea_P": dict(sdep=2.0), "land_S": dict(ipha=[-1, -1], rayps=[0.10, 0.12]),
        "sea_S_deconv": dict(sdep=1.0, ipha=[-1, -1], deconv_mode=1), "P_deconv": dict(deconv_mode=1),
        "common": dict(rayps=[0.06, 0.06], a_gus=[2.0, 4.0]), "vp1_tstart": dict(vp_mode=1, t_start=-3.0),
        # buried station (commented out in the reference: no reference output can exist)
        "buried_sea_P": dict(bdep=1.5, sdep=2.0), "buried_land_S": dict(bdep=6.0, ipha=[-1, -1], rayps=[0.10, 0.12]),
        "buried_half_space": dict(bdep=25.0),
    }
    for name, kw in cases.items():
        cfg = helpers.attach_obs_and_rinv(helpers.small_config(**kw))
        m = workloads.draw_models(cfg, 4, seed=11, dvs_scale=0.3)
        pc = helpers.py_config(cfg)
        flt = pyo.init_filter(pc)
        rinv = np.transpose(cfg.r_inv, (2, 1, 0))
        lls, rfts = [], []
        for i in range(4):
            ll, rft = pyo.calc_likelihood(pc, flt, rinv, int(m["k"][i]), m["z"][i], m["dvp"][i], m["dvs"][i], m["sig"][i])
            lls.append(ll); rfts.append(rft.T)
        out[name + "/obs"] = cfg.obs
        for key in ("k", "z", "dvp", "dvs", "sig"):
            out[f"{name}/{key}"] = m[key]
        out[name + "/logl"] = np.array(lls)
        out[name + "/rft"] = np.array(rfts)
    np.savez_compressed(os.path.join(HERE, "oracle_vectors.npz"), **out)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__":
    main(sys.argv[1])
