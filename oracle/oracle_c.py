"""ctypes loader for the C restatement ``oracle/rfinv_oracle.c`` (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py (observed traces, cpu_baseline / --impl reference legs) import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional

import numpy as np

from rf_inv_b200.config import RFConfig, RfinvConfigC

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "librfinv_oracle.so")
_lib = None

dp = C.POINTER(C.c_double)
i32p = C.POINTER(C.c_int32)
i64p = C.POINTER(C.c_int64)
i8p = C.POINTER(C.c_int8)
u8p = C.POINTER(C.c_uint8)


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "rfinv_oracle.c")
    hdr = os.path.join(_HERE, "..", "include", "rfinv_b200.h")
    stale = (not os.path.exists(_SO)) or any(
        os.path.exists(f) and os.path.getmtime(f) > os.path.getmtime(_SO) for f in (src, hdr))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        cfgp = C.POINTER(RfinvConfigC)
        L.orc_num_threads.restype = C.c_int32
        L.orc_vp_to_rho.restype = C.c_double
        L.orc_vp_to_rho.argtypes = [C.c_double]
        L.orc_format_model.restype = C.c_int32
        L.orc_format_model.argtypes = [cfgp, C.c_int32, dp, dp, dp, i32p, dp, dp, dp, dp]
        L.orc_init_filter.argtypes = [cfgp, dp]
        L.orc_eval_batch.restype = C.c_int32
        L.orc_eval_batch.argtypes = [cfgp, C.c_int32, i32p, dp, dp, dp, dp, dp, dp, u8p, C.c_int32]
        L.orc_eval_batch_cond.restype = C.c_int32
        L.orc_eval_batch_cond.argtypes = [cfgp, C.c_int32, i32p, dp, dp, dp, dp, dp, dp, u8p, C.c_int32, dp]
        L.orc_calc_rf_layers.restype = C.c_int32
        L.orc_calc_rf_layers.argtypes = [cfgp, C.c_int32, dp, dp, dp, dp, dp]
        L.orc_mt_sequence.argtypes = [C.c_uint32, C.c_int32, dp]
        L.orc_deviates.argtypes = [C.c_uint32, C.c_int32, C.c_int32, dp]
        L.orc_pt_create.restype = C.c_void_p
        L.orc_pt_create.argtypes = [cfgp, C.c_int32, C.c_int32]
        L.orc_pt_destroy.argtypes = [C.c_void_p]
        L.orc_pt_run.restype = C.c_int32
        L.orc_pt_run.argtypes = [C.c_void_p, C.c_int32, i8p, i8p, i32p, C.c_int32]
        L.orc_pt_ntype.restype = C.c_int32
        L.orc_pt_ntype.argtypes = [C.c_void_p]
        L.orc_pt_n_eval.restype = C.c_int64
        L.orc_pt_n_eval.argtypes = [C.c_void_p]
        L.orc_pt_get_state.argtypes = [C.c_void_p, i32p, dp, dp, dp, dp, dp, dp, dp]
        L.orc_pt_get_counters.argtypes = [C.c_void_p, i64p, i64p, dp, i64p]
        L.orc_pt_get_hist.argtypes = [C.c_void_p, i64p, i64p, i64p, i64p, i64p, i64p, i64p, dp, dp, dp]
        _lib = L
    return _lib


def _p(a, t):
    return a.ctypes.data_as(t) if a is not None else C.cast(None, t)


def num_threads() -> int:
    return int(lib().orc_num_threads())


def vp_to_rho(a: float) -> float:
    return float(lib().orc_vp_to_rho(a))


def mt_sequence(seed: int, count: int) -> np.ndarray:
    out = np.empty(count)
    lib().orc_mt_sequence(seed & 0xFFFFFFFF, count, _p(out, dp))
    return out


def deviates(seed: int, kind: str, count: int) -> np.ndarray:
    out = np.empty(count)
    lib().orc_deviates(seed & 0xFFFFFFFF, 1 if kind == "laplace" else 0, count, _p(out, dp))
    return out


def init_filter(cfg: RFConfig) -> np.ndarray:
    c = cfg.to_c()
    flt = np.empty((cfg.ntrc, cfg.nh))
    lib().orc_init_filter(C.byref(c), _p(flt, dp))
    return flt


def format_model(cfg: RFConfig, k: int, z, dvp, dvs):
    c = cfg.to_c()
    km = cfg.k_max
    z = np.ascontiguousarray(z, dtype=np.float64); dvp = np.ascontiguousarray(dvp, dtype=np.float64)
    dvs = np.ascontiguousarray(dvs, dtype=np.float64)
    nlay = C.c_int32(0)
    out = [np.zeros(km + 1) for _ in range(4)]
    ok = lib().orc_format_model(C.byref(c), int(k), _p(z, dp), _p(dvp, dp), _p(dvs, dp), C.byref(nlay),
                                *[_p(o, dp) for o in out])
    n = nlay.value
    return n, out[0][:n], out[1][:n], out[2][:n], out[3][:n], bool(ok)


def calc_rf_layers(cfg: RFConfig, alpha, beta, rho, h) -> np.ndarray:
    c = cfg.to_c()
    a, b, r, hh = (np.ascontiguousarray(x, dtype=np.float64) for x in (alpha, beta, rho, h))
    rft = np.empty((cfg.ntrc, cfg.nfft))
    lib().orc_calc_rf_layers(C.byref(c), len(a), _p(a, dp), _p(b, dp), _p(r, dp), _p(hh, dp), _p(rft, dp))
    return rft


def eval_batch(cfg: RFConfig, k, z, dvp, dvs, sig, want_rft: bool = True, nthreads: int = 0, want_cond: bool = False):
    """calc_likelihood over C models.  Layouts: z[C][k_max-1], dvp/dvs[C][k_max], sig[C][ntrc].
    Returns (logl[C], rft[C][ntrc][nfft] or None, is_valid[C]) -- and with want_cond the condition number
    max|rx| / maxval(rx) of the reference's normalisation per (model, trace) as a fourth item."""
    c = cfg.to_c()
    k = np.ascontiguousarray(k, dtype=np.int32)
    nC = k.shape[0]
    z = np.ascontiguousarray(z, dtype=np.float64); dvp = np.ascontiguousarray(dvp, dtype=np.float64)
    dvs = np.ascontiguousarray(dvs, dtype=np.float64); sig = np.ascontiguousarray(sig, dtype=np.float64)
    assert z.shape == (nC, cfg.k_max - 1) and dvp.shape == (nC, cfg.k_max) and sig.shape == (nC, cfg.ntrc)
    logl = np.empty(nC)
    rft = np.empty((nC, cfg.ntrc, cfg.nfft)) if want_rft else None
    valid = np.empty(nC, dtype=np.uint8)
    if want_cond:
        cond = np.ones((nC, cfg.ntrc))
        st = lib().orc_eval_batch_cond(C.byref(c), nC, _p(k, i32p), _p(z, dp), _p(dvp, dp), _p(dvs, dp), _p(sig, dp),
                                       _p(logl, dp), _p(rft, dp), _p(valid, u8p), int(nthreads), _p(cond, dp))
        if st != 0:
            raise RuntimeError("orc_eval_batch: obs / r_inv missing in config")
        return logl, rft, valid.astype(bool), cond
    st = lib().orc_eval_batch(C.byref(c), nC, _p(k, i32p), _p(z, dp), _p(dvp, dp), _p(dvs, dp), _p(sig, dp),
                              _p(logl, dp), _p(rft, dp), _p(valid, u8p), int(nthreads))
    if st != 0:
        raise RuntimeError("orc_eval_batch: obs / r_inv missing in config")
    return logl, rft, valid.astype(bool)


class OraclePT:
    """PT-MCMC restatement with ``nproc`` virtual MPI ranks (pt_mcmc.f90:468-576)."""

    def __init__(self, cfg: RFConfig, nproc: int, nthreads: int = 0):
        self.cfg = cfg
        self.nproc = nproc
        self._c = cfg.to_c()
        self._h = lib().orc_pt_create(C.byref(self._c), nproc, nthreads)
        if not self._h:
            raise RuntimeError("orc_pt_create failed (obs / r_inv missing?)")
        self.G = nproc * cfg.nchains
        self.ntype = int(lib().orc_pt_ntype(self._h))

    def close(self):
        if self._h:
            lib().orc_pt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, n_iter: int, log: bool = True, record: bool = False):
        flags = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        itypes = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        swaps = np.zeros((n_iter, 3), dtype=np.int32) if log else None
        lib().orc_pt_run(self._h, n_iter, _p(flags, i8p), _p(itypes, i8p), _p(swaps, i32p), int(record))
        return flags, itypes, swaps

    @property
    def n_eval(self) -> int:
        return int(lib().orc_pt_n_eval(self._h))

    def state(self, want_rft: bool = False):
        cfg, G = self.cfg, self.G
        out = dict(k=np.empty(G, dtype=np.int32), z=np.empty((G, cfg.k_max - 1)), dvp=np.empty((G, cfg.k_max)),
                   dvs=np.empty((G, cfg.k_max)), sig=np.empty((G, cfg.ntrc)), logl=np.empty(G), temps=np.empty(G))
        rft = np.empty((G, cfg.ntrc, cfg.nfft)) if want_rft else None
        lib().orc_pt_get_state(self._h, _p(out["k"], i32p), _p(out["z"], dp), _p(out["dvp"], dp), _p(out["dvs"], dp),
                               _p(out["sig"], dp), _p(out["logl"], dp), _p(out["temps"], dp), _p(rft, dp))
        if want_rft:
            out["rft"] = rft
        return out

    def counters(self, n_iter_done: int):
        nprop = np.zeros(self.ntype, dtype=np.int64); nacc = np.zeros(self.ntype, dtype=np.int64)
        hist = np.zeros(n_iter_done); nmod = C.c_int64(0)
        lib().orc_pt_get_counters(self._h, _p(nprop, i64p), _p(nacc, i64p), _p(hist, dp), C.byref(nmod))
        return dict(nprop=nprop, naccept=nacc, likelihood_hist=hist, nmod=nmod.value)

    def hist(self):
        c = self.cfg
        o = dict(nk=np.zeros(c.k_max, np.int64), nz=np.zeros(c.nbin_z, np.int64),
                 nsig=np.zeros((c.ntrc, c.nbin_sig), np.int64), namp=np.zeros((c.ntrc, c.nsmp, c.nbin_amp), np.int64),
                 nvpz=np.zeros((c.nbin_vp, c.nbin_z), np.int64), nvsz=np.zeros((c.nbin_vs, c.nbin_z), np.int64),
                 nvpvsz=np.zeros((c.nbin_vpvs, c.nbin_z), np.int64), vp_mean=np.zeros(c.nbin_z),
                 vs_mean=np.zeros(c.nbin_z), vpvs_mean=np.zeros(c.nbin_z))
        lib().orc_pt_get_hist(self._h, *[_p(o[n], i64p) for n in ("nk", "nz", "nsig", "namp", "nvpz", "nvsz", "nvpvsz")],
                              *[_p(o[n], dp) for n in ("vp_mean", "vs_mean", "vpvs_mean")])
        return o
