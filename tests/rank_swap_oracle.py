"""ctypes loader for tests/rank_swap_oracle.c: the C restatement's PT run with the even/odd swaps inside every virtual rank
(DESIGN.md 7c), and its Philox4x64-10.  TEST INFRASTRUCTURE ONLY.

The library is compiled from rank_swap_oracle.c -- which includes oracle/rfinv_oracle.c unchanged -- with the restatement's
compiler and flags, into the temporary directory (the source tree may be read-only), named after a hash of its inputs.  It
holds the same code as oracle_c's library, so a PT handle made by oracle_c.OraclePT is driven by rso_pt_run as it is."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_c

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_SOURCES = [os.path.join(_HERE, "rank_swap_oracle.c"), os.path.join(_ROOT, "oracle", "rfinv_oracle.c"),
            os.path.join(_ROOT, "include", "rfinv_b200.h")]
_CC = "/usr/bin/gcc"
_CFLAGS = ["-O3", "-march=x86-64-v3", "-ffp-contract=off", "-fopenmp", "-fPIC", "-std=gnu99", "-Wall", "-Wno-unused-function"]
_lib = None
u64p = C.POINTER(C.c_uint64)


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(" ".join([_CC] + _CFLAGS).encode())
        for f in _SOURCES:
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), f"rfinv_rank_swap_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call([_CC] + _CFLAGS + ["-shared", "-o", tmp, _SOURCES[0], "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.rso_philox4x64.argtypes = [u64p, u64p, u64p]
        L.rso_pt_run.restype = C.c_int32
        L.rso_pt_run.argtypes = [C.c_void_p, C.c_int32, oracle_c.i64p, oracle_c.i64p, C.c_int32, oracle_c.i8p, oracle_c.i8p,
                                 oracle_c.i32p, C.c_int32]
        _lib = L
    return _lib


def philox4x64(counter, key) -> np.ndarray:
    """The four output words of Philox4x64-10 for a 256-bit counter (word 0 least significant) and a 128-bit key."""
    ctr = np.ascontiguousarray(counter, dtype=np.uint64)
    k = np.ascontiguousarray(key, dtype=np.uint64)
    out = np.empty(4, dtype=np.uint64)
    lib().rso_philox4x64(ctr.ctypes.data_as(u64p), k.ctypes.data_as(u64p), out.ctypes.data_as(u64p))
    return out


class RankSwapOraclePT(oracle_c.OraclePT):
    """oracle_c.OraclePT whose runs include the rank sweep in mode 1; mode 0 (the default) is oracle_c.OraclePT's run."""

    def __init__(self, cfg, nproc: int, nthreads: int = 0):
        super().__init__(cfg, nproc, nthreads)
        self.mode = 0
        n = max(cfg.nchains - 1, 0)
        self.n_prop = np.zeros(max(n, 1), np.int64)
        self.n_acc = np.zeros(max(n, 1), np.int64)

    def set_rank_swaps(self, mode: int) -> None:
        self.mode = int(mode)

    def rank_swaps(self) -> dict:
        n = max(self.cfg.nchains - 1, 0)
        return dict(mode=self.mode, n_prop=self.n_prop[:n].copy(), n_acc=self.n_acc[:n].copy())

    def run(self, n_iter: int, log: bool = True, record: bool = False):
        flags = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        itypes = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        swaps = np.zeros((n_iter, 3), dtype=np.int32) if log else None
        p = oracle_c._p
        lib().rso_pt_run(self._h, self.mode, p(self.n_prop, oracle_c.i64p), p(self.n_acc, oracle_c.i64p), n_iter,
                         p(flags, oracle_c.i8p), p(itypes, oracle_c.i8p), p(swaps, oracle_c.i32p), int(record))
        return flags, itypes, swaps
