"""ctypes loader for tests/ladder_oracle.c (DESIGN.md 7d): the C restatement's PT run with the rank sweep and the tuning of
every rank's ladder at the tuning points, and the tuning of one rank on its own.  TEST INFRASTRUCTURE ONLY.

The library is compiled from ladder_oracle.c -- which includes rank_swap_oracle.c and with it oracle/rfinv_oracle.c, both
unchanged -- with the restatement's compiler and flags, into the temporary directory (the source tree may be read-only),
named after a hash of its inputs.  It holds the same code as oracle_c's library, so a PT handle made by oracle_c.OraclePT is
driven by lo_pt_run as it is."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle_c
import rank_swap_oracle as rso

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = [os.path.join(_HERE, "ladder_oracle.c")] + rso._SOURCES
COLD_EPS = float(np.float32(1.0e-6))
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(" ".join([rso._CC] + rso._CFLAGS).encode())
        for f in _SOURCES:
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), f"rfinv_ladder_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call([rso._CC] + rso._CFLAGS + ["-shared", "-o", tmp, _SOURCES[0], "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.lo_tune_rank.restype = C.c_int32
        L.lo_tune_rank.argtypes = [C.c_int32, oracle_c.dp, oracle_c.i64p, oracle_c.i64p, C.c_int64]
        L.lo_pt_run.restype = C.c_int32
        L.lo_pt_run.argtypes = [C.c_void_p, C.c_int32, C.c_int32, oracle_c.i64p, oracle_c.i64p, oracle_c.i64p, oracle_c.i64p,
                                oracle_c.i32p, C.c_int32, oracle_c.i8p, oracle_c.i8p, oracle_c.i32p, C.c_int32]
        _lib = L
    return _lib


def tune_rank(temps, acc, base, e):
    """lo_tune_rank on copies: (new temperatures, new base, changed)."""
    t = np.array(temps, dtype=np.float64)
    a = np.ascontiguousarray(acc, dtype=np.int64)
    b = np.array(base, dtype=np.int64)
    ch = lib().lo_tune_rank(len(t), t.ctypes.data_as(oracle_c.dp), a.ctypes.data_as(oracle_c.i64p),
                             b.ctypes.data_as(oracle_c.i64p), int(e))
    return t, b, bool(ch)


def tuning_points(nburn):
    e, out = 64, []
    while e <= nburn:
        out.append(e)
        e *= 2
    return out


class LadderOraclePT(rso.RankSwapOraclePT):
    """RankSwapOraclePT with the ladder tuning (off by default: then its runs are RankSwapOraclePT's)."""

    def __init__(self, cfg, nproc: int, nthreads: int = 0):
        super().__init__(cfg, nproc, nthreads)
        self.tune = 0
        n = max(cfg.nchains - 1, 1)
        self.rows = np.zeros(nproc * n, np.int64)
        self.base = np.zeros(nproc * n, np.int64)
        self._points = np.zeros(1, np.int32)

    def set_ladder_tuning(self, on) -> None:
        self.tune = int(on)

    def set_rank_swaps(self, mode: int) -> None:
        super().set_rank_swaps(mode)
        if int(mode) == 0:
            self.tune = 0

    def ladder_tuning(self):
        return bool(self.tune), int(self._points[0])

    def run(self, n_iter: int, log: bool = True, record: bool = False):
        flags = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        itypes = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        swaps = np.zeros((n_iter, 3), dtype=np.int32) if log else None
        p = oracle_c._p
        lib().lo_pt_run(self._h, self.mode, self.tune, p(self.n_prop, oracle_c.i64p), p(self.n_acc, oracle_c.i64p),
                        p(self.rows, oracle_c.i64p), p(self.base, oracle_c.i64p), p(self._points, oracle_c.i32p), n_iter,
                        p(flags, oracle_c.i8p), p(itypes, oracle_c.i8p), p(swaps, oracle_c.i32p), int(record))
        return flags, itypes, swaps
