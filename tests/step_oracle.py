"""ctypes loader for tests/step_oracle.c (DESIGN.md 7e): the C restatement's PT run with the rank sweep, the ladder tuning and
the tuning of every rank's random-walk widths per level, and the width tuning of one rank on its own.  TEST INFRASTRUCTURE ONLY.

The library is compiled from step_oracle.c -- which includes ladder_oracle.c, rank_swap_oracle.c and oracle/rfinv_oracle.c,
all unchanged -- with the restatement's compiler and flags, into the temporary directory (the source tree may be read-only),
named after a hash of its inputs.  It holds the same code as oracle_c's library, so a PT handle made by oracle_c.OraclePT is
driven by so_pt_run as it is."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import ladder_oracle as lo
import oracle_c
import rank_swap_oracle as rso

_HERE = os.path.dirname(os.path.abspath(__file__))
_SOURCES = [os.path.join(_HERE, "step_oracle.c")] + lo._SOURCES
MIN_PROPOSALS = 16
SCALE_MIN, SCALE_MAX = 2.0 ** -8, 2.0 ** 8
_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha1(" ".join([rso._CC] + rso._CFLAGS).encode())
        for f in _SOURCES:
            with open(f, "rb") as fh:
                h.update(fh.read())
        so = os.path.join(tempfile.gettempdir(), f"rfinv_step_oracle_{h.hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call([rso._CC] + rso._CFLAGS + ["-shared", "-o", tmp, _SOURCES[0], "-lm"])
            os.replace(tmp, so)
        L = C.CDLL(so)
        i64p, i32p, i8p, dp = oracle_c.i64p, oracle_c.i32p, oracle_c.i8p, oracle_c.dp
        L.so_step.restype = C.c_int32
        L.so_step.argtypes = [C.c_void_p, C.c_int32, C.c_int32, dp, C.c_int32, i32p]
        L.so_levels.argtypes = [C.c_void_p, i32p]
        L.so_tune_rank.restype = C.c_int32
        L.so_tune_rank.argtypes = [C.c_int32, dp, i64p, i64p, i32p, C.c_double]
        L.so_pt_run.restype = C.c_int32
        L.so_pt_run.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_double, i64p, i64p, i64p, i64p, i32p, dp, i64p,
                                i64p, i32p, i32p, i32p, C.c_int32, i8p, i8p, i32p, i8p, C.c_int32]
        _lib = L
    return _lib


def tune_rank(scale, n_prop, n_acc, proposed, target):
    """so_tune_rank on copies: (new scale, new n_prop, new n_acc), all [nc][4]."""
    s = np.array(scale, dtype=np.float64)
    p = np.array(n_prop, dtype=np.int64)
    a = np.array(n_acc, dtype=np.int64)
    pr = np.ascontiguousarray(proposed, dtype=np.int32)
    lib().so_tune_rank(s.shape[0], s.ctypes.data_as(oracle_c.dp), p.ctypes.data_as(oracle_c.i64p),
                       a.ctypes.data_as(oracle_c.i64p), pr.ctypes.data_as(oracle_c.i32p), float(target))
    return s, p, a


class StepOraclePT(lo.LadderOraclePT):
    """LadderOraclePT with the width tuning (off by default: then its runs are LadderOraclePT's)."""

    def __init__(self, cfg, nproc: int, nthreads: int = 0):
        super().__init__(cfg, nproc, nthreads)
        self.steps, self.target = 0, 0.0
        shape = (nproc, cfg.nchains, 4)
        self.scale = np.ones(shape)
        self.st_nprop = np.zeros(shape, np.int64)
        self.st_nacc = np.zeros(shape, np.int64)
        self.lvl = np.zeros(self.G, np.int32)
        self.pair = np.full(2, -1, np.int32)
        self._st_points = np.zeros(1, np.int32)
        self.dev = np.array([cfg.dev_z, cfg.dev_dvs, cfg.dev_dvp, cfg.dev_sig])

    def set_step_tuning(self, on, target: float = 0.44) -> None:
        if on:   # a fresh start, as rfinv_pt_set_step_tuning (only before the first iteration)
            self.scale[:] = 1.0
            self.st_nprop[:] = 0
            self.st_nacc[:] = 0
            self.pair[:] = -1
            self._st_points[0] = 0
            lib().so_levels(self._h, self.lvl.ctypes.data_as(oracle_c.i32p))
            self.target = float(target)
        self.steps = int(on)

    def set_rank_swaps(self, mode: int) -> None:
        super().set_rank_swaps(mode)
        if int(mode) == 0:
            self.steps = 0

    def step_tuning(self) -> dict:
        widths = self.dev * (self.scale if self.steps else np.ones_like(self.scale))
        return dict(on=bool(self.steps), target=self.target, n_points=int(self._st_points[0]), widths=widths,
                    n_prop=self.st_nprop.copy(), n_acc=self.st_nacc.copy())

    def run(self, n_iter: int, log: bool = True, record: bool = False):
        flags = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        itypes = np.empty((n_iter, self.G), dtype=np.int8) if log else None
        swaps = np.zeros((n_iter, 3), dtype=np.int32) if log else None
        self.pairlog = np.zeros((n_iter, self.G), dtype=np.int8) if log else None
        p = oracle_c._p
        lib().so_pt_run(self._h, self.mode, self.tune, self.steps, self.target, p(self.n_prop, oracle_c.i64p),
                        p(self.n_acc, oracle_c.i64p), p(self.rows, oracle_c.i64p), p(self.base, oracle_c.i64p),
                        p(self._points, oracle_c.i32p), p(self.scale, oracle_c.dp), p(self.st_nprop, oracle_c.i64p),
                        p(self.st_nacc, oracle_c.i64p), p(self.lvl, oracle_c.i32p), p(self.pair, oracle_c.i32p),
                        p(self._st_points, oracle_c.i32p), n_iter, p(flags, oracle_c.i8p), p(itypes, oracle_c.i8p),
                        p(swaps, oracle_c.i32p), p(self.pairlog, oracle_c.i8p), int(record))
        return flags, itypes, swaps
