"""The refusals of the multi-station driver (python -m rf_inv_b200.run a/params.in b/params.in ...) that happen before any
GPU work: two stations writing to the same OUT_DIR, and stations that differ in N_BURN, N_ITER or N_CORR (a group advances
its stations in lock step)."""
import os

import numpy as np
import pytest

from rf_inv_b200 import build as rbuild
from rf_inv_b200 import run as rrun
from rf_inv_b200 import workloads

# line of params.in (after the comment line) that holds each value; tests/test_gpu_checkpoint.py::_problem_dir writes them
PARAM_LINE = {"OUT_DIR": 1, "N_BURN": 2, "N_ITER": 3, "N_CORR": 4, "I_SEED": 8}


@pytest.fixture(scope="module", autouse=True)
def lib():
    rbuild.build()


def station_dirs(tmp_path, n, noise=0.0):
    """n problem directories in the format of tests/test_gpu_checkpoint.py::_problem_dir, each with its own I_SEED and, with
    noise > 0, its own observed traces.  Returns the params.in paths."""
    import helpers
    from test_gpu_checkpoint import _problem_dir
    paths = []
    for i in range(n):
        cfg = workloads.make_config("sample")
        if noise > 0:
            cfg = helpers.attach_obs_and_rinv(cfg, noise_seed=100 + i, noise=noise)
        else:
            cfg.obs = np.zeros((cfg.ntrc, cfg.nsmp))
        d = tmp_path / f"station{i}"
        _problem_dir(d, cfg)
        set_param(d / "params.in", "I_SEED", 12345678 + 1000 * i)
        paths.append(str(d / "params.in"))
    return paths


def set_param(path, name, value):
    lines = open(path).read().split("\n")
    lines[PARAM_LINE[name]] = str(value)
    open(path, "w").write("\n".join(lines))


def _refused(paths, words):
    with pytest.raises(ValueError) as e:
        rrun.main(list(paths) + ["--nproc", "4"])
    for w in words:
        assert w in str(e.value), (w, str(e.value))
    for p in paths:                                        # nothing was written: refused before any work
        assert not os.path.exists(os.path.join(os.path.dirname(p), "rslt"))


def test_stations_sharing_an_out_dir_are_refused(tmp_path):
    a, b, c = station_dirs(tmp_path, 3)
    _refused([a, b, a], ["stations 0", "and 2", "same OUT_DIR"])
    set_param(c, "OUT_DIR", f"'{os.path.join(os.path.dirname(a), 'rslt')}'")   # another file, the same directory
    _refused([a, b, c], ["stations 0", "and 2", "same OUT_DIR"])


@pytest.mark.parametrize("name", ["N_BURN", "N_ITER", "N_CORR"])
def test_stations_with_different_iteration_counts_are_refused(tmp_path, name):
    a, b, c = station_dirs(tmp_path, 3)
    set_param(b, name, 20)
    _refused([a, b, c], [name, f"{b}: 20"])
