"""Builds the in-tree CUDA shared library ``rf_inv_b200/librfinv_b200.so`` for sm_100a with nvcc.

No torch types cross the library boundary (plain C-ABI, include/rfinv_b200.h), so the extension is built
with nvcc directly instead of torch.utils.cpp_extension; nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "librfinv_b200.so")
SOURCES = ["capi.cu", "forward.cu", "forward_general.cu", "likelihood.cu", "pt.cu", "comm.cu", "checkpoint.cu", "fp64_peak.cu", "host_io.cu"]
HEADERS = ["rfinv_common.cuh", "rfinv_handle.h", "rfinv_pt.h", os.path.join("..", "..", "include", "rfinv_b200.h")]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return SO
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    nvcc = nvcc_path()
    objs = []
    procs = []
    env = dict(os.environ)
    # the image exports CC/CXX pointing at a gcc wrapper without OpenMP specs; use the system g++ as host compiler
    host_cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    for s in SOURCES:
        o = os.path.join(objdir, s.replace(".cu", ".o"))
        objs.append(o)
        cmd = [nvcc, "-ccbin", host_cxx] + NVCC_FLAGS + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, env=env, text=True)))
    log = []
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {s} ====\n{out}")
        failed |= p.returncode != 0
    with open(os.path.join(objdir, "build.log"), "w") as f:
        f.write("\n".join(log))
    if failed or verbose:
        sys.stderr.write("\n".join(log))
    if failed:
        raise RuntimeError("nvcc failed, see rf_inv_b200/build/build.log")
    cmd = [nvcc, "-ccbin", host_cxx, "-shared", "-o", SO] + objs + ["-lcudart", "-ldl"]
    subprocess.check_call(cmd, env=env)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
