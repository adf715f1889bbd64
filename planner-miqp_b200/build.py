"""Builds libmiqp_b200.so (hand-written sm_100a CUDA + host driver) in-tree with nvcc.

The shared library is the product: a C-ABI (include/miqp_b200.h) with no CPU fallback.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmiqp_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off", "-Xptxas", "-v"]
# formulation.cu is compared bit for bit with the oracle: no FMA contraction there
if os.environ.get("MIQP_PROF") == "1":      # per-phase cycle counters of the node kernel (miqp_b200_debug_profile)
    COMMON.append("-DMQ_PROF")
UNITS = [("formulation.cu", ["--fmad=false"]), ("bnb.cu", []), ("bnb_multi.cu", []), ("solver.cu", []), ("peaks.cu", [])]


def _newest_src() -> float:
    t = 0.0
    for root, _, files in os.walk(CSRC):
        for f in files:
            t = max(t, os.path.getmtime(os.path.join(root, f)))
    t = max(t, os.path.getmtime(os.path.join(HERE, "..", "include", "miqp_b200.h")))
    return t


HOST = os.path.join(HERE, "host")
CAPI_LIB = os.path.join(HERE, "libmiqp_planner_c_api.so")
HOST_UNITS = ["b200_wrapper.cpp", "miqp_planner.cpp", "miqp_planner_c_api.cpp"]


def build_host(force: bool = False) -> str:
    """libmiqp_planner_c_api.so: the C++ host side (planner facade + solver driver shaped like the reference's
    MiqpPlanner / CplexWrapper + the 17-function C API), g++, linked against libmiqp_b200.so next to it."""
    newest = max(os.path.getmtime(os.path.join(r, f)) for r, _, fs in os.walk(HOST) for f in fs)
    newest = max(newest, max(os.path.getmtime(os.path.join(HERE, "..", "include", f)) for f in os.listdir(os.path.join(HERE, "..", "include"))))
    if not force and os.path.exists(CAPI_LIB) and os.path.getmtime(CAPI_LIB) >= newest:
        return CAPI_LIB
    gen = os.path.join(HERE, "..", "tools", "gen_fitting_tables_inc.py")
    subprocess.run([sys.executable, gen], check=True, capture_output=True)
    cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-comment", "-DPLANNER_MIQP_CAPI_NO_APOLLO=0",
           "-o", CAPI_LIB] + [os.path.join(HOST, u) for u in HOST_UNITS] + [
           "-L" + HERE, "-lmiqp_b200", "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("host library build failed")
    return CAPI_LIB


def pymodule_path() -> str:
    import sysconfig
    return os.path.join(HERE, "miqp" + sysconfig.get_config_var("EXT_SUFFIX"))


def build_pymodule(force: bool = False) -> str:
    """pybind11 module `miqp` (host/python_module.cpp): the Python surface of the reference's test module
    (python/bindings/python_module.cpp) over the host classes, linked against libmiqp_planner_c_api.so."""
    import pybind11
    import sysconfig
    out = pymodule_path()
    src = os.path.join(HOST, "python_module.cpp")
    newest = max(os.path.getmtime(CAPI_LIB), max(os.path.getmtime(os.path.join(HOST, f)) for f in os.listdir(HOST) if f.endswith((".hpp", ".cpp"))))
    if not force and os.path.exists(out) and os.path.getmtime(out) >= newest:
        return out
    cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-comment", "-fvisibility=hidden",
           "-I" + pybind11.get_include(), "-I" + sysconfig.get_paths()["include"], src, "-o", out,
           "-L" + HERE, "-lmiqp_planner_c_api", "-lmiqp_b200", "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("pybind module build failed")
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= _newest_src():
        build_host(force=False)
        build_pymodule(force=False)
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    log = []
    for src, extra in UNITS:
        obj = os.path.join(CSRC, src.replace(".cu", ".o"))
        cmd = [nvcc] + ARCH + COMMON + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log.append(r.stderr)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed on {src}")
        objs.append(obj)
    cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        sys.stderr.write("\n".join(log))
    build_host(force=True)
    build_pymodule(force=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
