"""Builds and runs tests/cpp/test_host_api.cpp against libmiqp_planner_c_api.so (the C++ classes
MiqpPlanner / B200Wrapper a reference-side caller uses directly)."""
import os
import subprocess

import pytest

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
PKG = os.path.join(ROOT, "planner-miqp_b200")
EXE = os.path.join(ROOT, "tests", "cpp", "test_host_api")


def _build():
    import planner_miqp_b200  # noqa: F401  (makes sure the libraries exist)
    from planner_miqp_b200 import planner_capi
    planner_capi.load_library()
    src = EXE + ".cpp"
    hdrs = [os.path.join(PKG, "host", f) for f in os.listdir(os.path.join(PKG, "host")) if f.endswith(".hpp")]
    newest = max([os.path.getmtime(src), os.path.getmtime(planner_capi.library_path())] + [os.path.getmtime(h) for h in hdrs])
    if os.path.exists(EXE) and os.path.getmtime(EXE) >= newest:
        return
    subprocess.run(["g++", "-std=c++17", "-O1", "-Wall", "-Wno-comment", src, "-o", EXE, "-L" + PKG, "-lmiqp_planner_c_api",
                    "-lmiqp_b200", "-Wl,-rpath," + PKG], check=True)


def test_host_api_cpu(tmp_path):
    _build()
    r = subprocess.run([EXE, "cpu", os.path.abspath(ROOT), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_host_api_gpu(tmp_path):
    _build()
    r = subprocess.run([EXE, "gpu", os.path.abspath(ROOT), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
