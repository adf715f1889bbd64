"""Anytime runs without a device: the C ABI declares and exports the anytime entry points, and the Python wrapper's callbacks,
stop returns and exception handling work against a stand-in for the C calls."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import planner_miqp_b200 as P
from planner_miqp_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRY_POINTS = ("miqp_b200_batch_run_anytime", "miqp_b200_request_stop", "miqp_b200_stopped")


def test_entry_points_are_declared_exported_and_listed():
    hdr = open(os.path.join(ROOT, "include", "miqp_b200.h")).read()
    for name in ENTRY_POINTS:
        assert re.search(r"\bint " + name + r"\(", hdr), name
        assert name in P.DECLARED_SYMBOLS
        assert hasattr(P.load_library(), name)
    assert "typedef int (*MiqpB200IncumbentFound)(" in hdr
    assert "typedef struct MiqpB200Incumbent {" in hdr


def test_incumbent_struct_mirrors_the_header():
    # 6 doubles, 3 longs, 1 unsigned long long, no padding on LP64
    assert C.sizeof(capi.CIncumbent) == 6 * 8 + 3 * C.sizeof(C.c_long) + 8
    assert [f for f, _ in capi.CIncumbent._fields_] == ["objective", "max_violation", "search_value", "best_bound", "gap", "seconds",
                                                        "round", "nodes", "qp_iters", "uid"]


class FakeLib:
    """miqp_b200_batch_run_anytime of a batch whose incumbents are found in the given order of (k, round): calls the incumbent
    callback for each, then the plan callback (if any) for every plan; a nonzero return of the incumbent callback is a stop."""

    def __init__(self, found, shapes, rc=0):
        self.found, self.shapes, self.rc = found, shapes, rc
        self.calls = 0
        self.stops = []          # plans stopped through a callback's return or request_stop
        self.had_on_done = None

    def miqp_b200_batch_run_anytime(self, h, ifunc, dfunc, user, ms):
        self.calls += 1
        self.had_on_done = bool(dfunc)
        for j, (k, rnd) in enumerate(self.found):
            c, n = self.shapes[k]
            traj = (C.c_double * (c * n * 8))(*np.arange(c * n * 8, dtype=np.float64) + 1000 * k + j)
            inc = capi.CIncumbent()
            inc.objective, inc.search_value, inc.round, inc.nodes, inc.uid = 10.0 - j, 10.0 - j, rnd, 3 * rnd, 100 + j
            if ifunc(None, k, C.cast(traj, capi._dp), C.byref(inc)):
                self.miqp_b200_request_stop(h, k)
        if dfunc:
            for k, (c, n) in enumerate(self.shapes):
                traj = (C.c_double * (c * n * 8))()
                info = capi.CSolveInfo()
                info.status, info.objective = 0, float(k)
                dfunc(None, k, C.cast(traj, capi._dp), C.byref(info))
        C.cast(ms, C.POINTER(C.c_float))[0] = 7.5
        return self.rc

    def miqp_b200_request_stop(self, h, k):
        if not -1 <= k < len(self.shapes):
            return -2
        self.stops.append(k)
        return 0

    def miqp_b200_stopped(self, h, out):
        for k in range(len(self.shapes)):
            out[k] = 4 if k in self.stops else -1
        return 0

    def miqp_b200_last_error(self, h):
        return b"stand-in error"


def fake_solver(found, shapes, rc=0):
    s = capi.Solver.__new__(capi.Solver)
    s._lib = FakeLib(found, shapes, rc)
    s._h = None
    s._shapes = shapes
    s._batch = (len(shapes), [1] * len(shapes))
    return s


def test_run_anytime_passes_records_to_the_callback():
    shapes = [(1, 3), (2, 4), (1, 5)]
    s = fake_solver([(1, 2), (0, 3), (1, 4)], shapes)
    got = []
    ms = s.run_anytime(lambda k, t, inc: got.append((k, t, inc)))
    assert ms == 7.5
    assert [k for k, _, _ in got] == [1, 0, 1]
    for j, (k, t, inc) in enumerate(got):
        c, n = shapes[k]
        assert t.shape == (c, n, 8)
        assert np.array_equal(t.ravel(), np.arange(c * n * 8) + 1000 * k + j)   # a copy: the C buffer is gone by now
        assert isinstance(inc, P.Incumbent)
        assert inc.objective == 10.0 - j and inc.round == [2, 3, 4][j] and inc.uid == 100 + j
    assert s._lib.had_on_done is False      # on_plan=None: a NULL plan callback
    assert s._lib.stops == []               # None returned: nothing stopped


def test_truthy_return_stops_the_plan():
    s = fake_solver([(0, 1), (1, 1), (2, 1), (0, 2)], [(1, 2)] * 3)
    s.run_anytime(lambda k, t, inc: "stop" if k == 2 or inc.round == 2 else 0)
    assert s._lib.stops == [2, 0]
    assert list(s.stopped()) == [4, -1, 4]
    s.request_stop(1)
    s.request_stop()
    assert s._lib.stops == [2, 0, 1, -1]
    with pytest.raises(P.MiqpB200Error):
        s.request_stop(3)


def test_on_plan_gets_every_plan_after_the_incumbents():
    shapes = [(1, 2), (2, 3)]
    s = fake_solver([(1, 1), (0, 2)], shapes)
    seq = []
    s.run_anytime(lambda k, t, inc: seq.append(("inc", k)), lambda k, t, info: seq.append(("done", k, t.shape, info.objective)))
    assert s._lib.had_on_done is True
    assert seq == [("inc", 1), ("inc", 0), ("done", 0, (1, 2, 8), 0.0), ("done", 1, (2, 3, 8), 1.0)]


def test_exception_in_callback_is_raised_after_the_run():
    s = fake_solver([(k, 1) for k in range(4)], [(1, 2)] * 4)
    seen, plans = [], []

    def on_inc(k, t, inc):
        seen.append(k)
        if k == 1:
            raise ValueError("bad incumbent")
        return True

    with pytest.raises(ValueError, match="bad incumbent"):
        s.run_anytime(on_inc, lambda k, t, i: plans.append(k))
    assert seen == [0, 1]                  # no calls after the first exception, to either callback
    assert plans == []
    assert s._lib.stops == [0]             # the plan the exception was raised for is not stopped
    assert s._lib.calls == 1               # the run itself went to its end
    got = []
    s.run_anytime(lambda k, t, inc: got.append(k))   # and the solver is usable again
    assert got == [0, 1, 2, 3]


def test_exception_in_plan_callback_is_raised_after_the_run():
    s = fake_solver([(0, 1)], [(1, 2)] * 2)

    def on_plan(k, t, i):
        raise KeyError("plan callback")

    with pytest.raises(KeyError):
        s.run_anytime(lambda k, t, inc: None, on_plan)


def test_error_code_of_the_call_raises():
    s = fake_solver([(0, 1)], [(1, 2)], rc=-2)
    with pytest.raises(P.MiqpB200Error, match="stand-in error"):
        s.run_anytime(lambda k, t, inc: None)


# the batched host/device copy entry points of the CUDA runtime and driver (assembled here so that this file does not name them)
BATCHED_COPIES = [pre + "Memcpy" + d + "Batch" + "Async" for pre in ("cuda", "cu") for d in ("", "3D")]


def test_no_source_names_a_batched_copy():
    hits = []
    for top in ("planner-miqp_b200", "tools", "tests", "include", "oracle", "."):
        base = os.path.join(ROOT, top)
        for dirpath, dirs, files in os.walk(base):
            if top == ".":
                dirs[:] = []                # only the files at the root
            dirs[:] = [d for d in dirs if not d.startswith(".") and d != "__pycache__"]
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".cpp", ".hpp", ".h", ".c", ".sh")):
                    continue
                text = open(os.path.join(dirpath, f), errors="replace").read()
                hits += [(os.path.join(dirpath, f), n) for n in BATCHED_COPIES if n in text]
    assert hits == []
    solver = open(os.path.join(ROOT, "planner-miqp_b200", "csrc", "solver.cu")).read()
    assert "cudaMemcpyAsync(s->d_stop.p, s->h_stop.data()" in solver            # the stop mask: one plain async copy
    assert "cudaMemcpyAsync(s->h_airec.data(), s->ai_rec.p" in solver          # the incumbent records likewise


def ptxas_figures(srcs, tmp_path):
    """per kernel (mangled name): registers, stack bytes, spill store bytes, from nvcc -Xptxas -v with the library's flags"""
    import importlib.util
    import subprocess
    spec = importlib.util.spec_from_file_location("_miqp_build_flags", os.path.join(ROOT, "planner-miqp_b200", "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    procs = [subprocess.Popen([nvcc] + b.ARCH + b.COMMON + ["-c", os.path.join(b.CSRC, f), "-o", str(tmp_path / (f + ".o"))],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for f in srcs]
    log = ""
    for p in procs:
        out, _ = p.communicate()
        assert p.returncode == 0, out
        log += out
    figs, entry, props = {}, None, None   # (ptxas lists the frames of out-of-line callees under their own names too)
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            entry = m.group(1)
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            props = m.group(1)
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores", line)
        if props and m:
            figs.setdefault(props, {}).update(stack=int(m.group(1)), spill=int(m.group(2)))
        m = re.search(r"Used (\d+) registers", line)
        if entry and m:
            figs.setdefault(entry, {})["regs"] = int(m.group(1))
    return figs


def test_node_kernels_keep_their_registers_and_the_new_kernels_do_not_spill(tmp_path):
    figs = ptxas_figures(["bnb.cu", "bnb_multi.cu"], tmp_path)
    for nw in (2, 4, 8):
        f = next(v for k, v in figs.items() if "bnb_nodes_kernelILi%dE" % nw in k)
        assert f["regs"] == 255 and f["stack"] == 480 and 164 <= f["spill"] <= 212, (nw, f)
    f = next(v for k, v in figs.items() if "bnb_nodes_multi_kernel" in k)
    assert f["regs"] == 249 and f["spill"] == 0, f
    new = {k: v for k, v in figs.items() if "bnb_inc_" in k and "_kernel" in k}
    assert len(new) == 3
    assert all(v["spill"] == 0 for v in new.values()), new
