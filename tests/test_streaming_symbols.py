"""Streaming runs without a device: the C ABI declares and exports miqp_b200_batch_run_streaming, and the Python wrapper's
callback, queue and exception handling work against a stand-in for the C call."""
import ctypes as C
import os
import threading

import numpy as np
import pytest

import planner_miqp_b200 as P
from planner_miqp_b200 import capi

INCLUDE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")


def test_entry_point_is_declared_exported_and_listed():
    hdr = open(os.path.join(INCLUDE, "miqp_b200.h")).read()
    assert "miqp_b200_batch_run_streaming(" in hdr
    assert "typedef void (*MiqpB200PlanDone)(" in hdr
    assert "miqp_b200_batch_run_streaming" in P.DECLARED_SYMBOLS
    assert hasattr(P.load_library(), "miqp_b200_batch_run_streaming")


class FakeLib:
    """miqp_b200_batch_run_streaming of a batch whose plans finish in the given order: calls the C callback for each."""

    def __init__(self, order, shapes, rc=0):
        self.order, self.shapes, self.rc = order, shapes, rc
        self.calls = 0

    def miqp_b200_batch_run_streaming(self, h, cfunc, user, ms):
        self.calls += 1
        for rnd, k in enumerate(self.order):
            c, n = self.shapes[k]
            traj = (C.c_double * (c * n * 8))(*np.arange(c * n * 8, dtype=np.float64) + 1000 * k)
            info = capi.CSolveInfo()
            info.status, info.objective, info.rounds, info.nodes = 0, float(k), rnd + 1, 7
            cfunc(None, k, C.cast(traj, capi._dp), C.byref(info))
        C.cast(ms, C.POINTER(C.c_float))[0] = 12.5
        return self.rc

    def miqp_b200_last_error(self, h):
        return b"stand-in error"


def fake_solver(order, shapes, rc=0):
    s = capi.Solver.__new__(capi.Solver)
    s._lib = FakeLib(order, shapes, rc)
    s._h = None
    s._shapes = shapes
    s._batch = (len(shapes), [1] * len(shapes))
    return s


def test_run_streaming_copies_every_plan():
    shapes = [(1, 3), (2, 4), (1, 5)]
    s = fake_solver([2, 0, 1], shapes)
    got = []
    ms = s.run_streaming(lambda k, t, i: got.append((k, t, i)))
    assert ms == 12.5
    assert [k for k, _, _ in got] == [2, 0, 1]
    for k, t, i in got:
        c, n = shapes[k]
        assert t.shape == (c, n, 8)
        assert np.array_equal(t.ravel(), np.arange(c * n * 8) + 1000 * k)   # a copy: the C buffer is gone by now
        assert isinstance(i, P.SolveInfo) and i.objective == k and i.nodes == 7


def test_exception_in_callback_is_raised_after_the_run():
    s = fake_solver([0, 1, 2, 3], [(1, 2)] * 4)
    seen = []

    def on_plan(k, t, i):
        seen.append(k)
        if k == 1:
            raise ValueError("bad plan")

    with pytest.raises(ValueError, match="bad plan"):
        s.run_streaming(on_plan)
    assert seen == [0, 1]                  # no calls after the first exception
    assert s._lib.calls == 1               # the run itself went to its end
    got = []
    s.run_streaming(lambda k, t, i: got.append(k))   # and the solver is usable again
    assert got == [0, 1, 2, 3]


def test_error_code_of_the_call_raises():
    s = fake_solver([0], [(1, 2)], rc=-2)
    with pytest.raises(P.MiqpB200Error, match="stand-in error"):
        s.run_streaming(lambda k, t, i: None)


def test_generator_yields_every_plan_from_a_worker_thread():
    shapes = [(1, 2)] * 6
    s = fake_solver([3, 1, 5, 0, 2, 4], shapes)
    threads = set()
    gen = capi._stream_results(lambda on_plan: (threads.add(threading.current_thread().name), s.run_streaming(on_plan)))
    got = [k for k, _, _ in gen]
    assert got == [3, 1, 5, 0, 2, 4]
    assert threads == {"miqp_b200-streaming"}
    assert not any(t.name == "miqp_b200-streaming" for t in threading.enumerate())


def test_abandoned_generator_leaves_no_thread():
    s = fake_solver(list(range(50)), [(1, 2)] * 50)
    gen = capi._stream_results(s.run_streaming)
    first = next(gen)
    assert first[0] == 0
    gen.close()
    assert not any(t.name == "miqp_b200-streaming" for t in threading.enumerate())
    assert s._lib.calls == 1


def test_generator_raises_the_run_error():
    s = fake_solver([0, 1], [(1, 2)] * 2, rc=-1)
    gen = capi._stream_results(s.run_streaming)
    assert [k for k, _, _ in [next(gen), next(gen)]] == [0, 1]
    with pytest.raises(P.MiqpB200Error):
        next(gen)
