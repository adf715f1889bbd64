"""The pybind11 module `miqp` (planner-miqp_b200/host/python_module.cpp) against what the reference's Python tests do
with theirs (python/bindings/tests/python_import_test.py: import; test/py_convexified_map_test.py: decomposition of road
polygons succeeds; python_cplex_wrapper.cpp:19-69: CplexWrapper on a .dat file, SolutionProperties, enums)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "planner-miqp_b200")


@pytest.fixture(scope="module")
def miqp():
    import planner_miqp_b200  # noqa: F401  (builds the libraries if needed)
    import importlib.util
    spec = importlib.util.spec_from_file_location("_b", os.path.join(PKG, "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    b.build_pymodule()
    if PKG not in sys.path:
        sys.path.insert(0, PKG)
    import miqp as m
    return m


def area(v):
    x, y = v[:, 0], v[:, 1]
    return 0.5 * float(np.sum(x * np.roll(y, -1) - np.roll(x, -1) * y))


def is_convex_ccw(v, tol=1e-9):
    n = len(v)
    for k in range(n):
        a, b, c = v[k], v[(k + 1) % n], v[(k + 2) % n]
        if (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0]) < -tol:
            return False
    return True


def test_import_enums_and_solution_properties(miqp):
    assert int(miqp.OptimizationStatus.SUCCESS) == 0 and int(miqp.OptimizationStatus.FAILED_TIMEOUT) == 3
    assert miqp.SUCCESS == miqp.OptimizationStatus.SUCCESS                      # export_values, as in the reference
    assert int(miqp.WarmstartType.BOTH_WARMSTART_STRATEGIES) == 3 and int(miqp.ParallelMode.OPPORTUNISTIC) == -1
    sp = miqp.SolutionProperties()
    sp.objective, sp.status, sp.gap, sp.time = 1.5, 101, 0.0, 0.25
    assert (sp.objective, sp.status, sp.gap, sp.time) == (1.5, 101, 0.0, 0.25)


def test_convexified_map_decomposes_an_l_shaped_road(miqp):
    # L-shaped road, 10 m wide arms, given clockwise and closed (the planner accepts both conventions)
    poly = np.array([[0, 0], [0, 40], [10, 40], [10, 10], [50, 10], [50, 0], [0, 0]], dtype=float)
    r = 1.0
    cm = miqp.ConvexifiedMap(None, poly, r, 0.0, 2.0, 1e-9)
    assert cm.HasValidPolygon() and cm.Convert()
    cells = cm.map_convex_polygons
    assert 2 <= len(cells) <= 3                                   # Hertel-Mehlhorn: at most 4x the optimum (2)
    for v in cells.values():
        assert is_convex_ccw(v) and area(v) > 0
    total = sum(area(v) for v in cells.values())
    # the offset region of the L has area 8*38 + 40*8 - the rounded reflex corner; the cells cover it up to that corner piece
    assert 8 * 38 + 40 * 8 - 1.0 <= total <= 8 * 39 + 40 * 8 + 1e-9
    # every cell keeps the collision radius from the boundary of the input polygon
    edges = list(zip(poly[:-1], poly[1:]))
    for v in cells.values():
        for p in v:
            d = min(np.linalg.norm(p - (a + np.clip(np.dot(p - a, b - a) / np.dot(b - a, b - a), 0, 1) * (b - a))) for a, b in edges)
            assert d >= r - 1e-9
    # the cells overlap or touch (a car can pass from one arm into the other): the diagonal between them is not shrunk
    pts = [np.array([5.0, 5.0]), np.array([5.0, 9.5]), np.array([9.0, 5.0])]
    def inside(v, p):
        return all((v[(k + 1) % len(v)][0] - v[k][0]) * (p[1] - v[k][1]) - (v[(k + 1) % len(v)][1] - v[k][1]) * (p[0] - v[k][0]) >= -1e-9 for k in range(len(v)))
    for p in pts:
        assert any(inside(v, p) for v in cells.values())
    # reference along the lower arm only: the upper arm's cell is not selected when it is farther than the buffer
    sel = cm.GetIntersectingConvexPolygons(np.array([[30.0, 5.0], [45.0, 5.0]]))
    assert 1 <= len(sel) <= len(cells) and all(k in cells for k in sel)
    assert np.allclose(cm.map_nonconvex_polygon, poly)


def test_convexified_map_rejects_degenerate_polygons(miqp):
    assert not miqp.ConvexifiedMap(None, np.array([[0, 0], [1, 0], [2, 0]], dtype=float), 0.5, 0.0, 2.0, 1e-9).Convert()
    # narrower than twice the radius: nothing is left
    assert not miqp.ConvexifiedMap(None, np.array([[0, 0], [10, 0], [10, 1], [0, 1]], dtype=float), 1.0, 0.0, 2.0, 1e-9).Convert()
    # a convex polygon is one cell
    cm = miqp.ConvexifiedMap(None, np.array([[0, 0], [10, 0], [10, 6], [0, 6]], dtype=float), 1.0, 0.0, 2.0, 1e-9)
    assert cm.Convert() and len(cm.map_convex_polygons) == 1
    assert np.isclose(area(cm.map_convex_polygons[0]), 8 * 4)


def test_cplex_wrapper_surface_without_device(miqp):
    w = miqp.CplexWrapper("cplexmodel.mod", 12)
    w.setDebugOutputPrint(False)
    w.setDebugOutputFilePrefix("pytest_")
    assert w.getDebugOutputParameterFilePath() == ""
    w.setParameterDatFileAbsolute("/nonexistent/file.dat")
    assert w.callCplex(0.0) == miqp.FAILED_SEG_FAULT              # the solver could not run
    assert "nonexistent" in w.lastError() or w.lastError() != ""


@pytest.mark.gpu
def test_cplex_wrapper_solves_the_reference_fixture(miqp, tmp_path):
    w = miqp.CplexWrapper("cplexmodel.mod", 12)
    w.setParameterDatFileAbsolute(os.path.join(ROOT, "tests", "golden", "cplexmodel_testcase.dat"))
    assert w.callCplex(0.0) == miqp.OptimizationStatus.SUCCESS
    sp = w.getSolutionProperties()
    assert abs(sp.objective - 9.57603) <= 0.1 * 9.57603 and sp.gap <= 0.1 and sp.time > 0    # the file asks for a 10 % gap
    mst, lp = str(tmp_path / "miqp_b200_pybind.mst"), str(tmp_path / "miqp_b200_pybind.lp")
    assert w.writeMIPStarts(mst) and w.readMIPStarts(mst)
    assert w.exportModel(lp) and os.path.getsize(lp) > 100000


# ---- BehaviorMiqpAgent (host/behavior_miqp_agent.hpp: the planning cycle of src/behavior_miqp_agent.cpp:137-335 without BARK) ----
ROAD = np.array([[-20.0, -6.0], [150.0, -6.0], [150.0, 6.0], [-20.0, 6.0]])
LANE = np.array([[-20.0, 0.0], [150.0, 0.0]])


def _world(t, ego, others=()):
    return {"time": t, "road_polygon": ROAD,
            "ego": {"id": 1, "state": ego, "length": 4.0, "width": 2.0, "lane_center": LANE},
            "others": [{"id": 10 + k, "state": o, "length": 4.0, "width": 2.0, "lane_center": LANE + np.array([0.0, o[1]])}
                       for k, o in enumerate(others)]}


def test_behavior_agent_bookkeeping_and_failure_path(miqp):
    """without a CUDA device Plan() cannot succeed: the agent must report it the way the reference does (status EXPIRED,
    NaN solution time, the last trajectory -- src/behavior_miqp_agent.cpp:264-271) after having set up planner, map and obstacles"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("failure path needs a box without GPU")
    a = miqp.BehaviorMiqpAgent({"Miqp::NrSteps": 10, "Miqp::NrRegions": 16, "Miqp::DesiredVelocity": 6.0})
    assert a.behavior_status == miqp.BehaviorStatus.NOT_STARTED_YET
    tr = a.Plan(0.25, _world(0.0, [0, 0, 0, 5, 0], others=[[25, 0, 0, 2, 0]]))
    assert tr.shape == (0, 5) and not a.last_planning_success
    assert a.behavior_status == miqp.BehaviorStatus.EXPIRED and np.isnan(a.last_solution_time)
    assert a.car_idxs == {1: 0} and list(a.obstacle_ids) == [10]
    np.testing.assert_allclose(a.env_polygon, ROAD)
    # box environment (Miqp::UseBoxAsEnv): bounding box of an L-shaped road
    b = miqp.BehaviorMiqpAgent({"Miqp::NrSteps": 10, "Miqp::UseBoxAsEnv": True})
    w = _world(0.0, [0, 0, 0, 5, 0])
    w["road_polygon"] = np.array([[0, 0], [40, 0], [40, 30], [30, 30], [30, 10], [0, 10.0]])
    b.Plan(0.25, w)
    np.testing.assert_allclose(b.env_polygon, [[0, 0], [40, 0], [40, 30], [0, 30]])


@pytest.mark.gpu
def test_behavior_agent_follows_and_overtakes_over_several_cycles(miqp):
    """receding-horizon simulation: the ego (5 m/s) comes up behind a slow vehicle (2 m/s) that is predicted with constant
    velocity; every cycle plans, the ego state moves to step 1 of the plan"""
    a = miqp.BehaviorMiqpAgent({"Miqp::NrSteps": 20, "Miqp::NrRegions": 16, "Miqp::DesiredVelocity": 5.0, "Miqp::MaxSolutionTime": 5.0,
                                "Miqp::RelativeMIPGapTolerance": 1e-3, "Miqp::WarmstartType": 1, "Miqp::ObstaclesSoft": False})
    ego = [0.0, 0.0, 0.0, 5.0, 0.0]
    other = [18.0, 0.5, 0.0, 2.0, 0.0]
    dt = 0.25
    min_gap = 1e9
    for k in range(8):
        tr = a.Plan(dt, _world(k * dt, ego, others=[other]))
        assert a.last_planning_success and a.behavior_status == miqp.BehaviorStatus.VALID
        assert tr.shape[1] == 5 and tr.shape[0] >= 2 and tr[0, 0] == pytest.approx(k * dt)
        assert tr[0, 1] == pytest.approx(ego[0], abs=1e-3) and tr[0, 2] == pytest.approx(ego[1], abs=1e-3)
        acc, delta = a.last_action
        assert np.isfinite(acc) and np.isfinite(delta) and abs(delta) < 0.6
        assert a.last_solution_time > 0 and a.obstacle_ids == {10: 0}
        # predicted separation along the plan: rear-axle point stays out of the inflated box (collision radius 1 m)
        for i in range(tr.shape[0]):
            ox = other[0] + other[3] * dt * i
            inside = abs(tr[i, 1] - ox) < 2.0 and abs(tr[i, 2] - other[1]) < 1.0
            assert not inside
            min_gap = min(min_gap, np.hypot(tr[i, 1] - ox, tr[i, 2] - other[1]))
        accel = (tr[1, 4] - ego[3]) / dt
        ego = [tr[1, 1], tr[1, 2], tr[1, 3], tr[1, 4], accel]
        other = [other[0] + other[3] * dt, other[1], 0.0, other[3], 0.0]
    assert ego[0] > 5.0 and min_gap > 1.0


@pytest.mark.gpu
def test_behavior_agent_multi_agent_planning(miqp):
    """Miqp::MultiAgentPlanning: the other agent becomes a second car of the joint plan, re-added every cycle"""
    a = miqp.BehaviorMiqpAgent({"Miqp::NrSteps": 8, "Miqp::NrRegions": 16, "Miqp::DesiredVelocity": 5.0, "Miqp::MaxSolutionTime": 5.0,
                                "Miqp::RelativeMIPGapTolerance": 1e-2, "Miqp::MultiAgentPlanning": True})
    ego = [0.0, -2.5, 0.0, 5.0, 0.0]
    other = [2.0, 3.0, 0.0, 5.0, 0.0]
    for k in range(3):
        w = _world(k * 0.25, ego, others=[other])
        w["ego"]["lane_center"] = LANE + np.array([0.0, -2.5])
        tr = a.Plan(0.25, w)
        assert a.last_planning_success, k
        assert a.car_idxs == {1: 0, 10: 1} and a.obstacle_ids == {}
        ego = [tr[1, 1], tr[1, 2], tr[1, 3], tr[1, 4], 0.0]
        other = [other[0] + 5.0 * 0.25, other[1], 0.0, 5.0, 0.0]
