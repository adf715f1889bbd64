"""Solution pool (miqp_b200_set_solution_pool / pool_sizes / pool_fetch): the best distinct integer-feasible leaves the device
search solves, best first, through every layer -- C ABI / capi.Solver, B200Wrapper (pybind CplexWrapper), MiqpPlanner and the
planner C ABI.  The pool records leaves only: with it on or off the search and its results are the same."""
import os

import numpy as np
import pytest

import planner_miqp_b200 as P
from planner_miqp_b200.scenarios import obstacle_scenario, parallel_lanes, two_agent_merge, advance_obstacle_scenario
from oracle import oracle as O

pytestmark = pytest.mark.gpu

CAP = 8
NPLANS = 256
# seeds of obstacle_scenario tried for a rough first incumbent: the search stopped after the first of ROUGH_ROUNDS round counts
# that leaves an incumbent more than 1e-3 (relative) above the optimum
ROUGH_SEEDS = list(range(32))
ROUGH_ROUNDS = list(range(2, 25))


@pytest.fixture(scope="module")
def batch(testcase_problem):
    return [obstacle_scenario(k).build() for k in range(NPLANS)] + [testcase_problem]


def solve(ps, pool, **kw):
    s = P.Solver(solution_pool=pool, **kw)
    s.upload(ps, gap_tol=1e-4, time_limit=60)
    s.run()
    xs, infos = s.fetch()
    return s, xs, infos


def binaries(p, x):
    isb, _, _ = O.col_info(p)
    return np.asarray(x)[isb.astype(bool)]


def check_pool(s, k, p, info, cap, size, oracle=True, x_inc=None, traj_inc=None):
    """checks 2 and 3 of the pool of plan k"""
    ents = s.pool(k)
    assert len(ents) == size
    if info.status != 0:
        assert size == 0
        return ents
    assert 1 <= size <= cap
    e0 = ents[0]
    assert np.array_equal(e0.x, s.fetch_vector(k) if x_inc is None else x_inc)
    assert e0.objective == info.objective and e0.max_violation == info.max_violation
    if traj_inc is not None:
        assert np.array_equal(e0.traj, traj_inc)
    vals = [e.search_value for e in ents]
    assert all(a <= b for a, b in zip(vals, vals[1:])), vals
    bins = []
    for e in ents:
        assert e.max_violation <= 1e-6, (k, e)
        if oracle:
            assert O.objective(p, e.x) == pytest.approx(e.objective, rel=1e-9, abs=1e-12)
            rc, _, fixed = O.solve_fixed(p, e.x)
            assert rc == 0
            if e.converged:
                assert e.objective == pytest.approx(fixed, rel=1e-6, abs=1e-9), (k, e.objective, fixed)
            else:
                assert e.objective >= fixed - 1e-6 * abs(fixed) - 1e-9
        bins.append(binaries(p, e.x))
    for a in range(len(bins)):
        for b in range(a):
            assert not np.array_equal(bins[a], bins[b]), (k, a, b)
    return ents


def test_pool_changes_no_result_and_entry_zero_is_the_incumbent(batch):
    s0, xs0, in0 = solve(batch, 0)
    s1, xs1, in1 = solve(batch, CAP)
    for a, b, xa, xb in zip(in0, in1, xs0, xs1):
        assert np.array_equal(xa, xb)
        for f in ("status", "objective", "best_bound", "gap", "nodes", "qp_iters", "rounds"):
            va, vb = getattr(a, f), getattr(b, f)
            assert va == vb or (np.isnan(va) and np.isnan(vb)), f
    with pytest.raises(P.MiqpB200Error):
        s0.pool_sizes()                      # the pool was off for that batch
    sizes = s1.pool_sizes()
    tr, _ = s1.fetch_compact()
    for k, (p, info) in enumerate(zip(batch, in1)):
        # oracle checks on a share of the batch (the fixed-binary QP is a CPU solve per entry)
        check_pool(s1, k, p, info, CAP, sizes[k], oracle=(k < 24 or k == len(batch) - 1), x_inc=xs1[k], traj_inc=tr[k])
    hist = np.bincount(sizes, minlength=CAP + 1)
    print("pool size histogram (0..%d entries) over %d plans: %s" % (CAP, len(batch), hist.tolist()))
    assert sizes.max() >= 2
    s0.close(); s1.close()


def test_pool_keeps_the_mip_start_next_to_better_plans():
    found = 0
    for seed in ROUGH_SEEDS:
        p = obstacle_scenario(seed).build()
        so, xo, io = solve([p], 0)
        so.close()
        for rounds in ROUGH_ROUNDS:
            sr = P.Solver(max_rounds=rounds)
            xr, ir = sr.solve(p, gap_tol=1e-4, time_limit=60)
            sr.close()
            if ir.status == 0:
                break
        if ir.status != 0 or not ir.objective > io[0].objective * (1 + 1e-3):
            continue
        found += 1
        s = P.Solver(solution_pool=64)
        s.upload([p], gap_tol=1e-4, time_limit=60, warm=[xr])
        s.run()
        _, infos = s.fetch()
        ents = check_pool(s, 0, p, infos[0], 64, s.pool_sizes()[0])
        assert len(ents) >= 2
        br = binaries(p, xr)
        assert any(np.array_equal(binaries(p, e.x), br) and e.objective <= ir.objective * (1 + 1e-9) for e in ents), seed
        s.close()
    print("rough incumbents above the optimum: %d of %d seeds" % (found, len(ROUGH_SEEDS)))
    assert found >= 1


@pytest.mark.parametrize("make", [lambda: parallel_lanes(2, nr_steps=5), lambda: two_agent_merge(0, nr_steps=8),
                                  lambda: two_agent_merge(1, nr_steps=8)])
def test_multi_car_kernel(make):
    p = make().build()
    s, xs, infos = solve([p], CAP)
    assert infos[0].status == 0
    check_pool(s, 0, p, infos[0], CAP, s.pool_sizes()[0])
    s.close()


def test_cta_per_node_kernel_on_the_test_case(testcase_problem, monkeypatch):
    monkeypatch.setenv("MIQP_B200_FORCE_MULTI", "1")
    s, xs, infos = solve([testcase_problem], CAP)
    check_pool(s, 0, testcase_problem, infos[0], CAP, s.pool_sizes()[0])
    s.close()


def pools(s, n):
    return [[(e.search_value, e.uid, e.converged, e.round, e.objective, e.max_violation, e.x.tobytes()) for e in s.pool(k)]
            for k in range(n)]


def test_determinism_team_sizes_and_reset(batch, monkeypatch):
    ps = batch[:64]
    s, _, _ = solve(ps, CAP)
    first = pools(s, len(ps))
    s.run()                                   # a second run of the same upload restarts the pool
    assert pools(s, len(ps)) == first
    s2, _, _ = solve(ps, CAP)                 # another solver: byte-identical pools
    assert pools(s2, len(ps)) == first
    s2.close()
    monkeypatch.setenv("MIQP_NO_NARROW_TEAM", "1")
    monkeypatch.setenv("MIQP_NO_WIDE_TEAM", "1")
    s3, _, _ = solve(ps, CAP)
    other = pools(s3, len(ps))
    s3.close()
    # the same leaves (uids, integer assignments) with every team size; their relaxations run on 2, 4 or 8 warps, so the points
    # agree to the interior-point tolerance (as the incumbents do, test_gpu_solve.py::test_two_warp_teams_give_the_same_results)
    for a, b, p in zip(first, other, ps):
        assert [e[1] for e in a] == [e[1] for e in b]
        for ea, eb in zip(a, b):
            xa, xb = np.frombuffer(ea[6]), np.frombuffer(eb[6])
            assert np.array_equal(binaries(p, xa), binaries(p, xb))
            assert ea[4] == pytest.approx(eb[4], rel=1e-6)
            np.testing.assert_allclose(xa, xb, atol=1e-4)
    # receding horizon: the next cycle's pool is feasible for the next cycle's problems
    builders = [obstacle_scenario(k) for k in range(16)]
    ps = [b.build() for b in builders]
    s.upload(ps, gap_tol=1e-4, time_limit=60)
    s.run()
    xs, _ = s.fetch()
    nxt = [advance_obstacle_scenario(b, p, x).build() for b, p, x in zip(builders, ps, xs)]
    s.upload_replan(nxt, gap_tol=1e-4, time_limit=60)
    s.run()
    _, infos = s.fetch()
    sizes = s.pool_sizes()
    for k, p in enumerate(nxt):
        for e in check_pool(s, k, p, infos[k], CAP, sizes[k], oracle=False):
            viol, _ = O.max_violation(p, e.x)
            assert viol <= 1e-6
    s.close()


def test_arguments():
    s = P.Solver()
    for bad in (-1, 65):
        with pytest.raises(P.MiqpB200Error):
            s.set_solution_pool(bad)
    s.set_solution_pool(4)
    p = obstacle_scenario(0).build()
    s.upload([p], gap_tol=1e-4, time_limit=60)
    with pytest.raises(P.MiqpB200Error):
        s.pool_sizes()                        # before a run
    s.run()
    assert s.pool_sizes()[0] >= 1
    assert len(s.pool(0, vectors=False, max_entries=1)) == 1
    s.set_solution_pool(0)                    # takes effect at the next upload
    assert s.pool_sizes()[0] >= 1
    s.close()


# ---- host layers: B200Wrapper (pybind CplexWrapper), MiqpPlanner and the planner C ABI ---------------------------------------
def test_cplex_wrapper_pool_and_nr_solution_pool():
    import importlib.util
    import sys
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "planner-miqp_b200")
    spec = importlib.util.spec_from_file_location("_b", os.path.join(pkg, "build.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    b.build_pymodule()
    if pkg not in sys.path:
        sys.path.insert(0, pkg)
    import miqp
    w = miqp.CplexWrapper("cplexmodel.mod", 12)
    w.setParameterDatFileAbsolute(os.path.join(pkg, "..", "tests", "golden", "cplexmodel_testcase.dat"))
    assert not w.setSolutionPoolCapacity(65)
    assert w.callCplex(0.0) == miqp.OptimizationStatus.SUCCESS
    assert w.getSolutionProperties().NrSolutionPool == 1 and w.getSolutionPool() == []   # pool off: as before
    assert w.setSolutionPoolCapacity(4)
    assert w.callCplex(0.0) == miqp.OptimizationStatus.SUCCESS
    pool = w.getSolutionPool()
    assert w.getSolutionProperties().NrSolutionPool == len(pool) >= 1
    obj, viol, conv, x = pool[0]
    assert np.array_equal(x, w.getSolutionVector())
    assert obj == pytest.approx(w.getSolutionProperties().objective, rel=1e-12)
    assert all(v <= 1e-6 for _, v, _, _ in pool)


def _planner(k, cap):
    from planner_miqp_b200 import planner_capi as PC
    p = PC.CMiqpPlanner()
    assert p.set_solution_pool(cap)
    p.add_car([0, 3 + 0.5 * k, 0, 0.2 * k, 0.1, 0], [0, 0, 50, 0], 5, 1)
    p.add_obstacle([[[12, -1.5 + 0.3 * k], [15, -1.5 + 0.3 * k], [15, 1.5], [12, 1.5]]] * p.N, is_static=True)
    return p


def test_planner_c_abi_pool():
    p = _planner(0, 6)
    assert not p.set_solution_pool(-1)
    assert p.plan(0.0)
    n = p.solution_pool_size()
    assert 1 <= n <= 6
    obj0, rows0 = p.solution_pool_trajectory(0, 0, 1.5)
    assert np.array_equal(rows0, p.trajectory(0, 1.5))
    assert obj0 == p.solution_properties()["objective"]
    objs = [p.solution_pool_trajectory(j)[0] for j in range(n)]
    assert all(np.isfinite(objs))
    bad, rows = p.solution_pool_trajectory(n)
    assert np.isnan(bad) and rows.shape[0] == 0
    p.close()


def test_plan_batch_gives_every_planner_its_own_pool():
    from planner_miqp_b200 import planner_capi as PC
    caps = [3, 6, 0, 6]
    singles, want = [], []
    for k, c in enumerate(caps):
        p = _planner(k, c)
        assert p.plan(0.0)
        want.append([p.solution_pool_trajectory(j) for j in range(p.solution_pool_size())])
        singles.append(p)
    batch = [_planner(k, c) for k, c in enumerate(caps)]
    assert PC.plan_batch(batch, 0.0) == [True] * len(caps)
    for k, (p, w) in enumerate(zip(batch, want)):
        assert p.solution_pool_size() == len(w) <= caps[k]
        for j, (o, rows) in enumerate(w):   # the leaves' relaxations may run on other team sizes in a batch: solver tolerance
            oj, rj = p.solution_pool_trajectory(j)
            assert oj == pytest.approx(o, rel=1e-6)
            np.testing.assert_allclose(rj, rows, atol=1e-6)
    for p in singles + batch:
        p.close()
