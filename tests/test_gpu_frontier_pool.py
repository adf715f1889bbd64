"""Solution pools of a frontier-sharded search (miqp_b200_pool_export / miqp_b200_pool_merge, capi.Solver.pool_export /
pool_merge, sharding.solve_frontier_sharded(merge_pool=True)).

* one process, W = 2 and 3 emulated ranks (one solver each: upload, ramp-up, frontier_split(r, W), the rest of the search, no
  incumbent exchange): the merged pool equals the pool policy applied by the host to the union of the ranks' pools, every entry
  bit-identical to the rank's entry of the same uid, and passes the checks of test_gpu_solution_pool.py;
* the merge is deterministic (every rank, any rank order in the gathered buffer), a merge with itself changes nothing, host and
  device input give the same pool, and mismatched exports are refused with the pool unchanged;
* two processes on gloo sharing cuda:0, and two GPUs over NCCL: both ranks return the same merged pool, whose entry 0 is the
  combined incumbent, and nothing else of the result changes."""
import dataclasses
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import planner_miqp_b200 as P
from planner_miqp_b200.scenarios import obstacle_scenario, parallel_lanes
from planner_miqp_b200.sharding import solve_frontier_sharded
from oracle import oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAP = 1e-4
CAP = 8
RAMP = 5
NODE_SLOTS = 4096   # open-node slots per plan of each emulated rank (several solvers share the GPU)


def plans_for_test(testcase):
    # single-car plans with obstacles, a two-car plan (the CTA-per-node kernel's pool) and the reference's test case
    return [obstacle_scenario(k).build() for k in (1, 7, 11)] + [parallel_lanes(2, 6, 4.8, stagger=1.0).build(), testcase]


@pytest.fixture(scope="module")
def plans(testcase_problem):
    return plans_for_test(testcase_problem)


def binaries(p, x):
    isb, _, _ = O.col_info(p)
    return np.asarray(x)[isb.astype(bool)]


def rank_solver(ps, rank, world, cap=CAP):
    """one emulated rank: the search of frontier sharding without incumbent exchange (its pool is still a set of solved leaves)"""
    s = P.Solver(pool_capacity=NODE_SLOTS, solution_pool=cap)
    s.upload(ps, gap_tol=GAP, time_limit=120)
    s.frontier_start()
    s.frontier_rounds(RAMP)
    s.frontier_split(rank, world)
    s.frontier_rounds(-1)
    s.frontier_finish()
    return s


def emulate(ps, world):
    solvers = [rank_solver(ps, r, world) for r in range(world)]
    pools = [[s.pool(k) for k in range(len(ps))] for s in solvers]
    exports = [s.pool_export().clone() for s in solvers]
    return solvers, pools, exports


def fetch_all(s, n):
    """everything pool_fetch returns, as bytes"""
    return [[(e.search_value, e.uid, e.converged, e.round, e.objective, e.max_violation, e.x.tobytes(), e.traj.tobytes())
             for e in s.pool(k)] for k in range(n)]


def host_greedy(p, entries, cap):
    """the pool policy over a union of entries: (search_value, uid) order, the first entry of every binary assignment, cap of them"""
    out, seen = [], []
    for e in sorted(entries, key=lambda e: (e.search_value, e.uid)):
        b = binaries(p, e.x)
        if any(np.array_equal(b, o) for o in seen):
            continue
        out.append(e)
        seen.append(b)
        if len(out) == cap:
            break
    return out


def check_entries(p, ents, cap):
    """the pool checks of test_gpu_solution_pool.check_pool that do not need an incumbent of this solver"""
    assert 1 <= len(ents) <= cap
    vals = [e.search_value for e in ents]
    assert all(a <= b for a, b in zip(vals, vals[1:])), vals
    bins = []
    for e in ents:
        assert e.max_violation <= 1e-6, e
        assert O.objective(p, e.x) == pytest.approx(e.objective, rel=1e-9, abs=1e-12)
        rc, _, fixed = O.solve_fixed(p, e.x)
        assert rc == 0
        if e.converged:
            assert e.objective == pytest.approx(fixed, rel=1e-6, abs=1e-9), (e.objective, fixed)
        else:
            assert e.objective >= fixed - 1e-6 * abs(fixed) - 1e-9
        bins.append(binaries(p, e.x))
    for a in range(len(bins)):
        for b in range(a):
            assert not np.array_equal(bins[a], bins[b]), (a, b)


@pytest.mark.parametrize("world", [2, 3])
def test_merge_is_the_pool_of_the_union_of_the_ranks_leaves(plans, world):
    solvers, pools, exports = emulate(plans, world)
    gathered = torch.cat(exports)
    s = solvers[0]
    s.pool_merge(gathered, world)
    sizes = s.pool_sizes()
    for k, p in enumerate(plans):
        union = [e for r in range(world) for e in pools[r][k]]
        want = host_greedy(p, union, CAP)
        got = s.pool(k)
        assert [(e.search_value, e.uid) for e in got] == [(e.search_value, e.uid) for e in want], k
        assert sizes[k] == len(got) >= max(len(pools[r][k]) for r in range(world))
        by_uid = {e.uid: e for e in union}
        for e in got:
            assert np.array_equal(e.x, by_uid[e.uid].x) and np.array_equal(e.traj, by_uid[e.uid].traj)
            assert e.objective == by_uid[e.uid].objective and e.max_violation == by_uid[e.uid].max_violation
        check_entries(p, got, CAP)
    # the ranks searched different shares: their pools differ somewhere
    assert any(len({tuple(e.uid for e in pools[r][k]) for r in range(world)}) > 1 for k in range(len(plans)))

    # determinism: every rank's solver, and any rank order in the gathered buffer, give the same bytes
    want = fetch_all(s, len(plans))
    for r in range(1, world):
        solvers[r].pool_merge(gathered, world)
        assert fetch_all(solvers[r], len(plans)) == want
    perm = list(reversed(range(world)))
    solvers[-1].pool_merge(torch.cat([exports[r] for r in perm]), world)
    assert fetch_all(solvers[-1], len(plans)) == want
    for x in solvers:
        x.close()


def test_merge_with_itself_changes_nothing(plans):
    s = P.Solver(solution_pool=CAP)
    s.upload(plans, gap_tol=GAP, time_limit=120)
    s.run()
    before = fetch_all(s, len(plans))
    exp = s.pool_export().clone()
    s.pool_merge(exp, 1)
    assert fetch_all(s, len(plans)) == before
    s.pool_merge(torch.cat([exp, exp]), 2)
    assert fetch_all(s, len(plans)) == before
    s.pool_merge(torch.cat([exp, exp]).cpu(), 2)         # host input: copied to the device first
    assert fetch_all(s, len(plans)) == before
    s.pool_merge(s.pool_export(), 1)                     # the export buffer itself as input
    assert fetch_all(s, len(plans)) == before
    s.close()


def test_refusals_leave_the_pool_unchanged(plans):
    s = P.Solver(solution_pool=CAP)
    s.upload(plans, gap_tol=GAP, time_limit=120)
    with pytest.raises(P.MiqpB200Error):
        s.pool_merge(torch.zeros(64, dtype=torch.uint8), 1)          # before any run
    s.run()
    before = fetch_all(s, len(plans))
    own = s.pool_export().clone()

    other_cap = P.Solver(solution_pool=4)
    other_cap.upload(plans, gap_tol=GAP, time_limit=120)
    other_cap.run()
    other_shape = P.Solver(solution_pool=CAP)
    other_shape.upload(plans[:-1] + [obstacle_scenario(3, nr_steps=30).build()], gap_tol=GAP, time_limit=120)
    other_shape.run()
    for bad in (other_cap.pool_export().clone(), other_shape.pool_export().clone()):
        with pytest.raises(P.MiqpB200Error):
            s.pool_merge(bad, 1)
        with pytest.raises(P.MiqpB200Error):
            s.pool_merge(torch.cat([own, bad]), 2)                   # the second header is checked too
        assert fetch_all(s, len(plans)) == before
    with pytest.raises(P.MiqpB200Error):
        s.pool_merge(own, 0)
    assert fetch_all(s, len(plans)) == before

    off = P.Solver()
    off.upload(plans, gap_tol=GAP, time_limit=120)
    off.run()
    with pytest.raises(P.MiqpB200Error):
        off.pool_merge(own, 1)                                       # pool off at upload
    with pytest.raises(P.MiqpB200Error):
        off.pool_export()
    for x in (s, other_cap, other_shape, off):
        x.close()


# ---- two ranks: gloo on one GPU, NCCL on two -----------------------------------------------------------------------------------
def _worker(rank, world, port, backend, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle.dat_io import read_dat
    ps = plans_for_test(read_dat(os.path.join(ROOT, "tests", "golden", "cplexmodel_testcase.dat")))
    s = P.Solver(device=dev, solution_pool=CAP)
    kw = dict(gap_tol=GAP, time_limit=120, ramp_rounds=RAMP, exchange_every=3)
    st0, st1 = {}, {}
    xs0, infos0 = solve_frontier_sharded(s, ps, stats=st0, **kw)
    own_sizes = s.pool_sizes().tolist()
    xs1, infos1 = solve_frontier_sharded(s, ps, stats=st1, merge_pool=True, **kw)
    pools = fetch_all(s, len(ps))
    q.put((rank, [dataclasses.replace(i, seconds=0.0) for i in infos0], [dataclasses.replace(i, seconds=0.0) for i in infos1],
           [x.copy() for x in xs0], [x.copy() for x in xs1], own_sizes, s.pool_sizes().tolist(), pools, st0, st1))
    dist.barrier()
    dist.destroy_process_group()
    s.close()


def _run_two(backend):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 37500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, backend, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=900) for _ in procs), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, in0, in1, xs0, xs1, own, merged, pools, st0, st1 in res:
        assert st1["split"] and st1["pool_bytes"] > 0 and st1["pool_merge_ms"] >= 0.0 and "pool_bytes" not in st0
        assert in0 == in1                                       # the merge changes nothing else of the result
        assert all(np.array_equal(a, b) for a, b in zip(xs0, xs1))
        for k in range(len(in1)):
            assert merged[k] >= own[k]
            assert in1[k].status == 0
            e0 = pools[k][0]
            assert e0[4] == pytest.approx(in1[k].objective, rel=1e-9)
            if e0[4] == in1[k].objective:
                assert np.array_equal(np.frombuffer(e0[6]), xs1[k])
    assert res[0][7] == res[1][7]                               # bit-identical pools on both ranks
    assert res[0][6] == res[1][6]


def test_two_ranks_one_gpu_gloo():
    _run_two("gloo")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_two_gpus_nccl():
    _run_two("nccl")
