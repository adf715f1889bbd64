"""Incumbent deliveries and stops of a frontier-sharded search (miqp_b200_frontier_inc_export / _merge,
solve_frontier_sharded(on_incumbent=...)).  Two ranks are gloo processes that share cuda:0, as in tests/test_gpu_frontier.py;
the NCCL case needs two GPUs.

* the search is unchanged by deliveries that do not stop (world 1 and 2, bit for bit);
* at world 1 the deliveries are a subsequence of Solver.run_anytime's records of the same batch, with the same last one;
* at world 2 the deliveries fall strictly per plan, are feasible, and the last one is the combined result, the same on every
  rank with deliver_rank=None;
* a stop (callback return or request_stop on the non-delivering rank) ends the plan on both ranks at the same round; a frontier
  search without deliveries ignores stops, and no stop leaks into a later batch run;
* the merge refuses foreign headers, a wrong n_max and a call before frontier_start, and changes nothing then."""
import os
import sys
import threading
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import planner_miqp_b200 as P
from planner_miqp_b200.scenarios import intersection
from planner_miqp_b200.sharding import solve_frontier_sharded
from test_gpu_frontier import plans_for_test

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GAP = 1e-4
TRAJ_BLOCKS = [2, 3, 4, 5, 6, 7, 0, 1]   # [C][N][8] = (pos_x, vel_x, acc_x, pos_y, vel_y, acc_y, u_x, u_y): column blocks of x


def hard_plans():
    """a single-car plan and a four-car intersection that does not prove its gap within the limit"""
    return [plans_for_test()[0], intersection(3, n_cars=4, nr_steps=20, nr_regions=32).build()]


def traj_of(x, c, n):
    return np.stack([x[b * c * n:(b + 1) * c * n].reshape(c, n) for b in TRAJ_BLOCKS], axis=-1)


def stop_when_uploaded(s, k):
    """request_stop(k) as soon as the solver holds a batch (a thread's call before the upload is refused)"""
    while True:
        try:
            s.request_stop(k)
            return
        except P.MiqpB200Error:
            time.sleep(0.01)


def collect(out):
    def cb(k, t, inc):
        out.append((k, t, inc))
        return False
    return cb


def same_search(a, b):
    (xa, ia), (xb, ib) = a, b
    for x0, x1, i0, i1 in zip(xa, xb, ia, ib):
        assert np.array_equal(x0, x1)
        assert np.float64(i0.objective).tobytes() == np.float64(i1.objective).tobytes() and i0.nodes == i1.nodes
        assert i0.status == i1.status


def test_world1_search_unchanged_and_deliveries_are_a_subsequence_of_run_anytime():
    ps = plans_for_test()
    s = P.Solver()
    plain = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=120, exchange_every=3)
    got, st = [], {}
    res = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=120, exchange_every=3, on_incumbent=collect(got), stats=st)
    same_search(plain, res)
    assert st["inc_exchanges"] > 1 and st["delivered"] == len(got) and st["inc_gather_bytes"] > 0
    s.upload(ps, gap_tol=GAP, time_limit=120)
    recs = {}
    s.run_anytime(lambda k, t, inc: recs.setdefault(k, []).append((t, inc)) and False)
    for k in range(len(ps)):
        mine = [(t, i) for kk, t, i in got if kk == k]
        assert mine, k
        full = recs[k]
        j = 0
        for t, i in mine:                     # a subsequence: same uid, objective and trajectory bits
            while j < len(full) and full[j][1].uid != i.uid:
                j += 1
            assert j < len(full), (k, i)
            ft, fi = full[j]
            assert np.array_equal(ft, t) and np.float64(fi.objective).tobytes() == np.float64(i.objective).tobytes()
            assert fi.search_value == i.search_value and i.rank == 0
        assert mine[-1][1].uid == full[-1][1].uid
        assert np.float64(res[1][k].objective).tobytes() == np.float64(mine[-1][1].objective).tobytes()
    s.close()


def test_stops_and_no_leak_world1():
    ps = hard_plans()
    s = P.Solver()
    # a frontier search without deliveries ignores stop requests
    t = threading.Timer(1.0, stop_when_uploaded, args=(s, -1))
    t.start()
    solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=3)
    t.join()
    assert list(s.stopped()) == [-1, -1]
    # deliveries that stop every plan at once: the stops end the plans, and the requests do not outlive the run
    got = []
    _, infos = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=20, exchange_every=2,
                                      on_incumbent=lambda k, tr, inc: got.append(k) or True)
    stopped = s.stopped()
    assert stopped[1] >= 0 and infos[1].status == 0 and infos[1].seconds < 20
    a = s.solve_batch(plans_for_test(), gap_tol=GAP, time_limit=120)
    f = P.Solver()
    b = f.solve_batch(plans_for_test(), gap_tol=GAP, time_limit=120)
    same_search(a, b)
    s.close(), f.close()


def test_merge_refusals_leave_the_state_unchanged():
    ps = plans_for_test()
    s, other = P.Solver(), P.Solver()
    s.upload(ps, gap_tol=GAP, time_limit=120)
    with pytest.raises(P.MiqpB200Error):
        s.frontier_inc_export()
    other.upload(ps[:2], gap_tol=GAP, time_limit=120)
    other.frontier_start()
    other.frontier_rounds(4)
    obuf, osb, orb, on = other.frontier_inc_export()
    foreign = obuf[:osb + on * orb].clone()
    with pytest.raises(P.MiqpB200Error):            # before frontier_start
        s.frontier_inc_merge(foreign, 1, on)
    s.frontier_start()
    s.frontier_rounds(6)
    buf, sb, rb, n = s.frontier_inc_export()
    assert n >= 1
    block = buf[:sb + n * rb].clone()
    with pytest.raises(P.MiqpB200Error):            # another batch
        s.frontier_inc_merge(foreign, 1, on)
    with pytest.raises(P.MiqpB200Error):            # fewer than the block holds
        s.frontier_inc_merge(buf[:sb + (n - 1) * rb].clone(), 1, n - 1)
    with pytest.raises(P.MiqpB200Error):            # more than a block can hold
        s.frontier_inc_merge(torch.cat([block] * 2), 1, len(ps) + 1)
    with pytest.raises(P.MiqpB200Error):            # n_max too small: the second block's header is not where it says
        s.frontier_inc_merge(torch.cat([block] * 2), 2, n - 1)
    got = []
    assert s.frontier_inc_merge(block, 1, n, collect(got)) == n      # nothing was delivered by the refused calls
    assert [k for k, _, _ in got] == sorted(k for k, _, _ in got) and len(got) == n
    assert s.frontier_inc_merge(block.cpu(), 1, n, collect(got)) == 0    # the same records again (from the host): no improvement
    s.frontier_rounds(-1)
    s.frontier_finish()
    with pytest.raises(P.MiqpB200Error):            # after frontier_finish
        s.frontier_inc_export()
    s.close(), other.close()


def _worker(rank, world, port, backend, q, mode):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = rank if backend == "nccl" else 0
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", dev))
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    out = {"rank": rank}
    s = P.Solver(device=dev)
    got = []
    if mode == "deliver":
        ps = plans_for_test()
        plain = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=120, ramp_rounds=5, exchange_every=3)
        res = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=120, ramp_rounds=5, exchange_every=3,
                                     on_incumbent=collect(got), deliver_rank=None)
        same_search(plain, res)
    else:
        ps = hard_plans()
        timer = None
        if mode == "stop_cb":
            cb = lambda k, t, inc: got.append((k, t, inc)) or k == 1      # noqa: E731
        else:                                 # request_stop on rank 1, which does not deliver
            cb = collect(got)
            if rank == 1:
                timer = threading.Timer(1.5, stop_when_uploaded, args=(s, 1))
                timer.start()
        res = solve_frontier_sharded(s, ps, gap_tol=GAP, time_limit=20, ramp_rounds=5, exchange_every=3, on_incumbent=cb)
        if timer is not None:
            timer.join()
        out["stopped"] = s.stopped().tolist()
    xs, infos = res
    out.update(got=[(k, t, inc) for k, t, inc in got], xs=[x.copy() for x in xs], infos=infos,
               shapes=[(p.C, p.N) for p in ps])
    q.put(out)
    dist.barrier()
    dist.destroy_process_group()
    s.close()


def _run_two(backend, mode, base):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = base + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, backend, q, mode)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=900) for _ in procs), key=lambda r: r["rank"])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return res


def check_deliveries(r):
    last = {}
    for k, t, inc in r["got"]:
        assert inc.max_violation <= 1e-6 and inc.best_bound <= inc.objective and inc.rank in (0, 1), (k, inc)
        assert k not in last or inc.objective < last[k][1].objective, (k, inc)
        last[k] = (t, inc)
    for k, info in enumerate(r["infos"]):
        if info.status != 0:
            continue
        t, inc = last[k]
        assert inc.objective == info.objective and inc.max_violation == info.max_violation
        c, n = r["shapes"][k]
        assert np.array_equal(t, traj_of(r["xs"][k], c, n))
    return last


@pytest.mark.parametrize("backend", ["gloo", pytest.param("nccl", marks=pytest.mark.skipif(
    torch.cuda.device_count() < 2, reason="needs two GPUs"))])
def test_two_ranks_deliver_the_combined_result(backend):
    res = _run_two(backend, "deliver", 47500 if backend == "gloo" else 49500)
    for r in res:
        check_deliveries(r)
    key = lambda r: [(k, inc.uid, inc.objective, inc.rank, t.tobytes()) for k, t, inc in r["got"]]   # noqa: E731
    assert key(res[0]) and key(res[0]) == key(res[1])


@pytest.mark.parametrize("mode", ["stop_cb", "stop_request"])
def test_stop_reaches_both_ranks_at_the_same_round(mode):
    res = _run_two("gloo", mode, 51500 if mode == "stop_cb" else 53500)
    assert res[0]["stopped"] == res[1]["stopped"]
    assert res[0]["stopped"][1] >= 0, res[0]["stopped"]
    info = res[0]["infos"][1]
    assert info.seconds < 20
    if mode == "stop_cb" or info.status == 0:
        assert info.status == 0
        last = check_deliveries(res[0])
        assert last[1][1].objective == info.objective
