"""Host logic of the pool merge of frontier sharding (planner-miqp_b200/sharding.py:solve_frontier_sharded(merge_pool=True))
with world size 2 on the gloo backend.  The stand-in solver of tests/test_frontier_gloo.py gets a pool_export / pool_merge that
record what they are given, so what is checked here is the protocol: export and merge exactly once on every rank, only with
merge_pool=True and more than one rank, exports gathered in rank order, a refusal on every rank when a pool is off, and no
change to the combined result.  The device merge behind the same calls is covered by tests/test_gpu_frontier_pool.py."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXPORT_BYTES = 48


def make_pool_toy(rank, pool_on=True):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_frontier_gloo import make_toy
    from planner_miqp_b200.capi import MiqpB200Error

    class PoolToy(make_toy()):
        def __init__(self):
            self.exports, self.merges = 0, []

        def pool_export(self):
            if not pool_on:
                raise MiqpB200Error("pool off")
            self.exports += 1
            return torch.arange(EXPORT_BYTES, dtype=torch.uint8) + 100 * rank   # first byte names the rank

        def pool_merge(self, gathered, world):
            self.merges.append((world, gathered.numel(), gathered[::EXPORT_BYTES].tolist()))

    return PoolToy()


class _Plan:
    scal = {"relative_mip_gap_tolerance": 1e-9}


def _worker(rank, world, port, q, pool_on):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from planner_miqp_b200.capi import MiqpB200Error
    from planner_miqp_b200.sharding import solve_frontier_sharded
    out = {"rank": rank}
    plans = [_Plan() for _ in range(3)]
    plain = make_pool_toy(rank, pool_on)
    xs0, infos0 = solve_frontier_sharded(plain, plans, ramp_rounds=4, exchange_every=3)
    out["plain"] = (plain.exports, plain.merges)
    toy, st = make_pool_toy(rank, pool_on), {}
    try:
        xs1, infos1 = solve_frontier_sharded(toy, plans, ramp_rounds=4, exchange_every=3, stats=st, merge_pool=True)
        out["same_result"] = [x.tolist() for x in xs0] == [x.tolist() for x in xs1] and infos0 == infos1
    except MiqpB200Error as ex:
        out["error"] = str(ex)
    out["merge"] = (toy.exports, toy.merges, st.get("pool_bytes"), "pool_merge_ms" in st)
    q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def _run(pool_on):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 39500 + (os.getpid() % 2000) + (0 if pool_on else 17)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, pool_on)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=240) for _ in procs), key=lambda r: r["rank"])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def test_pools_are_gathered_in_rank_order_and_merged_once_on_every_rank():
    for r in _run(True):
        assert r["plain"] == (0, [])                                   # merge_pool=False: no export, no merge
        exports, merges, nbytes, timed = r["merge"]
        assert exports == 1 and nbytes == EXPORT_BYTES and timed
        assert merges == [(2, 2 * EXPORT_BYTES, [0, 100])]             # once, both exports, rank 0 first
        assert r["same_result"]


def test_pool_off_is_refused_on_every_rank():
    for r in _run(False):
        assert "error" in r and r["merge"][1] == []


def test_single_process_does_not_merge():
    sys.path.insert(0, ROOT)
    from planner_miqp_b200.sharding import solve_frontier_sharded
    toy, st = make_pool_toy(0), {}
    solve_frontier_sharded(toy, [_Plan()], stats=st, merge_pool=True)
    assert toy.exports == 0 and toy.merges == [] and "pool_bytes" not in st
