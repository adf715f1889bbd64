"""Host logic of the incumbent deliveries of frontier sharding (planner-miqp_b200/sharding.py:solve_frontier_sharded(on_incumbent=...))
with world size 2 on the gloo backend.  The stand-in solver of tests/test_frontier_gloo.py gets frontier_inc_export /
frontier_inc_merge / request_stop that log what they are given (records = the plans whose own incumbent improved since the last
export; merge = best (objective, rank) per plan, delivered when it improves), so what is checked here is the protocol: export
before the incumbent-objective exchange and once more before frontier_finish, blocks gathered in rank order with n_max from the
MAX all-reduce, the callback on the delivering rank only, a callback exception raised on its rank after both ranks completed
every collective, and an unchanged combined result.  The device export and merge are covered by tests/test_gpu_frontier_anytime.py."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_inc_toy(rank):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_frontier_gloo import make_toy
    from planner_miqp_b200.capi import Incumbent

    class IncToy(make_toy()):
        """summary = float64 [rank, n_records, stop[0..n)]; record = float64 [k, objective, rank]"""

        def __init__(self):
            self.log, self.merges = [], []

        def frontier_start(self):
            super().frontier_start()
            self.reported = np.full(self.n, np.inf)
            self.key = [None] * self.n
            self.stop_req = np.zeros(self.n)
            self.applied = set()

        def frontier_rounds(self, nrounds):
            self.log.append("rounds")
            for k in self.applied:
                self.open[k] = []
            return super().frontier_rounds(nrounds)

        def frontier_get_ub(self):
            self.log.append("get_ub")
            return super().frontier_get_ub()

        def frontier_finish(self):
            self.log.append("finish")
            return super().frontier_finish()

        def request_stop(self, k=-1):
            if k < 0:
                self.stop_req[:] = 1
            else:
                self.stop_req[k] = 1

        def frontier_inc_export(self):
            self.log.append("export")
            recs = [[k, self.own[k], rank] for k in range(self.n) if self.own[k] < self.reported[k]]
            for k, _, _ in recs:
                self.reported[k] = self.own[k]
            summary = np.concatenate([[rank, len(recs)], self.stop_req]).astype(np.float64)
            data = np.concatenate([summary, np.array(recs, dtype=np.float64).reshape(-1), np.zeros(3 * self.n)])
            buf = torch.from_numpy(data).view(torch.uint8)
            return buf, 8 * len(summary), 24, len(recs)

        def frontier_inc_merge(self, gathered, world, n_max, on_incumbent=None):
            self.log.append("merge")
            d = gathered.view(torch.float64).numpy()
            hdr = 2 + self.n
            blk = hdr + 3 * n_max
            assert d.size == world * blk
            assert n_max == max(int(d[r * blk + 1]) for r in range(world))   # the MAX all-reduce of the record counts
            self.merges.append((world, n_max, [float(d[r * blk]) for r in range(world)]))
            best = {}
            for r in range(world):
                b = d[r * blk:(r + 1) * blk]
                self.applied |= {k for k in range(self.n) if b[2 + k]}
                assert b[1] <= n_max
                for j in range(int(b[1])):
                    k, obj, rr = b[hdr + 3 * j: hdr + 3 * j + 3]
                    if int(k) not in best or (obj, rr) < best[int(k)]:
                        best[int(k)] = (obj, rr)
            got = 0
            for k in sorted(best):
                if self.key[k] is None or best[k] < self.key[k]:
                    self.key[k] = best[k]
                    got += 1
                    if on_incumbent is not None:
                        obj, rr = best[k]
                        inc = Incumbent(obj, 0.0, obj, obj, 0.0, 0.0, 0, 0, 0, 0, int(rr))
                        if on_incumbent(k, np.zeros((1, 1, 8)), inc):
                            self.request_stop(k)
            return got

    return IncToy()


class _Plan:
    scal = {"relative_mip_gap_tolerance": 1e-9}


def _worker(rank, world, port, q, mode):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from planner_miqp_b200.sharding import solve_frontier_sharded
    out = {"rank": rank}
    plans = [_Plan() for _ in range(3)]
    plain = make_inc_toy(rank)
    xs0, infos0 = solve_frontier_sharded(plain, plans, ramp_rounds=4, exchange_every=3)
    out["plain_log"] = list(plain.log)
    toy, st, got = make_inc_toy(rank), {}, []

    def cb(k, traj, inc):
        got.append((k, inc.objective, inc.rank))
        if mode == "raise" and rank == 1:
            raise ValueError("bad incumbent")
        return False

    kw = dict(deliver_rank=None) if mode in ("all", "raise") else {}
    try:
        xs1, infos1 = solve_frontier_sharded(toy, plans, ramp_rounds=4, exchange_every=3, stats=st, on_incumbent=cb, **kw)
        out["same_result"] = [x.tolist() for x in xs0] == [x.tolist() for x in xs1] and infos0 == infos1
        out["want"] = [i.objective for i in infos1]
    except ValueError as ex:
        out["error"] = str(ex)
    out.update(log=toy.log, merges=toy.merges, got=got, stats={k: v for k, v in st.items() if k.startswith("inc_") or k == "delivered"},
               stop_req=toy.stop_req.tolist())
    q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def _run(mode, base):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = base + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q, mode)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=240) for _ in procs), key=lambda r: r["rank"])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return res


def exchanges_of(log):
    """the calls between consecutive frontier_rounds (the ramp-up's and the loop's)"""
    out, cur = [], None
    for e in log:
        if e == "rounds":
            cur = []
            out.append(cur)
        elif cur is not None:
            cur.append(e)
    return out


def test_protocol_order_gather_and_delivering_rank():
    res = _run("rank0", 41500)
    for r in res:
        assert "export" not in r["plain_log"] and "merge" not in r["plain_log"]     # on_incumbent=None: nothing new
        assert r["same_result"]
        log = r["log"]
        assert log[-3:] == ["export", "merge", "finish"]                              # the final merge before finish
        loop = exchanges_of(log)[1:]                                                  # (the ramp-up is followed by the split)
        assert loop and all(x[:3] == ["export", "merge", "get_ub"] for x in loop), loop
        assert r["stats"]["inc_exchanges"] == log.count("export") and r["stats"]["inc_gather_bytes"] > 0 and r["stats"]["inc_ms"] >= 0
        for world, n_max, first in r["merges"]:
            assert world == 2 and first == [0.0, 1.0]                                 # blocks in rank order
    assert res[0]["merges"] == res[1]["merges"]                                       # the same n_max on both ranks
    # n_max is the larger record count of the two exports of that exchange: the toy counts its own improvements per export
    assert any(n_max > 0 for _, n_max, _ in res[0]["merges"])
    assert res[1]["got"] == [] and res[0]["got"]                                      # the callback on deliver_rank only
    assert res[0]["stats"]["delivered"] == res[1]["stats"]["delivered"] == len(res[0]["got"])
    last = {}
    for k, obj, rank in res[0]["got"]:
        assert k not in last or obj < last[k][0] or (obj == last[k][0] and rank < last[k][1])
        last[k] = (obj, rank)
    assert [last[k][0] for k in range(3)] == res[0]["want"]                           # the last delivery is the combined result


def test_every_rank_delivers_the_same():
    res = _run("all", 43500)
    assert res[0]["got"] and res[0]["got"] == res[1]["got"]


def test_callback_exception_is_raised_on_its_rank_after_the_protocol():
    res = _run("raise", 45500)
    assert "error" not in res[0] and res[1]["error"] == "bad incumbent"
    assert res[1]["got"] == res[0]["got"][:1]                                        # no calls after the exception
    assert res[0]["log"].count("export") == res[1]["log"].count("export")           # every collective on both ranks
    assert res[1]["log"][-1] == "finish" and res[1]["stop_req"] == [1.0, 1.0, 1.0]  # stops every plan on every rank


def test_single_process_exchanges_in_steps():
    sys.path.insert(0, ROOT)
    from planner_miqp_b200.sharding import solve_frontier_sharded
    toy, st, got = make_inc_toy(0), {}, []
    xs, infos = solve_frontier_sharded(toy, [_Plan()], stats=st, exchange_every=5,
                                       on_incumbent=lambda k, t, inc: got.append((k, inc.objective)))
    assert toy.log[-3:] == ["export", "merge", "finish"] and toy.log.count("rounds") > 1
    assert all(x[:2] == ["export", "merge"] for x in exchanges_of(toy.log))
    assert got and got[-1] == (0, infos[0].objective) and st["delivered"] == len(got)
