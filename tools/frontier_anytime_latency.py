"""Cost and benefit of incumbent deliveries on the frontier-sharded path (solve_frontier_sharded(on_incumbent=...)).

Workload: config 5 of bench.py, ONE joint plan of an 8-car intersection (scenarios.intersection(k, n_cars=8, nr_steps=40),
N = 40, R = 64), 5 s time limit, default ramp_rounds / exchange_every.  Seeds 0 .. --seeds-1; for every seed one plain search
(no on_incumbent) and one with deliveries (a no-op callback, no stops), alternating, so that both see the same machine state.
Reported per mode: node relaxations per second (all ranks' nodes over the wall time of the call), the time from the start of the
call to the first delivered incumbent against the time the combined result is available (the call's return), and per exchange
the host time of export, gather and merge and the bytes gathered.

One GPU: world 1 in this process.  With two or more GPUs the same over NCCL, one process per GPU (--world, default all GPUs).
The card's name and power limit are read in the same run.

    python tools/frontier_anytime_latency.py --out profiles/r3_frontier_anytime.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GAP = 1e-4


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return [dict(zip(("name", "power_limit", "sm_max_clock"), [v.strip() for v in line.split(",")])) for line in out]
    except Exception as ex:  # reported, not hidden
        return {"error": repr(ex)}


class Timed:
    """the solver with its export and merge calls timed (host clock; both end in a stream synchronise)"""

    def __init__(self, solver):
        self.solver, self.t_export, self.t_merge = solver, [], []

    def __getattr__(self, name):
        return getattr(self.solver, name)

    def frontier_inc_export(self):
        t0 = time.perf_counter()
        out = self.solver.frontier_inc_export()
        self.t_export.append(1e3 * (time.perf_counter() - t0))
        return out

    def frontier_inc_merge(self, *a, **kw):
        t0 = time.perf_counter()
        out = self.solver.frontier_inc_merge(*a, **kw)
        self.t_merge.append(1e3 * (time.perf_counter() - t0))
        return out


def one_search(solver, plan, args, deliver, group_world):
    import torch
    import torch.distributed as dist
    from planner_miqp_b200.sharding import solve_frontier_sharded
    timed = Timed(solver)
    first = []
    t0 = None

    def on_inc(k, traj, inc):
        if not first:
            first.append((time.perf_counter() - t0, inc.seconds, inc.objective))
        return False

    st = {}
    torch.cuda.synchronize()
    if group_world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    xs, infos = solve_frontier_sharded(timed, [plan], gap_tol=GAP, time_limit=args.time_limit, stats=st,
                                       on_incumbent=on_inc if deliver else None)
    wall = time.perf_counter() - t0
    i = infos[0]
    rec = {"wall_s": wall, "nodes_all_ranks": int(i.nodes), "nodes_per_s": i.nodes / wall, "objective": i.objective,
           "gap": i.gap, "status": i.status, "exchanges": st["exchanges"]}
    if deliver:
        n = max(st["inc_exchanges"], 1)
        export_ms, merge_ms = float(np.sum(timed.t_export)), float(np.sum(timed.t_merge))
        rec.update(first_delivery_s=first[0][0] if first else None, first_delivery_solver_clock_s=first[0][1] if first else None,
                   first_objective=first[0][2] if first else None, delivered=st["delivered"], inc_exchanges=st["inc_exchanges"],
                   export_ms_per_exchange=export_ms / n, merge_ms_per_exchange=merge_ms / n,
                   gather_ms_per_exchange=(st["inc_ms"] - export_ms - merge_ms) / n, bytes_per_exchange=st["inc_gather_bytes"] / n,
                   inc_ms_total=st["inc_ms"])
    return rec


def run(args, rank=0, world=1):
    import torch
    import planner_miqp_b200 as P
    from planner_miqp_b200.scenarios import intersection
    solver = P.Solver(device=rank)
    plans = [intersection(k, n_cars=8, nr_steps=40).build() for k in range(args.seeds)]
    one_search(solver, plans[0], argparse.Namespace(time_limit=1.0), True, world)    # warm-up of every path
    rows = []
    for k, p in enumerate(plans):
        for deliver in ((False, True) if k % 2 == 0 else (True, False)):
            r = one_search(solver, p, args, deliver, world)
            r.update(seed=k, mode="on_incumbent" if deliver else "plain")
            rows.append(r)
    solver.close()
    torch.cuda.synchronize()
    return rows


def summarize(rows):
    out = {}
    for mode in ("plain", "on_incumbent"):
        m = [r for r in rows if r["mode"] == mode]
        s = {"nodes_per_s_mean": float(np.mean([r["nodes_per_s"] for r in m])), "nodes_per_s": [r["nodes_per_s"] for r in m],
             "wall_s": [r["wall_s"] for r in m]}
        if mode == "on_incumbent":
            for f in ("first_delivery_s", "export_ms_per_exchange", "gather_ms_per_exchange", "merge_ms_per_exchange",
                      "bytes_per_exchange", "inc_exchanges", "delivered"):
                s[f] = [r[f] for r in m]
        out[mode] = s
    return out


def _worker(rank, world, port, args, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    rows = run(args, rank, world)
    if rank == 0:
        q.put(rows)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seeds", type=int, default=4)
    ap.add_argument("--time-limit", type=float, default=5.0)
    ap.add_argument("--world", type=int, default=0, help="GPUs of the NCCL run (0: all; skipped with fewer than 2)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing measured")
    res = {"gpus": gpu_info(), "workload": "config 5: 8-car intersection, N = 40, R = 64, one joint plan, gap 1e-4",
           "time_limit_s": args.time_limit, "seeds": args.seeds, "runs": {}}
    rows = run(args)
    res["runs"]["1gpu"] = {"summary": summarize(rows), "rows": rows}
    print(json.dumps(res["runs"]["1gpu"]["summary"], indent=1), flush=True)
    world = args.world or torch.cuda.device_count()
    if world >= 2 and torch.cuda.device_count() >= world:
        ctx = mp.get_context("spawn")
        q = ctx.Queue()
        procs = [ctx.Process(target=_worker, args=(r, world, 29500 + os.getpid() % 1000, args, q)) for r in range(world)]
        for p in procs:
            p.start()
        rows = q.get(timeout=3600)
        for p in procs:
            p.join()
        res["runs"][f"{world}gpu_nccl"] = {"summary": summarize(rows), "rows": rows}
        print(json.dumps(res["runs"][f"{world}gpu_nccl"]["summary"], indent=1), flush=True)
    else:
        res["runs"]["multi_gpu"] = f"not measured: {torch.cuda.device_count()} GPU(s) on this machine"
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
