#!/usr/bin/env python
"""bench.py -- MIQP plans/s at 1e-4 relative gap on N B200s (BASELINE.json metric).

Workload (config[1] of BASELINE.json): batch of single-agent plans with one static and one
dynamic-occupancy obstacle, N=40 steps, 32 fitted regions, reference default settings
(planner-miqp_b200/scenarios.py:obstacle_scenario, seeds rank*B .. rank*B+B-1).

One step = one pass of the hot path over one batch: every plan is solved to a proven
relative gap <= 1e-4 by the device branch and bound.  The scenario seeds rotate from step to
step (--shards distinct batches per rank); per-shard step times are reported.
  value : plans/s, whole job, batch already resident in HBM when the timed region starts
          (miqp_b200_batch_run; CUDA events on the solver stream, max over ranks)
  e2e   : plans/s through the C ABI with host buffers (miqp_b200_solve_batch: pack + H2D +
          solve + D2H of every solution vector inside the timed region)
Rank layout: one process per GPU, scenario sharding, no data-path collective ("weak").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (solution vectors and per-plan solve results of rank 0) as
.npy files, so that two builds can be compared output for output on identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if int(os.environ.get("WORLD_SIZE", "1")) > 1:
    # communicator lines ("... nranks N ... Init COMPLETE") go to stderr (fd 1 is redirected there, see emit()); NCCL reads the
    # variable once, at the first library call, which torch makes on import: set it before
    # (forced: the GPU boxes preset NCCL_DEBUG=VERSION, which prints the version line only)
    if not os.environ.get("MIQP_BENCH_KEEP_NCCL_DEBUG"):
        os.environ["NCCL_DEBUG"] = "INFO"
        os.environ["NCCL_DEBUG_SUBSYS"] = "INIT"

import numpy as np  # noqa: E402

# Everything libraries print to fd 1 (NCCL prints its version there at the first collective) goes to stderr;
# the one JSON line is written to the real stdout.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line: dict):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


GAP = 1e-4
WORKLOAD = "single agent, static + dynamic-occupancy obstacle, N=40, R=32 (BASELINE.json configs[1])"


def make_plans(first_seed: int, count: int):
    import planner_miqp_b200  # noqa: F401
    from planner_miqp_b200.scenarios import obstacle_scenario
    return [obstacle_scenario(first_seed + k).build() for k in range(count)]


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def algorithmic_flops(stats: dict, N: int) -> float:
    """Algorithmic FP64 flops of the node kernel (DESIGN.md section 5): per interior-point
    iteration 1000 flops per stage for the Riccati factorisation and sweeps, 60 flops per
    active inequality row for residuals, Hessian update, two gradients and two step lengths."""
    return 1000.0 * N * stats["qp_iters"] + 60.0 * stats["rows_visited"]


DUMP_BYTES = 64_000_000
DUMP_FIELDS = ("status", "proven", "objective", "best_bound", "gap", "max_violation")


def dump_outputs(out_dir: str, solver, seeds):
    """Writes the results the solver holds (its last batch run) as float64 .npy files: x.npy [plans, columns] (the solution
    vectors), plan_seed.npy (scenario seed of every row) and one array per solve-result field.  Search statistics (nodes,
    iterations, seconds) are left out: they say how the search went, not what it computed.  When the whole batch exceeds
    DUMP_BYTES, a fixed seeded sample of its plans is written."""
    xs, infos = solver.fetch()
    ncols = max(len(x) for x in xs)
    per_plan = 8 * (ncols + 1 + len(DUMP_FIELDS))
    keep = min(len(xs), (DUMP_BYTES - (1 << 16)) // per_plan)        # (1 << 16): room for the .npy headers
    idx = np.arange(len(xs))
    if keep < len(xs):
        idx = np.sort(np.random.default_rng(0).choice(len(xs), keep, replace=False))
    x = np.full((keep, ncols), np.nan)
    for row, k in enumerate(idx):
        x[row, :len(xs[k])] = xs[k]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), x)
    np.save(os.path.join(out_dir, "plan_seed.npy"), np.asarray(seeds, dtype=np.float64)[idx])
    for f in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f + ".npy"), np.array([float(getattr(infos[k], f)) for k in idx]))


def cpu_oracle_rate(plans, threads: int):
    """plans/s of the CPU oracle (oracle/, the checker) on `plans` with `threads` host threads."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as O
    O.lib()
    t0 = time.perf_counter()
    if threads <= 1:
        infos = [O.solve(p, gap_tol=GAP, time_limit=60.0)[1] for p in plans]
    else:
        with ThreadPoolExecutor(max_workers=threads) as ex:   # ctypes releases the GIL
            infos = [r[1] for r in ex.map(lambda p: O.solve(p, gap_tol=GAP, time_limit=60.0), plans)]
    dt = time.perf_counter() - t0
    ok = sum(1 for i in infos if i.status == 0)
    return len(plans) / dt, dt, ok


def bench_config(B: int) -> dict:
    """The `config` object, identical in both arms (the reference arm times bounded samples of the same workload); what is
    specific to a run (batches in flight, timing, cache handling of the leg that produced `value`) is in `run`."""
    return {"workload": WORKLOAD, "plans_per_gpu_per_step": B, "gap": GAP,
            "seeds": "shard s = scenario seeds s*B .. s*B+B-1 of scenarios.obstacle_scenario; rank r works on shards r, r + n_gpus, ...",
            "cache": "L2 flushed between steps (256 MiB write) when one batch runs at a time; batches in flight alternate over "
                     "different resident batches whose combined footprint exceeds the 126 MB L2 (see `run`)"}


def run_reference(args):
    """Reference arm: the CPU implementation of the path (the oracle port; CPLEX 12.10 is
    proprietary and absent, BASELINE.md section 4) on all host cores, same workload/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    sample = min(args.batch, max(4 * cores, 32))
    plans = make_plans(0, sample)
    for _ in range(args.warmup):
        cpu_oracle_rate(plans[:cores], cores)
    rates, times = [], []
    for _ in range(args.steps):
        r, dt, ok = cpu_oracle_rate(plans, cores)
        rates.append(r); times.append(dt)
    value = sample * args.steps / sum(times)
    line = {
        "impl": "reference", "metric": "MIQP plans/sec at 1e-4 gap", "value": value, "unit": "plans/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": bench_config(args.batch),
        "cpu_baseline": {"value": value, "unit": "plans/s", "cores": cores, "kind": "port",
                         "sample": f"every step solves the first {sample} plans of shard 0 of the workload (a bounded sample of the "
                                   f"{args.batch}-plan batch), one oracle solve per host thread; ms_per_step is the time of the sample"},
        "e2e": {"value": value, "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def replan_leg(solver, scenarios: int, cycles: int, device_shift: bool = True):
    """Config 2 as BASELINE.json names it: warm-started replanning.  `scenarios` config-2 scenarios are planned, then
    re-planned `cycles - 1` times in a receding horizon (state <- step 1 of the plan, obstacle predictions advance by one
    step, MIP start = previous solution shifted by one step: reference src/miqp_planner.cpp:787-1051,
    src/cplex_wrapper.cpp:494-639).  Timed: the C-ABI call on host buffers (pack + H2D + solve + D2H) of every cycle."""
    from planner_miqp_b200.scenarios import obstacle_scenario, advance_obstacle_scenario
    from planner_miqp_b200.results import shift_warmstart
    builders = [obstacle_scenario(k) for k in range(scenarios)]
    plans = [b.build() for b in builders]
    warm = None
    t_cold = t_warm = 0.0
    nodes_cold = nodes_warm = 0
    proven = 0
    for c in range(cycles):
        prep = solver.prepare(plans, gap_tol=GAP, time_limit=600.0, warm=None if device_shift else warm)
        t0 = time.perf_counter()
        if device_shift and c > 0:     # MIP starts = previous incumbents shifted on the device (miqp_b200_batch_upload_replan)
            solver.upload_replan_prepared(prep)
            solver.run()
            xs, infos = solver.fetch()
        else:
            xs, infos = solver.solve_prepared(prep)
        dt = time.perf_counter() - t0
        st = solver.run_stats()
        proven += sum(1 for i in infos if i.status == 0 and i.proven)
        if c == 0:
            t_cold, nodes_cold = dt, st["nodes"]
        else:
            t_warm += dt; nodes_warm += st["nodes"]
        if c + 1 < cycles:
            warm = [shift_warmstart(p, x) if i.status == 0 else None for p, x, i in zip(plans, xs, infos)]
            builders = [advance_obstacle_scenario(b, p, x) if i.status == 0 else b for b, p, x, i in zip(builders, plans, xs, infos)]
            plans = [b.build() for b in builders]
    return {"scenarios": scenarios, "cycles": cycles,
            "cold_plans_per_s": scenarios / t_cold, "warm_plans_per_s": scenarios * (cycles - 1) / t_warm if cycles > 1 else None,
            "all_cycles_plans_per_s": scenarios * cycles / (t_cold + t_warm),
            "nodes_per_plan_cold": nodes_cold / scenarios, "nodes_per_plan_warm": nodes_warm / (scenarios * max(cycles - 1, 1)),
            "proven_optimal": proven, "plans": scenarios * cycles,
            "warm_start": "previous incumbents shifted by one step on the device (miqp_b200_batch_upload_replan)" if device_shift
                          else "previous solution vectors shifted on the host (results.shift_warmstart), sent as MIP starts",
            "timed": "the C-ABI calls on host buffers per cycle (pack + H2D + solve + D2H); the scenario update (new states, "
                     "obstacle predictions one step ahead) runs on the host between the cycles, untimed"}


WORKLOADS = {
    "config3": "two-agent cooperative merge, joint MIQP with agent_collision_constraints, N=20, R=16 (BASELINE.json configs[2])",
    "config4": "randomised 1-4 agent scenarios, N=20, R=16, throughput mode (BASELINE.json configs[3])",
    "config5": "8-agent intersection, joint MIQP, N=40, R=64, B&B frontier sharded over the GPUs (BASELINE.json configs[4])",
}


def gap_histogram(infos, gap_tol):
    edges = [gap_tol, 1e-3, 1e-2, 1e-1, 1.0]
    names = [f"<={gap_tol:g}", "<=1e-3", "<=1e-2", "<=1e-1", "<=1", ">1"]
    h = {n: 0 for n in names}
    h["no incumbent"] = 0
    for i in infos:
        if i.status != 0 or not (i.gap == i.gap):
            h["no incumbent"] += 1
            continue
        for e, n in zip(edges, names):
            if i.gap <= e + 1e-15:
                h[n] += 1
                break
        else:
            h[names[-1]] += 1
    return h


def init_dist():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MIQP backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    return rank, local_rank, world


def run_multi_agent_batch(args):
    """configs 3 and 4: batches of joint multi-agent plans (scenario sharding, no data-path collective).  Multi-agent plans
    with active collision rows are not proven to 1e-4 within the time limit (DESIGN.md section 6): the line reports how many
    were, and the gap histogram of the rest."""
    import torch
    import torch.distributed as dist
    rank, local_rank, world = init_dist()
    import planner_miqp_b200 as P
    from planner_miqp_b200.scenarios import two_agent_merge, random_scenario
    B = args.batch if args.batch_given else (256 if args.workload == "config3" else 512)
    tl = args.time_limit or 2.0
    mk = (lambda k: two_agent_merge(k).build()) if args.workload == "config3" else (lambda k: random_scenario(k).build())
    S = max(1, min(args.shards, args.steps))
    shard_ids = [rank + k * world for k in range(S)]
    solver = P.Solver(device=local_rank)
    prepared = {}
    plans_of = {}
    for sid in shard_ids:
        plans_of[sid] = [mk(sid * B + k) for k in range(B)]
        prepared[sid] = solver.prepare(plans_of[sid], gap_tol=GAP, time_limit=tl)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(max(args.warmup, 1)):
        solver.upload_prepared(prepared[shard_ids[k % S]]); flush.fill_(1); solver.run()
    sampler = ClockSampler(local_rank)
    barrier(); sampler.start()
    dev_ms, launches, all_infos, nodes = [], 0, [], 0
    cars = {}
    for k in range(args.steps):
        sid = shard_ids[k % S]
        solver.upload_prepared(prepared[sid]); flush.fill_(1); torch.cuda.synchronize()
        dev_ms.append(solver.run())
        launches += solver.run_stats()["launches"]
        if k < S:
            xs, infos = solver.fetch()
            all_infos += infos
            nodes += solver.run_stats()["nodes"]
            for p in plans_of[sid]:
                cars[p.C] = cars.get(p.C, 0) + 1
    barrier()
    clocks = sampler.stop()
    e2e_s = 0.0
    for k in range(args.steps):
        flush.fill_(1); torch.cuda.synchronize()
        t0 = time.perf_counter()
        solver.solve_prepared(prepared[shard_ids[k % S]])
        e2e_s += time.perf_counter() - t0
    st2 = solver.run_stats()
    barrier()
    total_ms = sum(dev_ms)
    if world > 1:
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = (float(v) for v in t.tolist())
    if rank == 0:
        # parity sample against the oracle: the first plans of shard 0 (same gap, same time limit)
        from oracle import oracle as O
        sample = min(args.cpu_sample, 16, B)
        t0 = time.perf_counter()
        agree = worse = better = 0
        for k in range(sample):
            xo, io = O.solve(plans_of[shard_ids[0]][k], gap_tol=GAP, time_limit=tl)
            i = all_infos[k]
            if io.status != 0 or i.status != 0:
                agree += int(io.status != 0 and i.status != 0); worse += int(io.status == 0 and i.status != 0); better += int(io.status != 0 and i.status == 0)
            elif abs(io.objective - i.objective) <= max(i.gap, io.gap, GAP) * max(abs(io.objective), 1e-9) + 1e-9:
                agree += 1
            elif i.objective < io.objective:
                better += 1
            else:
                worse += 1
        cpu_dt = time.perf_counter() - t0
        viols = [i.max_violation for i in all_infos if i.status == 0]
        line = {
            "metric": "MIQP plans/sec at 1e-4 gap", "value": world * B * args.steps / (total_ms * 1e-3), "unit": "plans/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.workload], "plans_per_gpu_per_step": B, "gap": GAP, "time_limit_s": tl,
                       "cars_per_plan_rank0": {str(c): n for c, n in sorted(cars.items())},
                       "cache": "L2 flushed between steps (256 MiB write)",
                       "note": "a plan counts when it returns (proven, or time-limited with its incumbent and gap): see `solved`"},
            "clocks": clocks,
            "e2e": {"value": world * B * args.steps / e2e_s, "unit": "plans/s", "h2d_bytes_per_step": st2["h2d_bytes"],
                    "d2h_bytes_per_step": st2["d2h_bytes"], "ms_per_step": 1e3 * e2e_s / args.steps},
            "gpu_launches": launches,
            "solved": {"plans_rank0": len(all_infos), "proven_optimal": sum(1 for i in all_infos if i.status == 0 and i.proven),
                       "with_incumbent": sum(1 for i in all_infos if i.status == 0), "gap_histogram": gap_histogram(all_infos, GAP),
                       "worst_violation": max(viols) if viols else None, "nodes_per_plan": nodes / max(len(all_infos), 1)},
            "cpu_baseline": {"value": sample / cpu_dt, "unit": "plans/s", "cores": 1, "kind": "port",
                             "sample": f"first {sample} plans of shard 0, oracle/miqp_oracle_bnb.c, same gap and time limit, {cpu_dt:.1f} s",
                             "vs_device_on_sample": {"agree_within_gap": agree, "device_better": better, "device_worse": worse}},
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_frontier_workload(args):
    """config 5: ONE joint 8-agent plan per step, its branch-and-bound frontier sharded over the ranks
    (planner-miqp_b200/sharding.py:solve_frontier_sharded); NCCL carries the incumbent-objective min-all-reduce."""
    import torch
    import torch.distributed as dist
    rank, local_rank, world = init_dist()
    import planner_miqp_b200 as P
    from planner_miqp_b200.scenarios import intersection
    from planner_miqp_b200.sharding import solve_frontier_sharded
    tl = args.time_limit or 5.0
    n_cars, steps_h = args.cars, args.horizon
    solver = P.Solver(device=local_rank)
    S = max(1, min(args.shards, args.steps))
    plans = [intersection(k, n_cars=n_cars, nr_steps=steps_h).build() for k in range(S)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for k in range(max(args.warmup, 1)):
        solve_frontier_sharded(solver, [plans[k % S]], gap_tol=GAP, time_limit=min(tl, 1.0), ramp_rounds=args.ramp_rounds, exchange_every=args.exchange_every)
    sampler = ClockSampler(local_rank)
    barrier(); sampler.start()
    t0 = time.perf_counter()
    results, launches, dev_ms = [], 0, []
    for k in range(args.steps):
        st = {}
        barrier()
        t1 = time.perf_counter()
        xs, infos = solve_frontier_sharded(solver, [plans[k % S]], gap_tol=GAP, time_limit=tl, ramp_rounds=args.ramp_rounds,
                                           exchange_every=args.exchange_every, stats=st)
        barrier()
        dt = time.perf_counter() - t1
        dev_ms.append(st["device_ms"])
        rs = solver.run_stats()
        launches += rs["launches"]
        results.append((infos[0], st, dt, rs))
    total_s = time.perf_counter() - t0
    clocks = sampler.stop()
    dev_total = sum(dev_ms)
    if world > 1:
        t = torch.tensor([dev_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_total = float(t.item())
        own = torch.tensor([float(r[1]["nodes_this_rank"]) for r in results], dtype=torch.float64, device="cuda")
        gathered = [torch.zeros_like(own) for _ in range(world)]
        dist.all_gather(gathered, own)
        nodes_by_rank = [[int(v) for v in g.tolist()] for g in gathered]
    else:
        nodes_by_rank = [[int(r[1]["nodes_this_rank"]) for r in results]]
    if rank == 0:
        from oracle import oracle as O
        p0 = plans[0]
        sz = solver.sizes(p0)
        nodes = sum(r[0].nodes for r in results)
        line = {
            "metric": "MIQP plans/sec at 1e-4 gap", "value": args.steps / (dev_total * 1e-3), "unit": "plans/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dev_total / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS["config5"], "cars": n_cars, "N": steps_h, "R": p0.R, "gap": GAP, "time_limit_s": tl,
                       "model": {"rows": sz.nrows, "cols": sz.ncols, "binaries": sz.nbin},
                       "ramp_rounds": args.ramp_rounds, "exchange_every_rounds": args.exchange_every,
                       "collective": "min-all-reduce of the incumbent objective (8 bytes, in place on the solver's device array) every "
                                     f"{args.exchange_every} rounds + one sum-all-reduce of the unfinished-plan count; winner's vector once at the end",
                       "note": "every step ends at the time limit unless the gap is proven: plans/s is 1 / time limit then, and the figures "
                               "that scale with the GPUs are node relaxations per second and the gap reached (see `solved`)"},
            "clocks": clocks,
            "e2e": {"value": args.steps / total_s, "unit": "plans/s", "h2d_bytes_per_step": results[-1][3]["h2d_bytes"],
                    "d2h_bytes_per_step": results[-1][3]["d2h_bytes"], "ms_per_step": 1e3 * total_s / args.steps},
            "gpu_launches": launches,
            "solved": {"per_step": [{"status": r[0].status, "objective": r[0].objective, "best_bound": r[0].best_bound, "gap": r[0].gap,
                                     "proven": bool(r[0].proven), "nodes_all_ranks": r[0].nodes, "max_violation": r[0].max_violation,
                                     "exchanges": r[1]["exchanges"], "split": r[1]["split"], "wall_s": r[2]} for r in results],
                       "node_relaxations_per_s": nodes / (dev_total * 1e-3), "nodes_by_rank_per_step": nodes_by_rank},
        }
        if args.cpu_sample > 0:
            t1 = time.perf_counter()
            xo, io = O.solve(p0, gap_tol=GAP, time_limit=tl)
            cdt = time.perf_counter() - t1
            line["cpu_baseline"] = {"value": 1.0 / cdt, "unit": "plans/s", "cores": 1, "kind": "port",
                                    "sample": f"plan 0 with the same time limit, oracle/miqp_oracle_bnb.c, {cdt:.1f} s: status {io.status}, "
                                              f"objective {io.objective}, gap {io.gap}"}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config2", choices=["config2", "config3", "config4", "config5"])
    ap.add_argument("--time-limit", type=float, default=None, help="per-plan time limit of configs 3-5 (s)")
    ap.add_argument("--cars", type=int, default=8, help="config5: agents")
    ap.add_argument("--horizon", type=int, default=40, help="config5: steps")
    ap.add_argument("--ramp-rounds", type=int, default=8)
    ap.add_argument("--exchange-every", type=int, default=4)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=2048, help="plans per GPU per step")
    ap.add_argument("--shards", type=int, default=3, help="distinct scenario shards a rank cycles through (seeds rotate per step)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--nodes-per-round", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=48)
    ap.add_argument("--latency-plans", type=int, default=16)
    ap.add_argument("--replan-scenarios", type=int, default=256)
    ap.add_argument("--replan-cycles", type=int, default=8)
    ap.add_argument("--first-shard", type=int, default=0, help="offset of the scenario shards (knobs are tuned on held-out shards >= 100, the reported runs use 0)")
    ap.add_argument("--skip-extras", action="store_true", help="only the throughput legs (no latency, replanning, assembly, CPU baseline): for A/B runs")
    ap.add_argument("--in-flight", type=int, default=3, help="batches in flight on one GPU (solver instances / streams); 1 = one at a time")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the solution vectors and solve results of the last timed step (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl == "reference" or args.workload != "config2"):
        ap.error("--dump-outputs covers the device path of the default workload (config2)")
    args.batch_given = any(a == "--batch" or a.startswith("--batch=") for a in sys.argv[1:])
    if args.impl == "reference":
        return run_reference(args)
    if args.workload in ("config3", "config4"):
        return run_multi_agent_batch(args)
    if args.workload == "config5":
        return run_frontier_workload(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MIQP backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import planner_miqp_b200 as P
    if world > 1:
        # one process per GPU and several batches in flight per process share the host cores: keep the packing threads of all of
        # them within the core count (8 ranks x 3 batches x 8 threads on 16 cores otherwise)
        os.environ.setdefault("MIQP_PACK_THREADS", str(max(1, min(8, (os.cpu_count() or 8) // (world * max(args.in_flight, 1))))))
    B = args.batch
    S = max(1, min(args.shards, args.steps))
    shard_ids = [args.first_shard + rank + k * world for k in range(S)]          # rank r: shards r, r + world, ...
    solver = P.Solver(device=local_rank, nodes_per_round=args.nodes_per_round)
    shard_plans = {sid: make_plans(sid * B, B) for sid in shard_ids}
    prepared = {sid: solver.prepare(shard_plans[sid], gap_tol=GAP, time_limit=600.0) for sid in shard_ids}
    plans = shard_plans[shard_ids[0]]
    N = plans[0].N
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ------------------------------------------------------
    # every step solves another shard of the workload: upload (untimed; the batch is resident in HBM when the timed
    # region of the step starts), L2 flush, then the device solve, timed with CUDA events on the solver stream
    for k in range(args.warmup):
        solver.upload_prepared(prepared[shard_ids[k % S]])
        flush.fill_(1)
        solver.run()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    dev_ms, node_ms, launches = [], 0.0, 0
    per_shard = {sid: [] for sid in shard_ids}
    nodes_tot = iters_tot = rows_tot = 0
    n_ok = 0
    uncert = pool_ex = 0
    worst_viol = 0.0
    t_wall0 = time.perf_counter()
    for k in range(args.steps):
        sid = shard_ids[k % S]
        solver.upload_prepared(prepared[sid])
        flush.fill_(1)
        torch.cuda.synchronize()
        ms = solver.run()
        dev_ms.append(ms); per_shard[sid].append(ms)
        st = solver.run_stats()
        node_ms += st["node_kernel_ms"]; launches += st["launches"]
        if k < S:      # results of every distinct shard are fetched and checked once (outside the device-timed region)
            xs, infos = solver.fetch()
            stf = solver.run_stats()
            nodes_tot += stf["nodes"]; iters_tot += stf["qp_iters"]; rows_tot += stf["rows_visited"]
            n_ok += sum(1 for i in infos if i.status == 0 and i.proven)
            uncert += sum(i.uncertified for i in infos); pool_ex += sum(i.pool_exhausted for i in infos)
            worst_viol = max([worst_viol] + [i.max_violation for i in infos if i.status == 0])
            if sid == shard_ids[0]:
                infos0, st0 = infos, dict(stf)
                st0["node_kernel_ms"] = st["node_kernel_ms"]
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    total_ms = sum(dev_ms)
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
        ok_t = torch.tensor([n_ok, uncert, pool_ex], dtype=torch.int64, device="cuda")
        dist.all_reduce(ok_t)
        n_ok_all, uncert, pool_ex = (int(v) for v in ok_t.tolist())
    else:
        n_ok_all = n_ok
    value_seq = world * B * args.steps / (total_ms * 1e-3)
    seq_ms_per_step = total_ms / args.steps

    # ---- two batches in flight (two solver instances, two streams) ---------------------------
    # the tail rounds of one batch (a few hard plans, a near-empty GPU) overlap with the head rounds of the next one;
    # device time from the first launch to the last completion on either stream (CUDA events on the solvers' streams)
    def agree(flag: bool) -> bool:
        """True only if `flag` holds on every rank (keeps the collectives below in step when one rank fails a leg)"""
        if world == 1:
            return bool(flag)
        t = torch.tensor([1.0 if flag else 0.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item()) > 0.5

    pipe = None
    pipe_ms = None
    if args.in_flight > 1 and S > 1 and args.steps > 1:
        ok = True
        stagger = 0.5e-3 * seq_ms_per_step * (args.in_flight / 2.0)
        try:
            pipe = P.PipelinedSolver(device=local_rank, depth=args.in_flight, nodes_per_round=args.nodes_per_round)
            pipe.upload_resident([prepared[shard_ids[k % S]] for k in range(args.in_flight)])
            pipe.run_resident(max(args.warmup, args.in_flight), stagger)
        except Exception as ex:     # (e.g. not enough memory for a second node pool): the sequential figures stand
            sys.stderr.write(f"[bench] pipelined leg failed: {ex}\n")
            ok = False
        if agree(ok):
            barrier()
            try:
                pipe_ms, pipe_runs = pipe.timed_resident(args.steps, stagger)
                launches_pipe = int(sum(s_.run_stats()["launches"] for s_ in pipe.solvers) / len(pipe.solvers) * args.steps)
            except Exception as ex:
                sys.stderr.write(f"[bench] pipelined leg failed: {ex}\n")
                pipe_ms = None
            barrier()
        if world > 1:
            t = torch.tensor([pipe_ms if pipe_ms is not None else -1.0], dtype=torch.float64, device="cuda")
            tmin = t.clone()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
            pipe_ms = float(t.item()) if float(tmin.item()) > 0 else None
        if pipe_ms is None and pipe is not None:      # (on every rank alike)
            pipe.close()
            pipe = None
    value_pipe = world * B * args.steps / (pipe_ms * 1e-3) if pipe_ms else None
    use_pipe = value_pipe is not None and value_pipe > value_seq
    value = value_pipe if use_pipe else value_seq
    if use_pipe:
        total_ms = pipe_ms
    if args.dump_outputs and rank == 0:
        # results of the leg that gave `value`, as its last timed step left them: the sequential solver ran shard
        # shard_ids[(steps - 1) mod S] last; pipelined step (steps - 1) ran on instance (steps - 1) mod depth, which holds
        # shard_ids[instance mod S] (upload_resident above)
        if use_pipe:
            w = (args.steps - 1) % len(pipe.solvers)
            last_solver, last_sid = pipe.solvers[w], shard_ids[w % S]
        else:
            last_solver, last_sid = solver, shard_ids[(args.steps - 1) % S]
        dump_outputs(args.dump_outputs, last_solver, [last_sid * B + k for k in range(B)])

    # ---- end to end through the C ABI with host buffers ------------------------------------
    # the caller holds the batch as MiqpB200Problem structs over host arrays and receives every
    # solution vector in host arrays; timed: the C-ABI call (flatten + H2D + device solve + D2H)
    for k in range(2):
        solver.solve_prepared(prepared[shard_ids[k % S]])
    barrier()
    e2e_s = 0.0
    for k in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        solver.solve_prepared(prepared[shard_ids[k % S]])
        e2e_s += time.perf_counter() - t0
    barrier()
    st2 = solver.run_stats()
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_full = world * B * args.steps / e2e_s          # every OPL column vector returned (68 MB per 2048 plans)
    e2e_full_ms = 1e3 * e2e_s / args.steps
    d2h_full = st2["d2h_bytes"]
    # compact results: trajectories + status / objective / gap per plan; the full vectors stay on the device (fetch_vector on demand)
    solver.solve_prepared_compact(prepared[shard_ids[0]])
    barrier()
    e2e_s = 0.0
    for k in range(args.steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        solver.solve_prepared_compact(prepared[shard_ids[k % S]])
        e2e_s += time.perf_counter() - t0
    barrier()
    st2 = solver.run_stats()
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_seq = world * B * args.steps / e2e_s
    e2e_seq_ms = 1e3 * e2e_s / args.steps
    # the same calls with two batches in flight: pack + H2D of one batch and D2H + scatter of the other overlap with the search
    e2e_pipe = None
    if pipe is not None:          # (the same on every rank, see above)
        jobs = [prepared[shard_ids[k % S]] for k in range(args.steps)]
        ok = True
        try:
            pipe.solve_stream_compact(jobs[:args.in_flight], 0.5e-3 * e2e_seq_ms)
        except Exception as ex:
            sys.stderr.write(f"[bench] pipelined end-to-end leg failed: {ex}\n")
            ok = False
        if agree(ok):
            barrier()
            t0 = time.perf_counter()
            try:
                pipe.solve_stream_compact(jobs, 0.5e-3 * e2e_seq_ms)
            except Exception as ex:
                sys.stderr.write(f"[bench] pipelined end-to-end leg failed: {ex}\n")
                ok = False
            e2e_pipe_s = time.perf_counter() - t0
            barrier()
            if agree(ok):
                if world > 1:
                    t = torch.tensor([e2e_pipe_s], dtype=torch.float64, device="cuda")
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    e2e_pipe_s = float(t.item())
                e2e_pipe = world * B * args.steps / e2e_pipe_s
    if e2e_pipe is not None and e2e_pipe > e2e_seq:
        e2e_value, e2e_s = e2e_pipe, e2e_pipe_s
    else:
        e2e_value = e2e_seq
    if pipe is not None:
        pipe.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (bnb_nodes_kernel), first shard ----------------------
    st = st0
    fp64_peak = solver.measure_fp64_peak()
    flops = algorithmic_flops(st, N)
    node_ms_last = st["node_kernel_ms"]
    achieved_tf = flops / (node_ms_last * 1e-3) / 1e12 if node_ms_last > 0 else 0.0
    peaks = measured_peaks()
    # algorithmic HBM bytes: every node relaxation reads its record and writes its children
    ndec = 6 * N + 5 * plans[0].O * N
    node_bytes = 2.0 * (ndec + 32 + 64 * N)   # decisions + bookkeeping + the parent's relaxed optimum (8 N doubles), read once and written per child
    hbm_gbs = st["nodes"] * node_bytes / (node_ms_last * 1e-3) / 1e9 if node_ms_last > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "node_kernel_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get("dram_bytes_per_launch")
    roofline = {
        "kernel": "bnb_nodes_kernel", "bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
        "frac": achieved_tf / fp64_peak if fp64_peak else None, "traffic": traffic,
        "peak_source": "DFMA micro-benchmark in this run (MEASURED_PEAKS.json has no FP64 figure)",
        "kernel_share_of_step": node_ms / sum(dev_ms) if dev_ms else None,
        "note": "latency-bound FP64 kernel (one CTA of four warps per node relaxation, sequential Riccati recursion on one warp); see DESIGN.md section 4",
        "hbm": {"achieved": hbm_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": hbm_gbs / peaks["hbm_gbs"] if peaks["hbm_gbs"] else None, "peak_source": peaks["source"]},
        "nodes_per_s": st["nodes"] / (node_ms_last * 1e-3) if node_ms_last > 0 else None,
        "ipm_iters_per_node": st["qp_iters"] / max(st["nodes"], 1),
    }
    # assembly kernel (SURVEY section 8(d)(a)): HBM-write bound; bytes = CSR values + column indices + two row bounds + row pointers
    asm_ms, asm_rows, asm_nnz = solver.assemble_batch(plans, repeats=5)
    asm_bytes = 12.0 * asm_nnz + 16.0 * asm_rows + 8.0 * (asm_rows + B)
    asm_gbs = asm_bytes / (asm_ms * 1e-3) / 1e9 if asm_ms > 0 else 0.0
    roofline["assembly"] = {"kernel": "assemble_rows_kernel", "bound": "hbm", "achieved": asm_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": asm_gbs / peaks["hbm_gbs"] if peaks["hbm_gbs"] else None, "ms_per_batch": asm_ms,
                            "plans": B, "rows": asm_rows, "nnz": asm_nnz, "bytes": asm_bytes, "peak_source": peaks["source"],
                            "assemblies_per_s": B / (asm_ms * 1e-3) if asm_ms > 0 else None}

    if args.skip_extras:
        emit({"value": value, "ms_per_step": total_ms / args.steps, "batches_in_flight": args.in_flight if use_pipe else 1, "batch": B,
              "one_batch_at_a_time": {"value": value_seq, "ms_per_step": seq_ms_per_step, "e2e": e2e_seq, "e2e_full_vectors": e2e_full},
              "e2e": e2e_value, "steps": args.steps, "env": {k: v for k, v in os.environ.items() if k.startswith("MIQP_")}})
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- single-plan latency ----------------------------------------------------------------
    lat_e2e, lat_dev = [], []
    for k in range(min(args.latency_plans, B)):
        t0 = time.perf_counter()
        solver.solve(plans[k], gap_tol=GAP, time_limit=60.0)
        lat_e2e.append(1e3 * (time.perf_counter() - t0))
        lat_dev.append(solver.run_stats()["total_ms"])

    # ---- config 2 as named: warm-started replanning ---------------------------------------------
    replan = replan_leg(solver, min(args.replan_scenarios, B), args.replan_cycles) if args.replan_scenarios > 0 else None

    # ---- CPU baseline (rank 0, bounded sample, one core) --------------------------------------
    sample = min(args.cpu_sample, B)
    cpu_rate, cpu_dt, cpu_ok = cpu_oracle_rate(plans[:sample], 1)
    # parity spot check of the sample against the oracle (objective within 1e-4 relative)
    from oracle import oracle as O
    mism = 0
    for k in range(min(8, sample)):
        xo, io = O.solve(plans[k], gap_tol=GAP, time_limit=60.0)
        if io.status != infos0[k].status or (io.status == 0 and abs(io.objective - infos0[k].objective) > 1e-4 * max(abs(io.objective), 1e-9)):
            mism += 1

    shard_ms = {str(sid): {"min": min(v), "mean": sum(v) / len(v), "max": max(v), "steps": len(v)} for sid, v in per_shard.items() if v}
    cfg = bench_config(B)
    run = {"nodes_per_plan_per_round": args.nodes_per_round or "auto", "batches_in_flight": args.in_flight if use_pipe else 1,
           "first_shard": args.first_shard}
    if use_pipe:
        run["seeds"] = "solver instance w holds shard (rank + w * n_gpus) resident and re-runs it (steps alternate over the instances)"
        run["cache"] = "no flush between overlapping steps: the instances alternate over different resident batches (problem data + node pools > 126 MB L2)"
        run["timing"] = "CUDA events on the solvers' own streams: first launch of the first step to the last completion on any stream, max over ranks"
    else:
        run["seeds"] = "step k of rank r: shard (r + k * n_gpus) mod shards"
        run["cache"] = "L2 flushed between steps (256 MiB write)"
        run["timing"] = "CUDA events on the solver stream around every miqp_b200_batch_run, summed, max over ranks"
    line = {
        "metric": "MIQP plans/sec at 1e-4 gap", "value": value, "unit": "plans/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "run": run,
        "clocks": clocks,
        "one_batch_at_a_time": {"value": value_seq, "ms_per_step": seq_ms_per_step, "e2e_value": e2e_seq, "e2e_ms_per_step": e2e_seq_ms,
                                "e2e_full_vectors": {"value": e2e_full, "ms_per_step": e2e_full_ms, "d2h_bytes_per_step": d2h_full},
                                "note": "one solver, one stream: batch k + 1 starts when batch k has finished (L2 flushed in between); "
                                        "the roofline and per-shard figures below are from this leg"},
        "e2e": {"value": e2e_value, "unit": "plans/s", "h2d_bytes_per_step": st2["h2d_bytes"], "d2h_bytes_per_step": st2["d2h_bytes"],
                "ms_per_step": 1e3 * e2e_s / args.steps,
                "results": "compact: per plan the trajectory [C][N][8] and status / objective / bound / gap / violation (miqp_b200_solve_batch_compact); "
                           "the full column vectors stay on the device (miqp_b200_fetch_vector)",
                "host_ms_last_step": {"pack": st2.get("pack_ms"), "h2d_tables_pool": st2.get("upload_ms"), "d2h_scatter": st2.get("fetch_ms")}},
        "gpu_launches": launches_pipe if use_pipe else launches,
        "roofline": roofline,
        "cpu_baseline": {"value": cpu_rate, "unit": "plans/s", "cores": 1, "kind": "port",
                         "sample": f"first {sample} plans of the batch, oracle/miqp_oracle_bnb.c, {cpu_dt:.1f} s"},
        "latency_p50_ms": {"e2e": statistics.median(lat_e2e), "device": statistics.median(lat_dev), "plans": len(lat_e2e)},
        "shard_ms_rank0": shard_ms,
        "replan": replan,
        "solved": {"proven_optimal": n_ok_all, "plans": world * B * S, "worst_violation": worst_viol,
                   "oracle_mismatches_in_sample": mism, "nodes_per_plan": nodes_tot / (B * S), "rounds": st["rounds"],
                   "nodes_closed_without_certificate": uncert, "plans_with_exhausted_pool": pool_ex,
                   "note": "every distinct shard is fetched and checked once; counts are summed over ranks and shards"},
        "wall_s_timed_region": t_wall,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
