"""Cost and benefit of anytime runs (Solver.run_anytime) against plain and streaming runs.

overhead   bench.py's flagship workload: config 2 (one car, N = 40, R = 32), 2048 plans per batch, seeded shards 0..2, gap 1e-4.
           The same resident batches are run alternately plain (batch_run), streaming (a no-op on_plan) and anytime (a no-op
           incumbent callback, no stops), --runs times each.  Reported: device time per batch (CUDA events on the solver stream),
           whether every run's outputs are identical, records per plan, and the anytime kernels' share of kernel time (one
           separate torch.profiler run).
latency    config 4 (1-4 cars, 512 plans, 2 s limit): time from the start of the run to each plan's first incumbent callback,
           against the time its final result reaches on_plan (p50 / p90 / p99).
stop       config 4 again, the callback stopping a plan once its gap is <= 10 % (the reference's default tolerance): batch time
           and the plans' final gaps against the plain run.

The card's name and power limit are read in the same process.

    python tools/anytime_latency.py --out profiles/r3_anytime_latency.json
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import planner_miqp_b200 as P                                              # noqa: E402
from planner_miqp_b200.scenarios import obstacle_scenario, random_scenario   # noqa: E402

GAP = 1e-4
MODES = ("plain", "stream", "anytime")
STOP_GAP = 0.10


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [v.strip() for v in out[0].split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as ex:  # reported, not hidden
        return {"error": repr(ex)}


def pct(a, q):
    a = np.asarray(a, dtype=np.float64)
    a = a[np.isfinite(a)]
    return float(np.percentile(a, q)) if len(a) else None


def dist(a):
    a = np.asarray(a, dtype=np.float64)
    a = a[np.isfinite(a)]
    return {"n": int(len(a)), "p50": pct(a, 50), "p90": pct(a, 90), "p99": pct(a, 99), "max": float(np.max(a)) if len(a) else None}


def digest(tr, infos):
    """every output of a run except the host-clock fields (seconds) and the round count"""
    h = hashlib.sha256()
    for t in tr:
        h.update(np.ascontiguousarray(t).tobytes())
    for i in infos:
        h.update(np.array([i.status, i.proven, i.nodes, i.qp_iters, i.uncertified, i.pool_exhausted], dtype=np.int64).tobytes())
        h.update(np.array([i.objective, i.best_bound, i.gap, i.max_violation], dtype=np.float64).tobytes())
    return h.hexdigest()


def run_mode(s, mode):
    """one run of the resident batch: (device ms, number of incumbent records)"""
    if mode == "plain":
        return s.run(), 0
    if mode == "stream":
        return s.run_streaming(lambda k, t, i: None), 0
    n = [0]

    def on_inc(k, t, inc):
        n[0] += 1

    return s.run_anytime(on_inc), n[0]


def anytime_share(s):
    """kernel time of the incumbent harvest (bnb_inc_* and evaluate_list_kernel, which only it launches in an anytime run
    without on_plan) over all kernel time of one anytime run (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.run_anytime(lambda k, t, i: None)
        torch.cuda.synchronize()
    tot, ai, per = 0.0, 0.0, {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if us <= 0:
            continue
        tot += us
        if "bnb_inc_" in e.key or "evaluate_list" in e.key:
            ai += us
            per[e.key] = {"us": us, "count": e.count}
    return {"anytime_us": ai, "all_kernels_us": tot, "share": ai / tot if tot else None, "kernels": per}


def overhead(args):
    B, S = args.batch, args.shards
    s = P.Solver()
    prepared = [s.prepare([obstacle_scenario(sid * B + k).build() for k in range(B)], gap_tol=GAP, time_limit=600.0)
                for sid in range(S)]
    for mode in MODES:                    # warm-up: module loads, pool sizing, page-locked buffers of every mode
        s.upload_prepared(prepared[0])
        run_mode(s, mode)
    ms = {m: [] for m in MODES}
    recs_per_plan = []
    ref, identical = {}, True
    for r in range(args.runs):
        for sid in range(S):
            order = MODES[(r + sid) % 3:] + MODES[:(r + sid) % 3]   # rotate the order: no mode always runs first
            for mode in order:
                s.upload_prepared(prepared[sid])
                t, nrec = run_mode(s, mode)
                ms[mode].append(t)
                if mode == "anytime":
                    recs_per_plan.append(nrec / B)
                tr, infos = s.fetch_compact()
                d = digest(tr, infos)
                ref.setdefault(sid, d)
                identical &= (d == ref[sid])
    out = {
        "workload": f"config 2 (1 car, N=40, R=32), {B} plans per batch, scenario shards s*B .. s*B+B-1 of obstacle_scenario, "
                    f"s = 0..{S - 1}, gap {GAP}",
        "runs_per_mode_per_shard": args.runs,
        "outputs_identical_across_modes_and_runs": bool(identical),
        "batch_device_ms": {m: {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v)), "std": float(np.std(v)),
                                "all": v} for m, v in ms.items()},
        "overhead_vs_plain_device_ms": {m: float(np.mean(ms[m]) - np.mean(ms["plain"])) for m in MODES[1:]},
        "incumbent_records_per_plan": float(np.mean(recs_per_plan)),
    }
    if not args.no_profile:
        s.upload_prepared(prepared[0])
        try:
            out["anytime_kernel_share"] = anytime_share(s)
        except Exception as ex:
            out["anytime_kernel_share"] = {"error": repr(ex)}
    s.close()
    return out


def config4(args):
    B = args.batch4
    s = P.Solver()
    b = s.prepare([random_scenario(k).build() for k in range(B)], gap_tol=GAP, time_limit=args.time_limit)
    for warm in (lambda: s.run(), lambda: s.run_anytime(lambda k, t, i: None, lambda k, t, i: None)):
        s.upload_prepared(b)              # warm-up: the first anytime run of a solver allocates its record buffers
        warm()
    # plain
    s.upload_prepared(b)
    t0 = time.perf_counter()
    ms_plain = s.run()
    wall_plain = time.perf_counter() - t0
    _, in_plain = s.fetch_compact()
    st_plain = s.run_stats()
    # latency: first incumbent callback and final result (on_plan) of every plan
    first = np.full(B, np.nan)
    first_gap = np.full(B, np.nan)
    final = np.full(B, np.nan)
    nrec = np.zeros(B, dtype=np.int64)
    s.upload_prepared(b)
    t0 = time.perf_counter()

    def on_inc(k, t, inc):
        nrec[k] += 1
        if np.isnan(first[k]):
            first[k] = time.perf_counter() - t0
            first_gap[k] = inc.gap

    def on_plan(k, t, info):
        final[k] = time.perf_counter() - t0

    ms_any = s.run_anytime(on_inc, on_plan)
    wall_any = time.perf_counter() - t0
    st_any = s.run_stats()
    have = np.isfinite(first)
    latency = {
        "workload": f"config 4 (random_scenario, 1-4 cars, N=20, R=16), {B} plans, time limit {args.time_limit} s, gap {GAP}",
        "plans_with_incumbent": int(have.sum()),
        "first_incumbent_ms": dist(first * 1e3),
        "final_result_ms": dist(final[have] * 1e3),
        "first_over_final": dist(first[have] / final[have]),
        "gap_of_first_incumbent": dist(first_gap),
        "records_per_plan_with_incumbent": float(nrec[have].mean()) if have.any() else None,
        "batch_wall_ms": {"plain": 1e3 * wall_plain, "anytime": 1e3 * wall_any},
        "batch_device_ms": {"plain": ms_plain, "anytime": ms_any},
        # (the plans run to a wall-clock limit: how many rounds fit, and so the results, differ from run to run)
        "rounds": {"plain": st_plain["rounds"], "anytime": st_any["rounds"]},
    }
    # stop policy: a plan is stopped once its incumbent's gap is <= STOP_GAP
    s.upload_prepared(b)
    t0 = time.perf_counter()
    ms_stop = s.run_anytime(lambda k, t, inc: inc.gap <= STOP_GAP)
    wall_stop = time.perf_counter() - t0
    _, in_stop = s.fetch_compact()
    stopped = s.stopped()
    st_stop = s.run_stats()
    hit = stopped >= 0
    gaps = lambda infos: [i.gap if i.status == 0 else np.inf for i in infos]   # noqa: E731
    stop = {
        "policy": f"on_incumbent returns gap <= {STOP_GAP}",
        "plans_stopped": int((stopped >= 0).sum()),
        "batch_device_ms": {"plain": ms_plain, "stop_policy": ms_stop},
        "batch_wall_ms": {"plain": 1e3 * wall_plain, "stop_policy": 1e3 * wall_stop},
        "rounds": {"plain": st_plain["rounds"], "stop_policy": st_stop["rounds"]},
        "nodes": {"plain": st_plain["nodes"], "stop_policy": st_stop["nodes"]},
        "stopped_plans_seconds_ms": {"plain": dist([1e3 * in_plain[k].seconds for k in np.flatnonzero(hit)]),
                                     "stop_policy": dist([1e3 * in_stop[k].seconds for k in np.flatnonzero(hit)])},
        "stopped_plans_final_gap": dist([in_stop[k].gap for k in np.flatnonzero(hit)]),
        "final_gap": {"plain": dist(gaps(in_plain)), "stop_policy": dist(gaps(in_stop))},
        "plans_gap_le_10pct": {"plain": int(sum(g <= STOP_GAP for g in gaps(in_plain))),
                               "stop_policy": int(sum(g <= STOP_GAP for g in gaps(in_stop)))},
        "status_counts": {"plain": np.bincount([i.status for i in in_plain], minlength=4).tolist(),
                          "stop_policy": np.bincount([i.status for i in in_stop], minlength=4).tolist()},
    }
    s.close()
    return latency, stop


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--shards", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3, help="runs of every mode on every shard (overhead)")
    ap.add_argument("--batch4", type=int, default=512, help="plans of the config-4 batch (latency, stop policy)")
    ap.add_argument("--time-limit", type=float, default=2.0, help="time limit of the config-4 plans, seconds")
    ap.add_argument("--out", default=None, help="JSON file to write (also printed)")
    ap.add_argument("--no-profile", action="store_true", help="skip the torch.profiler run of the anytime kernels' share")
    args = ap.parse_args()
    out = {"tool": "tools/anytime_latency.py", "gpu": gpu_info()}
    out["overhead"] = overhead(args)
    out["latency"], out["stop_policy"] = config4(args)
    txt = json.dumps(out, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
