"""Per-plan delivery latency of streaming runs (Solver.run_streaming) against plain batch runs, on the flagship workload of
bench.py: config 2 (one car, N = 40, R = 32), 2048 plans per batch, the same seeded shards, gap 1e-4.

On one GPU, the same resident batches are run alternately plain (batch_run) and streaming, --runs times each.  Reported:
device time per batch (CUDA events) of both modes with its spread, per-plan latency from the start of the run to the callback
(p50 / p90 / p99 / max) next to the batch time and next to each plan's own `seconds`, rounds per batch, the harvest kernels'
share of device time (one separate torch.profiler run) and whether every run's outputs are identical.  The card's name and
power limit are read in the same process.

    python tools/stream_latency.py --out profiles/stream_latency_batch2048.json
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

import planner_miqp_b200 as P                                   # noqa: E402
from planner_miqp_b200.scenarios import obstacle_scenario        # noqa: E402

GAP = 1e-4
MODES = ("plain", "stream")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [v.strip() for v in out[0].split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as ex:  # reported, not hidden
        return {"error": repr(ex)}


def pct(a, q):
    return float(np.percentile(np.asarray(a, dtype=np.float64), q)) if len(a) else None


def dist(a):
    return {"p50": pct(a, 50), "p90": pct(a, 90), "p99": pct(a, 99), "max": float(np.max(a)) if len(a) else None}


def digest(tr, infos):
    """every output of a run except the host-clock fields (seconds) and the round count"""
    h = hashlib.sha256()
    for t in tr:
        h.update(np.ascontiguousarray(t).tobytes())
    for i in infos:
        h.update(np.array([i.status, i.proven, i.nodes, i.qp_iters, i.uncertified, i.pool_exhausted], dtype=np.int64).tobytes())
        h.update(np.array([i.objective, i.best_bound, i.gap, i.max_violation], dtype=np.float64).tobytes())
    return h.hexdigest()


def run_once(s, mode):
    """one run of the resident batch; returns (device ms, wall s, per-plan callback times from the start, streamed infos)"""
    if mode == "plain":
        t0 = time.perf_counter()
        ms = s.run()
        return ms, time.perf_counter() - t0, None, None
    n = s._batch[0]
    lat = np.full(n, np.nan)
    infos = [None] * n
    t0 = time.perf_counter()

    def on_plan(k, traj, info):
        lat[k] = time.perf_counter() - t0
        infos[k] = info

    ms = s.run_streaming(on_plan)
    wall = time.perf_counter() - t0
    return ms, wall, lat, infos


def harvest_share(s):
    """kernel time of the harvest kernels over all kernel time of one streaming run (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        s.run_streaming(lambda k, t, i: None)
        torch.cuda.synchronize()
    tot, hv, per = 0.0, 0.0, {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        if us <= 0:
            continue
        tot += us
        if "harvest" in e.key or "evaluate_list" in e.key:
            hv += us
            per[e.key] = {"us": us, "count": e.count}
    return {"harvest_us": hv, "all_kernels_us": tot, "share": hv / tot if tot else None, "kernels": per}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--shards", type=int, default=3)
    ap.add_argument("--runs", type=int, default=5, help="runs of every mode on every shard")
    ap.add_argument("--out", default=None, help="JSON file to write (also printed)")
    ap.add_argument("--no-profile", action="store_true", help="skip the torch.profiler run of the harvest share")
    args = ap.parse_args()
    B, S = args.batch, args.shards
    hw = gpu_info()
    s = P.Solver()
    prepared = [s.prepare([obstacle_scenario(sid * B + k).build() for k in range(B)], gap_tol=GAP, time_limit=600.0)
                for sid in range(S)]
    for mode in MODES:                    # warm-up: module loads, pool sizing, page-locked buffers of every mode
        s.upload_prepared(prepared[0])
        run_once(s, mode)
    rec = {m: {"ms": [], "wall_s": [], "rounds": []} for m in MODES}
    lat_all = {m: [] for m in MODES[1:]}
    after_seconds = {m: [] for m in MODES[1:]}
    seconds_all, lat_over_batch = [], {m: [] for m in MODES[1:]}
    ref_digest, identical, streamed_equal = {}, True, True
    for r in range(args.runs):
        for sid in range(S):
            order = MODES if (r + sid) % 2 == 0 else MODES[::-1]   # alternate the order: no mode always runs first
            for mode in order:
                s.upload_prepared(prepared[sid])
                ms, wall, lat, sinfos = run_once(s, mode)
                st = s.run_stats()
                rec[mode]["ms"].append(ms); rec[mode]["wall_s"].append(wall); rec[mode]["rounds"].append(st["rounds"])
                tr, infos = s.fetch_compact()
                d = digest(tr, infos)
                if sid not in ref_digest:
                    ref_digest[sid] = d
                identical &= (d == ref_digest[sid])
                if lat is not None:
                    assert not np.isnan(lat).any(), "a plan was not delivered"
                    sec = np.array([i.seconds for i in infos])
                    for k in range(len(infos)):
                        a, b = sinfos[k], infos[k]
                        streamed_equal &= all(np.float64(getattr(a, f)).tobytes() == np.float64(getattr(b, f)).tobytes()
                                              for f in ("objective", "best_bound", "gap", "seconds", "max_violation")) \
                            and (a.status, a.proven, a.nodes, a.qp_iters) == (b.status, b.proven, b.nodes, b.qp_iters)
                    lat_all[mode].extend((lat * 1e3).tolist())
                    after_seconds[mode].extend(((lat - sec) * 1e3).tolist())
                    lat_over_batch[mode].extend((lat / wall).tolist())
                    seconds_all.extend((sec * 1e3).tolist())
    out = {
        "tool": "tools/stream_latency.py",
        "gpu": hw,
        "workload": f"config 2 (1 car, N=40, R=32), {B} plans per batch, scenario shards s*B .. s*B+B-1 of obstacle_scenario, "
                    f"s = 0..{S - 1}, gap {GAP}",
        "runs_per_mode_per_shard": args.runs,
        "outputs_identical_across_modes_and_runs": bool(identical),
        "streamed_info_equals_fetch": bool(streamed_equal),
        "batch_device_ms": {m: {"mean": float(np.mean(v["ms"])), "min": float(np.min(v["ms"])), "max": float(np.max(v["ms"])),
                                "std": float(np.std(v["ms"])), "all": v["ms"]} for m, v in rec.items()},
        "batch_wall_ms": {m: {"mean": 1e3 * float(np.mean(v["wall_s"])), "min": 1e3 * float(np.min(v["wall_s"])),
                              "max": 1e3 * float(np.max(v["wall_s"]))} for m, v in rec.items()},
        "rounds_per_batch": {m: sorted(set(v["rounds"])) for m, v in rec.items()},
        "streaming_overhead_device_ms": {m: float(np.mean(rec[m]["ms"]) - np.mean(rec["plain"]["ms"])) for m in MODES[1:]},
        "per_plan_latency_ms": {m: dist(v) for m, v in lat_all.items()},
        "latency_over_batch_wall": {m: dist(v) for m, v in lat_over_batch.items()},
        "latency_after_plan_seconds_ms": {m: dist(v) for m, v in after_seconds.items()},
        "plan_seconds_ms": dist(seconds_all),
    }
    if not args.no_profile:
        s.upload_prepared(prepared[0])
        try:
            out["harvest_kernel_share"] = harvest_share(s)
        except Exception as ex:
            out["harvest_kernel_share"] = {"error": repr(ex)}
    s.close()
    txt = json.dumps(out, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
