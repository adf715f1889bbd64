"""Cost and contents of the solution pool on the flagship workload: config 2 (obstacle_scenario, N = 40, R = 32), shard 0
(seeds 0 .. B-1), one resident batch.

  * device time of batch_run with the pool off and on, alternated over --reps repetitions (CUDA events of the solver);
  * time of pool_fetch with vectors (full column vectors + trajectories + device evaluation) over every plan of the batch;
  * the pool-size histogram.

usage: python tools/pool_stats.py OUT_DIR [--batch 2048] [--capacity 8] [--reps 5]
Writes OUT_DIR/pool_stats.json with the GPU's name and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [f.strip() for f in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--capacity", type=int, default=8)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import planner_miqp_b200 as P
    from planner_miqp_b200.scenarios import obstacle_scenario
    plans = [obstacle_scenario(k).build() for k in range(a.batch)]
    off, on = P.Solver(), P.Solver(solution_pool=a.capacity)
    for s in (off, on):
        s.upload(plans, gap_tol=1e-4, time_limit=60)
        s.run()                                            # warm-up (module load, first touch of the pools)
    ms = {"off": [], "on": []}
    for _ in range(a.reps):
        ms["off"].append(off.run())
        ms["on"].append(on.run())
    _, info_off = off.fetch()
    _, info_on = on.fetch()
    same = all(x.objective == y.objective or (np.isnan(x.objective) and np.isnan(y.objective)) for x, y in zip(info_off, info_on))
    sizes = on.pool_sizes()
    t0 = time.perf_counter()
    entries = sum(len(on.pool(k, vectors=True, max_entries=a.capacity)) for k in range(a.batch))
    fetch_s = time.perf_counter() - t0
    res = dict(gpu_info(), workload="config2 shard 0 (obstacle_scenario seeds 0..%d), N=40, R=32" % (a.batch - 1),
               batch=a.batch, capacity=a.capacity, reps=a.reps,
               batch_run_ms_pool_off=ms["off"], batch_run_ms_pool_on=ms["on"],
               median_ms_off=float(np.median(ms["off"])), median_ms_on=float(np.median(ms["on"])),
               overhead_pct=100.0 * (np.median(ms["on"]) / np.median(ms["off"]) - 1.0),
               objectives_identical=bool(same),
               pool_fetch_with_vectors_ms_per_plan=1e3 * fetch_s / a.batch, pool_entries_fetched=int(entries),
               pool_size_histogram=np.bincount(sizes, minlength=a.capacity + 1).tolist())
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "pool_stats.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    off.close(); on.close()


if __name__ == "__main__":
    main()
