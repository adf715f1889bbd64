"""Cost of merging the solution pools of a frontier-sharded search (miqp_b200_pool_export / miqp_b200_pool_merge).

Two shapes:
  * config 5: one joint plan (intersection, 8 cars, N = 40, R = 64), pool capacities 16 and 64;
  * config 2: 2048 plans (obstacle_scenario seeds 0..2047, N = 40, R = 32), pool capacity 8;
each for world 2, 4 and 8.  On one GPU a world of W ranks is emulated: W sequential searches of the uploaded batch with
frontier_split(r, W) after the ramp-up (no incumbent exchange), their exports concatenated in rank order.  Recorded per case:
the export size (bytes of one rank, from the shapes: header + records + decisions + z), the entries the ranks' pools hold, the
merge time with CUDA events on the solver's stream (median of --reps merges of the same gathered buffer, after one warm-up
merge; the buffer stays on the device) and the host time of the call.  With at least W GPUs visible the NCCL all-gather of
W exports of that size is timed too (CUDA events, median of --reps); otherwise it is recorded as not measured.

usage: python tools/pool_merge_cost.py OUT_DIR [--reps 20] [--config5-time-limit 2.0]
Writes OUT_DIR/pool_merge_cost.json with the GPU's name and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
WORLDS = (2, 4, 8)


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [f.strip() for f in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def _allgather_worker(rank, world, port, nbytes, reps, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    src = torch.full((nbytes,), rank, dtype=torch.uint8, device="cuda")
    out = torch.empty(world * nbytes, dtype=torch.uint8, device="cuda")
    ms = []
    for r in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        a.record()
        dist.all_gather_into_tensor(out, src)
        b.record()
        torch.cuda.synchronize()
        if r > 0:
            ms.append(a.elapsed_time(b))
    if rank == 0:
        q.put(float(np.median(ms)))
    dist.destroy_process_group()


def allgather_ms(world, nbytes, reps):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        return None
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 41500 + (os.getpid() % 1000) + world
    procs = [ctx.Process(target=_allgather_worker, args=(r, world, port, nbytes, reps, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
    return res


def measure(name, plans, cap, time_limit, reps):
    import torch
    import planner_miqp_b200 as P
    s = P.Solver(solution_pool=cap)
    s.upload(plans, gap_tol=1e-4, time_limit=time_limit)
    p0 = plans[0]
    pairs = p0.C * (p0.C - 1) // 2
    out = []
    for world in WORLDS:
        exports, entries = [], []
        for r in range(world):
            s.frontier_start()
            s.frontier_rounds(6)
            s.frontier_split(r, world)
            s.frontier_rounds(-1)
            s.frontier_finish()
            entries.append(int(s.pool_sizes().sum()))
            exports.append(s.pool_export().clone())
        gathered = torch.cat(exports)
        del exports
        s.pool_merge(gathered, world)                     # warm-up
        dev_ms, host_ms = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            s.mark(0)
            s.pool_merge(gathered, world)
            s.mark(1)
            host_ms.append(1e3 * (time.perf_counter() - t0))
            dev_ms.append(s.elapsed_to(s))
        nbytes = gathered.numel() // world
        ag = allgather_ms(world, nbytes, reps)
        rec = dict(shape=name, plans=len(plans), pool_capacity=cap, world=world, export_bytes=nbytes,
                   gathered_bytes=int(gathered.numel()),
                   z_bytes_per_entry=8 * (p0.C * p0.N * 8 + 4 * pairs * p0.N),
                   pool_entries_per_rank=entries, merged_entries=int(s.pool_sizes().sum()),
                   merge_ms_cuda_events_median=float(np.median(dev_ms)), merge_ms_cuda_events_min=float(np.min(dev_ms)),
                   merge_ms_host_median=float(np.median(host_ms)),
                   allgather_ms_nccl_median=ag if ag is not None else "not measured: fewer than %d GPUs visible" % world)
        print(json.dumps(rec), flush=True)
        out.append(rec)
        del gathered
    s.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--config5-time-limit", type=float, default=2.0)
    a = ap.parse_args()
    from planner_miqp_b200.scenarios import intersection, obstacle_scenario
    import torch
    res = dict(gpu_info(), gpus_visible=torch.cuda.device_count(), reps=a.reps,
               emulation="world W on one GPU: W sequential searches with frontier_split(r, W) after 6 ramp-up rounds, "
                         "no incumbent exchange, exports concatenated in rank order",
               config5_time_limit_s=a.config5_time_limit, cases=[])
    c5 = [intersection(0, n_cars=8, nr_steps=40).build()]
    for cap in (16, 64):
        res["cases"] += measure("config5: intersection, 8 cars, N=40, R=64", c5, cap, a.config5_time_limit, a.reps)
    c2 = [obstacle_scenario(k).build() for k in range(2048)]
    res["cases"] += measure("config2: obstacle_scenario seeds 0..2047, N=40, R=32", c2, 8, 60.0, a.reps)
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "pool_merge_cost.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
