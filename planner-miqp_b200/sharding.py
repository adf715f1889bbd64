"""Scenario sharding across the GPUs of one box (SURVEY.md section 8(e).1).

Plans are independent units: plan s of a batch goes to rank s mod world.  There is no collective
on the data path; the per-plan results (status, objective, gap, solution vector) are gathered on
every rank at the end with one all_gather_object over the process group (NCCL ranks use a gloo
side group for Python objects; on CPU test boxes the group is gloo).  One process per GPU,
launched by torchrun (RANK / LOCAL_RANK / WORLD_SIZE / MASTER_* from the environment).
"""
from __future__ import annotations

import dataclasses
import os
import time
from typing import Callable, Sequence

from .capi import MiqpB200Error, _DevView


def shard_indices(count: int, rank: int, world: int) -> list[int]:
    """indices of the plans rank `rank` solves: s mod world == rank (round robin balances the
    mix of cheap and expensive scenarios better than contiguous blocks)"""
    return list(range(rank, count, world))


def default_solve_fn(gap_tol=None, time_limit=None):
    """solves a shard on this rank's GPU (LOCAL_RANK) through the C ABI; no CPU fallback"""
    from .capi import Solver
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    solver = Solver(device=dev)

    def fn(plans):
        if not plans:
            return [], []
        return solver.solve_batch(plans, gap_tol=gap_tol, time_limit=time_limit)
    return fn


def solve_sharded(problems: Sequence, solve_fn: Callable, group=None):
    """Every rank passes the same `problems`; returns (xs, infos) for ALL plans on every rank,
    in the order of `problems`."""
    import torch.distributed as dist
    if not dist.is_initialized():
        return solve_fn(list(problems))
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    mine = shard_indices(len(problems), rank, world)
    xs, infos = solve_fn([problems[k] for k in mine])
    payload = [(k, x, i) for k, x, i in zip(mine, xs, infos)]
    gathered = [None] * world
    dist.all_gather_object(gathered, payload, group=group)
    out_x, out_i = [None] * len(problems), [None] * len(problems)
    for part in gathered:
        for k, x, i in part:
            out_x[k], out_i[k] = x, i
    return out_x, out_i


# ---------------------------------------------------------------------------------------------------------------------
# Frontier sharding (SURVEY.md section 8(e).2): ONE plan (or a few), its open nodes distributed over the ranks
# ---------------------------------------------------------------------------------------------------------------------
def solve_frontier_sharded(solver, problems: Sequence, gap_tol=None, time_limit=None, warm=None, group=None,
                           ramp_rounds: int = 6, exchange_every: int = 4, stats: dict | None = None, merge_pool: bool = False):
    """Every rank passes the same `problems` and its own solver (one GPU each); returns (xs, infos) of ALL plans on every
    rank.  Each plan's branch-and-bound frontier is sharded over the ranks:

      1. every rank uploads the batch and runs the same `ramp_rounds` rounds (the search is deterministic, the open lists are
         identical; their fingerprints are compared with a min / max all-reduce and the split is skipped if they differ);
      2. frontier_split: rank r keeps the open nodes whose uid hashes to r -- subtree roots dealt by hash, nothing is sent;
      3. loop: `exchange_every` rounds, then ONE min-all-reduce of the incumbent objectives (8 bytes per plan; in place on the
         solver's device array over NCCL, through host buffers on gloo) and a sum-all-reduce of the unfinished-plan counts;
      4. results: best bound = min over ranks, incumbent = the best rank's vector (one sum-all-reduce of the masked vectors,
         i.e. the broadcast of the winner of every plan in a single collective).

    Node order depends on the rank count (like CPLEX's opportunistic mode); bounds stay valid: every open node lives on
    exactly one rank and pruned bounds are kept per rank.

    merge_pool (solution pool on at upload, world > 1): after the search every rank exports its pool, the exports are
    all-gathered (NCCL: straight from the device buffers; gloo: through the host) in rank order and merged, so that
    solver.pool(k) on every rank returns the same pool, that of the union of all ranks' leaves.  stats gains pool_bytes
    (one rank's export) and pool_merge_ms.  Nothing else of the result changes.
    """
    import numpy as np
    import torch
    import torch.distributed as dist

    sharded = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    rank = dist.get_rank(group) if sharded else 0
    world = dist.get_world_size(group) if sharded else 1
    on_nccl = sharded and dist.get_backend(group) == "nccl"
    dev = torch.device("cuda", torch.cuda.current_device()) if on_nccl else torch.device("cpu")

    def allreduce(arr, op):
        t = torch.from_numpy(np.array(arr, copy=True)).to(dev)      # (a copy: the caller keeps its array)
        dist.all_reduce(t, op=op, group=group)
        return t.cpu().numpy()

    n = len(problems)
    solver.upload(problems, gap_tol=gap_tol, time_limit=time_limit, warm=warm)
    solver.frontier_start()
    left = solver.frontier_rounds(ramp_rounds if sharded else -1)
    exchanges, split_done = 0, False
    if sharded:
        fp = solver.frontier_fingerprint()
        same = bool((allreduce(fp, dist.ReduceOp.MIN) == allreduce(fp, dist.ReduceOp.MAX)).all())
        if same:
            solver.frontier_split(rank, world)
            split_done = True
        ub_t = None
        if on_nccl:
            ptr, cnt = solver.frontier_ub_device()
            ub_t = torch.as_tensor(_DevView(ptr, cnt), device=dev)
        total_left = int(allreduce(np.array([left], dtype=np.int64), dist.ReduceOp.SUM)[0])
        while total_left > 0:
            left = solver.frontier_rounds(exchange_every) if left > 0 else 0
            if on_nccl:     # in place on the solver's incumbent objectives: no host copy
                dist.all_reduce(ub_t, op=dist.ReduceOp.MIN, group=group)
                torch.cuda.synchronize()
            else:
                solver.frontier_tighten(allreduce(solver.frontier_get_ub(), dist.ReduceOp.MIN))
            exchanges += 1
            total_left = int(allreduce(np.array([left], dtype=np.int64), dist.ReduceOp.SUM)[0])
    ms = solver.frontier_finish()
    xs, infos = solver.fetch()
    if stats is not None:
        stats.update(device_ms=ms, exchanges=exchanges, split=split_done, world=world, nodes_this_rank=sum(i.nodes for i in infos))
    if not sharded:
        return xs, infos

    if merge_pool:
        _merge_pools(solver, group, world, dev, on_nccl, allreduce, stats)

    # -- combine: objective and winner per plan, best bound, node counts
    big = 1e300
    own = np.array([i.objective if i.status == 0 else big for i in infos])
    best = allreduce(own, dist.ReduceOp.MIN)
    cand = np.where(own <= best, rank, world).astype(np.int64)
    winner = allreduce(cand, dist.ReduceOp.MIN)                       # lowest rank among the best
    bound = allreduce(np.array([i.best_bound if np.isfinite(i.best_bound) else big for i in infos]), dist.ReduceOp.MIN)
    counts = allreduce(np.array([[i.nodes, i.qp_iters, i.uncertified, i.pool_exhausted] for i in infos], dtype=np.int64).reshape(-1),
                       dist.ReduceOp.SUM).reshape(n, 4)
    viol = allreduce(np.array([i.max_violation if (i.status == 0 and winner[k] == rank) else 0.0 for k, i in enumerate(infos)]),
                     dist.ReduceOp.MAX)
    flat = np.concatenate([x if winner[k] == rank else np.zeros_like(x) for k, x in enumerate(xs)]) if n else np.zeros(0)
    flat = allreduce(flat, dist.ReduceOp.SUM)                         # "broadcast" of every plan's winning vector
    timed_out = allreduce(np.array([1 if i.status == 3 else 0 for i in infos], dtype=np.int64), dist.ReduceOp.MAX)
    out_x, out_i, off = [], [], 0
    for k, i in enumerate(infos):
        m = len(xs[k])
        out_x.append(flat[off:off + m].copy())
        off += m
        have = best[k] < big
        gtol = problems[k].scal["relative_mip_gap_tolerance"] if gap_tol is None else gap_tol
        lb = min(bound[k], best[k]) if have else bound[k]
        gap = abs(lb - best[k]) / (1e-10 + abs(best[k])) if have else float("nan")
        out_i.append(dataclasses.replace(i, status=0 if have else (3 if timed_out[k] else i.status),
                                objective=float(best[k]) if have else float("nan"), best_bound=float(lb), gap=float(gap),
                                proven=bool(have and gap <= gtol + 1e-15), nodes=int(counts[k, 0]), qp_iters=int(counts[k, 1]),
                                uncertified=int(counts[k, 2]), pool_exhausted=int(counts[k, 3] > 0),
                                max_violation=float(viol[k]) if have else float("nan")))
    return out_x, out_i


def _merge_pools(solver, group, world, dev, on_nccl, allreduce, stats):
    """every rank's pool export, all-gathered in rank order, merged on every rank (solve_frontier_sharded(merge_pool=True))"""
    import numpy as np
    import torch
    import torch.distributed as dist
    try:
        exp, err = solver.pool_export(), None
    except MiqpB200Error as ex:            # (pool off at upload) every rank learns of it before any rank raises
        exp, err = None, ex
    nbytes = 0 if exp is None else int(exp.numel())
    hi, neg_lo = allreduce(np.array([nbytes, -nbytes], dtype=np.int64), dist.ReduceOp.MAX)
    if err is not None:
        raise err
    if hi != -neg_lo or hi == 0:
        raise MiqpB200Error("solve_frontier_sharded(merge_pool=True): the solution pool was off or differs between the ranks "
                            "(set the same capacity on every rank before the upload)")
    if on_nccl:
        gathered = torch.empty(world * nbytes, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(gathered, exp, group=group)
        torch.cuda.synchronize()
    else:
        mine = exp.cpu()
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine, group=group)
        gathered = torch.cat(parts)
    t0 = time.perf_counter()
    solver.pool_merge(gathered, world)
    if stats is not None:
        stats.update(pool_bytes=nbytes, pool_merge_ms=1e3 * (time.perf_counter() - t0))
