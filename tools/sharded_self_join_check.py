"""ShardedFlatIP.range_self_join: parity with one GPU's self-join over the full matrix, and the time of its parts.

Cells: 1 M x 512 and 851 284 x 768 rows of the CLIP-like mixture of tools/range_search_timing.py, generated on the
device from a seed; two radii per cell, those of tools/range_self_join_timing.py: the median over 256 sampled rows of
the 10th- and of the 100th-best score to another row.

Under torchrun (one rank per GPU, NCCL) every rank builds the full matrix, keeps its block in a ShardedFlatIP and times,
per cell and radius:
  total_ms     ShardedFlatIP.range_self_join end to end (host clock around a device synchronise, max over ranks);
  local_ms     the rank's tasks of join_schedule on an index of the full matrix: the self-join keys of its window and
               its cross joins against the other rows, taken from the same index (no exchange; max over ranks);
  merge_ms     the merge of the rank's runs (max over ranks);
  exchange_ms  total - local - merge: the row and hit exchanges, the agreement all-gathers and the allocation checks.
Every rank's (lims, D, I) must equal the rows of rank 0's single-GPU join bit for bit (gathered with gather=True).

Without torchrun (one GPU) the ranks are windows of one index for --worlds (default 2, 8): after one warm-up pass over
every rank's tasks, each rank's tasks are timed in turn, --runs times (host clock around a device synchronise per task;
the medians are reported, per rank and per task with its operand order: other_is_lower).  The tool reports every
rank's time, their sum against the single-GPU join with the exact capacity (CUDA events, median of --runs; sharding
should add no work: within 10 %) and the slowest rank against the mean (within 15 %).  The merged result must equal
the single-GPU join bit for bit.  Both modes print the card's name and power limit.

    torchrun --nproc-per-node 8 tools/sharded_self_join_check.py [--cells 1M,851k] [--neighbours 10,100] [--runs 3]
    python tools/sharded_self_join_check.py [--worlds 2,8] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from range_search_timing import clip_like_dev, power_limit  # noqa: E402

CELLS = {"1M": (1_000_000, 512), "851k": (851_284, 768)}


def radii(X16, ks, torch):
    n = X16.shape[0]
    sample = torch.from_numpy(np.random.default_rng(0).choice(n, 256, replace=False)).cuda()
    s = X16[sample].float() @ X16.float().T
    s[torch.arange(256, device="cuda"), sample] = -math.inf
    best = torch.topk(s, max(ks), dim=1).values
    return {k: float(best[:, k - 1].median()) for k in ks}


def rank_tasks(idx, bounds, r, radius, times=None):
    """Rank r's tasks of join_schedule on `idx` (all rows, ids = stored rows): (runs over r's rows, runs over other
    ranks' rows as (peer, a, b, lims, keys)).  `times`: a list that receives (task, other_is_lower, ms) per task,
    host clock around a device synchronise."""
    import torch
    from ivr_b200.sharded import join_schedule
    tasks = join_schedule(bounds, r)
    lo, hi = tasks[0][:2]
    idx.set_window(lo, hi - lo)
    (L, K), ms = clock(lambda: idx.range_self_join_keys_tensor(radius), torch)
    mine, theirs = [(lo, hi, L, K)], []
    if times is not None:
        times.append(("diagonal", False, ms))
    for t, (a, b, p, c, d) in enumerate(tasks[1:], 1):
        def cross():
            other = idx.rows_f16_tensor(c, d - c)
            idx.set_window(a, b - a)
            return idx.range_cross_join_keys_tensor(other, c, radius, c < a)
        (ls, ks, lo_, ko), ms = clock(cross, torch)
        mine.append((a, b, ls, ks))
        theirs.append((p, c, d, lo_, ko))
        if times is not None:
            times.append((f"cross {t} (peer {p})", c < a, ms))
    idx.set_window()
    return mine, theirs


def merge(parts, lo, hi, torch):
    from ivr_b200.sharded import ShardedFlatIP, _cuda_range_merge
    return ShardedFlatIP._merge_runs(types.SimpleNamespace(_range_merge=_cuda_range_merge), parts, lo, hi,
                                     torch.device("cuda", torch.cuda.current_device()))


def clock(fn, torch):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, 1e3 * (time.perf_counter() - t)


def same(a, b, torch):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def exact_join(idx, radius, runs, torch):
    """The single-GPU join with the exact capacity (as tools/range_self_join_timing.py times it): its result and the
    median of `runs` CUDA-event-timed calls after one warm-up call."""
    from ivr_b200 import _native as nat
    from range_search_timing import timed
    ref = idx.range_self_join_tensor(radius)
    n, cap = idx.ntotal, max(int(ref[0][-1]), 1)
    L = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    D = torch.empty(cap, device="cuda")
    I = torch.empty(cap, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def join():
        nat.check(nat.lib.ivr_index_range_self_join_device(idx._handle(), radius, cap, L.data_ptr(), D.data_ptr(),
                                                           I.data_ptr(), st))
    ms = timed(join, runs, torch)
    del L, D, I
    return ref, ms


def single_gpu(args, torch, ivr_b200, dev):
    from ivr_b200.sharded import partition_rows
    results = []
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        X = torch.cat(list(clip_like_dev(n, d, seed=1, torch=torch)))
        idx = ivr_b200.IndexFlatIP(d, device=0)
        idx.add_tensor(X)
        rads = radii(X.half(), [int(v) for v in args.neighbours.split(",")], torch)
        del X
        for k, radius in rads.items():
            ref, n1_ms = exact_join(idx, radius, args.runs, torch)
            for world in (int(v) for v in args.worlds.split(",")):
                bounds = partition_rows(n, world)
                for r in range(world):                                 # warm-up: every rank's tasks once
                    rank_tasks(idx, bounds, r, radius)
                torch.cuda.empty_cache()
                samples = [[] for _ in range(world)]                   # [rank][run] = [(task, lower, ms)]
                for run in range(args.runs):
                    for r in range(world):
                        t = []
                        rank_tasks(idx, bounds, r, radius, t)
                        samples[r].append(t)
                rank_ms = [float(np.median([sum(ms for _, _, ms in t) for t in samples[r]])) for r in range(world)]
                tasks = [[(name, lower, float(np.median([t[i][2] for t in samples[r]])))
                          for i, (name, lower, _) in enumerate(samples[r][0])] for r in range(world)]
                parts = [[] for _ in range(world)]
                for r in range(world):
                    mine, theirs = rank_tasks(idx, bounds, r, radius)
                    parts[r] += mine
                    for p, a, b, L, K in theirs:
                        parts[p].append((a, b, L, K))
                ok = True
                for r in range(world):
                    lo, hi = int(bounds[r]), int(bounds[r + 1])
                    L, D, I = merge(parts[r], lo, hi, torch)
                    a, b = int(ref[0][lo]), int(ref[0][hi])
                    ok = ok and same((L, D, I), (ref[0][lo:hi + 1] - a, ref[1][a:b], ref[2][a:b]), torch)
                del parts
                torch.cuda.empty_cache()
                res = {"mode": "one_gpu", "rows": n, "dim": d, "neighbours": k, "radius": radius, "world": world,
                       "hits": int(ref[0][-1]), "runs": args.runs, "n1_ms": n1_ms, "rank_ms": rank_ms,
                       "sum_over_n1": sum(rank_ms) / n1_ms, "slowest_over_mean": max(rank_ms) / (sum(rank_ms) / world),
                       "rank_tasks_ms": tasks, "parity": ok, **dev}
                results.append(res)
                print(json.dumps(res), flush=True)
            del ref
        idx.close()
        torch.cuda.empty_cache()
    return results


def distributed(args, torch, ivr_b200, dev):
    import torch.distributed as dist
    from ivr_b200.sharded import ShardedFlatIP, partition_rows
    rank, world = dist.get_rank(), dist.get_world_size()
    results = []
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        X = torch.cat(list(clip_like_dev(n, d, seed=1, torch=torch)))
        full = ivr_b200.IndexFlatIP(d, device=torch.cuda.current_device())
        full.add_tensor(X)
        sh = ShardedFlatIP(d, device=torch.cuda.current_device())
        sh.add_global(X)
        bounds = partition_rows(n, world)
        rads = radii(X.half(), [int(v) for v in args.neighbours.split(",")], torch)
        del X
        for k, radius in rads.items():
            sh.range_self_join(radius)                                 # warm-up
            tot, loc, mrg = [], [], []
            for _ in range(args.runs):
                dist.barrier()
                got, ms = clock(lambda: sh.range_self_join(radius), torch)
                tot.append(ms)
                (mine, _), ms = clock(lambda: rank_tasks(full, bounds, rank, radius), torch)
                loc.append(ms)
                _, ms = clock(lambda: merge(mine, int(bounds[rank]), int(bounds[rank + 1]), torch), torch)
                mrg.append(ms)
                del mine
            mine = torch.tensor([np.median(tot), np.median(loc), np.median(mrg)], dtype=torch.float64, device="cuda")
            dist.all_reduce(mine, op=dist.ReduceOp.MAX)
            allg = sh.range_self_join(radius, gather=True)
            ok = torch.tensor([1], device="cuda")
            if rank == 0:
                ref = full.range_self_join_tensor(radius)
                ok[0] = int(same(allg, ref, torch))
                del ref
            dist.broadcast(ok, 0)
            lo, hi = int(bounds[rank]), int(bounds[rank + 1])
            a, b = int(allg[0][lo]), int(allg[0][hi])
            flag = torch.tensor([int(same(got, (allg[0][lo:hi + 1] - a, allg[1][a:b], allg[2][a:b]), torch))],
                                device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            t, l, m = (float(v) for v in mine.cpu())
            res = {"mode": "torchrun", "world": world, "rows": n, "dim": d, "neighbours": k, "radius": radius,
                   "hits": int(allg[0][-1]), "total_ms": t, "local_ms": l, "merge_ms": m, "exchange_ms": t - l - m,
                   "parity": bool(ok.item()) and bool(flag.item()), **dev}
            del allg, got
            torch.cuda.empty_cache()
            if rank == 0:
                results.append(res)
                print(json.dumps(res), flush=True)
        full.close()
        sh.close()
        torch.cuda.empty_cache()
    return results


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--cells", default="1M,851k")
    ap.add_argument("--neighbours", default="10,100")
    ap.add_argument("--worlds", default="2,8")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for sharded_self_join_check.json")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_self_join_check needs a CUDA device")
    import ivr_b200
    dev = {"gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    print(json.dumps(dev), flush=True)
    if "RANK" in os.environ:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
        try:
            results = distributed(args, torch, ivr_b200, dev)
        finally:
            dist.destroy_process_group()
        if int(os.environ["RANK"]) != 0:
            return
    else:
        results = single_gpu(args, torch, ivr_b200, dev)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "sharded_self_join_check.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
