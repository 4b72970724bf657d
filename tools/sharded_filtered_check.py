"""Filtered ShardedFlatIP.search / range_search: parity with one GPU's filtered search over the full matrix, and the
time of the parts.

Rows and queries are those of tools/sharded_range_check.py (the CLIP-like mixture, generated on the device block by
block from a seed).  Cells: 100 M x 512 and 10 M x 768 rows; nq in {1, 16, 128}; k = 100.  Selections of global ids:
contiguous 0.1 / 1 / 10 / 100 % (starting a third of the way in, not tile-aligned), random 1 %, and 1 % centred on
the boundary between ranks 0 and 1.  The range search of a cell uses radius = the median over the queries of the
100th-best filtered score, so about 100 hits per query.

Under torchrun (one rank per GPU, NCCL, static partition) every rank holds its block of rows and the tool times, per
cell, with the slowest rank's number:
  local_ms     the rank's filtered search_keys_tensor (CUDA events) / range_search_keys_tensor (host clock, its sizing
               read-back included);
  total_ms     ShardedFlatIP.search / range_search with params, end to end (host clock);
  exchange_merge_ms  total - local;
  n1_ms        rank 0's filtered search over the full matrix, which it also holds for the parity check.
Every rank's result must equal rank 0's full-matrix filtered search bit for bit (D and I; lims, D and I).

Without torchrun (one GPU) the ranks are windows of one index holding the full matrix, for --worlds (default 2, 8):
each window runs the filtered key calls under its window in turn (local_ms is the slowest window), the keys are
stacked as the exchange would leave them and merged (merge_ms, CUDA events); the exchange is not measured.  The merged
result must equal the full-matrix filtered search bit for bit.  Each window's selected row tiles and their bytes
(tiles x 128 x dpad x 2) are reported with the rate local_ms gives them.

    torchrun --nproc-per-node 8 tools/sharded_filtered_check.py [--cells 100M,10M] [--nq 1,16,128] [--runs 5]
    python tools/sharded_filtered_check.py [--worlds 2,8] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from sharded_range_check import (CELLS, add_rows, event_ms, host_ms, power_limit, rows_block, same,  # noqa: E402
                                 stacked)

K = 100


def selections(n, boundary):
    """name -> selector of global ids in [0, n)."""
    import ivr_b200
    rng = np.random.default_rng(n)
    out = {}
    for name, frac in (("contig 0.1%", 0.001), ("contig 1%", 0.01), ("contig 10%", 0.1), ("contig 100%", 1.0)):
        a = min(n // 3 + 37, n - int(n * frac)) if frac < 1.0 else 0
        out[name] = ivr_b200.IDSelectorRange(a, a + int(n * frac))
    out["random 1%"] = ivr_b200.IDSelectorBatch(rng.choice(n, n // 100, replace=False))
    out["1% across a boundary"] = ivr_b200.IDSelectorRange(boundary - n // 200, boundary + n // 200)
    return out


def tiles_in(mask, lo, hi):
    """Row tiles of the stored rows [lo, hi) that hold a selected row (the windows are cut the same way)."""
    m = mask[lo:hi]
    a = (-lo) % 128                                             # rows of the partial first tile
    head = int(m[:a].any()) if a else 0
    body = m[a:]
    full = body[:body.size // 128 * 128].reshape(-1, 128).any(axis=1).sum()
    tail = int(body[body.size // 128 * 128:].any())
    return int(head + full + tail)


def one_gpu(args, torch):
    import ivr_b200
    from ivr_b200.sharded import _cuda_merge, _cuda_range_merge, partition_rows
    results, ok = [], True
    worlds = [int(v) for v in args.worlds.split(",")]
    merge = _cuda_merge(0)
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        dpad = (d + 63) // 64 * 64
        full = ivr_b200.IndexFlatIP(d, device=0)
        full.reserve(n)
        add_rows(full.add_tensor, 0, n, n, d, torch)
        qall = rows_block(0, 128, d, torch, seed=100 + d)
        for name, sel in selections(n, int(partition_rows(n, 2)[1])).items():
            p = ivr_b200.SearchParameters(sel=sel)
            mask = sel._mask(n)
            for nq in (int(v) for v in args.nq.split(",")):
                q = qall[:nq].contiguous()
                want = full.search_tensor(q, K, params=p)
                radius = float(want[0][:, K - 1].median())
                want_r = full.range_search_tensor(q, radius, params=p)
                row = {"rows": n, "dim": d, "selection": name, "selected": int(mask.sum()), "nq": nq, "k": K,
                       "radius": radius, "range_hits": int(want_r[0][-1]),
                       "n1_topk_ms": event_ms(lambda: full.search_tensor(q, K, params=p), args.runs, torch),
                       "n1_range_ms": host_ms(lambda: full.range_search_tensor(q, radius, params=p), args.runs, torch),
                       **args.dev}
                for world in worlds:
                    off = partition_rows(n, world)
                    keys, runs, t_top, t_rng, tiles = [], [], [], [], []
                    for r in range(world):
                        full.set_window(int(off[r]), int(off[r + 1] - off[r]))
                        keys.append(full.search_keys_tensor(q, K, params=p))
                        runs.append(full.range_search_keys_tensor(q, radius, params=p))
                        t_top.append(event_ms(lambda: full.search_keys_tensor(q, K, params=p), args.runs, torch))
                        t_rng.append(host_ms(lambda: full.range_search_keys_tensor(q, radius, params=p), args.runs,
                                             torch))
                        tiles.append(tiles_in(mask, int(off[r]), int(off[r + 1])))
                    full.set_window()
                    parts = torch.stack(keys)
                    got = merge(parts, K)
                    rk, rl, total = stacked(runs, torch)
                    got_r = _cuda_range_merge(rk, rl, total)
                    good = same(got, want, torch) and same(got_r, want_r, torch)
                    ok = ok and good
                    slow = int(np.argmax(t_top))
                    gb = tiles[slow] * 128 * dpad * 2 / 1e9
                    row[f"n{world}"] = {
                        "local_topk_ms": max(t_top), "local_range_ms": max(t_rng),
                        "merge_topk_ms": event_ms(lambda: merge(parts, K), args.runs, torch),
                        "merge_range_ms": event_ms(lambda: _cuda_range_merge(rk, rl, total), args.runs, torch),
                        "tiles_per_window": tiles, "slowest_window_GB": gb,
                        "slowest_window_GBps": gb / (max(t_top) / 1e3) if max(t_top) > 0 else None,
                        "exchange_ms": "not measured (one GPU)", "equal_to_n1": good}
                results.append(row)
                print(json.dumps(row), flush=True)
            sel.close()
        full.close()
        torch.cuda.empty_cache()
    return results, ok


def distributed(args, torch):
    import torch.distributed as dist
    import ivr_b200
    from ivr_b200.sharded import partition_rows
    rank, world = dist.get_rank(), dist.get_world_size()
    results, ok = [], True

    def slowest(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()

    def bcast(want, like):
        """rank 0's tensors `want` on every rank (`like`: tensors of the same dtypes)."""
        shapes = [[list(t.shape) for t in want] if rank == 0 else None]
        dist.broadcast_object_list(shapes, 0)
        ref = [want[i] if rank == 0 else torch.empty(shapes[0][i], dtype=t.dtype, device="cuda")
               for i, t in enumerate(like)]
        for t in ref:
            dist.broadcast(t, 0)
        return ref

    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        off = partition_rows(n, world)
        lo, hi = int(off[rank]), int(off[rank + 1])
        sh = ivr_b200.ShardedFlatIP(d, device=torch.cuda.current_device())
        sh.local.reserve(hi - lo)
        add_rows(lambda x: sh.add_local(x, lo, n), lo, hi, n, d, torch)
        full = None
        if rank == 0:
            full = ivr_b200.IndexFlatIP(d, device=torch.cuda.current_device())
            full.reserve(n)
            add_rows(full.add_tensor, 0, n, n, d, torch)
        qall = rows_block(0, 128, d, torch, seed=100 + d)
        for name, sel in selections(n, int(off[1])).items():
            p = ivr_b200.SearchParameters(sel=sel)
            lp = ivr_b200.SearchParameters(sel=sel.shard(n, lo))
            for nq in (int(v) for v in args.nq.split(",")):
                q = qall[:nq].contiguous()
                got = sh.search(q, K, params=p)
                radius = torch.tensor([float(got[0][:, K - 1].median())], device="cuda")
                dist.broadcast(radius, 0)
                radius = float(radius.item())
                got_r = sh.range_search(q, radius, params=p)
                local = slowest(event_ms(lambda: sh.local.search_keys_tensor(q, K, id_offset=lo, params=lp),
                                         args.runs, torch))
                local_r = slowest(host_ms(lambda: sh.local.range_search_keys_tensor(q, radius, id_offset=lo,
                                                                                    params=lp),
                                          args.runs, torch, sync=barrier))
                total = slowest(host_ms(lambda: sh.search(q, K, params=p), args.runs, torch, sync=barrier))
                total_r = slowest(host_ms(lambda: sh.range_search(q, radius, params=p), args.runs, torch,
                                          sync=barrier))
                n1 = n1_r = -1.0
                want = want_r = got
                if rank == 0:
                    want = full.search_tensor(q, K, params=p)
                    want_r = full.range_search_tensor(q, radius, params=p)
                    n1 = event_ms(lambda: full.search_tensor(q, K, params=p), args.runs, torch)
                    n1_r = host_ms(lambda: full.range_search_tensor(q, radius, params=p), args.runs, torch)
                want = bcast(list(want), list(got))
                want_r = bcast(list(want_r), list(got_r))
                good = torch.tensor([int(same(got, want, torch) and same(got_r, want_r, torch))], device="cuda")
                dist.all_reduce(good, op=dist.ReduceOp.MIN)
                ok = ok and bool(good.item())
                if rank == 0:
                    row = {"world": world, "rows": n, "dim": d, "selection": name, "nq": nq, "k": K,
                           "radius": radius, "range_hits": int(got_r[0][-1]),
                           "local_topk_ms": local, "total_topk_ms": total, "exchange_merge_topk_ms": total - local,
                           "local_range_ms": local_r, "total_range_ms": total_r,
                           "exchange_merge_range_ms": total_r - local_r, "n1_topk_ms": n1, "n1_range_ms": n1_r,
                           "equal_to_n1_on_every_rank": bool(good.item()), **args.dev}
                    results.append(row)
                    print(json.dumps(row), flush=True)
            sel.close()
        if full is not None:
            full.close()
        sh.close()
        sh.local.close()
        torch.cuda.empty_cache()
    return results, ok


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--cells", default="100M,10M")
    ap.add_argument("--nq", default="1,16,128")
    ap.add_argument("--worlds", default="2,8", help="ranks simulated as row windows without torchrun")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for sharded_filtered_check.json (rank 0)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_filtered_check needs a CUDA device")
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        lr = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(lr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
        args.dev = {"gpu": torch.cuda.get_device_name(lr), "power_limit": power_limit()}
        results, ok = distributed(args, torch)
        rank = dist.get_rank()
        dist.destroy_process_group()
    else:
        args.dev = {"gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
        results, ok = one_gpu(args, torch)
        rank = 0
    if rank == 0:
        print(json.dumps(args.dev), flush=True)
        if args.out:
            os.makedirs(args.out, exist_ok=True)
            with open(os.path.join(args.out, "sharded_filtered_check.json"), "w") as f:
                json.dump(results, f, indent=1)
        print(f"sharded_filtered_check: every result equal to the full-matrix filtered search: {ok}", flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
