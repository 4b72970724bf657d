"""ShardedFlatIP.range_search: parity with one GPU's range search over the full matrix, and the time of its parts.

Rows and queries are the CLIP-like mixture of tools/range_search_timing.py, generated on the device from a seed, one
block of 2^20 rows at a time (block b has its own seed, so a rank generates just its own rows).  Cells: 100 M x 512
and 10 M x 768 rows, nq in {1, 16, 128}, two radii per cell: the median over the first 128 queries of the 100th- and
of the 10 000th-best exact fp32 score (about 100 and 10 k hits per query).

Under torchrun (one rank per GPU, NCCL) every rank holds its block of rows and the tool times, per cell:
  local_ms     the rank's range_search_keys_tensor, sizing read-back included (host clock, max over ranks);
  merge_ms     ivr_range_merge_keys_device on the gathered runs (CUDA events);
  total_ms     ShardedFlatIP.range_search end to end (host clock, max over ranks);
  exchange_ms  total - local - merge: the two all-gathers, the status checks and the allocation all-reduce;
  n1_ms        rank 0's range_search_tensor over the full matrix, which it also holds for the parity check.
Every rank's (lims, D, I) must equal rank 0's full-matrix result bit for bit.

Without torchrun (one GPU) the tool measures the same parts with the ranks as row windows of one index holding the
full matrix, for --worlds (default 2, 8): each window runs range_search_keys_tensor in turn (local_ms is the slowest
window), the runs are stacked as an all-gather would leave them and merged; the exchange is not measured.  The merged
result must equal the full-matrix range search bit for bit.

    torchrun --nproc-per-node 8 tools/sharded_range_check.py [--cells 100M,10M] [--nq 1,16,128] [--runs 10]
    python tools/sharded_range_check.py [--worlds 2,8] [--out DIR]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CELLS = {"100M": (100_000_000, 512), "10M": (10_000_000, 768)}
BLOCK = 1 << 20


def rows_block(b, n, d, torch, seed=1, n_centres=4096, centre_seed=1234, sigma_scale=0.5):
    """Rows [b * BLOCK, min(n, (b + 1) * BLOCK)) of the mixture, float32 on the current device."""
    g = torch.Generator(device="cuda").manual_seed(centre_seed)
    c = torch.randn((n_centres, d), generator=g, device="cuda")
    c = c / c.norm(dim=1, keepdim=True)
    g = torch.Generator(device="cuda").manual_seed(seed * 1_000_003 + b)
    m = min(BLOCK, n - b * BLOCK)
    z = torch.randint(0, n_centres, (m,), generator=g, device="cuda")
    x = c[z] + (sigma_scale / math.sqrt(d)) * torch.randn((m, d), generator=g, device="cuda")
    return x / x.norm(dim=1, keepdim=True)


def add_rows(add, lo, hi, n, d, torch):
    """add(x) of the global rows [lo, hi), block by block."""
    for b in range(lo // BLOCK, (hi + BLOCK - 1) // BLOCK):
        x = rows_block(b, n, d, torch)
        s = b * BLOCK
        add(x[max(lo, s) - s:min(hi, s + x.shape[0]) - s])
    torch.cuda.synchronize()


def radii(q, lo, hi, n, d, torch, targets=(100, 10_000)):
    """Median over the queries of the target-th best exact fp32 score over rows [lo, hi): (per target) the
    [len(q), max target] best scores of this row range, to be merged across ranks by the caller."""
    kmax = max(targets)
    best = None
    for b in range(lo // BLOCK, (hi + BLOCK - 1) // BLOCK):
        x = rows_block(b, n, d, torch)
        s = b * BLOCK
        x = x[max(lo, s) - s:min(hi, s + x.shape[0]) - s]
        t = torch.topk(q @ x.T, min(kmax, x.shape[0]), dim=1).values
        best = t if best is None else torch.topk(torch.cat([best, t], 1), min(kmax, best.shape[1] + t.shape[1]),
                                                 dim=1).values
    return best


def pick(best, targets=(100, 10_000)):
    return {t: float(best[:, t - 1].median()) for t in targets}


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def host_ms(fn, runs, torch, sync=None):
    """Median host time of fn() (which ends in a host wait), after 2 warm-up calls."""
    for _ in range(2):
        fn()
    ms = []
    for _ in range(runs):
        (sync or torch.cuda.synchronize)()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ms.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ms))


def event_ms(fn, runs, torch):
    for _ in range(2):
        fn()
    ms = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def same(a, b, torch):
    return all(x.shape == y.shape and torch.equal(x, y) for x, y in zip(a, b))


def stacked(runs, torch):
    """The runs as the all-gather of ShardedFlatIP.range_search leaves them: [world, longest] and [world, nq + 1]."""
    stride = max(int(k.numel()) for _, k in runs)
    keys = torch.zeros((len(runs), stride), dtype=torch.int64, device="cuda")
    for r, (_, k) in enumerate(runs):
        keys[r, :k.numel()] = k
    lims = torch.stack([l for l, _ in runs])
    return keys, lims, int(lims[:, -1].sum())


def one_gpu(args, torch):
    """The ranks as windows of one index on one GPU (no exchange)."""
    import ivr_b200
    from ivr_b200.sharded import _cuda_range_merge, partition_rows
    results, ok = [], True
    worlds = [int(v) for v in args.worlds.split(",")]
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        full = ivr_b200.IndexFlatIP(d, device=0)
        full.reserve(n)
        add_rows(full.add_tensor, 0, n, n, d, torch)
        qall = rows_block(0, 128, d, torch, seed=100 + d)
        r_of = pick(radii(qall, 0, n, n, d, torch))
        for nq in (int(v) for v in args.nq.split(",")):
            q = qall[:nq].contiguous()
            for target, radius in r_of.items():
                want = full.range_search_tensor(q, radius)
                n1 = host_ms(lambda: full.range_search_tensor(q, radius), args.runs, torch)
                row = {"rows": n, "dim": d, "nq": nq, "target_hits_per_query": target, "radius": radius,
                       "hits": int(want[0][-1]), "n1_ms": n1, **args.dev}
                for world in worlds:
                    off = partition_rows(n, world)
                    locs, runs = [], []
                    for r in range(world):
                        full.set_window(int(off[r]), int(off[r + 1] - off[r]))
                        runs.append(full.range_search_keys_tensor(q, radius))
                        locs.append(host_ms(lambda: full.range_search_keys_tensor(q, radius), args.runs, torch))
                    full.set_window()
                    keys, lims, total = stacked(runs, torch)
                    got = _cuda_range_merge(keys, lims, total)
                    merge = event_ms(lambda: _cuda_range_merge(keys, lims, total), args.runs, torch)
                    good = same(got, want, torch)
                    ok = ok and good
                    row[f"n{world}"] = {"local_ms": max(locs), "local_ms_per_window": locs, "merge_ms": merge,
                                        "exchange_ms": "not measured (one GPU)", "equal_to_n1": good}
                results.append(row)
                print(json.dumps(row), flush=True)
        full.close()
        torch.cuda.empty_cache()
    return results, ok


def distributed(args, torch):
    import torch.distributed as dist
    import ivr_b200
    from ivr_b200.sharded import _cuda_range_merge, partition_rows
    rank, world = dist.get_rank(), dist.get_world_size()
    results, ok = [], True

    def slowest(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()

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
        best = radii(qall, lo, hi, n, d, torch)
        parts = [torch.empty_like(best) for _ in range(world)]
        dist.all_gather(parts, best)
        r_of = pick(torch.topk(torch.cat(parts, 1), best.shape[1], dim=1).values)
        for nq in (int(v) for v in args.nq.split(",")):
            q = qall[:nq].contiguous()
            for target, radius in r_of.items():
                got = sh.range_search(q, radius)
                lims, keys = sh.local.range_search_keys_tensor(q, radius, id_offset=lo)
                rows = [torch.empty_like(lims) for _ in range(world)]
                dist.all_gather(rows, lims)
                stride = max(int(r[-1]) for r in rows)
                mine = torch.zeros(stride, dtype=torch.int64, device="cuda")
                mine[:keys.numel()] = keys
                gathered = torch.empty((world, stride), dtype=torch.int64, device="cuda")
                dist.all_gather_into_tensor(gathered.view(-1), mine)
                lims_parts = torch.stack(rows)
                total = int(lims_parts[:, -1].sum())
                local = slowest(host_ms(lambda: sh.local.range_search_keys_tensor(q, radius, id_offset=lo),
                                        args.runs, torch, sync=barrier))
                merge = slowest(event_ms(lambda: _cuda_range_merge(gathered, lims_parts, total), args.runs, torch))
                e2e = slowest(host_ms(lambda: sh.range_search(q, radius), args.runs, torch, sync=barrier))
                # every rank's result equals rank 0's full-matrix range search
                ref = [torch.empty(int(got[0][-1]) if i else nq + 1, dtype=t.dtype, device="cuda")
                       for i, t in enumerate(got)]
                n1 = -1.0
                if rank == 0:
                    want = full.range_search_tensor(q, radius)
                    good = same(got, want, torch)
                    ref = list(want)
                    n1 = host_ms(lambda: full.range_search_tensor(q, radius), args.runs, torch)
                for t in ref:
                    dist.broadcast(t, 0)
                good = torch.tensor([int(same(got, ref, torch))], device="cuda")
                dist.all_reduce(good, op=dist.ReduceOp.MIN)
                ok = ok and bool(good.item())
                if rank == 0:
                    row = {"world": world, "rows": n, "dim": d, "nq": nq, "target_hits_per_query": target,
                           "radius": radius, "hits": int(got[0][-1]), "local_ms": local, "merge_ms": merge,
                           "total_ms": e2e, "exchange_ms": e2e - local - merge, "n1_ms": n1,
                           "equal_to_n1_on_every_rank": bool(good.item()), **args.dev}
                    results.append(row)
                    print(json.dumps(row), flush=True)
        if full is not None:
            full.close()
        sh.local.close()
        torch.cuda.empty_cache()
    return results, ok


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--cells", default="100M,10M")
    ap.add_argument("--nq", default="1,16,128")
    ap.add_argument("--worlds", default="2,8", help="ranks simulated as row windows without torchrun")
    ap.add_argument("--runs", type=int, default=10)
    ap.add_argument("--out", default=None, help="directory for sharded_range_check.json (rank 0)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("sharded_range_check needs a CUDA device")
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
            with open(os.path.join(args.out, "sharded_range_check.json"), "w") as f:
                json.dump(results, f, indent=1)
        print(f"sharded_range_check: every result equal to the full-matrix range search: {ok}", flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
