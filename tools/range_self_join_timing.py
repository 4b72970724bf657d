"""Range self-join (IndexFlatIP.range_self_join) on one GPU: time, floors, the range-search route and a model check.

Cells: 1 M x 512, 851 284 x 768 (the reference's production cell) and 100 k x 512 rows of the CLIP-like mixture of
oracle/synth.py, generated on the device from a seed.  The first two exceed the 126 MB L2 (1 GB and 1.3 GB of fp16
rows); 100 k x 512 (102 MB) fits it.  Two radii per cell: the median over 256 sampled rows of the 10th- and of the
100th-best score to another row (about 10 and 100 neighbours per row).

Per cell: join time (CUDA events around ivr_index_range_self_join_device with the exact capacity, warmed up, median of
--runs), its hits; the time of the range-search route on the same index (the fp32 rows on the device as queries,
ivr_index_range_search_device, exact capacity) and the ratio; the join's share of its two floors, by arithmetic from
measured peaks of 6552.6 GB/s (HBM copy) and 1389.5 TFLOP/s (sustained fp16 tensor): HBM n^2 * dpad / npad bytes (every
B block streams the rows below it once, no L2 reuse), tensor n^2 * dpad FLOP (n^2 / 2 pairs, 2 * dpad each); the
range route's HBM floor ceil(n / chunk) * n * 2 * dpad bytes; and a model check of 256 sampled rows' lists against the
float64 product of the stored fp16 rows within the fp16 model's bound (oracle/fp16_model.py), symmetry included.

    python tools/range_self_join_timing.py [--runs 5] [--out DIR] [--cells 1M,851k,100k] [--neighbours 10,100]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from range_search_timing import clip_like_dev, power_limit, timed  # noqa: E402

COPY_PEAK_GBS = 6552.6
TENSOR_PEAK_TFLOPS = 1389.5
CELLS = {"1M": (1_000_000, 512), "851k": (851_284, 768), "100k": (100_000, 512)}
U, TINY = 2.0 ** -23, 2.0 ** -149


def model_check(X16, sample, radius, lims, D, I, dpad, torch):
    """Sampled rows' lists against the model: (violations, worst |D - m| / eps, pairs missing their mirror)."""
    bad, worst, asym = 0, 0.0, 0
    Xd = X16.double()
    Xa = Xd.abs()
    r = float(np.float32(radius))
    for i in sample.tolist():
        m = Xd @ Xd[i]
        eps = (dpad / 8 + 4) * (U * (Xa @ Xa[i]) + TINY) + TINY
        a, b = int(lims[i]), int(lims[i + 1])                 # lims, D, I on the host
        ids, d = I[a:b].cuda(), D[a:b].double().cuda()
        if (ids == i).any() or ids.unique().numel() != ids.numel() or (d <= r).any():
            bad += 1
        err = (d - m[ids]).abs()
        if ids.numel():
            worst = max(worst, float((err / eps[ids]).max()))
            if (err > eps[ids]).any():
                bad += 1
        low = m - eps
        low[ids] = -math.inf
        low[i] = -math.inf
        if float(low.max()) > r:
            bad += 1
        for j, s in zip(ids.tolist(), D[a:b].tolist()):
            a2, b2 = int(lims[j]), int(lims[j + 1])
            pos = (I[a2:b2] == i).nonzero()
            if pos.numel() != 1 or float(D[a2 + int(pos[0])]) != s:
                asym += 1
    return bad, worst, asym


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for range_self_join_timing.json")
    ap.add_argument("--cells", default="1M,851k,100k")
    ap.add_argument("--neighbours", default="10,100")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("range_self_join_timing needs a CUDA device")
    import ivr_b200
    from ivr_b200 import _native as nat

    dev = {"gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    print(json.dumps(dev), flush=True)
    results = []
    st = torch.cuda.current_stream().cuda_stream
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        X = torch.cat(list(clip_like_dev(n, d, seed=1, torch=torch)))
        idx = ivr_b200.IndexFlatIP(d, device=0)
        idx.add_tensor(X)
        X16 = X.half()
        torch.cuda.synchronize()
        dpad = (d + 63) // 64 * 64
        npad = min(128, 65536 // dpad // 16 * 16)
        sample = torch.from_numpy(np.random.default_rng(0).choice(n, 256, replace=False)).cuda()
        s = (X16[sample].float() @ X16.float().T)
        s[torch.arange(256, device="cuda"), sample] = -math.inf
        best = torch.topk(s, 100, dim=1).values
        del s
        for k in (int(v) for v in args.neighbours.split(",")):
            radius = float(best[:, k - 1].median())
            L = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
            box = {"cap": 0, "D": torch.empty(1, device="cuda"), "I": torch.empty(1, dtype=torch.int64, device="cuda")}

            def join():
                nat.check(nat.lib.ivr_index_range_self_join_device(idx._handle(), radius, box["cap"], L.data_ptr(),
                                                                   box["D"].data_ptr(), box["I"].data_ptr(), st))
            join()
            torch.cuda.synchronize()
            hits = int(L[n])
            box["cap"] = max(hits, 1)
            box["D"] = torch.empty(box["cap"], device="cuda")
            box["I"] = torch.empty(box["cap"], dtype=torch.int64, device="cuda")
            ms = timed(join, args.runs, torch)
            lims, D, I = L.clone(), box["D"][:hits].clone(), box["I"][:hits].clone()
            del box["D"], box["I"]
            # the range-search route: every row as an fp32 query, self-hits included
            LR = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
            rbox = {"cap": 0, "D": torch.empty(1, device="cuda"), "I": torch.empty(1, dtype=torch.int64, device="cuda")}

            def route():
                nat.check(nat.lib.ivr_index_range_search_device(idx._handle(), X.data_ptr(), n, radius, rbox["cap"],
                                                                LR.data_ptr(), rbox["D"].data_ptr(),
                                                                rbox["I"].data_ptr(), 0, st))
            route()
            torch.cuda.synchronize()
            rhits = int(LR[n])
            rbox["cap"] = max(rhits, 1)
            rbox["D"] = torch.empty(rbox["cap"], device="cuda")
            rbox["I"] = torch.empty(rbox["cap"], dtype=torch.int64, device="cuda")
            ms_route = timed(route, max(3, args.runs // 2), torch)
            del rbox["D"], rbox["I"]
            torch.cuda.empty_cache()
            hbm_floor_s = n * n * dpad / npad / (COPY_PEAK_GBS * 1e9)
            tensor_floor_s = n * n * dpad / (TENSOR_PEAK_TFLOPS * 1e12)
            route_floor_s = -(-n // npad) * n * 2 * dpad / (COPY_PEAK_GBS * 1e9)
            bad, worst, asym = model_check(X16, sample, radius, lims.cpu(), D.cpu(), I.cpu(), dpad, torch)
            r = {"rows": n, "dim": d, "in_l2": n * dpad * 2 < 126e6, "target_neighbours": k, "radius": radius,
                 "join_ms": ms, "join_hits": hits, "hits_per_row": hits / n, "route_ms": ms_route,
                 "route_hits": rhits, "join_over_route": ms / ms_route,
                 "hbm_floor_ms": 1e3 * hbm_floor_s, "tensor_floor_ms": 1e3 * tensor_floor_s,
                 "pct_hbm_floor": 100 * 1e3 * hbm_floor_s / ms, "pct_tensor_floor": 100 * 1e3 * tensor_floor_s / ms,
                 "route_hbm_floor_ms": 1e3 * route_floor_s, "route_pct_floor": 100 * 1e3 * route_floor_s / ms_route,
                 "model_rows": 256, "model_violations": bad, "worst_err_over_eps": worst,
                 "asymmetric_pairs": asym, **dev}
            results.append(r)
            print(json.dumps(r), flush=True)
        idx.close()
        del X, X16
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "range_self_join_timing.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
