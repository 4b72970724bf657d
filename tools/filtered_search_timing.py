"""Time filtered top-k search (SearchParameters(sel=...)) against the unfiltered search of the same batch.

For each shape, selection and batch size: the median of 20 device-event-timed calls of ``search_tensor`` after two
warm-up calls, filtered and unfiltered (auto path), plus -- for the 100 % selection -- the unfiltered search forced onto
the list mode of the small-batch kernel (IVR_MMA_MODE=3, IVR_SMALL_DUMP_MAX_KROWS=0), the path the filtered kernel
shares.  Rows are generated on the device (unit-norm Gaussian) and are far larger than the 126 MB L2, so every call
streams its rows from HBM.  The bytes column is the selected tiles' rows (tiles x 128 x dpad x 2); its share is of
6552.6 GB/s, the row-streaming rate measured in DESIGN.md section 6.  The card's name and power limit are read in the
same run and printed first.

    python tools/filtered_search_timing.py [--shapes 10000000x512,851284x768] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6552.6
RUNS, WARMUP = 20, 2
SELECTIONS = [("contig 0.1%", 0.001), ("contig 1%", 0.01), ("contig 10%", 0.1), ("contig 100%", 1.0),
              ("random 1%", -0.01)]


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in out.split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def build(n, d, seed=0):
    import torch
    import ivr_b200
    idx = ivr_b200.IndexFlatIP(d, device=0)
    idx.reserve(n)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for s in range(0, n, 1 << 20):
        m = min(1 << 20, n - s)
        x = torch.randn((m, d), generator=g, device="cuda")
        idx.add_tensor(x / x.norm(dim=1, keepdim=True))
    torch.cuda.synchronize()
    return idx


def selection(n, frac, seed=1):
    from ivr_b200 import faiss_compat as fc
    if frac > 0:
        a = int(n * 0.37) // 128 * 128 + 5 if frac < 1 else 0   # a run starting mid-index, not tile-aligned
        b = min(n, a + int(round(n * frac)))
        return fc.IDSelectorRange(a, b)
    rng = np.random.default_rng(seed)
    return fc.IDSelectorBatch(rng.choice(n, int(round(n * -frac)), replace=False))


def median_ms(fn):
    import torch
    for _ in range(WARMUP):
        fn()
    ts = []
    for _ in range(RUNS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    import torch
    from ivr_b200 import faiss_compat as fc
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="10000000x512,851284x768")
    ap.add_argument("--nq", default="1,16,128")
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}", flush=True)
    rows = []
    for shape in a.shapes.split(","):
        n, d = (int(v) for v in shape.split("x"))
        idx = build(n, d)
        dpad = (d + 63) // 64 * 64
        n_tiles = (n + 127) // 128
        qs = torch.randn((max(int(v) for v in a.nq.split(",")), d), generator=torch.Generator(device="cuda")
                         .manual_seed(7), device="cuda")
        qs = qs / qs.norm(dim=1, keepdim=True)
        for label, frac in SELECTIONS:
            sel = selection(n, frac)
            words = sel.words(n)
            tiles = int((np.bitwise_or.reduce(np.pad(words, (0, -words.size % 4)).reshape(-1, 4), axis=1) != 0).sum())
            p = fc.SearchParameters(sel=sel)
            for nq in (int(v) for v in a.nq.split(",")):
                q = qs[:nq].contiguous()
                ms_f = median_ms(lambda: idx.search_tensor(q, a.k, params=p))
                kern = idx.last_timing()["kernel"]
                ms_u = median_ms(lambda: idx.search_tensor(q, a.k))
                kern_u = idx.last_timing()["kernel"]
                ms_l = None
                if frac == 1.0 and nq > 1:
                    os.environ["IVR_MMA_MODE"], os.environ["IVR_SMALL_DUMP_MAX_KROWS"] = "3", "0"
                    ms_l = median_ms(lambda: idx.search_tensor(q, a.k))
                    del os.environ["IVR_MMA_MODE"], os.environ["IVR_SMALL_DUMP_MAX_KROWS"]
                gb = tiles * 128 * dpad * 2 / 1e9
                r = {"shape": shape, "selection": label, "selected_rows": sel.count(n), "tiles": tiles,
                     "tiles_share": tiles / n_tiles, "nq": nq, "k": a.k, "filtered_ms": ms_f[0],
                     "filtered_min_max": ms_f[1:], "kernel": kern, "unfiltered_ms": ms_u[0], "unfiltered_kernel": kern_u,
                     "unfiltered_list_ms": None if ms_l is None else ms_l[0], "ratio": ms_f[0] / ms_u[0],
                     "gb_streamed": gb, "hbm_share": gb / (ms_f[0] * 1e-3) / HBM_GBS}
                rows.append(r)
                print(f"{shape:>16} {label:>12} tiles {tiles:>7} ({r['tiles_share']:6.1%}) nq {nq:>3}: "
                      f"filtered {ms_f[0]:8.3f} ms  unfiltered {ms_u[0]:8.3f} ms ({kern_u})  "
                      f"ratio {r['ratio']:6.3f}"
                      + (f"  list-mode {ms_l[0]:8.3f} ms" if ms_l else "")
                      + f"  {gb:7.3f} GB = {r['hbm_share']:6.1%} of {HBM_GBS} GB/s", flush=True)
            sel.close()
        idx.close()
        del qs
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": info, "runs": RUNS, "warmup": WARMUP, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
