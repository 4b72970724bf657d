"""Range search (IndexFlatIP.range_search) on one GPU: time, bytes, achieved HBM rate and parity.

Cells: rows 10 M x 512 and 851 284 x 768 (the reference's production cell), nq in {1, 16, 128, 1024}, two radii per
query set: the median over queries of the 100th- and of the 10 000th-best fp32 score (about 100 and 10 k hits per
query).  Rows and queries are the CLIP-like mixture of oracle/synth.py (unit centres + isotropic noise,
L2-normalised), generated on the device from a seed.

Per cell: range-search time (CUDA events around the device entry point, warmed up, median of --runs), algorithmic
bytes (rows ntotal * dpad * 2 once per query chunk, plus 24 per hit: 12 to the pool, 12 to D / I), GB/s and its share
of the measured 6552.6 GB/s HBM copy rate, the search(k=100) time of the same batch, and a parity check of up to 256
queries against an exact fp32 scan with torch (worst score error, band substitutions).  The row sets exceed the
126 MB L2, so every timed pass streams from HBM.

    python tools/range_search_timing.py [--runs 20] [--out DIR] [--cells 10M,851k] [--nq 1,16,128,1024]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

COPY_PEAK_GBS = 6552.6
CELLS = {"10M": (10_000_000, 512), "851k": (851_284, 768)}


def clip_like_dev(n, d, seed, torch, n_centres=4096, centre_seed=1234, sigma_scale=0.5, block=1 << 20):
    """oracle/synth.clip_like's mixture, generated on the device: yields float32 [<=block, d] CUDA blocks."""
    g = torch.Generator(device="cuda").manual_seed(centre_seed)
    c = torch.randn((n_centres, d), generator=g, device="cuda")
    c = c / c.norm(dim=1, keepdim=True)
    g = torch.Generator(device="cuda").manual_seed(seed)
    for s in range(0, n, block):
        m = min(block, n - s)
        z = torch.randint(0, n_centres, (m,), generator=g, device="cuda")
        x = c[z] + (sigma_scale / math.sqrt(d)) * torch.randn((m, d), generator=g, device="cuda")
        yield x / x.norm(dim=1, keepdim=True)


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def timed(fn, runs, torch):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def parity(X, q, radius, lims, D, I, torch, orr, tol=1e-3):
    """Exact fp32 scan of the sampled queries; returns (worst |score error|, band substitutions, violations)."""
    nq = q.shape[0]
    refs = [[] for _ in range(nq)]
    for s in range(0, X.shape[0], 1 << 20):
        sc = q @ X[s:s + (1 << 20)].T
        qi, ri = torch.nonzero(sc > radius, as_tuple=True)
        v = sc[qi, ri]
        for qq in range(nq):
            sel = qi == qq
            refs[qq].append((v[sel].cpu().numpy(), (ri[sel] + s).cpu().numpy()))
    lims_r, D_r, I_r = [0], [], []
    for qq in range(nq):
        d = np.concatenate([a for a, _ in refs[qq]]).astype(np.float32)
        i = np.concatenate([b for _, b in refs[qq]]).astype(np.int64)
        o = np.lexsort((i, -d))
        D_r.append(d[o]); I_r.append(i[o]); lims_r.append(lims_r[-1] + d.size)
    lims_r, D_r, I_r = np.array(lims_r), np.concatenate(D_r), np.concatenate(I_r)

    def score_of(qq, ids):
        return (X[torch.from_numpy(ids).cuda()] @ q[qq]).cpu().numpy()

    bad = orr.compare_range(lims, D, I, lims_r, D_r, I_r, score_of, radius, tol)
    worst, subs = 0.0, 0
    for qq in range(nq):
        ids = I[lims[qq]:lims[qq + 1]]
        if ids.size:
            worst = max(worst, float(np.abs(D[lims[qq]:lims[qq + 1]] - score_of(qq, ids)).max()))
        subs += np.setxor1d(ids, I_r[lims_r[qq]:lims_r[qq + 1]]).size
    return worst, int(subs), bad


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--out", default=None, help="directory for range_search_timing.json")
    ap.add_argument("--cells", default="10M,851k")
    ap.add_argument("--nq", default="1,16,128,1024")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("range_search_timing needs a CUDA device")
    import ivr_b200
    from ivr_b200 import _native as nat
    from oracle import range_search as orr

    dev = {"gpu": torch.cuda.get_device_name(0), "power_limit": power_limit()}
    print(json.dumps(dev), flush=True)
    results = []
    st = torch.cuda.current_stream().cuda_stream
    for cell in args.cells.split(","):
        n, d = CELLS[cell]
        X = torch.cat(list(clip_like_dev(n, d, seed=1, torch=torch)))
        idx = ivr_b200.IndexFlatIP(d, device=0)
        idx.add_tensor(X)
        torch.cuda.synchronize()
        dpad = (d + 63) // 64 * 64
        chunk = min(128, 65536 // dpad // 16 * 16)
        for nq in (int(v) for v in args.nq.split(",")):
            q = next(clip_like_dev(nq, d, seed=100 + nq, torch=torch))
            # radii from the exact fp32 scores of up to 256 queries
            qs = q[:256]
            best = None
            for s in range(0, n, 1 << 20):
                t = torch.topk(qs @ X[s:s + (1 << 20)].T, min(10_000, min(1 << 20, n - s)), dim=1).values
                best = t if best is None else torch.topk(torch.cat([best, t], 1), 10_000, dim=1).values
            for target in (100, 10_000):
                radius = float(best[:, target - 1].median())
                L = torch.zeros(nq + 1, dtype=torch.int64, device="cuda")
                cap = 1
                Dd = torch.empty(cap, device="cuda")
                Id = torch.empty(cap, dtype=torch.int64, device="cuda")

                def call():
                    nat.check(nat.lib.ivr_index_range_search_device(idx._handle(), q.data_ptr(), nq, radius, cap,
                                                                    L.data_ptr(), Dd.data_ptr(), Id.data_ptr(), 0, st))
                call()
                torch.cuda.synchronize()
                hits = int(L[nq])
                cap = max(hits, 1)
                Dd = torch.empty(cap, device="cuda")
                Id = torch.empty(cap, dtype=torch.int64, device="cuda")
                ms = timed(call, args.runs, torch)
                Ds = torch.empty((nq, 100), device="cuda")
                Is = torch.empty((nq, 100), dtype=torch.int64, device="cuda")
                ms_search = timed(lambda: nat.check(nat.lib.ivr_index_search_device(
                    idx._handle(), q.data_ptr(), nq, 100, Ds.data_ptr(), Is.data_ptr(), 0, 0, st)), args.runs, torch)
                passes = -(-nq // chunk)
                row_bytes = n * dpad * 2 * passes
                byts = row_bytes + 24 * hits
                gbs = byts / ms / 1e6
                # parity on the first 256 queries: their slice of the result
                m = min(nq, 256)
                lims = L[:m + 1].cpu().numpy()
                D, I = Dd[:lims[m]].cpu().numpy(), Id[:lims[m]].cpu().numpy()
                worst, subs, bad = parity(X, q[:m], radius, lims, D, I, torch, orr)
                r = {"rows": n, "dim": d, "nq": nq, "target_hits_per_query": target, "radius": radius,
                     "hits": hits, "hits_per_query": hits / nq, "row_passes": passes, "range_ms": ms,
                     "bytes": byts, "GBps": gbs, "pct_copy_peak": 100 * gbs / COPY_PEAK_GBS,
                     "search_k100_ms": ms_search, "range_over_search": ms / ms_search,
                     "parity_queries": m, "worst_score_err": worst, "band_substitutions": subs,
                     "parity_violations": len(bad), **dev}
                results.append(r)
                print(json.dumps(r), flush=True)
                if bad:
                    print("  parity:", bad[:3], flush=True)
        idx.close()
        del X
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "range_search_timing.json"), "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
