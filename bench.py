#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native retrieval hot path.

Metric (BASELINE.json): top-100 queries/sec over N x 512 embeddings at 1/2/4/8 B200, with the
roofline fraction of the dominant kernel.  Workload: BASELINE config D -- 100 M x 512 synthetic
CLIP-like embeddings (fp16 rows, 102.4 GB: fits ONE B200), a batch of 4096 queries, k = 100.
Scaling is STRONG: the same 100 M rows are row-sharded over the N ranks (N=8 -> 12.5 M rows per
GPU, exactly config D), local top-k per GPU, packed 64-bit keys pushed into every peer's mailbox over NVLink
(csrc/exchange.cu; one NCCL all-gather where peers cannot be mapped), on-device k-way merge.  At N > 1 two searches
are in flight -- the exchange and merge of batch i run on a side stream while batch i+1 is being scored -- and the
shard boundaries follow each GPU's measured scoring speed (elastic boundaries: every rank also stores 4 % of either
neighbour's rows; `--equal-shards` turns that off).  Every batch is complete, merged and (e2e) back in host memory
before the closing timestamp.

    python bench.py --gpus 1 --steps K --warmup W          # our arm
    python bench.py --impl reference ...                   # the reference's own CPU code path

A "step" is one pass of the hot path over one query batch.  Prints ONE JSON line (rank 0).  ``--dump-outputs DIR``
also writes the scores and ids of the last timed step as .npy files; the inputs depend only on the arguments, so two
builds run with the same arguments can be compared output for output.

Reference arm: the reference's OWN batched entry point, ``core.FAISSRetriever.build_index`` + ``.search``
(core.py:758-930), imported unmodified from ``oracle/_ref`` (tools/make_ref.py) and run on every host core of
the box.  FAISS -- the un-vendored, absent library under it -- is replaced by the oracle's multi-threaded
restatement of the IndexFlatIP contract (oracle/flat_ip_mt.py).  A step is a BOUNDED sample of the workload
(``--cpu-sample-queries`` of the queries x ``--cpu-sample-rows`` of the rows); q/s for the full workload are
obtained by scaling the flat-search part linearly in rows (flat search is linear in N) and keeping the
reference's per-hit Python loop as measured (it does not depend on N).  Both the sample and the split are
printed.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

if "reference" in sys.argv:
    # The CPU arm uses every host core it may run on.  Launchers (torch.distributed.run) export OMP_NUM_THREADS=1,
    # which the OpenMP / BLAS pools read once at import: fix the environment BEFORE numpy / torch are imported
    # (oracle/flat_ip_mt.set_threads() then also sets the counts explicitly at run time).
    try:
        _cores = len(os.sched_getaffinity(0))
    except AttributeError:
        _cores = os.cpu_count() or 1
    for _v in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS"):
        os.environ[_v] = str(_cores)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "top-100 queries/sec over Nx512 embeddings"
GEN_CHUNK = 500_000              # rows generated per step; shard boundaries are multiples of it
N_CENTRES = 4096
CHECK_QUERIES = 256              # queries verified against an exact fp32 scan of the whole DB
TOL = 1e-3                       # north_star: ids identical except ties within 1e-3 of the k-th score
DUMP_BYTES = 64 << 20            # --dump-outputs: at most this much on disk


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--rows", type=int, default=int(os.environ.get("IVR_BENCH_ROWS", 100_000_000)))
    p.add_argument("--dim", type=int, default=512)
    p.add_argument("--nq", type=int, default=int(os.environ.get("IVR_BENCH_NQ", 4096)))
    p.add_argument("--k", type=int, default=100)
    p.add_argument("--path", type=int, default=int(os.environ.get("IVR_BENCH_PATH", 0)),
                   help="0 auto, 1 streaming (K3), 2 tcgen05 (K1+K2)")
    p.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    p.add_argument("--cpu-sample-queries", type=int, default=256)
    p.add_argument("--cpu-dedup-frames", type=int, default=10_000)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--equal-shards", action="store_true",
                   help="N > 1: static equal shards (no replicated boundary rows, no elastic boundaries)")
    p.add_argument("--shard-margin", type=float, default=0.04,
                   help="N > 1: fraction of a shard every rank also stores from either neighbour (elastic boundaries)")
    p.add_argument("--no-extras", action="store_true",
                   help="skip the informational legs (BASELINE configs A, B, C, the production-shaped cell)")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the top-k of the last timed step to DIR: scores.npy (float32 [m,k]), ids.npy (float64 "
                        "[m,k]) and query_rows.npy (float64 [m], the query of each row; a fixed sample when all nq "
                        "rows would exceed 64 MB)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes the outputs of --impl ours")
    return a


def workload_config(args):
    """The SAME dict in both arms (driver: same_config)."""
    return {"workload": f"BASELINE config D: flat inner-product top-{args.k} over {args.rows}x{args.dim} embeddings, "
                        f"batch {args.nq}",
            "rows": args.rows, "dim": args.dim, "nq": args.nq, "k": args.k, "n_gpus": args.gpus,
            "cache": "inputs larger than L2 (every DB shard >> 126 MB); no L2 flush needed"}


# ---------------------------------------------------------------------------- synthetic data
def centres(dim, device):
    import torch
    g = torch.Generator(device="cpu").manual_seed(1234)
    c = torch.randn(N_CENTRES, dim, generator=g, dtype=torch.float32)
    return torch.nn.functional.normalize(c, dim=1).to(device)


def gen_rows(chunk_idx, n, dim, cen, device, seed=77):
    """x = normalize(c[z] + sigma*g), sigma = 0.5/sqrt(d); deterministic per chunk index."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed * 1_000_003 + chunk_idx)
    z = torch.randint(0, N_CENTRES, (n,), generator=g, device=device)
    x = cen[z] + (0.5 / dim ** 0.5) * torch.randn(n, dim, generator=g, device=device, dtype=torch.float32)
    return torch.nn.functional.normalize(x, dim=1)


def gen_queries(nq, dim, cen_cpu):
    import torch
    g = torch.Generator(device="cpu").manual_seed(4321)
    z = torch.randint(0, N_CENTRES, (nq,), generator=g)
    q = cen_cpu[z] + (0.5 / dim ** 0.5) * torch.randn(nq, dim, generator=g, dtype=torch.float32)
    return torch.nn.functional.normalize(q, dim=1)


def gen_dedup_frames(n, d, dev, seed=7):
    """Scenes of geometric length (mean 20) around a per-scene base vector, un-normalised fp32 (SURVEY.md 8d)."""
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    lens = torch.distributions.Geometric(probs=torch.tensor(1.0 / 20)).sample((n // 10 + 16,)).to(torch.int64) + 1
    sid = torch.repeat_interleave(torch.arange(lens.numel()), lens)[:n].to(dev)
    base = torch.randn(int(sid.max().item()) + 1, d, generator=g, device=dev)
    sig = 0.10 + 0.25 * torch.rand(n, 1, generator=g, device=dev)
    return ((base[sid] + sig * torch.randn(n, d, generator=g, device=dev)) * 3.0).contiguous()


# ---------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------- CPU arm
def cpu_arm(args, xb, xq, steps, warmup):
    """The reference's CPU path on this box's host cores (see the module docstring).  ``xb`` / ``xq`` are the
    bounded sample (float32 NumPy).  Returns the ``cpu_baseline`` object plus ms_per_step of the sample."""
    from oracle import flat_ip_mt, ref_runner, ref_shims
    cores = flat_ip_mt.set_threads()                     # explicit: launchers export OMP_NUM_THREADS=1
    n_s, nq_s, n_total, k = len(xb), len(xq), args.rows, args.k
    grow = n_total / n_s
    if ref_shims.reference_available():
        r = ref_runner.time_faiss_retriever(xb, xq, k, steps=steps, warmup=warmup)
        loop_s = max(r["step_s"] - r["search_s"], 0.0)
        per_query = r["search_s"] / nq_s * grow + loop_s / nq_s
        raw_qps = nq_s / (r["search_s"] * grow)
        out = {"value": 1.0 / per_query, "unit": "queries/s", "cores": cores, "kind": "reference",
               "what": "the reference's own core.FAISSRetriever.search (core.py:848-930, unmodified, from oracle/_ref) "
                       "over oracle/flat_ip_mt.IndexFlatIP (FAISS, an un-vendored dependency, is absent)",
               "sample": f"{nq_s} of {args.nq} queries x {n_s} of {n_total} rows per step "
                         f"({r['step_s']:.2f} s of CPU work: {r['search_s']:.2f} s flat search on {cores} threads + "
                         f"{loop_s:.2f} s of the reference's per-hit Python loop); flat-search time scaled x{grow:g} "
                         f"in rows, the loop kept as measured",
               "raw_flat_search": {"value": raw_qps, "unit": "queries/s", "kind": "port", "cores": cores,
                                   "what": "oracle/flat_ip_mt alone: fp32 sgemm blocks + per-query top-k, all threads"}}
        return out, r["step_s"] * 1e3
    idx = flat_ip_mt.IndexFlatIP(xb.shape[1])
    idx.add(xb)
    for _ in range(warmup):
        idx.search(xq[:8], k)
    ts = []
    for _ in range(max(steps, 1)):
        t0 = time.perf_counter()
        idx.search(xq, k)
        ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    return ({"value": nq_s / (t * grow), "unit": "queries/s", "cores": cores, "kind": "port",
             "what": "oracle/flat_ip_mt (oracle/_ref is missing: run tools/make_ref.py where /root/reference exists)",
             "sample": f"{nq_s} of {args.nq} queries x {n_s} of {n_total} rows per step ({t:.2f} s), scaled x{grow:g} in rows"},
            t * 1e3)


def cpu_sample(args, device="cpu"):
    import torch
    dim = args.dim
    cen = centres(dim, device)
    n_s = min(args.cpu_sample_rows, args.rows)
    ch = min(GEN_CHUNK, n_s)
    xb = torch.cat([gen_rows(i, min(ch, n_s - i * ch), dim, cen, device).cpu()
                    for i in range((n_s + ch - 1) // ch)]).numpy()
    xq = gen_queries(args.nq, dim, cen.cpu())[:args.cpu_sample_queries].numpy()
    return xb, xq


def run_reference(args):
    if int(os.environ.get("RANK", 0)) != 0:
        return                                            # the CPU arm runs once, on rank 0
    xb, xq = cpu_sample(args)
    cpu, ms = cpu_arm(args, xb, xq, args.steps, min(args.warmup, 1))
    out = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": "queries/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args), "cpu_baseline": cpu,
           "e2e": {"value": cpu["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def measured_traffic(kernel, rows, dim, nq, k):
    """dram__bytes_read + dram__bytes_write of the dominant kernel from the committed ncu --set full
    captures of the same shape (profiles/*_traffic.json), per launch; None when no capture matches."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            table = json.load(open(os.path.join(ROOT, "profiles", name)))
        except Exception:
            continue
        for e in table:
            if (e["kernel"], e["rows"], e["dim"], e["nq"], e["k"]) == (kernel, rows, dim, nq, k):
                return e["dram_bytes"]
    return None


def hbm_roofline(gbs, peaks, bytes_per_launch, **extra):
    pk = peaks.get("hbm_gbs") or 6650.0
    r = {"bound": "hbm", "achieved": gbs, "peak": pk, "unit": "GB/s", "frac": gbs / pk,
         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks.get("hbm_gbs") else "fallback 6650 GB/s",
         "algorithmic_bytes_per_launch": bytes_per_launch}
    r.update(extra)
    return r


# ---------------------------------------------------------------------------- parity gate
def parity_report(Dn, In, Dr, Ir, k):
    """Ours (Dn, In) against the exact fp32 top-k (Dr, Ir) of the same queries over the whole DB.
    Raises SystemExit on a violation of the north-star rule; returns the evidence otherwise."""
    n_chk = len(In)
    worst, subs = 0.0, 0
    for q in range(n_chk):
        ref = dict(zip(Ir[q].tolist(), Dr[q].tolist()))
        s_k = Dr[q, -1]
        for i_, d_ in zip(In[q].tolist(), Dn[q].tolist()):
            if i_ in ref:
                err = abs(ref[i_] - d_)
                worst = max(worst, err)
                if err > TOL:
                    raise SystemExit(f"parity gate FAILED: q{q} id {i_} score {d_} vs exact {ref[i_]}")
            else:                                            # not in the exact list: must be a tie at the k-th score
                subs += 1
                if d_ < s_k - TOL or d_ > s_k + 2 * TOL:
                    raise SystemExit(f"parity gate FAILED: q{q} id {i_} score {d_} outside the tie band of s_k={s_k}")
        must = Ir[q][Dr[q] > s_k + TOL]
        miss = np.setdiff1d(must, In[q])
        if miss.size:
            raise SystemExit(f"parity gate FAILED: q{q} misses {miss.size} ids above s_k + tol")
        if np.any(np.diff(Dn[q]) > 0):
            raise SystemExit(f"parity gate FAILED: q{q} scores not sorted")
    from oracle import comparator
    return {"checked_queries": n_chk, "status": "ok", "tol": TOL,
            "max_abs_score_error_vs_exact_fp32": worst,
            "tie_band_substitutions": subs, "of_hits": n_chk * k,
            "recall_vs_exact_fp32": comparator.recall_at_k(In, Ir)}


# ---------------------------------------------------------------------------- extras (N=1 only)
def time_device_search(idx, qd, k, reps=10, warm=3):
    """Median whole-search device time (CUDA events on torch's stream) + the handle's own stage timing."""
    import torch
    for _ in range(warm):
        idx.search_tensor(qd, k)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        idx.search_tensor(qd, k)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    idx.set_timing(True)
    idx.search_tensor(qd, k)
    t = idx.last_timing()
    idx.set_timing(False)
    return statistics.median(ts), t


def time_host(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def dump_outputs(out_dir, D, I):
    """Writes what a caller of the timed path receives -- scores [nq,k] and global row ids [nq,k] -- so that two builds
    can be compared output for output.  Ids go out as float64 (exact below 2**53).  When every query row would not
    fit in DUMP_BYTES, a sample of query rows drawn with a fixed seed is written instead."""
    D, I = D.cpu().numpy(), I.cpu().numpy()
    nq, k = D.shape
    m = min(nq, (DUMP_BYTES - 4096) // (4 * k + 8 * k + 8))          # 4 KB: room for the three .npy headers
    rows = np.arange(nq) if m == nq else np.sort(np.random.default_rng(0).choice(nq, m, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "scores.npy"), D[rows].astype(np.float32))
    np.save(os.path.join(out_dir, "ids.npy"), I[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))


def run_extras(args, dev, peaks):
    """Informational legs (not the headline): BASELINE configs A / B / C and the reference's production-shaped cell."""
    import ctypes as C
    import torch
    import ivr_b200
    from ivr_b200 import _native as nat
    out = {}
    k = 100
    # ---- config C: single-query latency path ------------------------------------------
    n, d = 10_000_000, 768
    cen = centres(d, dev)
    idx = ivr_b200.IndexFlatIP(d, device=dev.index)
    idx.reserve(n)
    for c in range(n // GEN_CHUNK):
        idx.add(gen_rows(c, GEN_CHUNK, d, cen, dev, seed=79))
    q = gen_queries(16, d, cen.cpu())
    ms, t = time_device_search(idx, q[:1].to(dev), k)
    qn = q[:1].numpy()
    lat = time_host(lambda: idx.search(qn, k))
    gbs = n * d * 2 / (t["score_ms"] * 1e-3) / 1e9
    out["config_c_single_query_10Mx768"] = {
        "kernel": t["kernel"], "kernel_ms": t["score_ms"], "device_ms_per_query": ms,
        "e2e_latency_ms_host_buffers": lat * 1e3, "queries_per_s_e2e": 1.0 / lat,
        "roofline": hbm_roofline(gbs, peaks, n * d * 2)}
    ms, t = time_device_search(idx, q.to(dev), k)
    gbs = n * d * 2 / (t["score_ms"] * 1e-3) / 1e9
    out["config_c_16_queries_10Mx768"] = {
        "kernel": t["kernel"], "kernel_ms": t["score_ms"], "device_ms": ms, "queries_per_s_device": 16 / (ms * 1e-3),
        "roofline": hbm_roofline(gbs, peaks, n * d * 2,
                                 note="kernel_ms brackets the 2-3 seeded launches and their inter-launch merges")}
    # ---- the reference's production-shaped cell: ONE query over 851 284 x 768, k = 50 (logs/performance.log:8) ----
    n_p, k_p = 851_284, 50
    pidx = ivr_b200.IndexFlatIP(d, device=dev.index)
    pidx.reserve(n_p)
    done = 0
    while done < n_p:
        m = min(GEN_CHUNK, n_p - done)
        pidx.add(gen_rows(1000 + done // GEN_CHUNK, m, d, cen, dev, seed=79))
        done += m
    ms, t = time_device_search(pidx, q[:1].to(dev), k_p, reps=30)
    u = ivr_b200.UnifiedIndex(device=dev.index)
    u.faiss_index, u.is_loaded = pidx, True
    u.metadata_list = [{"frame_id": i} for i in range(n_p)]
    u.memory_maps = {"thumbnails": {}, "temporal": {}}
    lat = time_host(lambda: u.search_vectors(qn[0], k=k_p), reps=50)
    gbs = n_p * d * 2 / (ms * 1e-3) / 1e9
    out["production_cell_851284x768_1query_k50"] = {
        "kernel": t["kernel"], "device_ms": ms, "score_ms": t["score_ms"], "merge_ms": t["merge_ms"],
        "search_vectors_host_to_host_ms": lat * 1e3,
        "reference_logged_s": 7.23, "reference_source": "logs/performance.log:8 (text -> CLIP -> flat IP, first query)",
        "roofline": hbm_roofline(gbs, peaks, n_p * d * 2, note="whole search (prep + stream + merge) vs the HBM peak")}
    # the same index through the reference's persistence calls: faiss.write_index, then faiss.read_index (the payload is
    # memory-mapped and streamed page cache -> pinned double buffer -> HBM; the reference's .rvdb load took 29.0 s)
    try:
        import tempfile
        fpath = os.path.join(tempfile.gettempdir(), f"ivr_bench_{os.getpid()}.faiss")
        t0 = time.perf_counter()
        ivr_b200.faiss_compat.write_index(pidx, fpath)
        t_w = time.perf_counter() - t0
        nbytes = os.path.getsize(fpath)
        t0 = time.perf_counter()
        ridx = ivr_b200.faiss_compat.read_index(fpath, ivr_b200.faiss_compat.IO_FLAG_MMAP, device=dev.index)
        t_r = time.perf_counter() - t0
        same = bool(np.array_equal(ridx.search(qn, k_p)[1], pidx.search(qn, k_p)[1]))
        ridx.close()
        os.unlink(fpath)
        out["production_cell_851284x768_1query_k50"]["index_file_round_trip"] = {
            "bytes": nbytes, "write_index_s": t_w, "read_index_s": t_r, "read_gbs": nbytes / t_r / 1e9,
            "same_hits_after_reload": same, "reference_logged_load_s": 29.0,
            "reference_source": "logs/system_20250828.log:26 (.rvdb: FAISS deserialise + all vectors + LZ4/JSON metadata)",
            "note": "FAISS IndexFlatIP layout (IxFI header + float32 rows); page cache warm (the file was just written)"}
    except Exception as e:
        out["production_cell_851284x768_1query_k50"]["index_file_round_trip"] = {"error": repr(e)[:300]}
    u.faiss_index = None
    pidx.close()
    idx.close()
    del idx, pidx
    torch.cuda.empty_cache()
    # ---- config A: 100 k x 512, 1000 queries (the only config quoted as the reference's CPU path) ----------
    n, d = 100_000, 512
    cen = centres(d, dev)
    xa = gen_rows(0, n, d, cen, dev, seed=81)
    qa = gen_queries(1000, d, cen.cpu())
    aidx = ivr_b200.IndexFlatIP(d, device=dev.index)
    aidx.add(xa)
    ms, t = time_device_search(aidx, qa.to(dev), k)
    qan = qa.numpy()
    lat = time_host(lambda: aidx.search(qan, k), reps=10)
    fl = 2.0 * n * d * 1000
    out["config_a_100kx512_1000q"] = {
        "kernel": t["kernel"], "device_ms": ms, "queries_per_s_device": 1000 / (ms * 1e-3),
        "e2e_ms_host_buffers": lat * 1e3, "queries_per_s_e2e": 1000 / lat,
        "tflops": fl / (ms * 1e-3) / 1e12,
        "note": "102 GFLOP / 102 MB of rows: launch- and merge-latency bound, far below either roofline"}
    # the legacy retriever wrapper, host to host (SURVEY.md 3.2: the reference needed 0.467 s, 96 % in its Python loop)
    n_w = 20_000
    raw = xa[:n_w].cpu().numpy()
    kms = [ivr_b200.KeyframeMetadata(folder_name=f"L{i // 1000:02d}_V001", image_name=f"{i % 1000:04d}", frame_id=i % 1000,
                                     file_path=f"keyframes/L{i // 1000:02d}_V001/{i % 1000:04d}.jpg", clip_features=raw[i])
           for i in range(n_w)]
    fr = ivr_b200.FAISSRetriever(device=dev.index)
    fr.build_index(raw, kms, validate_consistency=False)
    lat = time_host(lambda: fr.search(qan[:64], k=100), reps=5, warm=1)
    out["faiss_retriever_wrapper_20kx512_64q_k100"] = {"host_to_host_s": lat, "hits": 6400,
                                                       "reference_same_shape_s": 0.467,
                                                       "reference_source": "SURVEY.md section 3.2 (authoring container)"}
    if not args.no_cpu_baseline:
        try:                                                 # the reference's own wrappers on config A, host cores
            from oracle import flat_ip_mt, ref_runner, ref_shims
            if ref_shims.reference_available():
                cores = flat_ip_mt.set_threads()
                xan = xa.cpu().numpy()
                r = ref_runner.time_faiss_retriever(xan, qan, k)
                sv = ref_runner.time_search_vectors(xan, qan[:200], k)
                out["config_a_100kx512_1000q"]["cpu_baseline"] = {
                    "kind": "reference", "cores": cores, "unit": "queries/s",
                    "faiss_retriever_search": {"value": 1000 / r["step_s"], "seconds": r["step_s"],
                                               "of_which_flat_search_s": r["search_s"]},
                    "search_vectors_one_query_per_call": {"value": 200 / sv["loop_s"], "sample": "200 of the 1000 queries"},
                    "what": "unmodified core.FAISSRetriever.search / unified_index.UnifiedIndex.search_vectors from "
                            "oracle/_ref over oracle/flat_ip_mt (FAISS absent)"}
        except Exception as e:
            out["config_a_100kx512_1000q"]["cpu_baseline"] = {"error": repr(e)[:300]}
    aidx.close()
    del aidx, xa
    torch.cuda.empty_cache()
    # ---- config B: near-duplicate pruning ----------------------------------------------
    n, d, w = 1_000_000, 512, 8
    x = gen_dedup_frames(n, d, dev)
    cos = torch.empty(n, dtype=torch.float32, device=dev)
    mask = torch.empty(n, dtype=torch.int32, device=dev)
    keep = torch.empty(n, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    nat.check(nat.lib.ivr_consecutive_cosine_device(dev.index, x.data_ptr(), n, d, cos.data_ptr(), st))
    torch.cuda.synchronize()
    cuts = torch.nonzero(cos[1:] < 0.75).flatten() + 1
    starts = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), cuts])
    ends = torch.cat([cuts, torch.tensor([n], device=dev)]) - 1
    ok = (ends - starts + 1) >= 2
    a, b = starts[ok].contiguous(), ends[ok].contiguous()
    nat.check(nat.lib.ivr_dedup_set_timing(1))
    ms2 = (C.c_float * 2)()
    runs = []
    for _ in range(12):
        nat.check(nat.lib.ivr_dedup_window_device(dev.index, x.data_ptr(), n, d, a.data_ptr(), b.data_ptr(),
                                                  a.numel(), w, C.c_float(0.95), keep.data_ptr(), cos.data_ptr(),
                                                  mask.data_ptr(), st))
        torch.cuda.synchronize()
        nat.check(nat.lib.ivr_dedup_last_timing(ms2))
        runs.append((ms2[0], ms2[1]))
    nat.check(nat.lib.ivr_dedup_set_timing(0))
    k_ms = statistics.median(r[0] for r in runs[2:])
    r_ms = statistics.median(r[1] for r in runs[2:])
    gbs = n * d * 4 / (k_ms * 1e-3) / 1e9
    leg = {"kernel": "banded_cosine_rw_kernel", "kernel_ms": k_ms, "resolve_ms": r_ms,
           "frames_per_s": n / ((k_ms + r_ms) * 1e-3), "kept": int(keep.sum().item()), "scenes": int(a.numel()),
           "roofline": hbm_roofline(gbs, peaks, n * d * 4)}
    # e2e: FrameFilter.apply_filters on PINNED host frames (2 GB H2D per call) -> kept indices on the host
    xh = torch.empty((n, d), dtype=torch.float32).pin_memory()
    xh.copy_(x)
    xnp = xh.numpy()
    ffl = ivr_b200.FrameFilter(window=w, threshold=0.95, transition_threshold=0.75, min_scene_length=2, device=dev.index)
    kept_e2e = ffl.apply_filters(xnp)
    t_e2e = time_host(lambda: ffl.apply_filters(xnp), reps=3, warm=1)
    leg["e2e"] = {"value": n / t_e2e, "unit": "frames/s", "seconds": t_e2e, "h2d_bytes_per_step": n * d * 4,
                  "d2h_bytes_per_step": int(n), "kept": int(len(kept_e2e)),
                  "h2d_gbs": n * d * 4 / t_e2e / 1e9,
                  "what": "FrameFilter.apply_filters(numpy float32 [n,d] in pinned host memory) -> kept indices"}
    if not args.no_cpu_baseline:
        try:                                                 # the reference's own filter.py on a bounded slice
            from oracle import ref_runner, ref_shims
            ns = min(args.cpu_dedup_frames, n)
            xs = xnp[:ns]
            if ref_shims.reference_available():
                r = ref_runner.time_filter_pipeline(xs, window=w, threshold=0.95, transition=0.75, min_scene=2)
                kept_gpu = ivr_b200.FrameFilter(window=w, threshold=0.95, transition_threshold=0.75, min_scene_length=2,
                                                device=dev.index).apply_filters(np.ascontiguousarray(xs))
                same = list(kept_gpu) == list(r["kept"])
                leg["cpu_baseline"] = {
                    "value": ns / r["seconds"], "unit": "frames/s", "cores": 1, "kind": "reference",
                    "what": "unmodified filter.py (142-315) from oracle/_ref: calculate_similarities -> scenes -> "
                            "filter_similar_frames_advanced; one Python thread by construction",
                    "sample": f"first {ns} of {n} frames ({r['seconds']:.1f} s of CPU work)",
                    "slice_parity": "ok (identical kept indices)" if same else
                                    f"differs ({len(kept_gpu)} vs {len(r['kept'])} kept; unguarded synthetic data may sit on a threshold)"}
        except Exception as e:
            leg["cpu_baseline"] = {"error": repr(e)[:300]}
    out["config_b_dedup_1Mx512_w8"] = leg
    return out


# ---------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    import ivr_b200
    from ivr_b200.sharded import ShardedFlatIP, partition_rows

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")        # one node: the controller's host-side group needs no
        dist.init_process_group("nccl", device_id=dev)           # resolvable hostname

    dim, k, nq, n_total = args.dim, args.k, args.nq, args.rows
    if n_total % GEN_CHUNK and n_total > GEN_CHUNK:
        raise SystemExit(f"--rows must be a multiple of {GEN_CHUNK}")
    chunk_rows = n_total if n_total < GEN_CHUNK else GEN_CHUNK

    cen = centres(dim, dev)
    q_host = gen_queries(nq, dim, cen.cpu()).pin_memory()
    q_dev = q_host.to(dev, non_blocking=True)
    n_chk = min(CHECK_QUERIES, nq)
    q_chk = q_dev[:n_chk]

    index = ShardedFlatIP(dim, device=local_rank) if world > 1 else None
    local = index.local if index else ivr_b200.IndexFlatIP(dim, device=local_rank)
    local.search_path = args.path
    torch.backends.cuda.matmul.allow_tf32 = False

    def build_shard(row0, row1, lo, hi):
        """Stores rows [lo, hi) of the synthetic matrix (generated chunk by chunk; a rank whose boundary falls inside
        a chunk keeps its part of it) and returns an exact fp32 top-k of the check queries over ITS OWN rows
        [row0, row1) -- the checker the parity gate merges across ranks."""
        local.reserve(hi - lo)
        bd = torch.full((n_chk, k), -float("inf"), device=dev)
        bi = torch.full((n_chk, k), -1, dtype=torch.int64, device=dev)
        for c in range(lo // chunk_rows, (hi + chunk_rows - 1) // chunk_rows):
            x = gen_rows(c, chunk_rows, dim, cen, dev)
            c0 = c * chunk_rows
            a, b = max(lo, c0), min(hi, c0 + chunk_rows)
            xs = x if b - a == chunk_rows else x[a - c0:b - c0].contiguous()
            if index:
                index.add_local(xs, lo, n_total)
            else:
                local.add(xs)
            a, b = max(row0, c0), min(row1, c0 + chunk_rows)
            if b > a:
                s = q_chk @ x[a - c0:b - c0].T
                d_, i_ = torch.topk(s, min(k, b - a), dim=1)
                cd, ci = torch.cat([bd, d_], 1), torch.cat([bi, i_ + a], 1)
                o = torch.argsort(cd, dim=1, descending=True, stable=True)[:, :k]
                bd, bi = torch.gather(cd, 1, o), torch.gather(ci, 1, o)
                del s
            del x, xs
        torch.cuda.synchronize()
        return bd, bi

    t_build = time.perf_counter()
    off = partition_rows(n_total, world)
    row0, row1 = int(off[rank]), int(off[rank + 1])
    # Elastic shard boundaries (N > 1): every rank also stores `margin` rows of either neighbour, so a boundary can
    # move between two searches without moving data; ShardedFlatIP's controller sizes the windows by the measured
    # scoring times (GPUs under the same power cap differ by a few per cent and drift with temperature).
    margin = 0 if (world == 1 or args.equal_shards) else int(args.shard_margin * (n_total // world)) // 1024 * 1024
    lo, hi = max(0, row0 - margin), min(n_total, row1 + margin)
    best_d, best_i = build_shard(row0, row1, lo, hi)
    if margin:
        index.enable_elastic(off, margin, period=8)
    t_build = time.perf_counter() - t_build

    def search_dev(q):
        return index.search(q, k) if index else local.search_tensor(q, k)

    def run_steps(n):
        """n searches back to back.  Sharded: two in flight -- the exchange + merge of search i run on the index's
        side stream while search i+1 is being scored (ShardedFlatIP.search_async); every result is complete and
        ordered into the timing stream before the closing event.  Returns the (D, I) of the last search."""
        out = None
        if not index:
            for _ in range(n):
                out = local.search_tensor(q_dev, k)
            return out
        prev = None
        for _ in range(n):
            h = index.search_async(q_dev, k)
            if prev is not None:
                prev.result(copy=False)
            prev = h
        return prev.result(copy=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity gate (outside every timed region) -------------------------------------
    D, I = search_dev(q_dev)
    torch.cuda.synchronize()
    if world > 1:                                                # exact reference: merge the per-rank exact lists
        gd = [torch.empty_like(best_d) for _ in range(world)]
        gi = [torch.empty_like(best_i) for _ in range(world)]
        dist.all_gather(gd, best_d); dist.all_gather(gi, best_i)
        cd, ci = torch.cat(gd, 1), torch.cat(gi, 1)
        o = torch.argsort(cd, dim=1, descending=True, stable=True)[:, :k]
        best_d, best_i = torch.gather(cd, 1, o), torch.gather(ci, 1, o)
    exact_d, exact_i = best_d.cpu().numpy(), best_i.cpu().numpy()
    parity = parity_report(D[:n_chk].cpu().numpy(), I[:n_chk].cpu().numpy(), exact_d, exact_i, k)
    del best_d, best_i

    # ---- value: whole-job throughput, inputs resident in HBM ---------------------------
    if margin:
        run_steps(4 * 8 + 2)                                     # four controller periods: the boundaries settle
    run_steps(args.warmup)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = run_steps(args.steps)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                          # before later searches can reuse the result buffers
        dump_outputs(args.dump_outputs, *last)
    del last
    ms_total = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_total, op=dist.ReduceOp.MAX)
    ms_step = ms_total.item() / args.steps
    value = nq / (ms_step * 1e-3)

    # ---- kernel roofline: score kernel duration from CUDA events on its launch stream ---
    local.set_timing(True)
    ks, merges, launches = [], [], None
    for _ in range(args.steps):
        search_dev(q_dev)
        t = local.last_timing()
        ks.append(t["score_ms"]); merges.append(t["merge_ms"])
        launches = t
    local.set_timing(False)
    k_ms = statistics.mean(ks)
    k_ranks = [k_ms]
    if world > 1:                                                # straggler spread: every rank's own scoring time
        kt = torch.tensor([k_ms], device=dev)
        kall = [torch.empty_like(kt) for _ in range(world)]
        dist.all_gather(kall, kt)
        k_ranks = [float(v.item()) for v in kall]
    rows_now = index.rows_per_rank if margin else None
    n_local = rows_now[rank] if margin else row1 - row0            # rows this rank scored in the last searches
    path = launches["path"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if path == "mma" and launches["kernel"] == "search_mma_small_kernel":
        # small batches: the tcgen05 kernel streams every row once for the whole batch -> HBM-bound
        ach = (float(n_local) * dim * 2) / (k_ms * 1e-3) / 1e9
        roofline = hbm_roofline(ach, peaks, float(n_local) * dim * 2,
                                traffic=measured_traffic(launches["kernel"], n_local, dim, nq, k),
                                kernel=launches["kernel"], kernel_ms=k_ms,
                                note="kernel_ms brackets the 2-3 seeded launches of one search and their merges")
    elif path == "mma":
        flops = 2.0 * n_local * dim * nq
        burst, sust = peaks.get("bf16_tflops") or 1590.0, peaks.get("bf16_tflops_sustained") or 1400.0
        ach = flops / (k_ms * 1e-3) / 1e12
        # the scoring stage runs back to back inside a seconds-long loop under the 1 kW cap: the sustained cuBLAS
        # figure is the comparable denominator; the burst fraction is printed beside it on every line
        roofline = {"bound": "tensor", "achieved": ach, "peak": sust, "unit": "TFLOP/s", "frac": ach / sust,
                    "frac_sustained": ach / sust, "frac_burst": ach / burst, "peak_burst": burst, "peak_sustained": sust,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained / bf16_tflops" if peaks.get("bf16_tflops")
                                   else "fallback 1400 / 1590 TFLOP/s",
                    "traffic": measured_traffic(launches["kernel"], n_local, dim, nq, k), "kernel": launches["kernel"],
                    "kernel_ms": k_ms, "algorithmic_flops_per_launch": flops,
                    "note": "kernel_ms brackets the whole scoring stage of one search: the short query-tile-resident "
                            "threshold-seeding launches (<1 %), the merges between launches (<1 %) and the "
                            "row-tile-resident launches (profiles/r2_launches_bench_n1.csv)"}
    else:
        passes = (nq + 3) // 4
        ach = (float(n_local) * dim * 2) / (k_ms * 1e-3) / 1e9   # events bracket the first pass of a multi-pass search
        roofline = hbm_roofline(ach, peaks, float(n_local) * dim * 2,
                                traffic=measured_traffic("search_stream_kernel", n_local, dim, nq, k),
                                kernel="search_stream_kernel", kernel_ms=k_ms, launches_per_step=passes)
    roofline["kernel_ms_per_rank"] = {"min": min(k_ranks), "max": max(k_ranks), "all": k_ranks}
    per_step_launches = launches["score_launches"] + launches["merge_launches"] + launches["prep_launches"]
    if world > 1:
        per_step_launches += 2 if index.exchange == "peer" else 1   # push kernel + the key merge after the exchange

    # ---- e2e: host buffers in, host results out, through the public API ----------------
    q_np = q_host.numpy()
    if world > 1:                                                # two steps in flight: device queries + pinned results x2
        qd2 = [torch.empty_like(q_dev) for _ in range(2)]
        res2 = [(torch.empty((nq, k), dtype=torch.float32).pin_memory(),
                 torch.empty((nq, k), dtype=torch.int64).pin_memory()) for _ in range(2)]

    def e2e_steps(n):
        """Every step: pinned host queries -> device, search, hits -> pinned host memory.  One GPU: the C ABI with HOST
        pointers (H2D + D2H inside the call).  Sharded: the D2H copies are queued behind the merge on the side
        stream and the host waits for step i after issuing step i+1 (two steps in flight)."""
        if world == 1:
            for _ in range(n):
                local.search(q_np, k)
            return
        prev = None
        for s_ in range(n):
            b = s_ % 2
            qd2[b].copy_(q_host, non_blocking=True)
            h = index.search_async(qd2[b], k).to_host(*res2[b])
            if prev is not None:
                prev.synchronize()
            prev = h
        prev.synchronize()

    e2e_steps(args.warmup)
    barrier()
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    barrier()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_val = nq / (t_e2e.item() / args.steps)

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only, bounded sample) -------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        xb_s, xq_s = cpu_sample(args, dev)
        cpu, _ = cpu_arm(args, xb_s, xq_s, steps=1, warmup=0)
        del xb_s

    balance = None
    if margin:
        # the same gate once more, with the shard boundaries where the controller has moved them (pipelined front end)
        D, I = index.search_async(q_dev, k).result(copy=True)
        torch.cuda.synchronize()
        again = parity_report(D[:n_chk].cpu().numpy(), I[:n_chk].cpu().numpy(), exact_d, exact_i, k)
        parity["after_the_boundaries_moved"] = {key: again[key] for key in
                                                ("status", "max_abs_score_error_vs_exact_fp32", "tie_band_substitutions")}
        log = index.balance_log
        balance = {"elastic_margin_rows": margin, "controller_period_searches": 8, "controller_steps": len(log),
                   "rows_per_rank_now": index.rows_per_rank,
                   "scoring_ms_per_rank_at_last_step": [round(t, 3) for t in log[-1][1]] if log else None,
                   "scoring_ms_per_rank_equal_shards": [round(t, 3) for t in log[0][1]] if log else None}
    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f16", "data": "synthetic",
               "config": workload_config(args),
               "run": {"storage": "fp16 rows, fp32 accumulate", "rows_per_gpu": n_local, "path": path,
                       "parallelism": (f"row-shard x{world}" if world > 1 else "one shard") + (
                           "" if world == 1 else
                           " + packed 64-bit keys pushed into peer mailboxes over NVLink (stream-ordered arrival wait)"
                           " + k-way merge; two searches in flight" if index.exchange == "peer" else
                           " + one all_gather of packed 64-bit keys + k-way merge"),
                       "exchange": index.exchange if index else None, "shard_balance": balance,
                       "rows_stored_per_gpu": hi - lo,
                       "build_s": round(t_build, 2)},
               "e2e": {"value": e2e_val, "unit": "queries/s", "h2d_bytes_per_step": nq * dim * 4,
                       "d2h_bytes_per_step": nq * k * 12},
               "gpu_launches": per_step_launches * args.steps,
               "roofline": roofline, "merge_ms": statistics.mean(merges),
               "outside_scoring_ms": ms_step - max(k_ranks),
               "clocks": clocks, "parity": parity}
        if cpu:
            out["cpu_baseline"] = cpu
        if world == 1 and not args.no_extras:
            local.close()                                            # free the 102 GB shard before the side legs
            torch.cuda.empty_cache()
            try:
                out["extras"] = run_extras(args, dev, peaks)
            except Exception as e:                                   # informational legs never sink the headline
                out["extras"] = {"error": repr(e)}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
