"""Oracle and comparator for FAISS's flat-index range query (TEST INFRASTRUCTURE ONLY).

``lims, D, I = index.range_search(x, radius)`` of ``faiss.IndexFlatIP`` -- not called by the reference.  Contract
restated (published FAISS behaviour): a row is a hit iff its fp32 inner product with the query is STRICTLY greater
than the radius (compared in float32, the type FAISS takes the radius in); query i's hits are
``D[lims[i]:lims[i+1]]`` / ``I[lims[i]:lims[i+1]]`` (the ``RangeSearchResult`` layout).  FAISS promises no order
within a query; this oracle orders by score descending, then lower id, so that its output is canonical.

PARITY UNPINNED against real FAISS (absent here; see oracle/__init__.py).

``compare_range`` reads the project's 1e-3 tolerance as a band around the radius: every returned id has an oracle
score > radius - tol, every oracle id with a score > radius + tol is returned, ids are unique per query, each score is
within tol of the oracle's, scores do not increase within a query, and ``lims`` is monotone from 0 with
``lims[-1] == len(D) == len(I)``.
"""
from __future__ import annotations

import numpy as np

TOL = 1e-3


def range_search(xb: np.ndarray, x: np.ndarray, radius: float, *, db_block: int = 1 << 18):
    """Exact fp32 range search of queries ``x`` [nq, d] over rows ``xb`` [n, d] (e.g. ``flat_ip.IndexFlatIP.xb``);
    ids are row positions.  Returns (lims int64 [nq + 1], D float32, I int64)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    xb = np.ascontiguousarray(xb, dtype=np.float32)
    if x.ndim != 2 or xb.ndim != 2 or x.shape[1] != xb.shape[1]:
        raise ValueError(f"range_search expects [nq,d] queries over [n,d] rows, got {x.shape} and {xb.shape}")
    r = np.float32(radius)
    nq = x.shape[0]
    ds, ids = [[] for _ in range(nq)], [[] for _ in range(nq)]
    for r0 in range(0, xb.shape[0], db_block):
        s = x @ xb[r0:r0 + db_block].T
        for q in range(nq):
            sel = np.nonzero(s[q] > r)[0]
            ds[q].append(s[q, sel])
            ids[q].append(sel.astype(np.int64) + r0)
    lims = np.zeros(nq + 1, np.int64)
    D, I = [], []
    for q in range(nq):
        d = np.concatenate(ds[q]).astype(np.float32) if ds[q] else np.zeros(0, np.float32)
        i = np.concatenate(ids[q]) if ids[q] else np.zeros(0, np.int64)
        order = np.lexsort((i, -d))
        D.append(d[order])
        I.append(i[order])
        lims[q + 1] = lims[q] + d.size
    return (lims, np.concatenate(D) if D else np.zeros(0, np.float32),
            np.concatenate(I) if I else np.zeros(0, np.int64))


def compare_range(lims, D, I, lims_ref, D_ref, I_ref, score_of, radius: float, tol: float = TOL):
    """Range-search parity (see the module docstring); returns a list of violations (empty list == parity).

    ``score_of(q, ids[m]) -> float32[m]`` gives the ORACLE's fp32 score of arbitrary ids for query q.
    """
    lims, D, I, lims_ref, D_ref, I_ref = map(np.asarray, (lims, D, I, lims_ref, D_ref, I_ref))
    bad = []
    if lims.shape != lims_ref.shape:
        return [f"lims has {lims.size} entries, oracle {lims_ref.size}"]
    if lims.size == 0 or lims[0] != 0 or np.any(np.diff(lims) < 0):
        return ["lims is not a monotone sequence starting at 0"]
    if not (int(lims[-1]) == D.size == I.size):
        return [f"lims[-1]={int(lims[-1])} but {D.size} scores and {I.size} ids"]
    if I.dtype != np.int64 or D.dtype != np.float32:
        bad.append(f"dtype mismatch D={D.dtype} I={I.dtype}")
    for q in range(lims.size - 1):
        ids, d = I[lims[q]:lims[q + 1]], D[lims[q]:lims[q + 1]]
        ref_ids, ref_d = I_ref[lims_ref[q]:lims_ref[q + 1]], D_ref[lims_ref[q]:lims_ref[q + 1]]
        if len(np.unique(ids)) != ids.size:
            bad.append(f"q{q}: duplicate ids")
        if np.any(d[1:] > d[:-1]):
            bad.append(f"q{q}: scores not non-increasing")
        os_ = np.asarray(score_of(q, ids), np.float32) if ids.size else np.zeros(0, np.float32)
        if np.any(os_ <= radius - tol):
            j = int(np.argmin(os_))
            bad.append(f"q{q}: id {ids[j]} has oracle score {os_[j]:.6f} <= radius-tol ({radius:.6f})")
        missing = np.setdiff1d(ref_ids[ref_d > radius + tol], ids)
        if missing.size:
            bad.append(f"q{q}: {missing.size} oracle ids above radius+tol missing, e.g. {missing[:3]}")
        err = np.abs(d - os_)
        if np.any(err > tol):
            j = int(np.argmax(err))
            bad.append(f"q{q}: score err {err[j]:.2e} at id {ids[j]}")
        if len(bad) > 20:
            bad.append("... (truncated)")
            break
    return bad
