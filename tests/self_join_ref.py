"""Model of the exact range self-join (``IndexFlatIP.range_self_join``) and the checker of its tests (TEST
INFRASTRUCTURE ONLY).

A self-join scores the stored fp16 rows against each other with no query scaling, so ``oracle/fp16_model`` applies at
scale 1: the model score of a pair is the float64 product of the two stored rows, and the kernel's fp32 accumulation
stays within the model's bound eps of it.  On ``fp16_model.exact_inputs`` rows every accumulation order is exact and
the kernel must reproduce the model bit for bit.
"""
from __future__ import annotations

import numpy as np

from oracle import fp16_model as fm


def model_scores(rows16, cols16=None):
    """(m, eps): model scores and bounds, float64 [len(rows16), len(cols16)], of stored fp16 rows against stored fp16
    rows (default: all of ``rows16``).  A pair with a row holding a NaN scores NaN."""
    rows16 = np.asarray(rows16, np.float16)
    cols16 = rows16 if cols16 is None else np.asarray(cols16, np.float16)
    x = rows16.astype(np.float64)
    x = np.where(np.isnan(x), 0.0, x)
    m, eps = fm._scores(x, np.ones(x.shape[0]), cols16)
    m[np.isnan(rows16.astype(np.float64)).any(axis=1)] = np.nan
    return m, eps


def model_join(rows16, radius: float, id_offset: int = 0):
    """(lims, D float64, I int64) of the model: row i's hits are the j != i with model score > radius (fp32 radius),
    ordered by score descending, then lower id."""
    m, _ = model_scores(rows16)
    n = m.shape[0]
    r = float(np.float32(radius))
    lims, D, I = [0], [], []
    for i in range(n):
        with np.errstate(invalid="ignore"):
            j = np.nonzero(m[i] > r)[0]
        j = j[j != i]
        o = np.lexsort((j, -m[i, j]))
        D.append(m[i, j[o]])
        I.append(j[o] + id_offset)
        lims.append(lims[-1] + j.size)
    return (np.array(lims, np.int64), np.concatenate(D) if D else np.zeros(0),
            np.concatenate(I).astype(np.int64) if I else np.zeros(0, np.int64))


def _pairs(lims, D, I, id_offset):
    i = np.repeat(np.arange(lims.size - 1, dtype=np.int64), np.diff(lims))
    return i, I - id_offset, np.ascontiguousarray(D, np.float32).view(np.uint32)


def symmetry_violations(lims, D, I, id_offset: int = 0, tag: str = ""):
    """j in row i's list iff i in row j's list, with the same score bits (over the whole output)."""
    lims, I = np.asarray(lims, np.int64), np.asarray(I, np.int64)
    i, j, bits = _pairs(lims, np.asarray(D, np.float32), I, id_offset)
    fwd = np.lexsort((bits, j, i))
    bwd = np.lexsort((bits, i, j))
    if not (np.array_equal(i[fwd], j[bwd]) and np.array_equal(j[fwd], i[bwd]) and
            np.array_equal(bits[fwd], bits[bwd])):
        return [f"{tag}: the result is not symmetric (a pair, or its score bits, appear in one direction only)"]
    return []


def check_join(lims, D, I, rows16, radius: float, id_offset: int = 0, exact: bool = False,
               sample=None, ratios: dict | None = None, tag: str = "", block: int = 4096):
    """Violations of a self-join result against the model (empty list == pass).

    ``lims`` monotone from 0, n + 1 entries, ending at len(D) == len(I); the result symmetric; and for every row of
    ``sample`` (default: all): no self-hit, no duplicate, key order, every hit D > radius (fp32) and |D - m| <= eps
    (``exact``: D == m), no hit with a NaN model score, no pair left out with m - eps > radius (``exact``: the hits
    are exactly the j != i with m > radius).  ``ratios[tag]`` keeps the largest |D - m| / eps seen."""
    rows16 = np.asarray(rows16, np.float16)
    lims, D, I = np.asarray(lims, np.int64), np.asarray(D, np.float32), np.asarray(I, np.int64)
    n = rows16.shape[0]
    r = float(np.float32(radius))
    if lims.shape != (n + 1,) or lims[0] != 0 or np.any(np.diff(lims) < 0):
        return [f"{tag}: lims is not a monotone sequence of n + 1 entries starting at 0"]
    if not (int(lims[-1]) == D.size == I.size):
        return [f"{tag}: lims[-1] = {int(lims[-1])} but {D.size} scores and {I.size} ids"]
    if I.size and ((I - id_offset).min() < 0 or (I - id_offset).max() >= n):
        return [f"{tag}: ids out of range"]
    bad = symmetry_violations(lims, D, I, id_offset, tag)
    rows = np.arange(n) if sample is None else np.asarray(sample, np.int64)
    worst = 0.0
    for b0 in range(0, rows.size, block):
        blk = rows[b0:b0 + block]
        m, eps = model_scores(rows16[blk], rows16)
        for t, i in enumerate(blk):
            tg = f"{tag} row {i}"
            a, z = lims[i], lims[i + 1]
            ids, d = I[a:z] - id_offset, D[a:z]
            if np.any(ids == i):
                bad.append(f"{tg}: a self-hit")
            if np.unique(ids).size != ids.size:
                bad.append(f"{tg}: duplicate ids")
            if np.any(~(d > np.float32(r))):
                bad.append(f"{tg}: a hit scores {d[~(d > np.float32(r))][0]!r}, not above the radius {r!r}")
            mh, eh = m[t, ids], eps[t, ids]
            if np.any(np.isnan(mh)):
                bad.append(f"{tg}: a pair with a NaN score is a hit")
            elif ids.size:
                err = np.abs(d.astype(np.float64) - mh)
                worst = max(worst, float((err / eh).max()))
                if exact and np.any(d != mh):
                    bad.append(f"{tg}: a hit's score differs from the model (exact inputs)")
                elif np.any(err > eh):
                    k = int(np.argmax(err / eh))
                    bad.append(f"{tg}: |D - m| = {err[k]:.3e} > eps {eh[k]:.3e} at id {ids[k]}")
            bad += fm._order_violations(tg, d, ids)
            out = np.ones(n, bool)
            out[ids] = False
            out[i] = False
            with np.errstate(invalid="ignore"):
                low = np.where(out & ~np.isnan(m[t]), m[t] - eps[t], -np.inf)
                if low.max(initial=-np.inf) > r:
                    bad.append(f"{tg}: pair ({i}, {int(np.argmax(low))}) with m - eps = {low.max()!r} > radius "
                               f"{r!r} is missing")
                if exact and np.any(out & (m[t] > r)):
                    bad.append(f"{tg}: {int(np.sum(out & (m[t] > r)))} pairs with a model score above the radius "
                               "are not hits")
            if len(bad) > 20:
                bad.append("... (truncated)")
                break
        if len(bad) > 20:
            break
    if ratios is not None:
        ratios[tag] = max(ratios.get(tag, 0.0), worst)
    return bad


def kth_radius(rows16, k: int, sample=None) -> float:
    """The median over (sampled) rows of the k-th best model score to another row: about k hits per row."""
    rows16 = np.asarray(rows16, np.float16)
    n = rows16.shape[0]
    rows = np.arange(n) if sample is None else np.asarray(sample)
    m, _ = model_scores(rows16[rows], rows16)
    m[np.arange(rows.size), rows] = -np.inf
    m = np.where(np.isnan(m), -np.inf, m)
    k = max(1, min(k, n - 1))
    return float(np.float32(np.median(-np.partition(-m, k - 1, axis=1)[:, k - 1])))
