"""The cosine arithmetic of ``dedup.cu`` and ``sequence.cu`` restated in float64, with proven error bounds
(TEST INFRASTRUCTURE ONLY).

The frame-filter, chain, sequence and clustering kernels make threshold decisions on fp32 cosines: ``cos >= thr``
(duplicate), ``cos < transition`` (scene cut, strict), ``1 - cos <= eps`` (neighbour), ``mean >= thr`` (sequence
hit).  The suite used to keep every cosine 1e-4 away from every threshold.  This module instead bounds how far each
kernel's cosine can lie from the exact one, so that a decision is checked wherever it is forced and counted as
"in the band" where either outcome is admissible.

Reference semantics (``exact_cos``; sklearn's ``cosine_similarity`` on fp32 rows, evaluated exactly): each row is
divided by its norm, a zero norm is replaced by 1 (cosine 0); a row whose sum of squares overflows fp32 divides by
inf and becomes a zero row (cosine 0); a NaN component, or an inf one (inf / inf), makes the row NaN and every
cosine with it NaN.  NaN fails every comparison: not a duplicate, not a cut, not a neighbour, not a hit.

The bounds (``pair_bound``).  u = 2^-24 is the unit roundoff of fp32; every correctly rounded operation (FMA, add,
multiply, divide, sqrt) returns v(1 + d) with |d| <= u, plus an absolute error of at most 2^-150 when the result is
subnormal.  A sum whose every term passes through at most n roundings is off by at most gamma_n * sum|terms|,
gamma_n = n u / (1 - n u) <= n U with U = 2^-23 (n u <= 1/2 throughout).  Each absolute subnormal error is bounded
by TINY = 2^-149 and there are fewer than d + 64 operations per sum.

1. Sum of squares, ``n_s`` roundings deep: fl(ss) = ss (1 + t), |t| <= theta = n_s U + (d + 64) TINY / ss.  All terms
   are positive, so the relative bound needs no Cauchy-Schwarz.  When ss is subnormal, TINY / ss is large: the bound
   widens with it, and at theta >= 1/2 (fl(ss) may be 0) it is infinite.
2. 1/||x|| from fl(ss): 1/sqrt(1 + t) - 1 <= theta / (2 (1 - theta)^1.5), then the ``extra`` roundings of sqrt,
   reciprocal or division, and of the multiply by the factor: x^_i = (x_i / ||x||)(1 + a_i), |a_i| <= rho =
   (1 + theta / (2 (1 - theta)^1.5)) (1 + U)^extra - 1.
3. The dot of two such rows, ``n_dot`` roundings deep: with Cauchy-Schwarz, sum |x_i y_i| / (||x|| ||y||) <= 1, so
       |cos_kernel - cos| <= ((1 + rho_x)(1 + rho_y) - 1) + n_dot U (1 + rho_x)(1 + rho_y) + (2d + 64) TINY,
   independent of the data except through theta.

Chains per kernel (``STEPS``; d = frame dimension):

- ``banded`` (``banded_cosine_kernel``, both DV > 0 and DV == 0) and ``chain`` (``chain_resolve_kernel``): a per-lane
  FMA chain of ceil(d/32), then 5 butterfly adds, for the sum of squares and for the dot; sqrtf, then 1/nrm and a
  multiply (DV > 0) or one division (DV == 0, and ``fmaf(p/ni, q/nq, acc)`` in the chain kernel): extra = 3 covers both.
- ``rw`` (``banded_cosine_rw_kernel``): two FFMA2 partial chains of d/64 per lane, their sum, 5 butterfly adds
  (n_s = d/64 + 6); the dot takes the same two chains, their sum and the 8-way transpose reduction (3 adds) plus 2
  more shuffle adds (n_dot = d/64 + 6).  The dot is taken with the RAW current row x and the normalised window row
  y^, then multiplied by 1/||x||: that is the same expression with x^ = x * inv, up to one more rounding, plus an
  absolute subnormal term (d + 64) TINY / ||x|| that matters only for tiny rows.  1/||x|| is rsqrt + one Newton step.
  If MUFU.RSQ is within 2^-12 relative (its documented bound is 2 ulp), the Newton step squares that error to below
  2^-24 and adds three roundings: about 2 U in all.  The claim is not measured, so ``K_RSQ`` gives the factor 8 U;
  the range outside the Newton path uses 1/sqrtf (2 roundings) and is covered by the same 8 U.
- ``seq`` (``seq_normalize_kernel`` + ``seq_cosine_kernel``): the normalisation is the banded one with a division
  (extra = 2), but the cosine is ONE sequential FMA chain over all d products: n_dot = d, a much wider bound.
- ``ref``: the reference's own fp32 evaluation (numpy einsum + sqrt + division, then a BLAS dot), order unknown:
  every path at most d + 1 roundings deep.

The sequence mean (``numpy_mean_f32``: pairwise sum of L cosines, then one division) adds
depth U sum|c_k| / L + U |mean| with depth = L for L < 8 and (L // 8 - 1) + 3 + L % 8 otherwise.

``exact_frames`` builds frames on which every kernel's arithmetic is exact (cosines j / 64), ``near_threshold_frames``
frames whose cosines sit within a few ulp of a threshold.  The checkers replay each greedy rule on the kernel's OWN
earlier decisions, so one admissible flip inside the band does not cascade, and report how many decisions fell
inside the band.
"""
from __future__ import annotations

import math
from typing import NamedTuple

import numpy as np

U = 2.0 ** -23                  # per-rounding relative bound (twice the unit roundoff of fp32)
TINY = 2.0 ** -149              # smallest fp32 subnormal
FLT_MAX = float(np.finfo(np.float32).max)
K_RSQ = 8                       # rounding units allowed for rsqrt + Newton (proven ~2, unmeasured: x4 slack)
EXACT_NNZ = 64                  # non-zeros of an exact frame: norm 8, cosines j / 64


def steps(kernel: str, d: int):
    """(n_s, extra, n_dot) of ``kernel`` at dimension d (see the module docstring)."""
    c32 = -(-d // 32)
    if kernel in ("banded", "chain"):
        return c32 + 5, 3, c32 + 5
    if kernel == "rw":
        if d % 128:
            raise ValueError("the register-window kernel takes d = 384 or 512")
        return d // 64 + 6, K_RSQ + 1, d // 64 + 6
    if kernel == "seq":
        return c32 + 5, 2, d
    if kernel == "ref":
        return d + 1, 2, d + 1
    raise ValueError(f"unknown kernel {kernel!r}")


# ---------------------------------------------------------------------------
# exact cosines (reference semantics)
# ---------------------------------------------------------------------------
class Rows(NamedTuple):
    xn: np.ndarray      # float64 [n, d] normalised rows (NaN rows NaN, zero / overflowed rows 0)
    ss: np.ndarray      # float64 [n] exact sum of squares (0 for non-finite rows)
    amb: np.ndarray     # bool [n]: the fp32 sum of squares may or may not overflow
    bad: np.ndarray     # bool [n]: a NaN or inf component


def rows(x) -> Rows:
    x = np.asarray(x, np.float32)
    if x.ndim == 1:
        x = x[None, :]
    x64 = x.astype(np.float64)
    bad = ~np.isfinite(x64).all(axis=1)
    x64 = np.where(bad[:, None], 0.0, x64)
    ss = np.einsum("ij,ij->i", x64, x64)
    slack = (x.shape[1] + 64) * U
    amb = (ss >= FLT_MAX * (1 - slack)) & (ss <= FLT_MAX * (1 + slack) + 2.0 ** 104)
    over = ss > FLT_MAX
    nrm = np.sqrt(np.where((ss == 0) | over, 1.0, ss))
    xn = x64 / nrm[:, None]
    xn[over] = 0.0
    xn[bad] = np.nan
    return Rows(xn, ss, amb, bad)


def exact_cos(x, y) -> float:
    """cos(x, y) of two fp32 rows with the reference's semantics, computed exactly (float64 on fp32 inputs)."""
    r = rows(np.stack([np.asarray(x, np.float32).reshape(-1), np.asarray(y, np.float32).reshape(-1)]))
    return float(r.xn[0] @ r.xn[1])


def pair_cos(r: Rows, i, j) -> np.ndarray:
    return np.einsum("ij,ij->i", r.xn[np.asarray(i)], r.xn[np.asarray(j)])


def _rho(r: Rows, idx, n_s: int, extra: int, d: int) -> np.ndarray:
    ss = r.ss[idx]
    with np.errstate(divide="ignore"):
        theta = n_s * U + np.where(ss > 0, (d + 64) * TINY / np.where(ss > 0, ss, 1.0), 0.0)
    exact_zero = (ss == 0) | (ss > FLT_MAX)                  # the kernel's row is exactly 0 (or NaN for bad rows)
    with np.errstate(invalid="ignore"):
        ra = theta / (2.0 * (1.0 - np.minimum(theta, 0.5)) ** 1.5)
    rho = (1.0 + ra) * (1.0 + U) ** extra - 1.0
    rho = np.where(theta >= 0.5, np.inf, rho)
    rho = np.where(exact_zero, 0.0, rho)
    return np.where(r.amb[idx], np.inf, rho)


def pair_bound(r: Rows, i, j, kernel: str) -> np.ndarray:
    """|cos_kernel(x_i, x_j) - cos_exact| bound per pair; for ``rw`` row i is the current (raw) frame."""
    i, j = np.asarray(i), np.asarray(j)
    d = r.xn.shape[1]
    n_s, extra, n_dot = steps(kernel, d)
    px, py = _rho(r, i, n_s, extra, d), _rho(r, j, n_s, extra, d)
    g = (1.0 + px) * (1.0 + py)
    b = (g - 1.0) + n_dot * U * g + (2 * d + 64) * TINY
    if kernel == "rw":
        nrm = np.sqrt(r.ss[i])
        with np.errstate(divide="ignore", invalid="ignore"):
            b = b + np.where(nrm > 0, (d + 64) * TINY * (1.0 + px) / np.where(nrm > 0, nrm, 1.0), 0.0) + TINY
    return b


def banded(r: Rows, window: int, kernel: str):
    """(E, B) float64 [n, window]: exact cos(e_i, e_{i-l}) and its bound at column l - 1 (NaN where i - l < 0)."""
    n = r.xn.shape[0]
    E = np.full((n, window), np.nan)
    B = np.full((n, window), np.nan)
    for l in range(1, window + 1):
        if l < n:
            i = np.arange(l, n)
            E[l:, l - 1] = pair_cos(r, i, i - l)
            B[l:, l - 1] = pair_bound(r, i, i - l, kernel)
    return E, B


def mean_depth(L: int) -> int:
    return L if L < 8 else (L // 8 - 1) + 3 + L % 8


def mean_f32(v) -> np.ndarray:
    """``numpy_mean_f32`` (sequence.cu) vectorised over the leading axes of float32 v [..., L]."""
    v = np.asarray(v, np.float32)
    f = np.float32
    L = v.shape[-1]
    if L < 8:
        res = np.zeros(v.shape[:-1], f)
        for k in range(L):
            res = (res + v[..., k]).astype(f)
    else:
        r8 = [v[..., k].copy() for k in range(8)]
        i = 8
        while i < L - L % 8:
            for k in range(8):
                r8[k] = (r8[k] + v[..., i + k]).astype(f)
            i += 8
        res = (((r8[0] + r8[1]).astype(f) + (r8[2] + r8[3]).astype(f)).astype(f) +
               ((r8[4] + r8[5]).astype(f) + (r8[6] + r8[7]).astype(f)).astype(f)).astype(f)
        while i < L:
            res = (res + v[..., i]).astype(f)
            i += 1
    return (res / f(L)).astype(f)


# ---------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------
def exact_frames(n: int, d: int, seed: int, moves=(0, 1, 2, 3, 4), p_new: float = 0.05, p_transition: float = 0.05):
    """Frames [n, d] (fp32) of EXACT_NNZ entries +-1 and zeros elsewhere: every norm is 8, every normalised entry
    +-1/8 and every partial sum of products a multiple of 1/64 below 2^7 -- exact in fp32 under any order, and the
    cosines are j / 64.  Each frame is the previous one with k entries moved to an unused coordinate (cosine
    (64 - k) / 64 to it), or exactly 16 moved (cosine 48/64 = 0.75), or a fresh frame."""
    if d < EXACT_NNZ + 16:
        raise ValueError(f"d >= {EXACT_NNZ + 16} needed")
    rng = np.random.default_rng(seed)
    x = np.zeros((n, d), np.float32)

    def fresh():
        v = np.zeros(d, np.float32)
        v[rng.choice(d, EXACT_NNZ, replace=False)] = rng.choice(np.float32([-1, 1]), EXACT_NNZ)
        return v

    cur = fresh()
    for i in range(n):
        if i:
            u = rng.random()
            if u < p_new:
                cur = fresh()
            else:
                k = 16 if u < p_new + p_transition else int(rng.choice(moves))
                cur = cur.copy()
                on = np.flatnonzero(cur)
                off = np.flatnonzero(cur == 0)
                src = rng.choice(on, k, replace=False)
                dst = rng.choice(off, k, replace=False)
                cur[dst] = rng.choice(np.float32([-1, 1]), k)
                cur[src] = 0
        x[i] = cur
    return x


def _toward(x, c, rng):
    """A float64 unit vector whose cosine to x is c: c x^ + sqrt(1 - c^2) z^, z orthogonal to x."""
    xh = x / np.linalg.norm(x)
    z = rng.standard_normal(x.shape[0])
    z -= (z @ xh) * xh
    z /= np.linalg.norm(z)
    return c * xh + math.sqrt(max(0.0, 1.0 - c * c)) * z


def near_threshold_frames(n: int, d: int, thr: float, transition: float, seed: int, window: int = 8,
                          scale: float = 3.0):
    """Frames [n, d] (fp32, scale ~3 like the synthetic dedup data) whose cosines lie within a few ulp of ``thr`` (to
    a random look-back 1..window) or of ``transition`` (to the previous frame), mixed with ordinary near-duplicates
    and fresh frames (scene cuts).  Solved in float64, rounded to fp32: the adversarial input the guard band avoided."""
    rng = np.random.default_rng(seed)
    x = np.zeros((n, d), np.float64)
    x[0] = rng.standard_normal(d)
    x[0] *= scale / np.linalg.norm(x[0])
    for i in range(1, n):
        u = rng.random()
        if u < 0.35:
            lag = int(rng.integers(1, window + 1)) if i >= window else int(rng.integers(1, i + 1))
            v = _toward(x[i - lag], thr, rng)
        elif u < 0.5:
            v = _toward(x[i - 1], transition, rng)
        elif u < 0.58:
            v = rng.standard_normal(d)
        else:
            v = _toward(x[i - 1], rng.uniform(thr - 0.04, 1.0), rng)
        x[i] = v / np.linalg.norm(v) * scale * rng.uniform(0.5, 2.0)
    return x.astype(np.float32)


# ---------------------------------------------------------------------------
# checkers
# ---------------------------------------------------------------------------
class Report(NamedTuple):
    violations: list    # empty == pass
    in_band: int        # decisions where both outcomes are admissible
    ties: int           # decisions whose exact value equals the threshold


def _decide_ge(e, b, t):
    """+1: e >= t is forced, -1: forbidden, 0: in the band.  NaN never passes."""
    if np.isnan(e):
        return -1
    if e - b >= t:
        return 1
    if e + b < t:
        return -1
    return 0


def _decide_lt(e, b, t):
    if np.isnan(e):
        return -1
    if e + b < t:
        return 1
    if e - b >= t:
        return -1
    return 0


def _scenes_from(cos_prev, n, transition, min_len):
    cuts = [i for i in range(1, n) if cos_prev[i] < np.float32(transition)]
    starts = [0] + cuts
    ends = cuts + [n]
    return [(s, e - 1) for s, e in zip(starts, ends) if e - s >= min_len]


def check_frame_filter(x, keep, cos_prev, stats, window: int, thr: float, transition: float, min_len: int,
                       kernel: str, exact: bool = False) -> Report:
    """``ivr_frame_filter`` output (keep [n], cos_prev [n], stats [scenes, frames]) against the model.

    cos_prev is within the bound of ``exact_cos`` (bit-equal with ``exact``); the scene split and ``stats`` follow
    bit-exactly from the returned cos_prev; inside each scene the window rule is replayed on the returned keep flags:
    a dropped frame needs a kept frame in its window whose cosine may be >= thr, a kept frame may have none whose
    cosine must be >= thr.  The look-back-1 decision follows bit-exactly from cos_prev (it is the same fp32 value)."""
    x = np.asarray(x, np.float32)
    n = x.shape[0]
    keep = np.asarray(keep).astype(bool)
    cp = np.asarray(cos_prev, np.float32)
    t32, tr32 = float(np.float32(thr)), float(np.float32(transition))
    r = rows(x)
    W = max(window, 1)
    E, B = banded(r, W, kernel)
    if exact:
        B = np.where(np.isnan(B), B, 0.0)
    v, band, ties = [], 0, 0
    if n and cp[0] != 1.0:
        v.append(f"frame 0: cos_prev {cp[0]} != 1")
    for i in range(1, n):
        e, b, c = E[i, 0], B[i, 0], float(cp[i])
        if np.isnan(e):
            if not np.isnan(c):
                v.append(f"frame {i}: cos_prev {c!r}, exact NaN")
        elif not (abs(c - e) <= b):
            v.append(f"frame {i}: cos_prev {c!r}, exact {e!r}, bound {b:.3g}")
        dec = _decide_lt(e, b, tr32)
        band += dec == 0
        ties += e == tr32
    scenes = _scenes_from(cp, n, transition, min_len)
    want_stats = [len(scenes), sum(e - s + 1 for s, e in scenes)]
    if stats is not None and [int(stats[0]), int(stats[1])] != want_stats:
        v.append(f"stats {[int(stats[0]), int(stats[1])]} != {want_stats} from the returned cos_prev")
    inside = np.zeros(n, bool)
    for s, e_ in scenes:
        inside[s:e_ + 1] = True
    for i in np.flatnonzero(keep & ~inside)[:5]:
        v.append(f"frame {i}: kept outside every scene")
    for s, e_ in scenes:
        for i in range(s, e_ + 1):
            if i == s or window <= 0:
                if not keep[i]:
                    v.append(f"frame {i}: {'scene start' if i == s else 'empty window'} dropped")
                continue
            must, can = False, False
            for j in range(max(s, i - window), i):
                if not keep[j]:
                    continue
                if i - j == 1:
                    dec = 1 if float(cp[i]) >= t32 else -1
                    d0 = _decide_ge(E[i, 0], B[i, 0], t32)
                    band += d0 == 0
                else:
                    dec = _decide_ge(E[i, i - j - 1], B[i, i - j - 1], t32)
                    band += dec == 0
                ties += E[i, i - j - 1] == t32
                must |= dec == 1
                can |= dec >= 0
            if keep[i] and must:
                v.append(f"frame {i}: kept, but a kept frame in its window must be a duplicate")
            if not keep[i] and not can:
                v.append(f"frame {i}: dropped, but no kept frame in its window can be a duplicate")
    return Report(v, int(band), int(ties))


def check_chain(x, keep, scenes, min_distance: int, thr: float, force_last: bool, fifo: int = 1,
                exact: bool = False) -> Report:
    """``ivr_dedup_chain`` (fifo = 1: last-kept rule, min_distance, force_last) and ``ivr_dedup_fifo`` (FIFO of the
    last ``fifo`` kept frames) replayed on the returned keep flags: a frame is unique iff its cosine to every FIFO
    entry is < thr.  (The kernel counts a NaN cosine as "not < thr"; frames here are finite.)"""
    x = np.asarray(x, np.float32)
    n = x.shape[0]
    keep = np.asarray(keep).astype(bool)
    t32 = float(np.float32(thr))
    r = rows(x)
    v, band, ties = [], 0, 0
    inside = np.zeros(n, bool)
    for a, b in scenes:
        a, b = max(a, 0), min(b, n - 1)
        if a > b:
            continue
        inside[a:b + 1] = True
        if not keep[a]:
            v.append(f"frame {a}: scene start dropped")
        fq, last = [a], a
        for i in range(a + 1, b + 1):
            forced = force_last and i == b
            if i - last < min_distance:
                if keep[i] != forced:
                    v.append(f"frame {i}: keep {int(keep[i])} inside min_distance of frame {last}")
                continue
            must, can = False, False
            for p in fq:
                e = float(pair_cos(r, [i], [p])[0])
                bnd = 0.0 if exact else float(pair_bound(r, [i], [p], "chain")[0])
                dec = _decide_ge(e, bnd, t32)
                band += dec == 0
                ties += e == t32
                must |= dec == 1
                can |= dec >= 0
            if not forced:
                if keep[i] and must:
                    v.append(f"frame {i}: kept, but it must duplicate a FIFO frame")
                if not keep[i] and not can:
                    v.append(f"frame {i}: dropped, but it cannot duplicate any FIFO frame")
            elif not keep[i]:
                v.append(f"frame {i}: last frame of the scene not kept")
            if keep[i]:
                last = i
                fq.append(i)
                if len(fq) > fifo:
                    fq.pop(0)
    for i in np.flatnonzero(keep & ~inside)[:5]:
        v.append(f"frame {i}: kept outside every scene")
    return Report(v, int(band), int(ties))


def window_sims(target, db, L: int, kernel: str = "seq"):
    """(M, Bm, C32): exact window means float64 [nt-L+1, nd-L+1], their bounds, and the exact cosines as fp32 means
    (``mean_f32`` of the exact cosines: bit-equal to the kernel on exact frames)."""
    rt, rd = rows(target), rows(db)
    nt, nd = rt.xn.shape[0] - L + 1, rd.xn.shape[0] - L + 1
    C = rt.xn @ rd.xn.T
    d = rt.xn.shape[1]
    n_s, extra, n_dot = steps(kernel, d)
    pt, pd = _rho(rt, np.arange(rt.xn.shape[0]), n_s, extra, d), _rho(rd, np.arange(rd.xn.shape[0]), n_s, extra, d)
    G = (1.0 + pt)[:, None] * (1.0 + pd)[None, :]
    Bc = (G - 1.0) + n_dot * U * G + (2 * d + 64) * TINY
    band = np.stack([C[k:k + nt, k:k + nd] for k in range(L)], axis=-1)
    bb = np.stack([Bc[k:k + nt, k:k + nd] for k in range(L)], axis=-1)
    M = band.mean(axis=-1)
    mb = bb.mean(axis=-1)
    sabs = np.abs(band).mean(axis=-1) + mb
    Bm = mb + mean_depth(L) * U * sabs + U * sabs * (1 + mean_depth(L) * U) + TINY
    with np.errstate(invalid="ignore"):
        M32 = mean_f32(band.astype(np.float32))
    return M, Bm, M32


def check_sequence_hits(target, db, L: int, thr: float, ht, hj, hs, ordered=None, exact: bool = False) -> Report:
    """Raw ``ivr_sequence_similarity`` hits (target start, db start, sim) against the model: no window twice; every
    sim >= thr (fp32) and within the bound of the exact mean (bit-equal to the fp32 mean of the exact cosines with
    ``exact``); every window whose exact mean is >= thr + bound present, none below thr - bound.  ``ordered``: the
    ``find_similar_sequences`` list [(db start, sim)], which must be the hits by sim descending, then target start,
    then db start."""
    ht, hj, hs = np.asarray(ht, np.int64), np.asarray(hj, np.int64), np.asarray(hs, np.float32)
    t32 = np.float32(thr)
    M, Bm, M32 = window_sims(target, db, L)
    if exact:
        Bm = np.zeros_like(Bm)
    v, band = [], 0
    got = np.zeros(M.shape, bool)
    for t, j, s in zip(ht, hj, hs):
        if not (0 <= t < M.shape[0] and 0 <= j < M.shape[1]):
            v.append(f"hit ({t}, {j}) outside the window grid")
            continue
        if got[t, j]:
            v.append(f"window ({t}, {j}) returned twice")
        got[t, j] = True
        if not s >= t32:
            v.append(f"window ({t}, {j}): sim {s!r} below the threshold")
        if exact:
            if s != M32[t, j]:
                v.append(f"window ({t}, {j}): sim {s!r} != fp32 mean of the exact cosines {M32[t, j]!r}")
        elif not abs(float(s) - M[t, j]) <= Bm[t, j]:
            v.append(f"window ({t}, {j}): sim {s!r}, exact {M[t, j]!r}, bound {Bm[t, j]:.3g}")
    ref = M32 if exact else M
    with np.errstate(invalid="ignore"):
        must = (ref - Bm >= t32) & ~np.isnan(ref)
        mustnot = (ref + Bm < t32) | np.isnan(ref)
    band = int((~must & ~mustnot).sum())
    ties = int((ref == t32).sum())
    for t, j in np.argwhere(must & ~got)[:5]:
        v.append(f"window ({t}, {j}): exact mean {M[t, j]!r} must be a hit")
    for t, j in np.argwhere(mustnot & got)[:5]:
        v.append(f"window ({t}, {j}): exact mean {M[t, j]!r} must not be a hit")
    if ordered is not None:
        order = sorted(range(len(hs)), key=lambda k: (-float(hs[k]), int(ht[k]), int(hj[k])))
        want = [(int(hj[k]), float(hs[k])) for k in order]
        if [(int(a), float(b)) for a, b in ordered] != want:
            v.append("find_similar_sequences order is not sim descending, target start, db start")
    return Report(v, band, ties)


def check_adjacency(x, eps: float, adj, exact: bool = False, block: int = 1024) -> Report:
    """``ivr_cosine_neighbors`` bits (uint32 [n, words]) against the rule fl(1 - cos) <= eps, per bit: forced where
    1 - exact +- (bound + rounding of the subtraction) stays on one side of eps."""
    x = np.asarray(x, np.float32)
    n = x.shape[0]
    bits = np.unpackbits(np.ascontiguousarray(adj, np.uint32).view(np.uint8), axis=1, bitorder="little")[:, :n]
    bits = bits.astype(bool)
    e32 = float(np.float32(eps))
    r = rows(x)
    d = x.shape[1]
    n_s, extra, n_dot = steps("seq", d)
    p = _rho(r, np.arange(n), n_s, extra, d)
    v, band, ties = [], 0, 0
    for i0 in range(0, n, block):
        C = r.xn[i0:i0 + block] @ r.xn.T
        dist = 1.0 - C
        if exact:
            Bt = np.zeros_like(C)
        else:
            G = (1.0 + p[i0:i0 + block])[:, None] * (1.0 + p)[None, :]
            Bc = (G - 1.0) + n_dot * U * G + (2 * d + 64) * TINY
            Bt = Bc + U * (np.abs(dist) + Bc)
        with np.errstate(invalid="ignore"):
            must = (dist + Bt <= e32) & ~np.isnan(dist)
            mustnot = (dist - Bt > e32) | np.isnan(dist)
        bb = bits[i0:i0 + block]
        band += int((~must & ~mustnot).sum())
        ties += int((dist == e32).sum())
        for a, b in np.argwhere(must & ~bb)[:3]:
            v.append(f"pair ({i0 + a}, {b}): 1 - cos = {dist[a, b]!r} must be a neighbour (eps {e32!r})")
        for a, b in np.argwhere(mustnot & bb)[:3]:
            v.append(f"pair ({i0 + a}, {b}): 1 - cos = {dist[a, b]!r} must not be a neighbour (eps {e32!r})")
    return Report(v, band, ties)
