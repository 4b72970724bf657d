"""The library's search arithmetic restated in float64 (TEST INFRASTRUCTURE ONLY).

The fp32 oracle (``flat_ip``, ``range_search``) is checked through a 1e-3 band, which at this suite's shapes holds
several rows around the k-th score.  This model is much tighter, because the library's arithmetic can be written down:

- rows are stored as fp16: NaN stays NaN, everything else is clamped to +-65504 and rounded to nearest even (``store``);
- the tcgen05 kernels (the batched, small-batch and range kernels) scale each query by 2^-e, e from ``frexp`` of its
  largest magnitude clamped to [-127, 127], round it to fp16 and multiply the fp32 result by 2^e; the streaming kernel
  (``search_stream_kernel``) keeps the fp32 query (``prepare_query``);
- an fp16 x fp16 product, and an fp16 x fp32 one, is exact in float64, so the only thing left out is the order and the
  rounding of the fp32 accumulation.

``scores`` bounds that: every fp32 step rounds (or truncates) by at most 2^-23 of its partial sum, or 2^-149 in the
subnormal range, and no kernel takes more than dpad / 8 + 4 dependent steps per score (the streaming kernel's
per-lane chain of dpad / 8 FMAs and 3 shuffle adds; a 16-wide MMA K-step adds once per 16 products).  The final
rescale by the power of two 2^e rounds only when the result is subnormal: one more 2^-149.

``exact_inputs`` builds rows and queries on which every accumulation order is exact in fp32, so that the kernels must
reproduce the model bit for bit.
"""
from __future__ import annotations

import numpy as np

F16_MAX = 65504.0
U = 2.0 ** -23                  # twice the unit roundoff of fp32: covers truncation as well as rounding
TINY = 2.0 ** -149              # smallest fp32 subnormal
FLT_MAX = float(np.finfo(np.float32).max)
_NORMAL_MIN = 2.0 ** -126


def pad_dim(d: int) -> int:
    return (d + 63) // 64 * 64


def store(x) -> np.ndarray:
    """fp32 -> the stored fp16 row: clamped to +-65504 (never inf), RNE, NaN kept."""
    x = np.asarray(x, np.float32)
    with np.errstate(invalid="ignore"):
        c = np.where(np.isnan(x), x, np.clip(x, -F16_MAX, F16_MAX)).astype(np.float32)
    return c.astype(np.float16)


def path_of(kernel: str) -> str:
    """The arithmetic family of ``last_timing()["kernel"]``: "stream" for search_stream_kernel, else "mma"."""
    return "stream" if kernel == "search_stream_kernel" else "mma"


def query_exponent(q) -> np.ndarray:
    """e per query: frexp of the largest finite magnitude, clamped to [-127, 127]; 0 for a zero or non-finite max."""
    q = np.asarray(q, np.float32)
    mx = np.fmax.reduce(np.abs(q), axis=1) if q.shape[1] else np.zeros(q.shape[0], np.float32)
    ok = (mx > 0) & np.isfinite(mx)
    e = np.frexp(np.where(ok, mx, np.float32(1)))[1].astype(np.int64)
    return np.where(ok, np.clip(e, -127, 127), 0)


def prepare_query(q, path: str):
    """(q~ as float64 [nq, d], scale float64 [nq]): the query operand the kernels multiply, and its rescale."""
    q = np.asarray(q, np.float32)
    if path == "stream":
        return q.astype(np.float64), np.ones(q.shape[0])
    if path != "mma":
        raise ValueError(f"unknown path {path!r}")
    e = query_exponent(q)
    down = np.ldexp(np.float32(1), -e).astype(np.float32)            # 2^-e, finite in fp32 for |e| <= 127
    with np.errstate(over="ignore", invalid="ignore"):
        qt = (q * down[:, None]).astype(np.float32).astype(np.float16)
    return qt.astype(np.float64), np.ldexp(1.0, e)


def _scores(qt, scale, rows16):
    """Model score and bound of prepared queries against stored rows (fp16 [n, d]); float64 [nq, n] each."""
    x = rows16.astype(np.float64)
    dpad = pad_dim(rows16.shape[1])
    nan_rows = np.isnan(x).any(axis=1)
    x = np.where(np.isnan(x), 0.0, x)
    with np.errstate(over="ignore", invalid="ignore"):
        m = (qt @ x.T) * scale[:, None]
        a = np.abs(qt) @ np.abs(x).T
        eps = (dpad / 8 + 4) * (U * a + TINY) * scale[:, None] + TINY
    m[:, nan_rows] = np.nan
    return m, eps


def scores(q, rows16, path: str):
    """(m, eps): the model score (q~ . x~) * scale and its bound, float64 [nq, n], for fp32 queries ``q`` and
    stored rows ``rows16`` (``store`` output).  A row holding a NaN scores NaN."""
    qt, scale = prepare_query(q, path)
    return _scores(qt, scale, rows16)


def exact_inputs(n: int, d: int, nq: int, seed: int, query_exp: int = 0):
    """Rows [n, d] and queries [nq, d] (fp32) of integers in [-8, 8] x 2^-4, the queries times 2^query_exp.

    Each product is a multiple of 2^-8 (times 2^query_exp) of magnitude <= 2^-2, every partial sum is at most 2^10 of
    those units for d <= 4096: any accumulation order is exact in fp32, and so is the tcgen05 query scaling.  The
    scores have massive exact ties, zeros and negative values."""
    rng = np.random.default_rng(seed)
    xb = (rng.integers(-8, 9, size=(n, d)) / 16.0).astype(np.float32)
    xq = np.ldexp(rng.integers(-8, 9, size=(nq, d)) / 16.0, query_exp).astype(np.float32)
    return xb, xq


def f2ord(D) -> np.ndarray:
    """The kernels' order-preserving map of fp32 scores to uint32 (the high half of a result key)."""
    u = np.ascontiguousarray(D, np.float32).view(np.uint32)
    return np.where(u & 0x80000000, ~u, u | 0x80000000).astype(np.uint32)


def keys_to_DI(keys, id_offset: int = 0):
    """Packed result keys (int64 ``ord(score) << 32 | ~id``, 0 = padding) -> (D, I) with -FLT_MAX / -1 padding."""
    k = np.asarray(keys).view(np.uint64)
    o = (k >> np.uint64(32)).astype(np.uint32)
    u = np.where(o & 0x80000000, o & 0x7fffffff, ~o).astype(np.uint32)
    D = u.view(np.float32).copy()
    I = (~(k & np.uint64(0xffffffff)).astype(np.uint32)).astype(np.int64)
    pad = k == 0
    D[pad] = -FLT_MAX
    I[pad] = -1
    return D, I


def _order_violations(tag, d, ids):
    """Key order: scores non-increasing (as fp32 keys: -0 below +0); equal normal scores in ascending id order.
    (Scores rescaled into the subnormal range, or to zero, can collide after the rescale: their order is the
    kernels' unrounded one.)"""
    if d.size < 2:
        return []
    o = f2ord(d).astype(np.int64)
    if np.any(o[1:] > o[:-1]):
        return [f"{tag}: scores not non-increasing"]
    same = (o[1:] == o[:-1]) & (np.abs(d[1:].astype(np.float64)) >= _NORMAL_MIN)
    if np.any(same & (ids[1:] < ids[:-1])):
        return [f"{tag}: equal scores not in ascending id order"]
    return []


def _model_blocks(q, rows16, path, block):
    qt, scale = prepare_query(q, path)
    for r0 in range(0, rows16.shape[0], block):
        m, eps = _scores(qt, scale, rows16[r0:r0 + block])
        yield r0, m, eps


def check_topk(D, I, q, rows16, path: str, id_offset: int = 0, exact: bool = False, ratios: dict | None = None,
               tag: str = "", block: int = 1 << 16):
    """Violations of top-k result (D, I) [nq, k] against the model (empty list == pass).

    1. |D - m(id)| <= eps(id) for every hit (``exact``: D == m);
    2. key order (``_order_violations``);
    3. no row outside the result has m - eps > D[k'-1], k' = min(k, rows with a non-NaN model score);
       (``exact``: the hits' scores are the k' largest model scores);
    4. ids unique and in range, k' hits then -1 / -FLT_MAX padding, no NaN-score row returned.
    ``ratios[tag]`` keeps the largest |D - m| / eps seen."""
    D, I = np.asarray(D, np.float32), np.asarray(I, np.int64)
    nq, k = I.shape
    n = rows16.shape[0]
    rows = I - id_offset
    valid = I >= 0
    m_hit = np.full((nq, k), np.nan)
    e_hit = np.ones((nq, k))
    out_max = np.full(nq, -np.inf)
    n_fin = np.zeros(nq, np.int64)
    tops = [[] for _ in range(nq)] if exact else None
    for r0, m, eps in _model_blocks(q, rows16, path, block):
        nb = m.shape[1]
        inb = valid & (rows >= r0) & (rows < r0 + nb)
        qi, kj = np.nonzero(inb)
        m_hit[qi, kj] = m[qi, rows[qi, kj] - r0]
        e_hit[qi, kj] = eps[qi, rows[qi, kj] - r0]
        fin = ~np.isnan(m)
        n_fin += fin.sum(axis=1)
        low = np.where(fin, m - eps, -np.inf)
        low[qi, rows[qi, kj] - r0] = -np.inf
        out_max = np.maximum(out_max, low.max(axis=1, initial=-np.inf))
        if exact:
            for qq in range(nq):
                s = m[qq][fin[qq]]
                tops[qq].append(np.sort(s)[::-1][:k])
    bad = []
    worst = 0.0
    for qq in range(nq):
        kp = int(min(k, n_fin[qq]))
        t = f"{tag} q{qq}"
        nv = int(valid[qq].sum())
        if nv != kp or not valid[qq, :kp].all():
            bad.append(f"{t}: {nv} valid hits, expected {kp}")
            continue
        if kp < k and not (np.all(I[qq, kp:] == -1) and np.all(D[qq, kp:] == -FLT_MAX)):
            bad.append(f"{t}: padding is not -1 / -FLT_MAX")
        ids = rows[qq, :kp]
        if np.any(ids >= n) or len(np.unique(ids)) != kp:
            bad.append(f"{t}: ids out of range or duplicated")
            continue
        if kp == 0:
            continue
        mh, eh, d = m_hit[qq, :kp], e_hit[qq, :kp], D[qq, :kp].astype(np.float64)
        if np.any(np.isnan(mh)):
            bad.append(f"{t}: a row with a NaN score was returned (id {ids[np.isnan(mh)][0]})")
            continue
        with np.errstate(invalid="ignore"):
            err = np.abs(d - mh)
        r = err / eh
        worst = max(worst, float(np.nanmax(r)))
        if exact and np.any(d != mh):
            j = int(np.argmax(err))
            bad.append(f"{t}: score {d[j]!r} of id {ids[j]} != model {mh[j]!r} (exact inputs)")
        elif np.any(~(err <= eh)):
            j = int(np.nanargmax(r))
            bad.append(f"{t}: |D - m| = {err[j]:.3e} > eps {eh[j]:.3e} at id {ids[j]}")
        bad += _order_violations(t, D[qq, :kp], ids)
        if out_max[qq] > d[kp - 1]:
            bad.append(f"{t}: a row outside the result scores >= {out_max[qq]!r} > the k-th score {d[kp - 1]!r}")
        if exact:
            want = np.sort(np.concatenate(tops[qq]))[::-1][:kp]
            if not np.array_equal(np.sort(d)[::-1], want):
                bad.append(f"{t}: scores are not the {kp} largest model scores")
        if len(bad) > 20:
            bad.append("... (truncated)")
            break
    if ratios is not None:
        ratios[tag] = max(ratios.get(tag, 0.0), worst)
    return bad


def check_range(lims, D, I, q, rows16, path: str, radius: float, id_offset: int = 0, exact: bool = False,
                ratios: dict | None = None, tag: str = "", block: int = 1 << 16):
    """Violations of range result (lims, D, I) against the model (empty list == pass): ``lims`` monotone from 0 and
    ending at len(D) == len(I); every hit has D > radius (fp32) and |D - m| <= eps (``exact``: D == m); key order; ids
    unique and in range; no NaN-score row is a hit; no row left out has m - eps > radius (``exact``: the hits are
    exactly the rows with m > radius)."""
    lims, D, I = np.asarray(lims, np.int64), np.asarray(D, np.float32), np.asarray(I, np.int64)
    nq = np.asarray(q).shape[0]
    n = rows16.shape[0]
    r = float(np.float32(radius))
    if lims.shape != (nq + 1,) or lims[0] != 0 or np.any(np.diff(lims) < 0):
        return [f"{tag}: lims is not a monotone sequence of nq + 1 entries starting at 0"]
    if not (int(lims[-1]) == D.size == I.size):
        return [f"{tag}: lims[-1] = {int(lims[-1])} but {D.size} scores and {I.size} ids"]
    hit = np.zeros((nq, n), bool)
    qid = np.repeat(np.arange(nq), np.diff(lims))
    rows = I - id_offset
    if rows.size and (rows.min() < 0 or rows.max() >= n):
        return [f"{tag}: ids out of range"]
    hit[qid, rows] = True
    m_hit = np.full(D.size, np.nan)
    e_hit = np.ones(D.size)
    missed = np.full(nq, -np.inf)
    extra = np.zeros(nq, np.int64)
    for r0, m, eps in _model_blocks(q, rows16, path, block):
        nb = m.shape[1]
        sel = (rows >= r0) & (rows < r0 + nb)
        m_hit[sel] = m[qid[sel], rows[sel] - r0]
        e_hit[sel] = eps[qid[sel], rows[sel] - r0]
        h = hit[:, r0:r0 + nb]
        with np.errstate(invalid="ignore"):
            if exact:
                extra += ((m > r) & ~h).sum(axis=1)
            low = np.where(np.isnan(m) | h, -np.inf, m - eps)
        missed = np.maximum(missed, low.max(axis=1, initial=-np.inf))
    bad = []
    worst = 0.0
    for qq in range(nq):
        t = f"{tag} q{qq}"
        a, b = lims[qq], lims[qq + 1]
        ids, d, mh, eh = rows[a:b], D[a:b], m_hit[a:b], e_hit[a:b]
        if len(np.unique(ids)) != ids.size:
            bad.append(f"{t}: duplicate ids")
        if np.any(~(d > np.float32(r))):
            bad.append(f"{t}: a hit scores {d[~(d > np.float32(r))][0]!r}, not above the radius {r!r}")
        if np.any(np.isnan(mh)):
            bad.append(f"{t}: a row with a NaN score is a hit")
        elif ids.size:
            err = np.abs(d.astype(np.float64) - mh)
            worst = max(worst, float((err / eh).max()))
            if exact and np.any(d != mh):
                bad.append(f"{t}: a hit's score differs from the model (exact inputs)")
            elif np.any(err > eh):
                j = int(np.argmax(err / eh))
                bad.append(f"{t}: |D - m| = {err[j]:.3e} > eps {eh[j]:.3e} at id {ids[j]}")
        bad += _order_violations(t, d, ids)
        if missed[qq] > r:
            bad.append(f"{t}: a row left out has m - eps = {missed[qq]!r} > radius {r!r}")
        if exact and extra[qq]:
            bad.append(f"{t}: {extra[qq]} rows with a model score above the radius are not hits")
        if len(bad) > 20:
            bad.append("... (truncated)")
            break
    if ratios is not None:
        ratios[tag] = max(ratios.get(tag, 0.0), worst)
    return bad
