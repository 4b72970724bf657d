"""CPU: the fp32 cosine model of the frame-filter, sequence and clustering kernels (oracle/fp32_model.py).

The bounds are checked against NumPy float32 emulations of each kernel's order of operations, the exact frames
against several summation orders, ``exact_cos`` against the reference restated (oracle.dedup.cos1), and every
checker against outputs that are wrong on purpose."""
import ctypes as C

import numpy as np
import pytest

from oracle import dedup as od, fp32_model as fm, synth
from oracle import temporal as ot

f32 = np.float32


# ---------------------------------------------------------------------------
# float32 emulation of the kernels' orders (FMA: exact product and sum in float64, one rounding to fp32)
# ---------------------------------------------------------------------------
def fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)


def butterfly(acc, order=(16, 8, 4, 2, 1)):
    lanes = np.arange(32)
    for o in order:
        acc = (acc + acc[:, lanes ^ o]).astype(f32)
    return acc[:, 0]


def lane_dot(A, B):
    """Per-lane FMA chain (float4 layout when d % 128 == 0, else element c on lane c % 32), then 5 xor adds."""
    P, d = A.shape
    if d % 128 == 0:
        A4, B4 = A.reshape(P, d // 128, 32, 4), B.reshape(P, d // 128, 32, 4)
        seq = [(j, c) for j in range(d // 128) for c in range(4)]
        acc = np.zeros((P, 32), f32)
        for j, c in seq:
            acc = fma32(A4[:, j, :, c], B4[:, j, :, c], acc)
    else:
        k = -(-d // 32)
        Ap, Bp = np.zeros((P, k * 32), f32), np.zeros((P, k * 32), f32)
        Ap[:, :d], Bp[:, :d] = A, B
        acc = np.zeros((P, 32), f32)
        for s in range(k):
            acc = fma32(Ap[:, s * 32:(s + 1) * 32], Bp[:, s * 32:(s + 1) * 32], acc)
    return butterfly(acc)


def emulate_banded(X, Y, divide: bool):
    def unit(Z):
        nrm = np.sqrt(lane_dot(Z, Z))
        nrm = np.where(nrm == 0, f32(1), nrm).astype(f32)
        if divide:
            return (Z / nrm[:, None]).astype(f32)
        return (Z * (f32(1) / nrm)[:, None]).astype(f32)
    return lane_dot(unit(X), unit(Y)).astype(np.float64)


def _rw_inv(ss):
    ss = ss.astype(f32)
    with np.errstate(over="ignore", divide="ignore", invalid="ignore"):      # lanes outside the Newton range
        y0 = (1.0 / np.sqrt(ss.astype(np.float64)) * (1 + 2.0 ** -22)).astype(f32)     # a 2-ulp-off rsqrt
        inv = (y0 * fma32(f32(-0.5) * ss, (y0 * y0).astype(f32), np.full_like(ss, 1.5))).astype(f32)
        alt = (f32(1) / np.sqrt(ss)).astype(f32)
    ok = (ss >= f32(2.0 ** -126)) & (ss < f32(2.0 ** 126))
    return np.where(ok, inv, np.where(ss == 0, f32(1), alt)).astype(f32)


def _rw_pair_chains(A, B):
    P, d = A.shape
    A4, B4 = A.reshape(P, d // 128, 32, 4), B.reshape(P, d // 128, 32, 4)
    a0, a1 = np.zeros((P, 32), f32), np.zeros((P, 32), f32)
    for j in range(d // 128):
        a0 = fma32(A4[:, j, :, 0], B4[:, j, :, 0], a0)
        a1 = fma32(A4[:, j, :, 1], B4[:, j, :, 1], a1)
        a0 = fma32(A4[:, j, :, 2], B4[:, j, :, 2], a0)
        a1 = fma32(A4[:, j, :, 3], B4[:, j, :, 3], a1)
    return (a0 + a1).astype(f32)


def emulate_rw(X, Y):
    """banded_cosine_rw_kernel: window row Y normalised by inv_y, dot with the RAW row X, times inv_x."""
    inv_x = _rw_inv(butterfly(_rw_pair_chains(X, X)))
    inv_y = _rw_inv(butterfly(_rw_pair_chains(Y, Y)))
    Yh = (Y * inv_y[:, None]).astype(f32)
    acc = butterfly(_rw_pair_chains(X, Yh), order=(4, 2, 1, 8, 16))
    return (acc * inv_x).astype(f32).astype(np.float64)


def emulate_seq(X, Y):
    def unit(Z):
        nrm = np.sqrt(lane_dot(Z, Z))
        nrm = np.where(nrm == 0, f32(1), nrm).astype(f32)
        return (Z / nrm[:, None]).astype(f32)
    Xh, Yh = unit(X), unit(Y)
    acc = np.zeros(X.shape[0], f32)
    for k in range(X.shape[1]):
        acc = fma32(Xh[:, k], Yh[:, k], acc)
    return acc.astype(np.float64)


def _frames(kind, d):
    if kind == "random":
        return (3 * np.random.default_rng(d).standard_normal((160, d))).astype(f32)
    if kind == "clip":
        return synth.clip_like(160, d, seed=d, n_centres=8)
    if kind == "near":
        return fm.near_threshold_frames(160, d, 0.95, 0.75, seed=d)
    if kind == "tiny":                     # sums of squares subnormal, squares subnormal
        return (np.ldexp(fm.near_threshold_frames(160, d, 0.95, 0.75, seed=d + 1).astype(np.float64), -66)).astype(f32)
    raise ValueError(kind)


@pytest.mark.parametrize("d", [64, 100, 384, 512, 768, 1024])
@pytest.mark.parametrize("kind", ["random", "clip", "near", "tiny"])
def test_bounds_hold_against_float32_emulation_of_each_kernel(kind, d):
    x = _frames(kind, d)
    if kind == "tiny":
        ss = np.einsum("ij,ij->i", x.astype(np.float64), x.astype(np.float64))
        assert (ss < 2.0 ** -126).all() and (ss > 0).all()
    r = fm.rows(x)
    n = len(x)
    i = np.concatenate([np.arange(1, n), np.arange(8, n)])
    j = np.concatenate([np.arange(0, n - 1), np.arange(0, n - 8)])
    exact = fm.pair_cos(r, i, j)
    cases = [("banded", emulate_banded(x[i], x[j], divide=d % 128 != 0)),
             ("chain", emulate_banded(x[i], x[j], divide=True)),
             ("seq", emulate_seq(x[i], x[j]))]
    if d % 128 == 0:
        cases.append(("rw", emulate_rw(x[i], x[j])))
    for kernel, got in cases:
        b = fm.pair_bound(r, i, j, kernel)
        assert np.isfinite(b).all() and (b < (1e-2 if kind == "tiny" else 1e-3)).all(), kernel
        err = np.abs(got - exact)
        assert (err <= b).all(), (kernel, float((err / b).max()))
    # the sequence mean: per-position emulated cosines through numpy_mean_f32
    got = emulate_seq(x[i], x[j]).astype(f32)
    b = fm.pair_bound(r, i, j, "seq")
    for L in (1, 7, 8, 9, 64, 127, 128):
        m = len(got) // L * L
        if m == 0:
            continue
        cv, ev, bv = got[:m].reshape(-1, L), exact[:m].reshape(-1, L), b[:m].reshape(-1, L)
        sim = np.array([ot.numpy_mean_f32(row) for row in cv], np.float64)
        assert np.array_equal(fm.mean_f32(cv).astype(np.float64), sim)
        mb = bv.mean(axis=1)
        sabs = np.abs(ev).mean(axis=1) + mb
        bound = mb + fm.mean_depth(L) * fm.U * sabs + fm.U * sabs * (1 + fm.mean_depth(L) * fm.U) + fm.TINY
        assert (np.abs(sim - ev.mean(axis=1)) <= bound).all(), L


@pytest.mark.parametrize("d", [100, 128, 384, 512, 1024])
def test_exact_frames_are_exact_under_any_summation_order(d):
    x = fm.exact_frames(120, d, seed=d)
    assert ((x != 0).sum(axis=1) == fm.EXACT_NNZ).all()
    r = fm.rows(x)
    assert (r.ss == fm.EXACT_NNZ).all()
    i, j = np.arange(1, 120), np.arange(0, 119)
    exact = fm.pair_cos(r, i, j)
    assert np.array_equal(exact * 64, np.round(exact * 64))
    got = [emulate_banded(x[i], x[j], True), emulate_banded(x[i], x[j], False), emulate_seq(x[i], x[j])]
    if d % 128 == 0:
        got.append(emulate_rw(x[i], x[j]))
    xn = (x / f32(8)).astype(f32)
    for order in (np.arange(d), np.arange(d)[::-1], np.random.default_rng(1).permutation(d)):
        acc = np.zeros(len(i), f32)
        for k in order:
            acc = fma32(xn[i, k], xn[j, k], acc)
        got.append(acc.astype(np.float64))
    got.append(np.array([od.cos1(x[a], x[b]) for a, b in zip(i, j)], np.float64))
    for g in got:
        assert np.array_equal(g, exact)
    # the walk produces the values the GPU tests rely on: 61/64 ties and 48/64 transitions
    assert (exact == 61 / 64).any() and (exact == 0.75).any()


def test_exact_cos_follows_the_reference():
    rng = np.random.default_rng(5)
    for d in (64, 100, 512):
        x = (3 * rng.standard_normal((40, d))).astype(f32)
        r = fm.rows(x)
        for a in range(1, 40):
            ref = float(od.cos1(x[a], x[a - 1]))
            ex = fm.exact_cos(x[a], x[a - 1])
            assert abs(ref - ex) <= fm.pair_bound(r, [a], [a - 1], "ref")[0]
        v = x[0]
        z = np.zeros(d, f32)
        nan = v.copy(); nan[3] = np.nan
        inf = v.copy(); inf[5] = np.inf
        big = (v.astype(np.float64) * 2.0 ** 66).astype(f32)          # finite, sum of squares overflows fp32
        assert np.isfinite(big).all() and not np.isfinite(np.einsum("i,i->", big, big))
        with np.errstate(all="ignore"):
            for a, b in ((z, v), (v, z), (z, z), (big, v), (v, big), (big, big), (nan, v), (v, inf), (inf, z),
                         (nan, big)):
                ref = float(od.cos1(a, b))
                ex = fm.exact_cos(a, b)
                assert (np.isnan(ref) and np.isnan(ex)) or ref == ex, (ref, ex)
        assert fm.exact_cos(z, v) == 0.0 and fm.exact_cos(big, v) == 0.0 and np.isnan(fm.exact_cos(v, inf))


# ---------------------------------------------------------------------------
# the checkers reject wrong outputs
# ---------------------------------------------------------------------------
THR, TR = 61 / 64, 0.75


def _frame_filter_ref(x, window, thr, transition, min_len):
    cp = od.consecutive_cosines_fast(x)
    scenes = od.scenes_from_cosines(cp, len(x), transition, min_len)
    keep = od.window_keep_mask(x, scenes, window, thr)
    return keep, np.concatenate([[f32(1)], cp]).astype(f32), [len(scenes), sum(e - s + 1 for s, e in scenes)], scenes


def test_frame_filter_checker_accepts_the_reference_and_rejects_wrong_outputs():
    x = fm.exact_frames(400, 128, seed=3)
    W = 8
    keep, cp, stats, scenes = _frame_filter_ref(x, W, THR, TR, 2)
    rep = fm.check_frame_filter(x, keep, cp, stats, W, THR, TR, 2, "banded", exact=True)
    assert rep.violations == [] and rep.ties > 0 and rep.in_band == 0
    assert fm.check_frame_filter(x, keep, cp, stats, W, THR, TR, 2, "banded").violations == []

    def bad(k=keep, c=cp, s=stats, exact=True):
        return fm.check_frame_filter(x, k, c, s, W, THR, TR, 2, "banded", exact=exact).violations

    # a duplicate flipped outside the band
    r = fm.rows(x)
    E, _ = fm.banded(r, W, "banded")
    dropped = [i for i in np.flatnonzero(keep == 0) if any(keep[i - l] and E[i, l - 1] > 0.97 for l in (1, 2)
                                                           if i - l >= 0)]
    k2 = keep.copy(); k2[dropped[0]] = 1
    assert bad(k2, exact=False)
    # '>' instead of '>=' on exact ties
    k3 = od.window_keep_mask(x, scenes, W, np.nextafter(f32(THR), f32(2)))
    assert not np.array_equal(k3, keep) and bad(k3)
    # '<=' instead of '<' for the cut
    scenes_le = od.scenes_from_cosines(cp[1:], len(x), np.nextafter(f32(TR), f32(2)), 2)
    assert scenes_le != scenes
    k4 = od.window_keep_mask(x, scenes_le, W, THR)
    assert bad(k4, s=[len(scenes_le), sum(e - s + 1 for s, e in scenes_le)])
    # a scene off by one: the first cut one frame late
    s0 = scenes[0]
    shifted = [(s0[0], s0[1] + 1), (scenes[1][0] + 1, scenes[1][1])] + scenes[2:]
    assert bad(od.window_keep_mask(x, shifted, W, THR))
    # wrong stats
    assert bad(s=[stats[0], stats[1] + 1]) and bad(s=[stats[0] - 1, stats[1]])
    # a cos_prev off by one ulp on exact data, and far off in bound mode
    c2 = cp.copy(); c2[5] = np.nextafter(c2[5], f32(2))
    assert bad(c=c2)
    c3 = cp.copy(); c3[5] += f32(1e-3)
    assert bad(c=c3, exact=False)


def test_frame_filter_checker_counts_the_band_on_the_references_own_fp32_output():
    x = fm.near_threshold_frames(600, 384, 0.95, 0.75, seed=11)
    keep, cp, stats, _ = _frame_filter_ref(x, 8, 0.95, 0.75, 2)
    rep = fm.check_frame_filter(x, keep, cp, stats, 8, 0.95, 0.75, 2, "ref")
    assert rep.violations == [] and rep.in_band > 0


def test_chain_checker_accepts_the_reference_and_rejects_wrong_outputs():
    x = fm.exact_frames(300, 128, seed=4, moves=(0, 1, 2, 3))
    n = len(x)
    kept = od.extract_unique_rule(list(x), THR)
    keep = np.zeros(n, np.uint8); keep[kept] = 1
    rep = fm.check_chain(x, keep, [(0, n - 1)], 1, THR, False, 1, exact=True)
    assert rep.violations == [] and rep.ties > 0
    gt = od.extract_unique_rule(list(x), float(np.nextafter(f32(THR), f32(2))))    # '>' instead of '>='
    k2 = np.zeros(n, np.uint8); k2[gt] = 1
    assert not np.array_equal(k2, keep) and fm.check_chain(x, k2, [(0, n - 1)], 1, THR, False, 1, exact=True).violations
    i = next(i for i in np.flatnonzero(keep == 0) if fm.exact_cos(x[i], x[i - 1]) == 1.0 and keep[i - 1])
    k3 = keep.copy(); k3[i] = 1
    assert fm.check_chain(x, k3, [(0, n - 1)], 1, THR, False, 1).violations
    # FIFO of 10 kept frames, and the scene rule with min_distance 2 and a forced last frame
    kf = od.temporal_window_filter(list(x), THR, 10)
    k4 = np.zeros(n, np.uint8); k4[kf] = 1
    assert fm.check_chain(x, k4, [(0, n - 1)], 1, THR, False, 10, exact=True).violations == []
    assert fm.check_chain(x, keep, [(0, n - 1)], 1, THR, False, 10, exact=True).violations or \
        np.array_equal(keep, k4)
    cfg = dict(enable_similarity_filtering=True, similarity_threshold=THR, min_frame_distance=2)
    rows = od.filter_similar_frames_in_scene(list(x[:150]), list(range(150)), cfg)
    k5 = np.zeros(n, np.uint8); k5[rows] = 1
    assert fm.check_chain(x, k5, [(0, 149)], 2, THR, True, 1, exact=True).violations == []
    k6 = k5.copy(); k6[149] = 0
    assert fm.check_chain(x, k6, [(0, 149)], 2, THR, True, 1, exact=True).violations


def test_sequence_checker_accepts_exact_hits_and_rejects_wrong_ones():
    t = fm.exact_frames(30, 128, seed=6)
    db = np.concatenate([t[5:25], fm.exact_frames(40, 128, seed=7)])
    L = 4
    M, Bm, M32 = fm.window_sims(t, db, L)
    thr = float(np.sort(M32.ravel())[-40])
    ht, hj = np.nonzero(M32 >= f32(thr))
    hs = M32[ht, hj]
    order = sorted(range(len(hs)), key=lambda k: (-float(hs[k]), ht[k], hj[k]))
    ordered = [(int(hj[k]), float(hs[k])) for k in order]
    rep = fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, ordered, exact=True)
    assert rep.violations == [] and rep.ties > 0
    assert fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, ordered).violations == []
    top = int(np.argmax(hs))
    drop = np.arange(len(hs)) != top
    assert fm.check_sequence_hits(t, db, L, thr, ht[drop], hj[drop], hs[drop]).violations     # missing hit
    a, b = np.nonzero(M32 < f32(thr))
    below = (np.append(ht, a[0]), np.append(hj, b[0]), np.append(hs, f32(thr)))
    assert fm.check_sequence_hits(t, db, L, thr, *below).violations                           # hit below thr
    if len(set(hs.tolist())) > 1:
        swapped = list(reversed(ordered))
        assert fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, swapped).violations          # wrong order
    tie = [k for k in range(len(ordered) - 1) if ordered[k][1] == ordered[k + 1][1] and ordered[k][0] != ordered[k + 1][0]]
    if tie:
        o2 = list(ordered); o2[tie[0]], o2[tie[0] + 1] = o2[tie[0] + 1], o2[tie[0]]
        assert fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, o2).violations              # tie order
    hs2 = hs.copy(); hs2[top] = np.nextafter(hs2[top], f32(-2))
    assert fm.check_sequence_hits(t, db, L, thr, ht, hj, hs2, exact=True).violations          # sim one ulp off


def test_adjacency_checker_accepts_exact_bits_and_rejects_a_flipped_bit():
    x = fm.exact_frames(70, 128, seed=8)
    eps = 3 / 64
    xn = fm.rows(x).xn
    inb = (1.0 - xn @ xn.T) <= eps
    words = (70 + 31) // 32
    pad = np.zeros((70, words * 32), bool); pad[:, :70] = inb
    adj = np.packbits(pad, axis=1, bitorder="little").view(np.uint32)
    rep = fm.check_adjacency(x, eps, adj, exact=True)
    assert rep.violations == [] and rep.ties > 0
    assert fm.check_adjacency(x, eps, adj).violations == []
    far = np.argwhere((1.0 - xn @ xn.T) > 0.5)[0]
    pad[far[0], far[1]] = True
    assert fm.check_adjacency(x, eps, np.packbits(pad, axis=1, bitorder="little").view(np.uint32)).violations


# ---------------------------------------------------------------------------
# argument checks that need no device
# ---------------------------------------------------------------------------
def test_frame_kernel_limits_are_refused_before_any_device_work():
    from ivr_b200 import _native as nat
    x = np.ones((4, 8), np.float32)
    keep = np.zeros(70000, np.uint8)
    one = np.zeros(1, np.int64)
    stats = (C.c_int64 * 2)()
    assert nat.lib.ivr_frame_filter(0, x.ctypes.data, 4, 8, nat.IVR_MAX_WINDOW + 1, C.c_float(0.9), C.c_float(0.7), 2,
                                    keep.ctypes.data, None, stats) == nat.IVR_EUNSUPPORTED
    for fifo in (0, 17):
        assert nat.lib.ivr_dedup_fifo(0, x.ctypes.data, 4, 8, one.ctypes.data, one.ctypes.data, 1, fifo,
                                      C.c_float(0.9), keep.ctypes.data) == nat.IVR_EUNSUPPORTED
        assert "fifo" in nat.last_error()
    n = C.c_int64(7)
    ht, hj, hs = np.zeros(1, np.int32), np.zeros(1, np.int64), np.zeros(1, np.float32)
    for L in (0, 129):
        assert nat.lib.ivr_sequence_similarity(0, x.ctypes.data, 4, x.ctypes.data, 4, 8, L, C.c_float(0.5), 1,
                                               ht.ctypes.data, hj.ctypes.data, hs.ctypes.data,
                                               C.byref(n)) == nat.IVR_EUNSUPPORTED
    for nt, L in ((65536, 1), (65537, 2), (65663, 128)):                # 65536 target windows: one grid row too many
        assert nat.lib.ivr_sequence_similarity(0, x.ctypes.data, nt, x.ctypes.data, 4, 8, L, C.c_float(0.5), 1,
                                               ht.ctypes.data, hj.ctypes.data, hs.ctypes.data,
                                               C.byref(n)) == nat.IVR_EUNSUPPORTED
        assert "65535" in nat.last_error()
    adj = np.zeros(1, np.uint32)
    assert nat.lib.ivr_cosine_neighbors(0, x.ctypes.data, 8193, 8, C.c_float(0.05),
                                        adj.ctypes.data) == nat.IVR_EUNSUPPORTED
