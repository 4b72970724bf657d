"""GPU: the frame-filter, chain, sequence and clustering kernels against the fp32 model (oracle/fp32_model.py),
without guard bands: bit for bit on exact frames (ties included), through the bounded replay checkers on frames that
sit on the thresholds, and at extreme frame scales and non-finite frames."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import cluster as oc, dedup as od, fp32_model as fm  # noqa: E402

THR, TR = 61 / 64, 0.75          # exact cosines on fm.exact_frames
RW = ("rw", "0")                 # banded_cosine_rw_kernel (default for d = 384 / 512, window <= 8)
GEN = ("banded", "2")            # banded_cosine_kernel (DV > 0 for d % 128 == 0, else DV == 0)


@pytest.fixture
def kernel(monkeypatch, request):
    model, env = request.param
    monkeypatch.setenv("IVR_DEDUP_KERNEL", env)
    return model


def frame_filter(x, window, thr, transition, min_len):
    from ivr_b200 import _native as nat
    x = np.ascontiguousarray(x, np.float32)
    n, d = x.shape
    keep = np.zeros(n, np.uint8)
    cosp = np.zeros(n, np.float32)
    stats = (C.c_int64 * 2)()
    nat.check(nat.lib.ivr_frame_filter(0, x.ctypes.data, n, d, window, C.c_float(thr), C.c_float(transition), min_len,
                                       keep.ctypes.data, cosp.ctypes.data, stats))
    return keep, cosp, [stats[0], stats[1]]


def sequence_hits(t, db, L, thr, cap=1 << 17):
    from ivr_b200 import _native as nat
    t, db = np.ascontiguousarray(t, np.float32), np.ascontiguousarray(db, np.float32)
    ht, hj, hs = np.empty(cap, np.int32), np.empty(cap, np.int64), np.empty(cap, np.float32)
    n = C.c_int64(0)
    nat.check(nat.lib.ivr_sequence_similarity(0, t.ctypes.data, len(t), db.ctypes.data, len(db), t.shape[1], L,
                                              C.c_float(thr), cap, ht.ctypes.data, hj.ctypes.data, hs.ctypes.data,
                                              C.byref(n)))
    assert n.value <= cap
    return ht[:n.value], hj[:n.value], hs[:n.value]


def neighbors(x, eps):
    from ivr_b200 import _native as nat
    x = np.ascontiguousarray(x, np.float32)
    adj = np.empty((len(x), (len(x) + 31) // 32), np.uint32)
    nat.check(nat.lib.ivr_cosine_neighbors(0, x.ctypes.data, len(x), x.shape[1], C.c_float(eps), adj.ctypes.data))
    return adj


def chunk_frames(d):
    return (64 << 20) // (d * 4)           # ivr_frame_filter's H2D chunk


# ---------------------------------------------------------------------------
# exact frames: ties resolve bit for bit as in the reference
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,d", [(RW, 384), (RW, 512), (GEN, 384), (GEN, 512), (GEN, 768), (GEN, 1024),
                                      (GEN, 100)], indirect=["kernel"])
def test_exact_ties_in_the_banded_kernels(kernel, d):
    from ivr_b200 import frame_filter as ff
    x = fm.exact_frames(3000, d, seed=d)
    r = fm.rows(x)
    exact = fm.pair_cos(r, np.arange(1, len(x)), np.arange(len(x) - 1))
    assert (exact == THR).sum() > 10 and (exact == TR).sum() > 10
    keep, cosp, stats = frame_filter(x, 8, THR, TR, 2)
    rep = fm.check_frame_filter(x, keep, cosp, stats, 8, THR, TR, 2, kernel, exact=True)
    assert rep.violations == [], (kernel, d, rep.violations[:5])
    assert rep.ties > 0
    assert np.array_equal(cosp[1:].astype(np.float64), exact)                      # cos == thr: duplicate, == 0.75: no cut
    sims = np.asarray(ff.calculate_similarities(x), np.float32)
    assert np.array_equal(sims.astype(np.float64), exact)
    scenes = od.scenes_from_cosines(exact, len(x), TR, 2)
    k2, c2 = ff._dedup_window(x, scenes, 8, THR)
    assert np.array_equal(k2, od.window_keep_mask(x, scenes, 8, THR))
    assert np.array_equal(c2[1:].astype(np.float64), exact)


def test_exact_ties_in_the_chain_fifo_neighbour_and_sequence_kernels(monkeypatch):
    from ivr_b200 import frame_filter as ff
    from ivr_b200.temporal import TemporalAnalyzer
    x = fm.exact_frames(1500, 128, seed=21, moves=(0, 1, 2, 3))
    n = len(x)
    want = od.extract_unique_rule(list(x), THR)
    got = ff.extract_unique_frames_rule(x, THR)
    assert got == want
    keep = np.zeros(n, np.uint8); keep[got] = 1
    rep = fm.check_chain(x, keep, [(0, n - 1)], 1, THR, False, 1, exact=True)
    assert rep.violations == [] and rep.ties > 0
    for tw in (10, 16):
        got = ff.temporal_window_filter(x, THR, tw)
        assert got == od.temporal_window_filter(list(x), THR, tw)
    adj = neighbors(x[:1000], 3 / 64)                                      # 1 - cos == eps is a neighbour
    rep = fm.check_adjacency(x[:1000], 3 / 64, adj, exact=True)
    assert rep.violations == [] and rep.ties > 0
    t = x[:200]
    db = np.concatenate([x[700:900], x[40:190], x[1000:1300]])
    ta = TemporalAnalyzer(device=0)
    for L in (1, 7, 8, 9, 64, 127, 128):
        _, _, M32 = fm.window_sims(t, db, L)
        thr = float(np.sort(M32.ravel())[-200])                             # a mean that occurs exactly
        ht, hj, hs = sequence_hits(t, db, L, thr)
        ordered = ta.find_similar_sequences(t, db, L, thr)
        rep = fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, ordered, exact=True)
        assert rep.violations == [] and rep.ties > 0, (L, rep.violations[:5])


# ---------------------------------------------------------------------------
# frames on the thresholds, no guard band
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kernel,n,d,window,min_len", [
    (RW, 40_000, 512, 8, 2),          # two H2D chunks: the look-back crosses the chunk boundary
    (GEN, 40_000, 512, 8, 2),
    (RW, 5_000, 384, 5, 1), (GEN, 5_000, 384, 5, 1),
    (GEN, 3_000, 100, 12, 2),          # DV == 0, window above the register window
    (GEN, 3_000, 64, 8, 2), (GEN, 2_000, 768, 3, 5)], indirect=["kernel"])
def test_near_threshold_frame_filter(kernel, n, d, window, min_len):
    x = fm.near_threshold_frames(n, d, 0.95, 0.75, seed=n + d + window, window=window)
    keep, cosp, stats = frame_filter(x, window, 0.95, 0.75, min_len)
    rep = fm.check_frame_filter(x, keep, cosp, stats, window, 0.95, 0.75, min_len, kernel)
    assert rep.violations == [], (kernel, rep.violations[:5])
    assert rep.in_band > 0
    print(f"{kernel} n={n} d={d} W={window}: {rep.in_band} decisions in the band")


@pytest.mark.parametrize("n,d", [(40_000, 512), (5_000, 384)])
def test_register_window_and_generic_kernels_agree_within_both_bounds(monkeypatch, n, d):
    x = fm.near_threshold_frames(n, d, 0.95, 0.75, seed=7 * d)
    out = {}
    for model, env in (RW, GEN):
        monkeypatch.setenv("IVR_DEDUP_KERNEL", env)
        out[model] = frame_filter(x, 8, 0.95, 0.75, 2)
        rep = fm.check_frame_filter(x, *out[model], 8, 0.95, 0.75, 2, model)
        assert rep.violations == [] and rep.in_band > 0, (model, rep.violations[:5])
    r = fm.rows(x)
    i = np.arange(1, n)
    b = fm.pair_bound(r, i, i - 1, "rw") + fm.pair_bound(r, i, i - 1, "banded")
    diff = np.abs(out["rw"][1][1:].astype(np.float64) - out["banded"][1][1:])
    assert (diff <= b).all()
    print(f"n={n} d={d}: {int((out['rw'][0] != out['banded'][0]).sum())} keep flags differ, all admissible")


def test_near_threshold_chain_and_fifo_rules():
    from ivr_b200 import frame_filter as ff
    x = fm.near_threshold_frames(2000, 128, 0.95, 0.75, seed=31)
    n = len(x)
    band = 0
    keep = np.zeros(n, np.uint8); keep[ff.extract_unique_frames_rule(x, 0.95)] = 1
    rep = fm.check_chain(x, keep, [(0, n - 1)], 1, 0.95, False, 1)
    assert rep.violations == [], rep.violations[:5]
    band += rep.in_band
    scenes = [(0, 99), (100, 100), (150, 1999)]
    for md in (1, 2, 3):
        cfg = dict(enable_similarity_filtering=True, similarity_threshold=0.95, min_frame_distance=md,
                   use_advanced_similarity_filtering=False, similarity_window_size=5)
        _, rows, _ = ff.apply_similarity_filtering_to_scenes(list(x), list(range(n)), scenes, cfg)
        keep = np.zeros(n, np.uint8); keep[rows] = 1
        rep = fm.check_chain(x, keep, scenes, md, 0.95, True, 1)
        assert rep.violations == [], (md, rep.violations[:5])
        band += rep.in_band
    for tw in (3, 10, 16):
        keep = np.zeros(n, np.uint8); keep[ff.temporal_window_filter(x, 0.95, tw)] = 1
        rep = fm.check_chain(x, keep, [(0, n - 1)], 1, 0.95, False, tw)
        assert rep.violations == [], (tw, rep.violations[:5])
        band += rep.in_band
    assert band > 0


@pytest.mark.parametrize("n,d", [(1200, 384), (1000, 100), (8192, 64)])      # 8192 = IVR_MAX_CLUSTER_FRAMES
def test_near_threshold_neighbours_and_clustering(n, d):
    from ivr_b200 import frame_filter as ff
    x = fm.near_threshold_frames(n, d, 0.95, 0.75, seed=n + d)
    eps = 0.05
    adj = neighbors(x, eps)
    rep = fm.check_adjacency(x, eps, adj)
    assert rep.violations == [] and rep.in_band > 0, rep.violations[:5]
    bits = np.unpackbits(adj.view(np.uint8), axis=1, bitorder="little")[:, :n].astype(bool)
    labels = oc.dbscan_labels([np.flatnonzero(row) for row in bits], 3)
    assert ff.cluster_similar_frames(x, eps=eps, min_samples=3) == oc.groups_from_labels(labels)


def _sequence_case(seed, d=128, thr=0.9):
    rng = np.random.default_rng(seed)
    t = fm.near_threshold_frames(90, d, thr, 0.75, seed=seed)
    near = np.stack([fm._toward(t[k].astype(np.float64), thr, rng) * 3 for k in range(90)]).astype(np.float32)
    db = np.concatenate([fm.near_threshold_frames(70, d, thr, 0.75, seed=seed + 1), near, t[10:60]])
    return t, db


def test_near_threshold_sequence_hits_and_forced_chunking(monkeypatch):
    from ivr_b200.temporal import TemporalAnalyzer
    t, db = _sequence_case(41)
    thr = 0.9
    ta = TemporalAnalyzer(device=0)
    for L in (1, 8, 13):
        ht, hj, hs = sequence_hits(t, db, L, thr)
        rep = fm.check_sequence_hits(t, db, L, thr, ht, hj, hs, ta.find_similar_sequences(t, db, L, thr))
        assert rep.violations == [] and rep.in_band > 0, (L, rep.violations[:5])
        monkeypatch.setenv("IVR_SEQ_BLOCK_COLS", "64")
        h2 = sequence_hits(t, db, L, thr)
        monkeypatch.delenv("IVR_SEQ_BLOCK_COLS")
        assert sorted(zip(*[a.tolist() for a in h2])) == sorted(zip(ht.tolist(), hj.tolist(), hs.tolist()))


# ---------------------------------------------------------------------------
# scale: powers of two change nothing; extreme and non-finite frames follow the reference
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", [RW, GEN], indirect=True)
def test_power_of_two_scaling_is_bit_identical(kernel):
    x = fm.near_threshold_frames(5000, 512, 0.95, 0.75, seed=51)
    base = frame_filter(x, 8, 0.95, 0.75, 2)
    for k in (-40, -20, 20, 40):
        xs = np.ldexp(x.astype(np.float64), k).astype(np.float32)
        ss = np.einsum("ij,ij->i", xs.astype(np.float64), xs.astype(np.float64))
        assert (ss > 2.0 ** -126).all() and (ss < 2.0 ** 126).all()
        got = frame_filter(xs, 8, 0.95, 0.75, 2)
        assert np.array_equal(got[0], base[0]) and got[2] == base[2], (kernel, k)
        assert np.array_equal(got[1].view(np.uint32), base[1].view(np.uint32)), (kernel, k)
    t, db = _sequence_case(52)
    h0 = sequence_hits(t, db, 8, 0.9)
    for k in (-30, 30):
        h = sequence_hits(np.ldexp(t, k), np.ldexp(db, k), 8, 0.9)
        assert sorted(zip(*[a.tolist() for a in h])) == sorted(zip(*[a.tolist() for a in h0])), k


EXTREMES = ("over", "sub", "zero", "nan", "inf")


def _insert_extremes(x, positions, rng):
    x = x.copy()
    kinds = {}
    for p in positions:
        kind = EXTREMES[len(kinds) % len(EXTREMES)]
        v = x[p].astype(np.float64)
        if kind == "over":                # finite components, sum of squares overflows fp32
            v = np.ldexp(v, 66)
        elif kind == "sub":               # sum of squares subnormal
            v = np.ldexp(v, -66)
        elif kind == "zero":
            v = np.zeros_like(v)
        elif kind == "nan":
            v[int(rng.integers(len(v)))] = np.nan
        else:
            v[int(rng.integers(len(v)))] = np.inf
        x[p] = v.astype(np.float32)
        kinds[p] = kind
    return x, kinds


@pytest.mark.parametrize("kernel,d", [(RW, 512), (RW, 384), (GEN, 512), (GEN, 100)], indirect=["kernel"])
def test_extreme_scales_and_non_finite_frames(kernel, d):
    """Frames whose sum of squares overflows (cosine 0 in the reference) or is subnormal, zero, NaN and inf frames:
    in runs, at the run end, on the H2D chunk boundary and inside the 8-frame window of later frames."""
    ch = chunk_frames(d)
    n = ch + 300
    rng = np.random.default_rng(d)
    x = fm.near_threshold_frames(n, d, 0.95, 0.75, seed=61 + d)
    pos = sorted({5, 6, 7, 8, 9, 10, 20, 23, 29, 100, 101, 140, 400, 1000, 1004,
                  ch - 9, ch - 8, ch - 2, ch - 1, ch, ch + 1, ch + 7, ch + 8, n - 3, n - 1})
    x, kinds = _insert_extremes(x, pos, rng)
    assert {kinds[p] for p in pos} == set(EXTREMES)
    keep, cosp, stats = frame_filter(x, 8, 0.95, 0.75, 2)
    rep = fm.check_frame_filter(x, keep, cosp, stats, 8, 0.95, 0.75, 2, kernel)
    assert rep.violations == [], (f"kernel {kernel}, d {d}: {len(rep.violations)} violations", rep.violations[:8],
                                  {p: kinds[p] for p in pos})
    r = fm.rows(x)
    exact = fm.pair_cos(r, np.arange(1, n), np.arange(n - 1))
    assert np.array_equal(np.isnan(cosp[1:]), np.isnan(exact))
    zero = np.isin(np.arange(1, n), [p for p in pos if kinds[p] in ("over", "zero")]) & (exact == 0)
    assert zero.sum() >= 5 and (cosp[1:][zero] == 0).all()                      # an overflowed norm: cosine 0, not NaN


def test_extreme_frames_give_the_same_results_on_both_banded_kernels(monkeypatch):
    d = 512
    x = fm.near_threshold_frames(3000, d, 0.95, 0.75, seed=71)
    x, kinds = _insert_extremes(x, [3, 4, 5, 6, 7, 300, 308, 316, 1500, 1501, 1502, 1503, 1504, 2999],
                                np.random.default_rng(3))
    out = {}
    for model, env in (RW, GEN):
        monkeypatch.setenv("IVR_DEDUP_KERNEL", env)
        out[model] = frame_filter(x, 8, 0.95, 0.75, 2)
    a, b = out["rw"][1], out["banded"][1]
    assert np.array_equal(np.isnan(a), np.isnan(b)), np.flatnonzero(np.isnan(a) != np.isnan(b))[:8]
    r = fm.rows(x)
    i = np.arange(1, len(x))
    bnd = fm.pair_bound(r, i, i - 1, "rw") + fm.pair_bound(r, i, i - 1, "banded")
    ok = np.isnan(a[1:]) | (np.abs(a[1:].astype(np.float64) - b[1:]) <= bnd)
    assert ok.all(), np.flatnonzero(~ok)[:8] + 1


# ---------------------------------------------------------------------------
# size edges
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", [RW, GEN], indirect=True)
def test_frame_filter_size_edges(kernel):
    d = 512
    x = fm.exact_frames(chunk_frames(d) + 1, d, seed=81)
    for n in (1, 2, 9, chunk_frames(d) + 1):                  # window + 1, one frame past a chunk
        keep, cosp, stats = frame_filter(x[:n], 8, THR, TR, 1)
        rep = fm.check_frame_filter(x[:n], keep, cosp, stats, 8, THR, TR, 1, kernel, exact=True)
        assert rep.violations == [], (kernel, n, rep.violations[:5])


def test_sequence_similarity_at_65535_target_windows():
    from ivr_b200 import _native as nat
    d = 16
    e1, e2 = np.zeros(d, np.float32), np.zeros(d, np.float32)
    e1[0], e2[1] = 1.0, 1.0
    t = np.tile(e1, (65535, 1))
    db = np.stack([e1] + [e2] * 7)
    ht, hj, hs = sequence_hits(t, db, 1, 0.5, cap=65535)
    assert len(ht) == 65535 and (hj == 0).all() and (hs == 1.0).all()
    assert np.array_equal(np.sort(ht), np.arange(65535))
    t2 = np.tile(e1, (65536, 1))
    with pytest.raises(nat.NativeError) as e:
        sequence_hits(t2, db, 1, 0.5, cap=16)
    assert e.value.code == nat.IVR_EUNSUPPORTED
