"""CPU: pin the float64 model of the library's arithmetic (oracle/fp16_model.py) and show what it catches that the
1e-3 comparators do not."""
import numpy as np
import pytest

from oracle import comparator, flat_ip, fp16_model as fm, range_search, synth


def test_store_hand_cases():
    x = np.array([65504, 65519, 65520, 1e9, -65520, -np.inf, np.inf, 1 + 2 ** -11, 1 + 3 * 2 ** -11,
                  2 ** -24, 2 ** -25, 3 * 2 ** -26, 2 ** -14, -0.0, np.nan], np.float32)
    s = fm.store(x).astype(np.float32)
    want = [65504, 65504, 65504, 65504, -65504, -65504, 65504, 1.0, 1 + 2 ** -9,   # clamped, never inf; RNE ties
            2 ** -24, 0.0, 2 ** -24, 2 ** -14, -0.0]                               # fp16 subnormals, RNE tie to 0
    np.testing.assert_array_equal(s[:-1], np.array(want, np.float32))
    assert np.signbit(s[13]) and np.isnan(s[14])


def test_prepare_query_scales():
    q = np.zeros((8, 4), np.float32)
    q[1, 0] = 0.5
    q[2, 1] = 1.0
    q[3, 2] = 2.0 ** -126
    q[4, 3] = np.float32(2.0 ** -130)
    q[5, 0] = np.float32(3.2e38)
    q[6] = [-0.25, -0.75, -3.0, -1.0]
    q[7] = [np.float32(2.0 ** -140), 0, 0, np.float32(-2.0 ** -141)]
    qt, scale = fm.prepare_query(q, "mma")
    assert np.all(np.isfinite(qt)) and np.all(np.isfinite(scale))
    np.testing.assert_array_equal(np.log2(scale), [0, 0, 1, -125, -127, 127, 2, -127])
    assert qt[0].tolist() == [0, 0, 0, 0]
    assert qt[1, 0] == 0.5 and qt[2, 1] == 0.5 and qt[3, 2] == 0.5
    assert qt[4, 3] == 2.0 ** -3                                   # clamped exponent: max below 0.5
    assert qt[5, 0] == np.float64(np.float16(np.float32(3.2e38) / np.float32(2.0 ** 127)))   # in [1, 2)
    assert qt[6].tolist() == [-1 / 16, -3 / 16, -0.75, -0.25]
    assert qt[7].tolist() == [2.0 ** -13, 0, 0, -2.0 ** -14]
    # the model score is q . x up to fp16 rounding of the query, at either end of the float range
    x = np.ones((1, 4), np.float16)
    m, eps = fm._scores(qt, scale, x)
    np.testing.assert_allclose(m[:, 0], q.astype(np.float64).sum(axis=1), rtol=2 ** -10)
    qs, ss = fm.prepare_query(q, "stream")
    assert np.array_equal(qs, q.astype(np.float64)) and np.all(ss == 1)


def _fp32_sums(p):
    """fp32 sums of the products p [..., d] in three orders: sequential, 16-wide blocks, pairwise."""
    p = p.astype(np.float32)
    seq = np.zeros(p.shape[:-1], np.float32)
    for i in range(p.shape[-1]):
        seq = (seq + p[..., i]).astype(np.float32)
    blk = np.zeros(p.shape[:-1], np.float32)
    for i in range(0, p.shape[-1], 16):
        part = np.zeros(p.shape[:-1], np.float32)
        for j in range(i, min(i + 16, p.shape[-1])):
            part = (part + p[..., j]).astype(np.float32)
        blk = (blk + part).astype(np.float32)
    pw = p
    while pw.shape[-1] > 1:
        if pw.shape[-1] % 2:
            pw = np.concatenate([pw, np.zeros(pw.shape[:-1] + (1,), np.float32)], axis=-1)
        pw = (pw[..., 0::2] + pw[..., 1::2]).astype(np.float32)
    return seq, blk, pw[..., 0]


@pytest.mark.parametrize("d,qe", [(4096, 0), (1024, -140), (512, 100)])
def test_exact_inputs_are_exact_in_any_order(d, qe):
    xb, xq = fm.exact_inputs(64, d, 3, seed=d, query_exp=qe)
    for path in ("mma", "stream"):
        qt, scale = fm.prepare_query(xq, path)
        np.testing.assert_array_equal(qt * scale[:, None], xq.astype(np.float64))
    m, _ = fm.scores(xq, fm.store(xb), "mma")
    prods = xq[:, None, :].astype(np.float32) * xb[None, :, :]
    for s in _fp32_sums(prods):
        np.testing.assert_array_equal(s.astype(np.float64), m)
    assert np.any(m < 0) and np.any(m > 0)


def _r32(v, truncate):
    """float64 -> fp32, rounded to nearest or truncated toward zero."""
    f = v.astype(np.float32)
    if truncate:
        over = np.abs(f.astype(np.float64)) > np.abs(v)
        f = np.where(over, np.nextafter(f, np.float32(0)), f)
    return f.astype(np.float64)


def _emulate(qt, x, scheme, truncate):
    """fp32 accumulation of the exact products in a kernel's order: "lanes" -- 8 lanes each chain every 8th group of
    8 products with one rounding per product, then 3 pairwise adds (the streaming kernel); "block16" / "block8" -- the
    exact sum of each 16 / 8 consecutive products added to the accumulator with one rounding (MMA K-steps)."""
    p = qt[:, None, :] * x[None, :, :]                       # float64, exact
    d = p.shape[-1]
    if scheme == "lanes":
        lanes = []
        for lane in range(8):
            acc = np.zeros(p.shape[:-1])
            for c in range(0, d, 64):
                for j in range(c + lane * 8, min(c + lane * 8 + 8, d)):
                    acc = _r32(acc + p[..., j], truncate)
            lanes.append(acc)
        while len(lanes) > 1:
            lanes = [_r32(lanes[i] + lanes[i + 1], truncate) for i in range(0, len(lanes), 2)]
        return lanes[0]
    w = 16 if scheme == "block16" else 8
    acc = np.zeros(p.shape[:-1])
    for i in range(0, d, w):
        acc = _r32(acc + p[..., i:i + w].sum(axis=-1), truncate)
    return acc


@pytest.mark.parametrize("truncate", [False, True], ids=["nearest", "truncate"])
def test_bound_holds_for_kernel_accumulation_orders(truncate):
    xb = fm.store(synth.clip_like(300, 512, seed=5, n_centres=16))
    xq = synth.clip_like(4, 512, seed=6, n_centres=16) * np.float32(7.3)
    worst = 0.0
    for path, schemes in (("stream", ("lanes",)), ("mma", ("block16", "block8"))):
        qt, scale = fm.prepare_query(xq, path)
        m, eps = fm._scores(qt, scale, xb)
        for scheme in schemes:
            got = _emulate(qt, xb.astype(np.float64), scheme, truncate) * scale[:, None]
            worst = max(worst, float((np.abs(got - m) / eps).max()))
    print(f"largest |emulated - m| / eps ({'truncated' if truncate else 'rounded'} fp32 steps): {worst:.4f}")
    assert worst <= 1.0


def test_keys_round_trip():
    D = np.array([[3.5, 0.0, -0.0, -2.0]], np.float32)
    I = np.array([[7, 2, 9, 0]], np.int64)
    o = fm.f2ord(D).astype(np.uint64)
    keys = ((o << np.uint64(32)) | (~(I.astype(np.uint64) + np.uint64(5)) & np.uint64(0xffffffff))).view(np.int64)
    keys[0, 3] = 0
    D2, I2 = fm.keys_to_DI(keys)
    np.testing.assert_array_equal(D2[0, :3], D[0, :3])
    assert np.signbit(D2[0, 2]) and D2[0, 3] == -fm.FLT_MAX
    assert I2.tolist() == [[12, 7, 14, -1]]


def _setup(n=30000, d=512, nq=16, k=100):
    xb = synth.clip_like(n, d, seed=11)
    xq = synth.clip_like(nq, d, seed=12)
    rows16 = fm.store(xb)
    ref = flat_ip.IndexFlatIP(d)
    ref.add(rows16.astype(np.float32))                            # the oracle over the stored rows
    return xq, rows16, ref


def test_model_accepts_exact_result_and_rejects_next_row():
    """The demonstration: a result that swaps its k-th row for the (k+1)-th passes the 1e-3 comparator and fails the
    model check."""
    k = 100
    xq, rows16, ref = _setup(k=k)
    m, eps = fm.scores(xq, rows16, "mma")
    order = np.lexsort((np.broadcast_to(np.arange(m.shape[1]), m.shape), -m), axis=1)
    I = order[:, :k].astype(np.int64)
    D = np.take_along_axis(m, I, 1).astype(np.float32)
    assert not fm.check_topk(D, I, xq, rows16, "mma")
    I2, D2 = I.copy(), D.copy()
    I2[:, k - 1] = order[:, k]
    D2[:, k - 1] = np.take_along_axis(m, order[:, k:k + 1], 1)[:, 0].astype(np.float32)
    # the dropped row is provably better wherever its lower bound clears the substitute's score
    low = np.take_along_axis(m - eps, order[:, k - 1:k], 1)[:, 0]
    wide = low > D2[:, k - 1]
    assert wide.sum() >= len(xq) // 2
    Dr, Ir = ref.search(xq, k)
    assert not comparator.compare_topk(D2, I2, Dr, Ir, lambda ids: ref.scores_of(xq, ids))
    bad = fm.check_topk(D2, I2, xq, rows16, "mma")
    flagged = {int(b.split()[0][1:-1]) for b in bad if "outside the result" in b}
    assert flagged == set(np.nonzero(wide)[0].tolist())


def test_model_rejects_range_result_missing_a_hit_above_radius():
    xq, rows16, ref = _setup(nq=4)
    m, eps = fm.scores(xq, rows16, "mma")
    radius = float(np.float32(np.sort(m[0])[-50] - 2e-4))          # row 50 of query 0 lies 2e-4 above the radius
    lims, D, I = range_search.range_search(rows16.astype(np.float32), xq, radius)
    # the model's D: the oracle's hit set, scored by the model (exact result)
    D = np.concatenate([m[q, I[lims[q]:lims[q + 1]]] for q in range(4)]).astype(np.float32)
    for q in range(4):                                       # key order of the model's scores
        a, b = lims[q], lims[q + 1]
        o = np.lexsort((I[a:b], -D[a:b]))
        D[a:b], I[a:b] = D[a:b][o], I[a:b][o]
    keep = np.ones(D.size, bool)
    a = lims[0]
    j = a + int(np.argmin(np.abs(D[a:lims[1]] - (radius + 2e-4))))
    keep[j] = False
    assert not fm.check_range(lims, D, I, xq, rows16, "mma", radius)
    lims2 = lims.copy()
    lims2[1:] -= 1
    D2, I2 = D[keep], I[keep]
    assert not range_search.compare_range(lims2, D2, I2, lims, D, I,
                                          lambda q, ids: ref.scores_of(xq[q:q + 1], ids[None])[0], radius)
    bad = fm.check_range(lims2, D2, I2, xq, rows16, "mma", radius)
    assert any("left out" in b and b.split()[0] == "q0:" for b in bad)
