"""GPU: filtered search (SearchParameters(sel=...)) against the float64 model of the library's arithmetic.

The model is oracle/fp16_model.py, unchanged: the rows left out of the selection are set to NaN in the model's copy
of the stored rows, so ``check_topk`` / ``check_range`` with ``path="mma"`` state exactly "the k best selected rows"
and "every selected row above the radius".  On ``fm.exact_inputs`` every accumulation order is exact and the results
must match the model bit for bit."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import fp16_model as fm, synth  # noqa: E402

SEL_KERNEL = "search_mma_small_sel_kernel"


def make_index(xb):
    import ivr_b200
    idx = ivr_b200.IndexFlatIP(xb.shape[1])
    idx.set_timing(True)
    idx.add(xb)
    return idx


def data(kind, n, d, nq, seed):
    if kind == "exact":
        return fm.exact_inputs(n, d, nq, seed)
    return synth.clip_like(n, d, seed, n_centres=256), synth.clip_like(nq, d, seed + 1, n_centres=256)


def selector(name, n, seed=0):
    """(selector, bool mask [n]) of the named selection over n rows."""
    from ivr_b200 import faiss_compat as fc
    rng = np.random.default_rng(seed)
    mask = np.zeros(n, bool)
    if name == "empty":
        sel = fc.IDSelectorBatch([])
    elif name == "one":
        sel = fc.IDSelectorBatch([n // 3])
    elif name == "video":                            # one contiguous, tile-unaligned run
        a, b = n // 5 + 37, n // 5 + 37 + max(n // 40, 300)
        sel = fc.IDSelectorRange(a, b)
    elif name == "ranges":
        runs = [(5, 77), (n // 2 - 100, n // 2 + 150), (n - 200, n - 3)]
        m = np.zeros(n, bool)
        for a, b in runs:
            m[a:b] = True
        sel = fc.IDSelectorBitmap(np.packbits(m, bitorder="little"))
    elif name == "rand1":
        sel = fc.IDSelectorBatch(rng.choice(n, max(n // 100, 1), replace=False))
    elif name == "rand50":
        sel = fc.IDSelectorNot(fc.IDSelectorBatch(rng.choice(n, n // 2, replace=False)))
    elif name == "all":
        sel = fc.IDSelectorRange(0, n)
    elif name == "beyond":                           # ids past ntotal are ignored
        sel = fc.IDSelectorRange(n - 500, n + 100_000)
    else:
        raise ValueError(name)
    mask[:] = sel._mask(n)
    return sel, mask


def masked(rows16, mask):
    r = rows16.copy()
    r[~mask] = np.nan
    return r


def params(sel):
    from ivr_b200 import faiss_compat as fc
    return fc.SearchParameters(sel=sel)


def check_search(idx, rows16, mask, sel, xq, k, exact=False, device=False, id_offset=0):
    import torch
    if device:
        D, I = idx.search_tensor(torch.from_numpy(xq).cuda(), k, id_offset=id_offset, params=params(sel))
        D, I = D.cpu().numpy(), I.cpu().numpy()
    else:
        D, I = idx.search(xq, k, params=params(sel))
    bad = fm.check_topk(D, I, xq, masked(rows16, mask), "mma", id_offset=id_offset, exact=exact, tag="sel")
    assert not bad, "\n".join(bad[:10])
    t = idx.last_timing()
    if mask[:idx.ntotal].any():
        assert t["kernel"] == SEL_KERNEL and t["score_launches"] >= 1
    else:
        assert t["path"] == "empty" and t["score_launches"] == 0
    return D, I


def check_range(idx, rows16, mask, sel, xq, radius, exact=False, device=False):
    import torch
    if device:
        lims, D, I = (t.cpu().numpy() for t in idx.range_search_tensor(torch.from_numpy(xq).cuda(), radius,
                                                                         params=params(sel)))
    else:
        lims, D, I = idx.range_search(xq, radius, params=params(sel))
    bad = fm.check_range(lims, D, I, xq, masked(rows16, mask), "mma", radius, exact=exact, tag="sel_range")
    assert not bad, "\n".join(bad[:10])
    return lims, D, I


SELECTIONS = ["empty", "one", "video", "ranges", "rand1", "rand50", "all", "beyond"]


@pytest.mark.parametrize("kind", ["exact", "clip"])
@pytest.mark.parametrize("name", SELECTIONS)
def test_selections(name, kind):
    d, n = 512, 100_000                              # 782 row tiles: the broad selections run seeded launches
    xb, xq = data(kind, n, d, 300, seed=11)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    sel, mask = selector(name, n, seed=12)
    for nq in (1, 17, 129):
        check_search(idx, rows16, mask, sel, xq[:nq], 100, exact=kind == "exact")
    m, _ = fm.scores(xq[:17], masked(rows16, mask), "mma")
    fin = np.where(np.isnan(m), -np.inf, m)
    radius = float(np.float32(np.median(np.sort(fin, axis=1)[:, -30]))) if mask.any() else 0.0
    if not np.isfinite(radius):
        radius = -1.0
    check_range(idx, rows16, mask, sel, xq[:17], radius, exact=kind == "exact")
    sel.close()


@pytest.mark.parametrize("nq", [1, 16, 17, 128, 129, 300])
def test_query_counts(nq):
    d, n = 512, 30_000
    xb, xq = data("clip", n, d, nq, seed=nq)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    for name in ("video", "rand1"):
        sel, mask = selector(name, n, seed=nq)
        check_search(idx, rows16, mask, sel, xq, 100)
        check_search(idx, rows16, mask, sel, xq, 100, device=True, id_offset=1000)


@pytest.mark.parametrize("kind", ["exact", "clip"])
@pytest.mark.parametrize("d", [64, 512, 768, 1024])
def test_dims_and_k(d, kind):
    n = 20_000
    xb, xq = data(kind, n, d, 130, seed=d)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    sel, mask = selector("video", n)
    cnt = int(mask.sum())
    for k in (1, 100, cnt + 50, 2048):
        for nq in (16, 130):
            check_search(idx, rows16, mask, sel, xq[:nq], k, exact=kind == "exact")
    D, I = idx.search(xq[:16], cnt + 50, params=params(sel))
    assert np.all(I[:, cnt:] == -1) and np.all(D[:, cnt:] == -np.finfo(np.float32).max)
    m, _ = fm.scores(xq, masked(rows16, mask), "mma")
    radius = float(np.float32(np.median(np.sort(np.nan_to_num(m, nan=-np.inf), axis=1)[:, -20])))
    check_range(idx, rows16, mask, sel, xq, radius, exact=kind == "exact")


def test_nan_rows_inside_and_outside():
    d, n = 256, 20_000
    xb, xq = data("clip", n, d, 24, seed=5)
    sel, mask = selector("video", n)
    inside = np.nonzero(mask)[0]
    nan_at = np.concatenate([inside[[0, 1, 31, 32, 127, -1]], [0, 127, 128, n - 1]])
    xb[nan_at, 3] = np.nan
    rows16 = fm.store(xb)
    idx = make_index(xb)
    for k in (100, int(mask.sum())):
        check_search(idx, rows16, mask, sel, xq, k)
    check_range(idx, rows16, mask, sel, xq, -1.0)    # every finite selected row is a hit


SCALES = [2.0 ** -140, 1.5 * 2.0 ** -128, 1e-30, 1e30]


def test_query_magnitudes():
    d = 512
    xb = synth.clip_like(20000, d, seed=21, n_centres=256)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    sel, mask = selector("ranges", 20000)
    base = synth.clip_like(6, d, seed=22, n_centres=256)
    sub = base.copy()
    sub[:, 1::2] *= np.float32(2.0 ** -20)
    onehot = np.zeros((1, d), np.float32)
    onehot[0, 5] = np.float32(3.2e38)
    batches = [(base * np.float32(s)).astype(np.float32) for s in SCALES] + [onehot, np.zeros((1, d), np.float32), sub]
    for xq in batches:
        check_search(idx, rows16, mask, sel, np.resize(xq, (8, d)).astype(np.float32), 100)
        check_range(idx, rows16, mask, sel, xq, 0.0)
    xb2, xq2 = fm.exact_inputs(5000, d, 8, seed=24, query_exp=-140)
    idx2, rows2 = make_index(xb2), fm.store(xb2)
    sel2, mask2 = selector("rand50", 5000)
    check_search(idx2, rows2, mask2, sel2, xq2, 100, exact=True)
    check_range(idx2, rows2, mask2, sel2, xq2, 0.0, exact=True)


@pytest.mark.parametrize("nq", [2, 16, 100, 128])
def test_all_selected_equals_unfiltered(nq, monkeypatch):
    """Every row selected: the filtered kernel streams the same tiles in the same launches as the list mode of
    search_mma_small_kernel, so D and I agree bit for bit; range search with every row selected is range_search."""
    from ivr_b200 import faiss_compat as fc
    monkeypatch.setenv("IVR_MMA_MODE", "3")
    monkeypatch.setenv("IVR_SMALL_DUMP_MAX_KROWS", "0")
    for n in (30_000, 100_000):                      # one launch; two seeded launches
        xb, xq = data("clip", n, 512, nq, seed=n + nq)
        idx = make_index(xb)
        D0, I0 = idx.search(xq, 100)
        assert idx.last_timing()["kernel"] == "search_mma_small_kernel"
        launches = idx.last_timing()["score_launches"]
        sel = fc.IDSelectorRange(0, n)
        D, I = idx.search(xq, 100, params=fc.SearchParameters(sel=sel))
        assert idx.last_timing()["kernel"] == SEL_KERNEL and idx.last_timing()["score_launches"] == launches
        assert np.array_equal(D, D0) and np.array_equal(I, I0)
        radius = float(np.float32(np.median(np.sort(xq @ xb.T, axis=1)[:, -40])))
        r0 = idx.range_search(xq, radius)
        r1 = idx.range_search(xq, radius, params=fc.SearchParameters(sel=sel))
        assert all(np.array_equal(a, b) for a, b in zip(r0, r1))
        sel.close()


@pytest.mark.parametrize("name", ["video", "ranges", "rand1", "rand50"])
def test_range_equals_filtered_unfiltered(name):
    """Filtered range search == range_search with the unselected hits dropped on the host, bit for bit."""
    import torch
    n, d = 50_000, 768
    xb, xq = data("clip", n, d, 100, seed=3)
    idx = make_index(xb)
    sel, mask = selector(name, n, seed=4)
    radius = float(np.float32(np.median(np.sort(xq @ xb.T, axis=1)[:, -200])))
    lims0, D0, I0 = idx.range_search(xq, radius)
    keep = mask[I0]
    q_of = np.repeat(np.arange(len(xq)), np.diff(lims0))
    want_lims = np.concatenate([[0], np.cumsum(np.bincount(q_of[keep], minlength=len(xq)))])
    lims, D, I = idx.range_search(xq, radius, params=params(sel))
    assert np.array_equal(lims, want_lims) and np.array_equal(D, D0[keep]) and np.array_equal(I, I0[keep])
    lt, Dt, It = idx.range_search_tensor(torch.from_numpy(xq).cuda(), radius, params=params(sel))
    assert np.array_equal(lt.cpu().numpy(), lims) and np.array_equal(Dt.cpu().numpy(), D)
    assert np.array_equal(It.cpu().numpy(), I)


def test_host_and_tensor_agree_and_window_raises():
    import torch
    from ivr_b200 import _native as nat
    n, d = 20_000, 512
    xb, xq = data("clip", n, d, 40, seed=8)
    idx = make_index(xb)
    sel, _ = selector("rand1", n)
    D, I = idx.search(xq, 50, params=params(sel))
    Dt, It = idx.search_tensor(torch.from_numpy(xq).cuda(), 50, params=params(sel))
    assert np.array_equal(D, Dt.cpu().numpy()) and np.array_equal(I, It.cpu().numpy())
    idx.set_window(100, 5000)
    with pytest.raises(nat.NativeError) as e:
        idx.search(xq, 50, params=params(sel))
    assert e.value.code == nat.IVR_EINVAL and "window" in str(e.value)
    with pytest.raises(nat.NativeError) as e:
        idx.range_search(xq, 0.5, params=params(sel))
    assert e.value.code == nat.IVR_EINVAL and "window" in str(e.value)
    idx.set_window()
    D2, I2 = idx.search(xq, 50, params=params(sel))
    assert np.array_equal(D, D2) and np.array_equal(I, I2)


def test_selection_longer_than_ntotal_and_count():
    """A bitmap over more rows than the index holds: the rows at or past ntotal are ignored."""
    from ivr_b200 import _native as nat
    n, d = 5000, 512
    xb, xq = data("exact", n, d, 16, seed=9)
    rows16 = fm.store(xb)
    idx = make_index(xb)
    n_rows = n + 3000
    words = np.full((n_rows + 31) // 32, 0xAAAAAAAA, np.uint32)      # odd rows, also in the last partial word
    h = ctypes.c_void_p()
    nat.check(nat.lib.ivr_selection_create(0, words.ctypes.data, n_rows, ctypes.byref(h)))
    try:
        assert nat.lib.ivr_selection_count(h) == n_rows // 2
        D = np.empty((16, 100), np.float32)
        I = np.empty((16, 100), np.int64)
        nat.check(nat.lib.ivr_index_search_selected(idx._handle(), h, xq.ctypes.data, 16, 100, D.ctypes.data,
                                                    I.ctypes.data))
        mask = (np.arange(n) & 1).astype(bool)
        bad = fm.check_topk(D, I, xq, masked(rows16, mask), "mma", exact=True, tag="beyond")
        assert not bad, "\n".join(bad[:10])
    finally:
        nat.lib.ivr_selection_destroy(h)


def test_empty_index():
    import ivr_b200
    from ivr_b200 import faiss_compat as fc
    idx = ivr_b200.IndexFlatIP(512)
    idx.set_timing(True)
    xq = synth.clip_like(3, 512, seed=1)
    D, I = idx.search(xq, 10, params=fc.SearchParameters(sel=fc.IDSelectorRange(0, 100)))
    assert np.all(I == -1) and np.all(D == -np.finfo(np.float32).max)
    assert idx.last_timing()["score_launches"] == 0
    lims, D, I = idx.range_search(xq, 0.0, params=fc.SearchParameters(sel=fc.IDSelectorRange(0, 100)))
    assert lims.tolist() == [0, 0, 0, 0] and D.size == 0


def test_search_vectors_videos():
    """videos= returns the k best frames of those videos; the filter_func post-filter of the global top-k finds fewer."""
    from ivr_b200.unified_index import UnifiedIndex
    n, d, k = 40_000, 512, 50
    xb = synth.clip_like(n, d, seed=31, n_centres=256)
    folders = [f"video_{i // 400:03d}" for i in range(n)]          # 100 videos of 400 frames
    u = UnifiedIndex()
    u.build_from_embeddings(xb, [{"folder_name": f, "frame_id": i} for i, f in enumerate(folders)])
    q = synth.clip_like(1, d, seed=32, n_centres=256)[0]
    want_videos = ["video_007", "video_042"]
    got = u.search_vectors(q, k=k, videos=want_videos)
    post = u.search_vectors(q, k=k, filter_func=lambda m: m["folder_name"] in want_videos)
    assert len(got) == k and len(post) < k
    assert [r["rank"] for r in got] == list(range(k))
    assert all(r["metadata"]["folder_name"] in want_videos for r in got)
    rows = u.video_rows(want_videos)
    xn = xb / np.linalg.norm(xb, axis=1, keepdims=True)
    qn = q / np.linalg.norm(q)
    best = rows[np.argsort(-(xn[rows] @ qn), kind="stable")[:k]]
    assert len(set(r["index"] for r in got) & set(best.tolist())) >= k - 2    # fp16 rows: ties near the k-th
    assert {r["index"] for r in post} <= {r["index"] for r in got}
    # filter_func still applies, ranks stay those of the filtered top-k
    odd = u.search_vectors(q, k=k, videos=want_videos, filter_func=lambda m: m["frame_id"] % 2 == 1)
    assert [r["index"] for r in odd] == [r["index"] for r in got if r["index"] % 2 == 1]
    assert [r["rank"] for r in odd] == [r["rank"] for r in got if r["index"] % 2 == 1]
    assert u.search_vectors(q, k=k, videos=["no_such_video"]) == []
    batch = u.search_vectors_batch(np.stack([q, q]), k=k, videos=want_videos)
    assert [r["index"] for r in batch[0]] == [r["index"] for r in got] == [r["index"] for r in batch[1]]
    assert u.search_vectors(q, k=k) == u.search_vectors(q, k=k, videos=None)
