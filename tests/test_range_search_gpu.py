"""GPU: exact range search (IndexFlatIP.range_search) against the fp32 oracle under the radius band of
oracle/range_search.py (compare_range)."""
import ctypes

import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat
from oracle import comparator, flat_ip, synth
from oracle import range_search as orr

pytestmark = pytest.mark.gpu
TOL = 1e-3


def build(xb):
    idx = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
    idx.add(xb)
    return idx


def check(lims, D, I, xb, xq, radius, tol=TOL, id_shift=0):
    lims_r, D_r, I_r = orr.range_search(xb, xq, radius)
    bad = orr.compare_range(lims, D, I - id_shift, lims_r, D_r, I_r,
                            lambda q, ids: xb[ids] @ xq[q], radius, tol)
    assert not bad, bad[:5]
    return lims_r


def kth_radius(xb, xq, kth):
    """median over queries of the kth-best fp32 score: about kth hits per query"""
    s = np.sort(xq @ xb.T, axis=1)[:, ::-1]
    return float(np.median(s[:, min(kth, s.shape[1]) - 1]))


@pytest.mark.parametrize("d", [64, 100, 384, 512, 768, 1024])
@pytest.mark.parametrize("nq", [1, 2, 16, 17, 128, 129, 300])
def test_range_search_dims_and_batches(d, nq):
    n = 3000
    xb = synth.clip_like(n, d, seed=d)
    xq = synth.clip_like(nq, d, seed=1000 + nq)
    idx = build(xb)
    s = xq @ xb.T
    radii = {"none": float(s.max()) + 0.01, "about_10": kth_radius(xb, xq, 10),
             "about_1000": kth_radius(xb, xq, 1000), "all": float(s.min()) - 0.01}
    for name, r in radii.items():
        lims, D, I = idx.range_search(xq, r)
        lims_r = check(lims, D, I, xb, xq, r)
        if name == "none":
            assert lims[-1] == 0
        if name == "all":
            assert lims_r[-1] == nq * n and lims[-1] == nq * n


def test_range_search_infinite_radii():
    xb = synth.clip_like(1000, 128, seed=3)
    xq = synth.clip_like(5, 128, seed=4)
    idx = build(xb)
    lims, D, I = idx.range_search(xq, np.inf)
    assert lims.tolist() == [0] * 6 and D.size == 0
    lims, D, I = idx.range_search(xq, -np.inf)
    assert np.all(np.diff(lims) == 1000)
    check(lims, D, I, xb, xq, -np.inf)
    with pytest.raises(ValueError):
        idx.range_search(xq, float("nan"))


def test_range_search_empty_index_no_queries_and_tiny_index():
    idx = ivr_b200.IndexFlatIP(64, device=0)
    xq = synth.clip_like(3, 64, seed=5)
    lims, D, I = idx.range_search(xq, -np.inf)
    assert lims.tolist() == [0, 0, 0, 0] and D.size == 0 and I.size == 0
    xb = synth.clip_like(50, 64, seed=6)                      # one partial 128-row tile
    idx.add(xb)
    lims, D, I = idx.range_search(np.zeros((0, 64), np.float32), 0.0)
    assert lims.tolist() == [0] and D.size == 0
    for r in (-np.inf, kth_radius(xb, xq, 10), 0.9):
        lims, D, I = idx.range_search(xq, r)
        check(lims, D, I, xb, xq, r)


def test_range_search_dimension_too_wide_is_unsupported():
    idx = ivr_b200.IndexFlatIP(4160, device=0)
    with pytest.raises(nat.NativeError) as e:
        idx.range_search(np.zeros((1, 4160), np.float32), 0.0)
    assert e.value.code == nat.IVR_EUNSUPPORTED
    idx = ivr_b200.IndexFlatIP(4096, device=0)                # the widest that fits: 16 queries per launch
    xb = synth.clip_like(300, 4096, seed=7)
    idx.add(xb)
    xq = synth.clip_like(20, 4096, seed=8)
    r = kth_radius(xb, xq, 30)
    lims, D, I = idx.range_search(xq, r)
    check(lims, D, I, xb, xq, r)


def test_range_search_overflow_reports_the_total_and_the_retry_matches_one_shot():
    import torch
    xb = synth.clip_like(4000, 256, seed=9)
    xq = synth.clip_like(20, 256, seed=10)
    idx = build(xb)
    r = kth_radius(xb, xq, 200)
    lims1, D1, I1 = idx.range_search(xq, r)
    total = int(lims1[-1])
    assert total > 10
    # host entry point, capacity 10: lims[nq] is the exact total, D / I untouched
    lims = np.full(21, -7, np.int64)
    D = np.full(10, 42.0, np.float32)
    I = np.full(10, -9, np.int64)
    nat.check(nat.lib.ivr_index_range_search(idx._handle(), xq.ctypes.data, 20, r, 10, lims.ctypes.data,
                                             D.ctypes.data, I.ctypes.data))
    assert lims[20] == total
    assert np.all(D == 42.0) and np.all(I == -9)
    D = np.empty(total, np.float32)
    I = np.empty(total, np.int64)
    nat.check(nat.lib.ivr_index_range_search(idx._handle(), xq.ctypes.data, 20, r, total, lims.ctypes.data,
                                             D.ctypes.data, I.ctypes.data))
    np.testing.assert_array_equal(lims, lims1)
    np.testing.assert_array_equal(D, D1)
    np.testing.assert_array_equal(I, I1)
    # device entry point, same contract
    q = torch.from_numpy(xq).cuda()
    L = torch.full((21,), -7, dtype=torch.int64, device="cuda")
    Dd = torch.full((10,), 42.0, device="cuda")
    Id = torch.full((10,), -9, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    nat.check(nat.lib.ivr_index_range_search_device(idx._handle(), q.data_ptr(), 20, r, 10, L.data_ptr(),
                                                    Dd.data_ptr(), Id.data_ptr(), 0, st))
    torch.cuda.synchronize()
    assert int(L[20]) == total
    assert bool((Dd == 42.0).all()) and bool((Id == -9).all())
    # the Python retry path: a first capacity below the total
    from ivr_b200 import faiss_compat
    orig = faiss_compat._range_capacity
    faiss_compat._range_capacity = lambda nq, ntotal: 7
    try:
        lims2, D2, I2 = idx.range_search(xq, r)
        Lt, Dt, It = idx.range_search_tensor(q, r)
    finally:
        faiss_compat._range_capacity = orig
    np.testing.assert_array_equal(lims2, lims1)
    np.testing.assert_array_equal(I2, I1)
    np.testing.assert_array_equal(It.cpu().numpy(), I1)


def test_range_search_scaled_queries():
    xb = synth.clip_like(5000, 512, seed=11)
    xq = synth.clip_like(16, 512, seed=12)
    idx = build(xb)
    r = kth_radius(xb, xq, 100)
    lims, D, I = idx.range_search(xq * np.float32(1e3), r * 1e3)
    check(lims, D, I, xb, xq * np.float32(1e3), r * 1e3, tol=TOL * 1e3)


def test_range_search_copies_are_all_returned_in_id_order():
    base = synth.clip_like(50, 128, seed=13)
    xb = np.tile(base, (40, 1))                                  # row i == row i + 50 j
    xq = synth.clip_like(3, 128, seed=14)
    idx = build(xb)
    r = kth_radius(base, xq, 5)
    lims, D, I = idx.range_search(xq, r)
    check(lims, D, I, xb, xq, r)
    for q in range(3):
        d, i = D[lims[q]:lims[q + 1]], I[lims[q]:lims[q + 1]]
        assert d.size % 40 == 0
        base_ids = np.unique(i % 50)
        assert d.size == 40 * base_ids.size                      # every copy of every hit
        for b in base_ids:
            run = np.nonzero(i % 50 == b)[0]
            assert np.all(np.diff(run) == 1)                     # copies are adjacent (equal scores) ...
            assert np.all(np.diff(i[run]) > 0)                   # ... ordered by id
            assert np.all(d[run] == d[run[0]])


def test_range_search_window_and_id_offset():
    import torch
    xb = synth.clip_like(6000, 384, seed=15)
    xq = synth.clip_like(17, 384, seed=16)
    idx = build(xb)
    first, count, off = 1234, 2500, 10_000
    win = xb[first:first + count]
    r = kth_radius(win, xq, 50)
    idx.set_window(first, count)
    try:
        L, Dt, It = idx.range_search_tensor(torch.from_numpy(xq).cuda(), r, id_offset=off)
    finally:
        idx.set_window()
    lims, D, I = L.cpu().numpy(), Dt.cpu().numpy(), It.cpu().numpy()
    assert np.all((I >= off + first) & (I < off + first + count))
    check(lims, D, I, win, xq, r, id_shift=off + first)


def test_range_search_prefix_agrees_with_search():
    xb = synth.clip_like(8000, 512, seed=17)
    xq = synth.clip_like(40, 512, seed=18)
    idx = build(xb)
    k = 100
    s = np.sort(xq @ xb.T, axis=1)[:, ::-1]
    r = float(s[:, k + 50].min())                                # every query has more than k hits
    lims, D, I = idx.range_search(xq, r)
    assert np.all(np.diff(lims) >= k)
    Dk = np.stack([D[lims[q]:lims[q] + k] for q in range(40)])
    Ik = np.stack([I[lims[q]:lims[q] + k] for q in range(40)])
    Ds, Is = idx.search(xq, k)
    ref = flat_ip.IndexFlatIP(512)
    ref.add(xb)
    bad = comparator.compare_topk(Dk, Ik, Ds, Is, lambda ids: ref.scores_of(xq, ids), TOL)
    assert not bad, bad[:5]


@pytest.mark.parametrize("nq", [3, 200])
def test_range_search_host_and_device_agree(nq):
    import torch
    xb = synth.clip_like(7000, 768, seed=19)
    xq = synth.clip_like(nq, 768, seed=20)
    idx = build(xb)
    r = kth_radius(xb, xq, 300)
    lims, D, I = idx.range_search(xq, r)
    L, Dt, It = idx.range_search(torch.from_numpy(xq).cuda(), r)          # CUDA tensor -> tensor variant
    assert L.is_cuda and Dt.is_cuda and It.is_cuda
    np.testing.assert_array_equal(L.cpu().numpy(), lims)
    np.testing.assert_array_equal(Dt.cpu().numpy(), D)
    np.testing.assert_array_equal(It.cpu().numpy(), I)
    check(lims, D, I, xb, xq, r)
