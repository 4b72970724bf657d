"""GPU: the exact range self-join (IndexFlatIP.range_self_join) against the model of tests/self_join_ref.py: bit for
bit on fp16_model.exact_inputs rows, within the fp16 model's bound on CLIP-like rows."""
import ctypes

import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat
from oracle import fp16_model as fm
from oracle import synth

import self_join_ref as sj

pytestmark = pytest.mark.gpu


def build(xb):
    idx = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
    idx.add(xb)
    return idx


def rows_of(kind, n, d, seed):
    if kind == "exact":
        return fm.exact_inputs(n, d, 1, seed=seed)[0]
    return synth.clip_like(n, d, seed=seed)


def radius_for(rows16, k=10):
    n = rows16.shape[0]
    if n < 2:
        return 0.0
    sample = np.random.default_rng(n).choice(n, 256, replace=False) if n > 1000 else None
    return sj.kth_radius(rows16, k, sample)


def join_and_check(idx, rows16, radius, exact, tag, **kw):
    lims, D, I = idx.range_self_join(radius)
    bad = sj.check_join(lims, D, I, rows16, radius, exact=exact, tag=tag, **kw)
    assert not bad, bad[:5]
    return lims, D, I


@pytest.mark.parametrize("d", [64, 512, 768, 1024, 4096])
@pytest.mark.parametrize("n", [0, 1, 2, 127, 128, 129, 255, 257, 1000, 4097])
def test_range_self_join_sizes_and_dims(n, d):
    for kind in ("exact", "clip"):
        xb = rows_of(kind, n, d, seed=n + d)
        rows16 = fm.store(xb)
        idx = build(xb)
        r = radius_for(rows16)
        lims, D, I = join_and_check(idx, rows16, r, kind == "exact", f"{kind} n={n} d={d}")
        if n < 2:
            assert lims.tolist() == [0] * (n + 1) and D.size == 0
        idx.close()


@pytest.mark.parametrize("d", [1, 63, 65, 100, 513, 1280])
def test_range_self_join_odd_dims(d):
    for kind in ("exact", "clip"):
        xb = rows_of(kind, 300, d, seed=d)
        rows16 = fm.store(xb)
        idx = build(xb)
        join_and_check(idx, rows16, radius_for(rows16), kind == "exact", f"{kind} d={d}")
        idx.close()


def _without_diagonal(lims, D, I):
    n = lims.size - 1
    row = np.repeat(np.arange(n), np.diff(lims))
    keep = I != row
    counts = np.bincount(row[keep], minlength=n)
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int64), D[keep], I[keep]


@pytest.mark.parametrize("d", [512, 768])
def test_range_self_join_equals_range_search_of_the_rows(d):
    xb = rows_of("exact", 1000, d, seed=7)
    idx = build(xb)
    rows16 = fm.store(xb)
    for r in (radius_for(rows16, 10), radius_for(rows16, 100)):
        got = idx.range_self_join(r)
        want = _without_diagonal(*idx.range_search(idx.reconstruct_n(), r))
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)                  # bit for bit on exact inputs
    xb = rows_of("clip", 1000, d, seed=8)
    idx = build(xb)
    r = radius_for(fm.store(xb))
    lims, D, I = idx.range_self_join(r)
    lims_r, D_r, I_r = _without_diagonal(*idx.range_search(idx.reconstruct_n(), r))
    ka = set(zip(np.repeat(np.arange(1000), np.diff(lims)).tolist(), I.tolist(), D.view(np.uint32).tolist()))
    kb = set(zip(np.repeat(np.arange(1000), np.diff(lims_r)).tolist(), I_r.tolist(), D_r.view(np.uint32).tolist()))
    print(f"clip-like d={d}: {len(ka ^ kb)} of {len(ka | kb)} (row, id, score) entries differ between the join and "
          "range_search of the reconstructed rows (different fp32 accumulation orders)")


def test_range_self_join_duplicated_rows_and_ties():
    d = 768                                                          # npad = 80: blocks and 128-row tiles misalign
    xb = rows_of("exact", 400, d, seed=21)
    copies = {5: [70, 300, 301], 10: [200], 3: [50], 79: [80], 159: [160, 399]}
    for src, dst in copies.items():
        xb[dst] = xb[src]
    rows16 = fm.store(xb)
    idx = build(xb)
    self_score = float((rows16[5].astype(np.float64) ** 2).sum())
    r = radius_for(rows16)
    lims, D, I = join_and_check(idx, rows16, r, True, "duplicates")
    for src, dst in copies.items():
        group = [src] + dst
        for a in group:
            ids = I[lims[a]:lims[a + 1]]
            assert all(b in ids for b in group if b != a), (a, group)
    ids, d5 = I[lims[5]:lims[5 + 1]], D[lims[5]:lims[5 + 1]]
    tied = ids[d5 == np.float32(self_score)]
    assert tied.tolist() == sorted(tied.tolist()) and {70, 300, 301} <= set(tied.tolist())


def test_range_self_join_nan_rows_and_infinite_radii():
    xb = rows_of("clip", 300, 512, seed=4)
    xb[[7, 150]] = np.nan
    xb[200, 3] = np.nan
    rows16 = fm.store(xb)
    idx = build(xb)
    nan_rows = [7, 150, 200]
    lims, D, I = join_and_check(idx, rows16, radius_for(rows16), False, "nan rows")
    for i in nan_rows:
        assert lims[i + 1] == lims[i]
    assert not np.isin(I, nan_rows).any()
    lims, D, I = idx.range_self_join(np.inf)
    assert lims.tolist() == [0] * 301 and D.size == 0
    lims, D, I = join_and_check(idx, rows16, -np.inf, False, "-inf")
    assert lims[-1] == 297 * 296
    with pytest.raises(ValueError):
        idx.range_self_join(float("nan"))
    with pytest.raises(ValueError):
        idx.range_self_join_tensor(float("nan"))
    small = build(rows_of("exact", 50, 64, seed=5))
    lims, D, I = small.range_self_join(-np.inf)
    assert lims[-1] == 50 * 49 and np.all(np.diff(lims) == 49)


def test_range_self_join_overflow_reports_the_total_and_retries():
    import torch
    xb = rows_of("exact", 1000, 512, seed=9)
    idx = build(xb)
    r = radius_for(fm.store(xb), 20)
    lims_w, D_w, I_w = idx.range_self_join(r)
    total = int(lims_w[-1])
    assert total > 10
    st = torch.cuda.current_stream().cuda_stream
    lims = torch.zeros(1001, dtype=torch.int64, device="cuda")
    D = torch.full((10,), -7.0, device="cuda")
    I = torch.full((10,), -9, dtype=torch.int64, device="cuda")
    nat.check(nat.lib.ivr_index_range_self_join_device(idx._handle(), r, 10, lims.data_ptr(), D.data_ptr(),
                                                       I.data_ptr(), st))
    assert int(lims[-1]) == total                                    # the exact total, D / I untouched
    assert torch.all(D == -7.0) and torch.all(I == -9)
    L = np.zeros(1001, np.int64)
    Dh, Ih = np.full(10, -7.0, np.float32), np.full(10, -9, np.int64)
    nat.check(nat.lib.ivr_index_range_self_join(idx._handle(), r, 10, L.ctypes.data, Dh.ctypes.data, Ih.ctypes.data))
    assert L[-1] == total and np.all(Dh == -7.0) and np.all(Ih == -9)
    D = torch.empty(total, device="cuda")
    I = torch.empty(total, dtype=torch.int64, device="cuda")
    nat.check(nat.lib.ivr_index_range_self_join_device(idx._handle(), r, total, lims.data_ptr(), D.data_ptr(),
                                                       I.data_ptr(), st))
    np.testing.assert_array_equal(lims.cpu().numpy(), lims_w)
    np.testing.assert_array_equal(D.cpu().numpy(), D_w)
    np.testing.assert_array_equal(I.cpu().numpy(), I_w)


def test_range_self_join_of_a_window():
    xb = rows_of("exact", 1000, 768, seed=12)
    rows16 = fm.store(xb)
    idx = build(xb)
    first, count = 300, 400
    idx.set_window(first, count)
    r = radius_for(rows16[first:first + count])
    lims, D, I = idx.range_self_join(r)
    assert lims.shape == (count + 1,)
    assert I.size == 0 or (I.min() >= first and I.max() < first + count)
    bad = sj.check_join(lims, D, I, rows16[first:first + count], r, id_offset=first, exact=True, tag="window")
    assert not bad, bad[:5]
    lt, Dt, It = idx.range_self_join_tensor(r)
    assert lt.numel() == count + 1
    np.testing.assert_array_equal(lt.cpu().numpy(), lims)
    np.testing.assert_array_equal(It.cpu().numpy(), I)
    alone = build(xb[first:first + count])
    la, Da, Ia = alone.range_self_join(r)
    np.testing.assert_array_equal(la, lims)
    np.testing.assert_array_equal(Da, D)
    np.testing.assert_array_equal(Ia + first, I)
    idx.set_window()
    assert idx.range_self_join(r)[0].shape == (1001,)


@pytest.mark.parametrize("kind", ["exact", "clip"])
def test_range_self_join_host_and_device_variants_agree(kind):
    xb = rows_of(kind, 2000, 1024, seed=13)
    idx = build(xb)
    r = radius_for(fm.store(xb), 30)
    lims, D, I = idx.range_self_join(r)
    lt, Dt, It = idx.range_self_join_tensor(r)
    assert lt.is_cuda and Dt.is_cuda and It.is_cuda
    np.testing.assert_array_equal(lt.cpu().numpy(), lims)
    np.testing.assert_array_equal(Dt.cpu().numpy().view(np.uint32), D.view(np.uint32))
    np.testing.assert_array_equal(It.cpu().numpy(), I)


def test_range_self_join_shares_the_workspace_with_searches():
    xb = rows_of("clip", 3000, 512, seed=14)
    idx = build(xb)
    r = radius_for(fm.store(xb))
    first = idx.range_self_join(r)
    xq = synth.clip_like(40, 512, seed=15)
    D1, I1 = idx.search(xq, 50)
    R1 = idx.range_search(xq, r)
    again = idx.range_self_join(r)
    for a, b in zip(first, again):
        np.testing.assert_array_equal(a, b)
    D2, I2 = idx.search(xq, 50)
    R2 = idx.range_search(xq, r)
    np.testing.assert_array_equal(D1, D2)
    np.testing.assert_array_equal(I1, I2)
    for a, b in zip(R1, R2):
        np.testing.assert_array_equal(a, b)


def test_range_self_join_many_ctas():
    n, d = 300_000, 512
    xb = synth.clip_like(n, d, seed=16)
    rows16 = fm.store(xb)
    idx = build(xb)
    sample = np.random.default_rng(0).choice(n, 256, replace=False)
    r = sj.kth_radius(rows16, 10, sample)
    lims, D, I = idx.range_self_join_tensor(r)
    lims, D, I = lims.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy()
    assert lims.shape == (n + 1,) and lims[0] == 0 and np.all(np.diff(lims) >= 0)
    assert lims[-1] == D.size == I.size and lims[-1] % 2 == 0
    assert not sj.symmetry_violations(lims, D, I, tag="300k")
    bad = sj.check_join(lims, D, I, rows16, r, sample=sample, block=64, tag="300k")
    assert not bad, bad[:5]
    print(f"300k x 512: {int(lims[-1])} hits, {lims[-1] / n:.1f} per row")
