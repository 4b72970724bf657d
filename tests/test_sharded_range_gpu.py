"""GPU: range search across row shards with several RANKS IN ONE PROCESS on one device.

Every rank runs its local ``range_search_keys_tensor`` (a shard index of its own, or a window of one index with an
id offset, as the elastic boundaries use it); the all-gather of ``ShardedFlatIP.range_search`` is replaced by a
``torch.stack`` of the runs padded to the longest, and every rank merges the stack with ``ivr_range_merge_keys_device``
itself.  The result must pass ``compare_range`` against the fp32 oracle, be identical on every rank, equal the host
restatement of the merge, and equal ``IndexFlatIP.range_search`` over the unsharded rows bit for bit: a row's score
depends only on its own fp16 values and the query, whichever rank scores it.
"""
import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat
from oracle import flat_ip, synth
from oracle import range_search as orr
from range_merge_ref import merge_range_parts

pytestmark = pytest.mark.gpu
TOL = 1e-3
BASE = 5000                     # global id of the first row in the window layout


def _rows(n, d, off):
    """CLIP-like rows whose last 5 rows before every inner shard boundary are copied right after it: equal scores
    on two ranks."""
    xb = synth.clip_like(n, d, seed=d + 1)
    for b in off[1:-1]:
        if 5 <= b <= n - 5:
            xb[b:b + 5] = xb[b - 5:b]
    return xb


def _local_runs(xb, off, q, radius, layout):
    """Each rank's (lims, keys) with global ids: 'shards' = one index per rank and id_offset = its first row;
    'windows' = one index of every row, rank r's window [off[r], off[r+1]) and id_offset = BASE."""
    runs = []
    if layout == "shards":
        for r in range(len(off) - 1):
            idx = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
            idx.add(xb[off[r]:off[r + 1]])
            runs.append(idx.range_search_keys_tensor(q, radius, id_offset=int(off[r])))
    else:
        idx = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
        idx.add(xb)
        for r in range(len(off) - 1):
            idx.set_window(int(off[r]), int(off[r + 1] - off[r]))
            runs.append(idx.range_search_keys_tensor(q, radius, id_offset=BASE))
        idx.set_window()
    return runs


def _exchange_and_merge(runs):
    """The two all-gathers as a stack of the padded runs, then the merge on every rank."""
    import torch
    from ivr_b200.sharded import _cuda_range_merge
    stride = max(int(k.numel()) for _, k in runs)
    keys_parts = torch.zeros((len(runs), stride), dtype=torch.int64, device="cuda")
    for r, (_, k) in enumerate(runs):
        keys_parts[r, :k.numel()] = k
    lims_parts = torch.stack([l for l, _ in runs])
    total = int(lims_parts[:, -1].sum())
    out = [_cuda_range_merge(keys_parts, lims_parts, total) for _ in runs]
    torch.cuda.synchronize()
    return out, keys_parts, lims_parts


def _kth_radius(xb, xq, kth):
    s = np.sort(xq @ xb.T, axis=1)[:, ::-1]
    return float(np.median(s[:, min(kth, s.shape[1]) - 1]))


@pytest.mark.parametrize("layout", ["shards", "windows"])
@pytest.mark.parametrize("nq", [1, 7, 130])
@pytest.mark.parametrize("d", [512, 768])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_range_merge_equals_the_unsharded_index(world, d, nq, layout):
    import torch
    from ivr_b200.sharded import partition_rows
    n = 6000
    off = partition_rows(n, world)
    xb = _rows(n, d, off)
    xq = synth.clip_like(nq, d, seed=2000 + nq)
    q = torch.from_numpy(xq).cuda()
    full = ivr_b200.IndexFlatIP(d, device=0)
    full.add(xb)
    shift = BASE if layout == "windows" else 0
    for radius in (_kth_radius(xb, xq, 10), _kth_radius(xb, xq, 1000), np.inf, -np.inf):
        runs = _local_runs(xb, off, q, radius, layout)
        out, keys_parts, lims_parts = _exchange_and_merge(runs)
        lims, D, I = (t.cpu().numpy() for t in out[0])
        for o in out[1:]:                                       # every rank holds the same result, bit for bit
            assert all(torch.equal(a, b) for a, b in zip(o, out[0]))
        lims_h, D_h, I_h = merge_range_parts(lims_parts.cpu().numpy(),
                                         [k[:l[-1]] for k, l in zip(keys_parts.cpu().numpy(),
                                                                    lims_parts.cpu().numpy())])
        np.testing.assert_array_equal(lims, lims_h)
        np.testing.assert_array_equal(I, I_h)
        np.testing.assert_array_equal(D, D_h)
        lims_f, D_f, I_f = full.range_search(xq, radius)        # the unsharded index: bit for bit
        np.testing.assert_array_equal(lims, lims_f)
        np.testing.assert_array_equal(I - shift, I_f)
        np.testing.assert_array_equal(D, D_f)
        lims_r, D_r, I_r = orr.range_search(xb, xq, radius)
        bad = orr.compare_range(lims, D, I - shift, lims_r, D_r, I_r, lambda qq, ids: xb[ids] @ xq[qq], radius, TOL)
        assert not bad, bad[:5]
        if radius == -np.inf:
            assert lims[-1] == nq * n


def test_overlapping_windows_stay_a_permutation():
    """Two ranks that both score rows [2000, 3000) (a caller bug): every hit of both runs is in the output once, an
    equal key of rank 0 before rank 1's."""
    import torch
    d, n, nq = 512, 4000, 9
    xb = synth.clip_like(n, d, seed=61)
    xq = synth.clip_like(nq, d, seed=62)
    radius = _kth_radius(xb, xq, 300)
    runs = _local_runs(xb, np.array([0, 3000, 4000]), torch.from_numpy(xq).cuda(), radius, "windows")
    idx = ivr_b200.IndexFlatIP(d, device=0)
    idx.add(xb)
    idx.set_window(2000, 2000)
    runs[1] = idx.range_search_keys_tensor(torch.from_numpy(xq).cuda(), radius, id_offset=BASE)
    out, keys_parts, lims_parts = _exchange_and_merge(runs)
    lims_h, D_h, I_h = merge_range_parts(lims_parts.cpu().numpy(),
                                         [k[:l[-1]] for k, l in zip(keys_parts.cpu().numpy(),
                                                                    lims_parts.cpu().numpy())])
    np.testing.assert_array_equal(out[0][0].cpu().numpy(), lims_h)
    np.testing.assert_array_equal(out[0][1].cpu().numpy(), D_h)
    np.testing.assert_array_equal(out[0][2].cpu().numpy(), I_h)
    I = out[0][2].cpu().numpy() - BASE
    assert np.sum((I >= 2000) & (I < 3000)) > 0 and lims_h[-1] == sum(int(l[-1]) for l, _ in runs)


def test_local_capacity_overflow_retries_to_the_same_runs():
    import torch
    from ivr_b200 import faiss_compat
    d, n, nq = 512, 6000, 20
    xb = synth.clip_like(n, d, seed=71)
    xq = torch.from_numpy(synth.clip_like(nq, d, seed=72)).cuda()
    idx = ivr_b200.IndexFlatIP(d, device=0)
    idx.add(xb)
    radius = _kth_radius(xb, xq.cpu().numpy(), 200)
    L1, K1 = idx.range_search_keys_tensor(xq, radius, id_offset=11)
    orig = faiss_compat._range_capacity
    faiss_compat._range_capacity = lambda nq, ntotal: 7
    try:
        L2, K2 = idx.range_search_keys_tensor(xq, radius, id_offset=11)
    finally:
        faiss_compat._range_capacity = orig
    assert int(L1[-1]) > 7
    assert torch.equal(L1, L2) and torch.equal(K1, K2)


def test_keys_unpack_to_the_range_search_result_and_the_id_limit():
    import torch
    d, n, nq = 768, 7000, 33
    xb = synth.clip_like(n, d, seed=81)
    xq = torch.from_numpy(synth.clip_like(nq, d, seed=82)).cuda()
    idx = ivr_b200.IndexFlatIP(d, device=0)
    idx.add(xb)
    radius = _kth_radius(xb, xq.cpu().numpy(), 100)
    for off in (0, 123_456, (1 << 32) - n):
        L, D, I = idx.range_search_tensor(xq, radius, id_offset=off)
        Lk, K = idx.range_search_keys_tensor(xq, radius, id_offset=off)
        Dk, Ik = flat_ip.unpack_keys(K.cpu().numpy().view(np.uint64))
        assert torch.equal(L, Lk)
        np.testing.assert_array_equal(Dk, D.cpu().numpy())
        np.testing.assert_array_equal(Ik, I.cpu().numpy())
    with pytest.raises(nat.NativeError) as e:
        idx.range_search_keys_tensor(xq, radius, id_offset=(1 << 32) - n + 1)
    assert e.value.code == nat.IVR_EUNSUPPORTED
    with pytest.raises(ValueError):
        idx.range_search_keys_tensor(xq, float("nan"))
    Lk, K = idx.range_search_keys_tensor(xq[:0], radius)
    assert Lk.tolist() == [0] and K.numel() == 0


def test_single_rank_sharded_range_search_is_the_local_range_search():
    import torch
    d, n, nq = 512, 9000, 12
    xb = synth.clip_like(n, d, seed=91)
    xq = synth.clip_like(nq, d, seed=92)
    sh = ivr_b200.ShardedFlatIP(d, device=0)
    assert sh.world == 1
    sh.add_global(xb)
    idx = ivr_b200.IndexFlatIP(d, device=0)
    idx.add(xb)
    radius = _kth_radius(xb, xq, 50)
    L, D, I = sh.range_search(torch.from_numpy(xq).cuda(), radius)
    assert L.is_cuda and D.is_cuda and I.is_cuda
    lims, Dr, Ir = idx.range_search(xq, radius)
    np.testing.assert_array_equal(L.cpu().numpy(), lims)
    np.testing.assert_array_equal(D.cpu().numpy(), Dr)
    np.testing.assert_array_equal(I.cpu().numpy(), Ir)
