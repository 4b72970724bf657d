"""GPU: the range self-join across row shards with several RANKS IN ONE PROCESS on one device.

Every rank runs the tasks of ``join_schedule`` on its local index (a window of one index of all rows, or an index of
its block plus a margin of each neighbour, as the elastic boundaries use it): the self-join keys of its window, then
the cross join against the rows of another rank, taken with ``rows_f16_tensor``.  The runs of the other side go to
their owner, and each rank merges its runs with ``ShardedFlatIP._merge_runs`` on the CUDA merge.  The result must
equal ``IndexFlatIP.range_self_join_tensor`` over the unsharded rows bit for bit: a pair's score depends only on the
two stored fp16 rows, and the lower row is on the streamed operand in both kernels.
"""
import os
import types

import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat
from ivr_b200.sharded import ShardedFlatIP, _cuda_range_merge, join_schedule, partition_rows
from oracle import flat_ip, synth
from oracle import fp16_model as fm

import self_join_ref as sj

pytestmark = pytest.mark.gpu
MARGIN = 300


class _Ranks:
    """The local indexes of `world` ranks over the rows xb with boundaries `bounds`; layout 'windows' or 'margins'."""

    def __init__(self, xb, bounds, layout):
        n, d = xb.shape
        self.bounds, self.world = bounds, len(bounds) - 1
        if layout == "windows":
            full = ivr_b200.IndexFlatIP(d, device=0)
            full.add(xb)
            self.idx, self.off = [full] * self.world, [0] * self.world
        else:
            self.idx, self.off = [], []
            for r in range(self.world):
                lo, hi = max(0, int(bounds[r]) - MARGIN), min(n, int(bounds[r + 1]) + MARGIN)
                ix = ivr_b200.IndexFlatIP(d, device=0)
                ix.add(xb[lo:hi])
                self.idx.append(ix)
                self.off.append(lo)

    def window(self, r, a, b):
        self.idx[r].set_window(a - self.off[r], b - a)

    def join(self, radius):
        """Every rank's merged (lims, D, I) over its window."""
        parts = [[] for _ in range(self.world)]
        for r in range(self.world):
            tasks = join_schedule(self.bounds, r)
            lo, hi = tasks[0][:2]
            self.window(r, lo, hi)
            parts[r].append((lo, hi) + tuple(self.idx[r].range_self_join_keys_tensor(radius, id_offset=self.off[r])))
            for a, b, p, c, d in tasks[1:]:
                other = self.idx[p].rows_f16_tensor(c - self.off[p], d - c)
                self.window(r, a, b)
                ls, ks, lo_, ko = self.idx[r].range_cross_join_keys_tensor(other, c, radius, c < a,
                                                                           id_offset=self.off[r])
                parts[r].append((a, b, ls, ks))
                parts[p].append((c, d, lo_, ko))
        ns = types.SimpleNamespace(_range_merge=_cuda_range_merge)
        import torch
        return [ShardedFlatIP._merge_runs(ns, parts[r], int(self.bounds[r]), int(self.bounds[r + 1]),
                                          torch.device("cuda", 0)) for r in range(self.world)]


def _cat(results):
    """The ranks' results in global row order."""
    import torch
    lims, D, I, base = [], [], [], 0
    for L, Dr, Ir in results:
        lims.append(L[:-1] + base)
        base += int(L[-1])
        D.append(Dr)
        I.append(Ir)
    lims.append(torch.tensor([base], dtype=torch.int64, device=results[0][0].device))
    return torch.cat(lims).cpu().numpy(), torch.cat(D).cpu().numpy(), torch.cat(I).cpu().numpy()


def _reference(xb, radius):
    full = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
    full.add(xb)
    return tuple(t.cpu().numpy() for t in full.range_self_join_tensor(radius))


def _assert_same(got, want):
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)


def _bounds(n, world, seed):
    """Boundaries off every 128-row tile and npad block edge."""
    w = 1.0 + 0.3 * np.random.default_rng(seed).random(world)
    b = partition_rows(n, world, weights=w)
    b[1:-1] += (b[1:-1] % 16 == 0)
    return b


def _radius(xb, k):
    rows16 = fm.store(xb)
    return sj.kth_radius(rows16, k, sample=np.arange(0, xb.shape[0], 41))


@pytest.mark.parametrize("layout", ["windows", "margins"])
@pytest.mark.parametrize("d", [64, 333, 512, 768, 1024])
@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_sharded_join_equals_the_unsharded_join(world, d, layout):
    n = 2411
    bounds = _bounds(n, world, seed=world * d)
    xb = synth.clip_like(n, d, seed=d + world)
    for b in bounds[1:-1]:                                  # rows duplicated across every shard boundary
        xb[b:b + 4] = xb[b - 4:b]
    ranks = _Ranks(xb, bounds, layout)
    for radius in (_radius(xb, 10), _radius(xb, 200)):
        got = _cat(ranks.join(radius))
        _assert_same(got, _reference(xb, radius))
        assert not sj.symmetry_violations(*got)
        assert got[0][-1] > 0


def test_sharded_join_agrees_with_the_model():
    n, d, world = 3001, 512, 4
    xb = synth.clip_like(n, d, seed=5)
    radius = _radius(xb, 50)
    got = _cat(_Ranks(xb, _bounds(n, world, 1), "margins").join(radius))
    bad = sj.check_join(*got, fm.store(xb), radius, sample=np.arange(0, n, 13))
    assert not bad, bad[:5]
    xe, _ = fm.exact_inputs(1500, 256, 1, seed=9)          # exact inputs: the model bit for bit
    radius = sj.kth_radius(fm.store(xe), 20)
    got = _cat(_Ranks(xe, _bounds(1500, 3, 2), "windows").join(radius))
    assert not sj.check_join(*got, fm.store(xe), radius, exact=True)


@pytest.mark.parametrize("radius", [-np.inf, -0.05, np.inf])
def test_nan_rows_and_extreme_radii(radius):
    n, d, world = 700, 768, 4
    xb = synth.clip_like(n, d, seed=17)
    xb[[3, 200, 201, 511], 5] = np.nan                     # NaN rows on several ranks and next to a boundary
    bounds = _bounds(n, world, 3)
    got = _cat(_Ranks(xb, bounds, "margins").join(radius))
    _assert_same(got, _reference(xb, radius))
    if radius == -np.inf:
        assert got[0][-1] == (n - 4) * (n - 5)


def _pair(d=512, n_self=900, n_other=300, seed=0):
    import torch
    xs = synth.clip_like(n_self, d, seed=seed + 1)
    xo = synth.clip_like(n_other, d, seed=seed + 2)
    xo[:5] = xs[:5]                                         # exact duplicates on both sides
    me = ivr_b200.IndexFlatIP(d, device=0)
    me.add(xs)
    oth = ivr_b200.IndexFlatIP(d, device=0)
    oth.add(xo)
    return me, oth, oth.rows_f16_tensor(0, n_other), torch


@pytest.mark.parametrize("lower", [0, 1])
@pytest.mark.parametrize("d", [512, 768, 1024])
def test_cross_join_equals_range_search_of_the_other_rows(lower, d):
    """Both sides of the cross join against range search with the other set's stored rows as fp32 queries."""
    me, oth, other, torch = _pair(d)
    first_other, off = (100, 5000) if lower else (9000, 200)
    radius = _radius(np.concatenate([me.reconstruct_n(), oth.reconstruct_n()]), 30)
    ls, ks, lo, ko = me.range_cross_join_keys_tensor(other, first_other, radius, bool(lower), id_offset=off)
    q_self = torch.from_numpy(me.reconstruct_n()).cuda()
    q_oth = torch.from_numpy(oth.reconstruct_n()).cuda()
    Lr, Kr = oth.range_search_keys_tensor(q_self, radius, id_offset=first_other)
    assert torch.equal(ls, Lr) and torch.equal(ks, Kr)
    Lr, Kr = me.range_search_keys_tensor(q_oth, radius, id_offset=off)
    assert torch.equal(lo, Lr) and torch.equal(ko, Kr)
    assert int(ls[-1]) == int(lo[-1]) > 0


def test_cross_join_small_and_empty_other_sets():
    me, oth, other, torch = _pair(768, n_self=1000, n_other=300)
    radius = -np.inf
    for m in (0, 1, 17, 79, 80, 81):                       # npad is 80 at 768 dims
        ls, ks, lo, ko = me.range_cross_join_keys_tensor(other[:m], 2000, radius, False)
        assert ls.numel() == 1001 and lo.numel() == m + 1
        assert int(ls[-1]) == int(lo[-1]) == 1000 * m and ks.numel() == ko.numel() == 1000 * m
        if m:
            D, I = flat_ip.unpack_keys(ks[:m].cpu().numpy().view(np.uint64))
            assert set(I.tolist()) == set(range(2000, 2000 + m))
    empty = ivr_b200.IndexFlatIP(768, device=0)
    ls, ks, lo, ko = empty.range_cross_join_keys_tensor(other, 0, radius, False)
    assert ls.tolist() == [0] and lo.tolist() == [0] * 301 and ks.numel() == ko.numel() == 0


def test_cross_join_capacity_retry_and_multi_launch_split():
    from ivr_b200 import faiss_compat
    me, oth, other, torch = _pair(512, n_self=5000, n_other=700)
    radius = _radius(me.reconstruct_n(), 40)
    want = me.range_cross_join_keys_tensor(other, 0, radius, True, id_offset=700)
    assert int(want[0][-1]) > 64
    orig = faiss_compat._cross_capacity
    faiss_compat._cross_capacity = lambda n, m: 64
    try:
        got = me.range_cross_join_keys_tensor(other, 0, radius, True, id_offset=700)
    finally:
        faiss_compat._cross_capacity = orig
    assert all(torch.equal(a, b) for a, b in zip(got, want))
    os.environ["IVR_JOIN_MAX_UNITS"] = "3"                  # 5000 rows of B = 40 units: 14 launches
    try:
        got = me.range_cross_join_keys_tensor(other, 0, radius, True, id_offset=700)
    finally:
        del os.environ["IVR_JOIN_MAX_UNITS"]
    assert all(torch.equal(a, b) for a, b in zip(got, want))


def test_argument_checks_that_need_an_index():
    import ctypes
    import torch
    me, oth, other, _ = _pair(512, n_self=100, n_other=50)
    L = torch.zeros(200, dtype=torch.int64, device="cuda")
    K = torch.zeros(16, dtype=torch.int64, device="cuda")

    def cross(n_other=50, first=0, cap=16, off=0, idx=me):
        return nat.lib.ivr_index_range_cross_join_keys_device(idx._handle(), other.data_ptr(), n_other, first, 0, 0.5,
                                                              cap, L.data_ptr(), K.data_ptr(), off, None)
    assert cross(cap=1 << 31) == nat.IVR_EUNSUPPORTED and "2^31-1" in nat.last_error()
    assert cross(n_other=(1 << 31) - 100) == nat.IVR_EUNSUPPORTED and "rows" in nat.last_error()
    assert cross(off=(1 << 32) - 99) == nat.IVR_EUNSUPPORTED and "2^32" in nat.last_error()
    assert cross(off=-1) == nat.IVR_EUNSUPPORTED
    assert cross(first=(1 << 32) - 49) == nat.IVR_EUNSUPPORTED and "2^32" in nat.last_error()
    assert cross(first=-1) == nat.IVR_EUNSUPPORTED
    assert cross(off=(1 << 32) - 100, first=(1 << 32) - 50) == nat.IVR_OK
    wide = ivr_b200.IndexFlatIP(4100, device=0)
    assert cross(idx=wide) == nat.IVR_EUNSUPPORTED and "4096" in nat.last_error()
    assert nat.lib.ivr_index_range_self_join_keys_device(me._handle(), 0.5, 16, L.data_ptr(), K.data_ptr(),
                                                         (1 << 32) - 99, None) == nat.IVR_EUNSUPPORTED
    with pytest.raises(nat.NativeError):
        me.rows_f16_tensor(90, 11)
    assert me.dpad == 512 and wide.dpad == 4160
    np.testing.assert_array_equal(me.rows_f16_tensor(7, 3).cpu().numpy()[:, :512], fm.store(me.reconstruct_n(7, 3)))


def test_single_rank_sharded_join_is_the_local_join():
    n, d = 3000, 512
    xb = synth.clip_like(n, d, seed=91)
    sh = ivr_b200.ShardedFlatIP(d, device=0)
    assert sh.world == 1
    sh.add_local(xb, id_offset=777, ntotal_global=n + 777)
    radius = _radius(xb, 20)
    L, D, I = sh.range_self_join(radius)
    assert L.is_cuda and D.is_cuda and I.is_cuda
    lims, Dr, Ir = _reference(xb, radius)
    _assert_same((L.cpu().numpy(), D.cpu().numpy(), I.cpu().numpy() - 777), (lims, Dr, Ir))

