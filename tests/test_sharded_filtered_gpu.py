"""GPU: filtered search across row shards with several RANKS IN ONE PROCESS on one device.

Every rank runs the windowed filtered key calls (``search_keys_tensor`` / ``range_search_keys_tensor`` with
``params``): either as a window of one index holding every row, with an id offset, or as a shard index of its own that
also stores ``MARGIN`` rows of each neighbour, searched under its window with the selector's slice of its stored rows
(what ``ShardedFlatIP`` does).  The exchange is a ``torch.stack`` of the keys; the merge is the CUDA merge kernel.  The
merged D / I must equal ``IndexFlatIP.search`` / ``range_search`` with the same selector on the unsharded index bit for
bit: a row's score depends only on its fp16 values and the query, whichever rank scores it, and the windows report
every selected row exactly once.  Boundaries are not 128-row aligned."""
import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat
from oracle import flat_ip, synth
from test_filtered_search_gpu import SELECTIONS, selector

pytestmark = pytest.mark.gpu
SEL_KERNEL = "search_mma_small_sel_kernel"
BASE = 7000                     # global id of stored row 0 in the window layout
MARGIN = 333                    # rows of each neighbour a shard also stores


def _params(sel):
    return ivr_b200.SearchParameters(sel=sel)


def _index(xb, timing=False):
    idx = ivr_b200.IndexFlatIP(xb.shape[1], device=0)
    idx.set_timing(timing)
    idx.add(xb)
    return idx


class _Ranks:
    """world ranks over the rows of xb, boundaries off: 'windows' = windows of one index (ids + BASE), 'shards' = one
    index per rank holding [off[r] - MARGIN, off[r+1] + MARGIN), searched under the window [off[r], off[r+1])."""

    def __init__(self, xb, off, layout, full=None):
        self.off, self.layout, self.n = off, layout, xb.shape[0]
        if layout == "windows":
            self.idx = [full]
            self.lo = [0] * (len(off) - 1)
        else:
            self.lo = [max(0, int(off[r]) - MARGIN) for r in range(len(off) - 1)]
            hi = [min(self.n, int(off[r + 1]) + MARGIN) for r in range(len(off) - 1)]
            self.idx = [_index(xb[a:b]) for a, b in zip(self.lo, hi)]

    def each(self, sel, call):
        """call(index, params, id_offset) on every rank under its window; the global ids of 'windows' are + BASE."""
        out = []
        for r in range(len(self.off) - 1):
            idx = self.idx[0] if self.layout == "windows" else self.idx[r]
            idx.set_window(int(self.off[r]) - self.lo[r], int(self.off[r + 1] - self.off[r]))
            if self.layout == "windows":
                out.append(call(idx, _params(sel), BASE))
            else:
                out.append(call(idx, _params(sel.shard(self.n, self.lo[r])), self.lo[r]))
            idx.set_window()
        return out

    def shift(self):
        return BASE if self.layout == "windows" else 0


def _merge_topk(parts, k):
    import torch
    from ivr_b200.sharded import _cuda_merge
    D, I = _cuda_merge(0)(torch.stack(parts), k)
    return D.cpu().numpy(), I.cpu().numpy()


def _merge_range(runs):
    import torch
    from ivr_b200.sharded import _cuda_range_merge
    stride = max(int(k.numel()) for _, k in runs)
    keys = torch.zeros((len(runs), stride), dtype=torch.int64, device="cuda")
    for r, (_, k) in enumerate(runs):
        keys[r, :k.numel()] = k
    lims = torch.stack([l for l, _ in runs])
    return [t.cpu().numpy() for t in _cuda_range_merge(keys, lims, int(lims[:, -1].sum()))]


def _radius(xq, xb, mask, kth=40):
    """About kth hits per query among the selected rows (0.0 when nothing is selected)."""
    if not mask.any():
        return 0.0
    s = np.sort(xq @ xb[mask].T, axis=1)
    return float(np.float32(np.median(s[:, -min(kth, s.shape[1])])))


def _check(ranks, full, xb, xq, q, sel, mask, nq, k):
    import torch
    want = full.search_tensor(q[:nq], k, params=_params(sel))
    got = _merge_topk(ranks.each(sel, lambda idx, p, off: idx.search_keys_tensor(q[:nq], k, id_offset=off, params=p)),
                      k)
    D0, I0 = (t.cpu().numpy() for t in want)
    I = np.where(got[1] >= 0, got[1] - ranks.shift(), -1)
    assert np.array_equal(got[0], D0) and np.array_equal(I, I0), (nq, k)
    radius = _radius(xq[:nq], xb, mask)
    lims0, Dr0, Ir0 = full.range_search(xq[:nq], radius, params=_params(sel))
    lims, Dr, Ir = _merge_range(ranks.each(sel, lambda idx, p, off: idx.range_search_keys_tensor(
        q[:nq], radius, id_offset=off, params=p)))
    assert np.array_equal(lims, lims0) and np.array_equal(Dr, Dr0) and np.array_equal(Ir - ranks.shift(), Ir0), nq
    torch.cuda.synchronize()


@pytest.mark.parametrize("layout", ["windows", "shards"])
@pytest.mark.parametrize("d", [512, 768])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_filtered_search_equals_the_unsharded_index(world, d, layout):
    import torch
    from ivr_b200.sharded import partition_rows
    n = 20_011
    off = partition_rows(n, world)
    assert any(int(b) % 128 for b in off[1:-1])
    xb = synth.clip_like(n, d, seed=d + world, n_centres=256)
    for b in off[1:-1]:                                            # equal scores on both sides of every boundary
        xb[b:b + 5] = xb[b - 5:b]
    xq = synth.clip_like(128, d, seed=d + 1, n_centres=256)
    q = torch.from_numpy(xq).cuda()
    full = _index(xb)
    ranks = _Ranks(xb, off, layout, full)
    for name in SELECTIONS:
        sel, mask = selector(name, n, seed=world)
        for nq in (1, 16, 100, 128):
            for k in (1, 100):
                _check(ranks, full, xb, xq, q, sel, mask, nq, k)
        sel.close()


def test_windows_with_seeded_launches():
    """Windows of 100 k rows (781 tiles): the filtered top-k runs its seeded launches inside each window."""
    import torch
    from ivr_b200.sharded import partition_rows
    n, d = 200_003, 512
    xb = synth.clip_like(n, d, seed=5, n_centres=256)
    xq = synth.clip_like(16, d, seed=6, n_centres=256)
    full = _index(xb)
    ranks = _Ranks(xb, partition_rows(n, 2), "windows", full)
    for name in ("all", "rand50", "video"):
        sel, mask = selector(name, n, seed=7)
        _check(ranks, full, xb, xq, torch.from_numpy(xq).cuda(), sel, mask, 16, 100)
        sel.close()


def test_windows_never_report_a_row_outside_them():
    """Overlapping windows over every row selected: the keys of a window name exactly its rows, also in its partial
    first and last tiles (k and a radius of -inf that return every row of the window)."""
    import torch
    n, d = 5000, 512
    xb = synth.clip_like(n, d, seed=9)
    q = torch.from_numpy(synth.clip_like(16, d, seed=10)).cuda()
    idx = _index(xb)
    sel = ivr_b200.IDSelectorRange(0, n)
    for first, count in ((0, 1), (1, 130), (127, 2), (130, 300), (200, 56), (1000, 1000), (4999, 1), (3, n - 4),
                         (128, 128), (0, n)):
        idx.set_window(first, count)
        k = min(count + 7, nat.IVR_MAX_K)
        keys = idx.search_keys_tensor(q, k, id_offset=11, params=_params(sel))
        _, I = flat_ip.unpack_keys(keys.cpu().numpy().view(np.uint64))
        if count < k:                                              # every row of the window, then padding
            assert np.all(I[:, count:] == -1), (first, count)
            assert all(sorted(r[:count].tolist()) == list(range(first + 11, first + count + 11)) for r in I)
        else:
            assert np.all((I >= first + 11) & (I < first + count + 11)), (first, count)
        lims, keys = idx.range_search_keys_tensor(q, -np.inf, id_offset=11, params=_params(sel))
        _, I = flat_ip.unpack_keys(keys.cpu().numpy().view(np.uint64))
        assert lims.cpu().numpy().tolist() == [count * i for i in range(17)], (first, count)
        assert np.array_equal(np.sort(I.reshape(16, count), axis=1),
                              np.broadcast_to(np.arange(first + 11, first + count + 11), (16, count)))
    idx.set_window(4000, 1001)                                     # past ntotal
    with pytest.raises(nat.NativeError) as e:
        idx.search_keys_tensor(q, 10, params=_params(sel))
    assert e.value.code == nat.IVR_EINVAL and "window" in str(e.value)
    with pytest.raises(nat.NativeError) as e:
        idx.range_search_keys_tensor(q, 0.5, params=_params(sel))
    assert e.value.code == nat.IVR_EINVAL and "window" in str(e.value)


@pytest.mark.parametrize("name", SELECTIONS)
def test_without_a_window_the_keys_are_the_filtered_search(name):
    """Window cleared: the key calls unpack to search_selected / range_search_selected bit for bit."""
    import torch
    n, d, off = 30_000, 768, 123_456
    xb = synth.clip_like(n, d, seed=12, n_centres=256)
    xq = synth.clip_like(130, d, seed=13, n_centres=256)
    q = torch.from_numpy(xq).cuda()
    idx = _index(xb, timing=True)
    sel, mask = selector(name, n, seed=14)
    for nq in (1, 16, 130):
        D, I = (t.cpu().numpy() for t in idx.search_tensor(q[:nq], 100, id_offset=off, params=_params(sel)))
        keys = idx.search_keys_tensor(q[:nq], 100, id_offset=off, params=_params(sel))
        t = idx.last_timing()
        if mask.any():
            assert t["kernel"] == SEL_KERNEL and t["score_launches"] >= 1
        else:
            assert t["path"] == "empty" and t["score_launches"] == 0
        Dk, Ik = flat_ip.unpack_keys(keys.cpu().numpy().view(np.uint64))
        assert np.array_equal(Dk, D) and np.array_equal(Ik, I)
    radius = _radius(xq, xb, mask)
    lims, Dr, Ir = (t.cpu().numpy() for t in idx.range_search_tensor(q, radius, id_offset=off, params=_params(sel)))
    lk, keys = idx.range_search_keys_tensor(q, radius, id_offset=off, params=_params(sel))
    Dk, Ik = flat_ip.unpack_keys(keys.cpu().numpy().view(np.uint64))
    assert np.array_equal(lk.cpu().numpy(), lims) and np.array_equal(Dk, Dr) and np.array_equal(Ik, Ir)
    sel.close()


def test_a_window_without_selected_rows_launches_nothing():
    import torch
    n, d = 4000, 512
    xb = synth.clip_like(n, d, seed=15)
    q = torch.from_numpy(synth.clip_like(16, d, seed=16)).cuda()
    idx = _index(xb, timing=True)
    # selected rows 1000..1009 share row tile 7 (896..1023) with the window's first rows, 1010..1023
    sel = ivr_b200.IDSelectorRange(1000, 1010)
    for first, count in ((1010, 300), (0, 1000), (1500, 2500), (700, 300)):
        idx.set_window(first, count)
        keys = idx.search_keys_tensor(q, 10, params=_params(sel))
        t = idx.last_timing()
        assert t["path"] == "empty" and t["score_launches"] == 0, (first, count, t)
        assert not keys.any()
        lims, keys = idx.range_search_keys_tensor(q, -np.inf, params=_params(sel))
        assert not lims.any() and keys.numel() == 0
    idx.set_window(1005, 300)                                      # five selected rows inside: the filtered kernel
    keys = idx.search_keys_tensor(q, 10, params=_params(sel))
    assert idx.last_timing()["kernel"] == SEL_KERNEL
    _, I = flat_ip.unpack_keys(keys.cpu().numpy().view(np.uint64))
    assert all(sorted(r[:5].tolist()) == list(range(1005, 1010)) for r in I) and np.all(I[:, 5:] == -1)


def test_single_rank_sharded_filtered_search_is_the_local_search_shifted():
    import torch
    n, d, first = 9000, 512, 40_000
    xb = synth.clip_like(n, d, seed=17)
    xq = synth.clip_like(12, d, seed=18)
    q = torch.from_numpy(xq).cuda()
    sh = ivr_b200.ShardedFlatIP(d, device=0)
    assert sh.world == 1
    sh.add_local(xb, id_offset=first, ntotal_global=first + n + 500)
    idx = _index(xb)
    sel = ivr_b200.IDSelectorRange(first - 100, first + 4321)
    local = ivr_b200.IDSelectorRange(0, 4321)
    D, I = sh.search(q, 100, params=_params(sel))
    Dl, Il = idx.search(xq, 100, params=_params(local))
    np.testing.assert_array_equal(D.cpu().numpy(), Dl)
    np.testing.assert_array_equal(I.cpu().numpy(), np.where(Il >= 0, Il + first, -1))
    radius = _radius(xq, xb, np.arange(n) < 4321)
    L, D, I = sh.range_search(q, radius, params=_params(sel))
    Ll, Dl, Il = idx.range_search(xq, radius, params=_params(local))
    np.testing.assert_array_equal(L.cpu().numpy(), Ll)
    np.testing.assert_array_equal(D.cpu().numpy(), Dl)
    np.testing.assert_array_equal(I.cpu().numpy(), Il + first)
