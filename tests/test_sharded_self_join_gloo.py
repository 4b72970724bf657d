"""CPU: the range self-join across row shards (``ShardedFlatIP.range_self_join``) at world sizes 2, 3 and 4 over gloo.

The local index is a NumPy stand-in that speaks the join protocol of faiss_compat.IndexFlatIP: a search window
(``set_window``), ``dpad``, ``rows_f16_tensor``, ``range_self_join_tensor``, ``range_self_join_keys_tensor`` and
``range_cross_join_keys_tensor``.  The rows hold small integers, so every inner product is exact in float16 and
float32 whatever the summation order, and the sharded join must equal a direct scan of all pairs exactly, ties
(lower id first) included.  The CUDA kernels behind the real calls are covered by tests/test_sharded_self_join_gpu.py.
"""
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import flat_ip
from range_merge_ref import merge_range_parts


class _NumpyLocal:
    """The local join protocol on the host.  ``max_hits``: a cross join with more hits raises OverflowError (as the
    real call does above 2^31-1); ``fail``: every cross join raises."""

    def __init__(self, d, max_hits=None, fail=False):
        self.d, self.xb, self.first, self.count = d, np.zeros((0, d), np.float32), 0, -1
        self.max_hits, self.fail, self.windows = max_hits, fail, []

    @property
    def ntotal(self):
        return self.xb.shape[0]

    @property
    def dpad(self):
        return self.d

    def add(self, x):
        self.xb = np.concatenate([self.xb, np.asarray(x, np.float32)])

    def set_window(self, first=0, count=-1):
        assert count < 0 or 0 <= first and first + count <= self.ntotal
        self.first, self.count = (first, count) if count >= 0 else (0, -1)
        self.windows.append((self.first, self.count))

    def _win(self):
        return (0, self.ntotal) if self.count < 0 else (self.first, self.first + self.count)

    def rows_f16_tensor(self, first, n):
        assert 0 <= first and first + n <= self.ntotal
        return torch.from_numpy(self.xb[first:first + n].astype(np.float16))

    def range_self_join_keys_tensor(self, radius, id_offset=0):
        a, b = self._win()
        x = self.xb[a:b]
        s = x @ x.T
        np.fill_diagonal(s, -np.inf)
        lims, D, I = _range(s, np.arange(a, b) + id_offset, radius)
        return torch.from_numpy(lims), torch.from_numpy(flat_ip.pack_keys(D, I).view(np.int64))

    def range_self_join_tensor(self, radius):
        lims, keys = self.range_self_join_keys_tensor(radius)
        D, I = flat_ip.unpack_keys(keys.numpy().view(np.uint64))
        return lims, torch.from_numpy(D), torch.from_numpy(I)

    def range_cross_join_keys_tensor(self, other_rows, other_first_id, radius, other_is_lower, id_offset=0):
        if self.fail:
            raise RuntimeError("injected failure")
        a, b = self._win()
        ids = np.arange(a, b) + id_offset
        oid = np.arange(other_rows.shape[0]) + other_first_id
        assert bool(other_is_lower) == (oid.size > 0 and ids.size > 0 and oid[0] < ids[0]) or not oid.size \
            or not ids.size
        s = self.xb[a:b] @ other_rows.numpy().astype(np.float32).T
        ls, Ds, Is = _range(s, oid, radius)
        lo, Do, Io = _range(s.T, ids, radius)
        if self.max_hits is not None and ls[-1] + lo[-1] > self.max_hits:
            raise OverflowError("too many hits")
        pk = lambda D, I: torch.from_numpy(flat_ip.pack_keys(D, I).view(np.int64))
        return torch.from_numpy(ls), pk(Ds, Is), torch.from_numpy(lo), pk(Do, Io)


def _range(s, ids, radius):
    lims, D, I = [0], [], []
    for q in range(s.shape[0]):
        hit = np.nonzero(s[q] > np.float32(radius))[0]
        order = hit[np.lexsort((ids[hit], -s[q, hit].astype(np.float64)))]
        D.extend(s[q, order])
        I.extend(ids[order])
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D, np.float32), np.array(I, np.int64)


def _scan(xb, radius):
    """The join by a direct scan of all pairs of the global rows."""
    s = xb @ xb.T
    np.fill_diagonal(s, -np.inf)
    return _range(s, np.arange(xb.shape[0]), radius)


def _rows_of(scan, lo, hi):
    lims, D, I = scan
    return lims[lo:hi + 1] - lims[lo], D[lims[lo]:lims[hi]], I[lims[lo]:lims[hi]]


def _range_merge(keys_parts, lims_parts, total):
    lims, D, I = merge_range_parts(lims_parts.numpy(), keys_parts.numpy())
    assert lims[-1] == total
    return torch.from_numpy(lims), torch.from_numpy(D), torch.from_numpy(I)


def _sharded(d, **kw):
    from ivr_b200.sharded import ShardedFlatIP
    return ShardedFlatIP(d, local_index=_NumpyLocal(d, **kw), merge=lambda *a: None, range_merge=_range_merge)


def _rows(n, d, seed, copy_at=()):
    """Small-integer rows (exact products); the 6 rows before every position in copy_at are repeated right after it,
    so equal scores and exact ties sit on both sides of a shard boundary."""
    x = np.random.default_rng(seed).integers(-3, 4, (n, d)).astype(np.float32)
    for b in copy_at:
        x[b:b + 6] = x[b - 6:b]
    return x


def _same(got, want):
    return all(np.array_equal(g.numpy(), w) for g, w in zip(got, want))


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _spawn(fn, world, timeout=180.0):
    """Runs fn(rank, world, port, out) on `world` processes; fails instead of hanging when a rank is left waiting."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = mp.Manager().dict()
    ctx = mp.spawn(fn, args=(world, port, out), nprocs=world, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=max(0.1, deadline - time.monotonic())):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail(f"a rank was still waiting after {timeout:.0f} s")
    return dict(out)


def _radii(xb):
    s = xb @ xb.T
    np.fill_diagonal(s, -np.inf)
    srt = np.sort(s, axis=1)
    return [-np.inf, float(np.median(srt[:, -5])), float(np.median(srt[:, -40])), -2.0, np.inf]


def _static_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        from ivr_b200.sharded import partition_rows
        n, d = 211, 16
        res = {}
        for weights in (None, list(range(1, world + 1))):
            off = partition_rows(n, world, weights)
            xb = _rows(n, d, seed=7, copy_at=[int(b) for b in off[1:-1] if b >= 6])
            sh = _sharded(d)
            sh.add_global(xb, weights=weights)
            for radius in _radii(xb):
                want = _scan(xb, radius)
                got = sh.range_self_join(radius)
                res[(str(weights), radius, "local")] = _same(got, _rows_of(want, int(off[rank]), int(off[rank + 1])))
                res[(str(weights), radius, "gather")] = _same(sh.range_self_join(radius, gather=True), want)
            res[(str(weights), "window")] = sh.local.count < 0           # a static shard is left without a window
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_self_join_equals_a_direct_scan(world):
    out = _spawn(_static_worker, world)
    assert all(out[r] == out[0] for r in range(world))
    bad = [key for key, ok in out[0].items() if not ok]
    assert not bad and len(out[0]) == 2 * (2 * 5 + 1), bad


def _elastic_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        from ivr_b200.sharded import partition_rows
        n, d, margin = 300, 16, 40
        nominal = partition_rows(n, world)
        moved = nominal.copy()
        moved[1:-1] += np.array([(-1) ** r * (13 + 7 * r) for r in range(world - 1)])
        xb = _rows(n, d, seed=11, copy_at=[int(b) for b in moved[1:-1]] + [int(b) for b in nominal[1:-1]])
        sh = _sharded(d, max_hits=400)                  # small cross calls: the other rows are split in halves
        sh.add_global(xb, margin=margin)
        ok = True
        for bounds in (nominal, moved):
            sh._bounds = bounds.copy()
            before = (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
            for radius in _radii(xb)[1:4]:
                want = _scan(xb, radius)
                got = sh.range_self_join(radius)
                ok = ok and _same(got, _rows_of(want, int(bounds[rank]), int(bounds[rank + 1])))
                ok = ok and _same(sh.range_self_join(radius, gather=True), want)
            lo = int(bounds[rank]) - sh.id_offset
            ok = ok and sh.local.windows[-1] == (lo, int(bounds[rank + 1] - bounds[rank]))   # restored
            ok = ok and before == (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
        out[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_self_join_on_elastic_margins_and_moved_boundaries(world):
    """Each rank stores 40 rows of either neighbour; the join follows the current boundaries (nominal, then moved off
    the nominal partition and off any alignment), restores the window of the current boundaries and leaves the
    elastic controller alone.  Cross calls holding more than 400 hits raise OverflowError and are split."""
    out = _spawn(_elastic_worker, world)
    assert all(out[r] for r in range(world)), out


def _error_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        n, d = 120, 16
        xb = _rows(n, d, seed=21)
        res = {}
        sh = _sharded(d)
        sh.add_global(xb)
        try:                                            # another radius on the last rank: every rank raises
            sh.range_self_join(1.0 if rank < world - 1 else 2.0)
            res["radius"] = "no error"
        except ValueError as e:
            res["radius"] = str(e)
        try:
            sh.range_self_join(float("nan"))            # before any collective, on every rank
            res["nan"] = "no error"
        except ValueError as e:
            res["nan"] = type(e).__name__
        bad = _sharded(d, fail=(rank == 1))             # a local failure on rank 1 only
        bad.add_global(xb)
        try:
            bad.range_self_join(1.0)
            res["fail"] = "no error"
        except RuntimeError as e:
            res["fail"] = str(e)
        def merge_fails(keys_parts, lims_parts, total):
            raise RuntimeError("injected merge failure")
        from ivr_b200.sharded import ShardedFlatIP
        unmerged = ShardedFlatIP(d, local_index=_NumpyLocal(d), merge=lambda *a: None,
                                 range_merge=merge_fails if rank == 1 else _range_merge)
        unmerged.add_global(xb)
        for gather in (False, True):                    # the merge fails on rank 1 only: nobody waits in the gather
            try:
                unmerged.range_self_join(1.0, gather=gather)
                res[("merge", gather)] = "no error"
            except RuntimeError as e:
                res[("merge", gather)] = str(e)
        res["after"] = _same(sh.range_self_join(1.0, gather=True), _scan(xb, 1.0))   # the group is still in step
        out[rank] = res
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_self_join_errors_are_raised_on_every_rank(world):
    out = _spawn(_error_worker, world)
    assert all(out[r] == out[0] for r in range(world)), out
    assert f"rank {world - 1} was called with radius=2.0" in out[0]["radius"], out[0]
    assert out[0]["nan"] == "ValueError"
    assert "failed on rank 1" in out[0]["fail"], out[0]
    assert all("rank 1 could not merge its runs" in out[0][("merge", g)] for g in (False, True)), out[0]
    assert out[0]["after"]


def test_single_rank_self_join_is_the_local_join_with_global_ids():
    from ivr_b200.sharded import ShardedFlatIP
    n, d, first = 90, 16, 5000
    xb = _rows(n, d, seed=31)
    sh = ShardedFlatIP(d, local_index=_NumpyLocal(d), merge=lambda *a: None, range_merge=_range_merge)
    assert sh.world == 1
    sh.add_local(xb, id_offset=first, ntotal_global=first + n)
    lims, D, I = _scan(xb, 3.0)
    assert _same(sh.range_self_join(3.0), (lims, D, I + first))


def test_too_many_ranks_for_one_merge_are_refused_before_any_collective():
    """64 ranks give each rank 65 runs (its window's join, then two per round): more than one merge takes.  The check
    depends on the world size alone, so every rank refuses before the first collective."""
    from ivr_b200.sharded import ShardedFlatIP
    sh = ShardedFlatIP(16, local_index=_NumpyLocal(16), merge=lambda *a: None, range_merge=_range_merge)
    sh.add_local(_rows(10, 16, seed=1), id_offset=0, ntotal_global=10)
    sh.world = 64                                       # no process group: a collective here would fail, not wait
    with pytest.raises(ValueError, match="65 runs"):
        sh.range_self_join(1.0)
    sh.world = 63
    with pytest.raises(Exception) as e:                 # 63 passes the check and reaches the first collective
        sh.range_self_join(1.0)
    assert "runs" not in str(e.value)
