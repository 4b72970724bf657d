"""CPU: filtered search (``params=SearchParameters(sel=...)``) across row shards at world size 2 over gloo.

The local index is a NumPy stand-in that speaks the extended protocol of faiss_compat.IndexFlatIP: a search window
(``set_window``), and ``search_keys_tensor`` / ``range_search_keys_tensor`` with ``params`` whose selector selects
STORED rows and is honoured inside the window only.  The rows hold small integers, so every inner product is exact in
float32 whatever the summation order, and the sharded results must equal a direct scan of the selected global ids
exactly, ties (lower id first) included.  The CUDA kernels behind the real calls are covered by
tests/test_sharded_filtered_gpu.py."""
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

NEG = np.float32(-3.402823466e+38)


class _NumpyLocal:
    """The local index protocol, on the host: stored rows, a search window, selectors of stored rows."""

    def __init__(self, d):
        self.d, self.xb, self.first, self.count = d, np.zeros((0, d), np.float32), 0, -1

    @property
    def ntotal(self):
        return self.xb.shape[0]

    def add(self, x):
        self.xb = np.concatenate([self.xb, np.asarray(x, np.float32)])

    def set_window(self, first=0, count=-1):
        assert count < 0 or 0 <= first and first + count <= self.ntotal
        self.first, self.count = (first, count) if count >= 0 else (0, -1)

    def _ids(self, params):
        """The stored rows a search reports: the window's, and of them the selected ones."""
        a, b = (0, self.ntotal) if self.count < 0 else (self.first, self.first + self.count)
        ids = np.arange(a, b)
        if params is not None and params.sel is not None:
            ids = ids[params.sel._mask(self.ntotal)[a:b]]
        return ids

    def search_keys_tensor(self, q, k, id_offset=0, out=None, params=None):
        ids = self._ids(params)
        D, I = _topk(q.numpy() @ self.xb[ids].T, ids + id_offset, k)
        keys = torch.from_numpy(flat_ip.pack_keys(D, I).view(np.int64))
        if out is None:
            return keys
        out.copy_(keys)
        return out

    def search_tensor(self, q, k, id_offset=0, params=None):
        assert self.count < 0, "search_tensor is the world-size-1 call: no window"
        D, I = flat_ip.unpack_keys(self.search_keys_tensor(q, k, id_offset, params=params).numpy().view(np.uint64))
        return torch.from_numpy(D), torch.from_numpy(I)

    def range_search_keys_tensor(self, q, radius, id_offset=0, params=None):
        ids = self._ids(params)
        lims, D, I = _range(q.numpy() @ self.xb[ids].T, ids + id_offset, radius)
        return torch.from_numpy(lims), torch.from_numpy(flat_ip.pack_keys(D, I).view(np.int64))

    def range_search_tensor(self, q, radius, id_offset=0, params=None):
        lims, keys = self.range_search_keys_tensor(q, radius, id_offset, params=params)
        D, I = flat_ip.unpack_keys(keys.numpy().view(np.uint64))
        return lims, torch.from_numpy(D), torch.from_numpy(I)


def _topk(s, ids, k):
    """k best columns of every row of s (score descending, then lower id), padded with -FLT_MAX / -1."""
    nq = s.shape[0]
    D, I = np.full((nq, k), NEG, np.float32), np.full((nq, k), -1, np.int64)
    for q in range(nq):
        order = np.lexsort((ids, -s[q].astype(np.float64)))[:k]
        D[q, :order.size], I[q, :order.size] = s[q, order], ids[order]
    return D, I


def _range(s, ids, radius):
    lims, D, I = [0], [], []
    for q in range(s.shape[0]):
        hit = np.nonzero(s[q] > np.float32(radius))[0]
        order = hit[np.lexsort((ids[hit], -s[q, hit].astype(np.float64)))]
        D.extend(s[q, order])
        I.extend(ids[order])
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D, np.float32), np.array(I, np.int64)


def _scan_topk(xb, xq, sel, k):
    ids = np.nonzero(sel._mask(xb.shape[0]))[0]
    return _topk(xq @ xb[ids].T, ids, k)


def _scan_range(xb, xq, sel, radius):
    ids = np.nonzero(sel._mask(xb.shape[0]))[0]
    return _range(xq @ xb[ids].T, ids, radius)


def _merge(keys_parts, k):
    D_all, I_all = zip(*(flat_ip.unpack_keys(p) for p in keys_parts.numpy().view(np.uint64)))
    D, I = flat_ip.merge_shard_results(list(D_all), list(I_all), k)
    return torch.from_numpy(D), torch.from_numpy(I)


def _range_merge(keys_parts, lims_parts, total):
    lims, D, I = merge_range_parts(lims_parts.numpy(), keys_parts.numpy())
    assert lims[-1] == total
    return torch.from_numpy(lims), torch.from_numpy(D), torch.from_numpy(I)


def _sharded(d):
    from ivr_b200.sharded import ShardedFlatIP
    return ShardedFlatIP(d, local_index=_NumpyLocal(d), merge=_merge, range_merge=_range_merge)


def _rows(n, d, seed, copy_at=()):
    """Small-integer rows (exact float32 inner products); the 8 rows before every position in copy_at are repeated
    right after it, so equal scores sit on both sides of a shard boundary."""
    x = np.random.default_rng(seed).integers(-3, 4, (n, d)).astype(np.float32)
    for b in copy_at:
        x[b:b + 8] = x[b - 8:b]
    return x


def _selectors(n, cut):
    """Named selectors of global ids; most hold runs that cross the shard boundary `cut`."""
    from ivr_b200 import faiss_compat as fc
    rng = np.random.default_rng(n)
    m = np.zeros(n, bool)
    m[cut - 37:cut + 45] = True
    m[5:9] = True
    return {"across": fc.IDSelectorRange(cut - 100, cut + 77),
            "bitmap": fc.IDSelectorBitmap(np.packbits(m, bitorder="little")),
            "rand": fc.IDSelectorBatch(rng.choice(n, n // 20, replace=False)),
            "not": fc.IDSelectorNot(fc.IDSelectorRange(0, cut - 3)),
            "one": fc.IDSelectorBatch([cut]),
            "empty": fc.IDSelectorBatch([]),
            "beyond": fc.IDSelectorRange(n - 10, n + 1000)}


def _same_topk(got, want):
    return np.array_equal(got[0].numpy(), want[0]) and np.array_equal(got[1].numpy(), want[1])


def _same_range(got, want):
    return all(np.array_equal(g.numpy(), w) for g, w in zip(got, want))


def _no_duplicates(I):
    """No id twice in a query's top-k row."""
    return all(len(set(r[r >= 0].tolist())) == int((r >= 0).sum()) for r in np.asarray(I))


def _no_duplicate_hits(lims, I):
    """No id twice among a query's range hits."""
    return all(np.unique(I[a:b]).size == b - a for a, b in zip(lims[:-1], lims[1:]))


def _init(rank, world, port):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _spawn(fn, timeout=180.0):
    """Runs fn(rank, world, port, out) on 2 processes; fails instead of hanging when a rank is left waiting."""
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = mp.Manager().dict()
    ctx = mp.spawn(fn, args=(2, port, out), nprocs=2, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=max(0.1, deadline - time.monotonic())):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail(f"a rank was still waiting after {timeout:.0f} s")
    return dict(out)


def _static_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        from ivr_b200 import faiss_compat as fc
        from ivr_b200.sharded import partition_rows
        n, d = 1003, 16
        res = {}
        for weights in (None, [1.0, 3.0]):
            off = partition_rows(n, world, weights)
            xb = _rows(n, d, seed=3, copy_at=[int(off[1])])
            xq = torch.from_numpy(_rows(6, d, seed=4))
            sh = _sharded(d)
            sh.add_global(xb, weights=weights)
            for name, sel in _selectors(n, int(off[1])).items():
                p = fc.SearchParameters(sel=sel)
                for k in (1, 10, 200):
                    got = sh.search(xq, k, params=p)
                    res[(str(weights), name, "topk", k)] = (_same_topk(got, _scan_topk(xb, xq.numpy(), sel, k))
                                                            and _no_duplicates(got[1].numpy()))
                s = xq.numpy() @ xb.T
                for radius in (-np.inf, float(np.median(np.sort(s, 1)[:, -60])), np.inf):
                    got = sh.range_search(xq, radius, params=p)
                    res[(str(weights), name, "range", radius)] = (
                        _same_range(got, _scan_range(xb, xq.numpy(), sel, radius))
                        and _no_duplicate_hits(got[0].numpy(), got[2].numpy()))
            # params=None and a SearchParameters without a selector are the unfiltered search
            full = _topk(xq.numpy() @ xb.T, np.arange(n), 10)
            res[(str(weights), "none")] = (_same_topk(sh.search(xq, 10), full)
                                           and _same_topk(sh.search(xq, 10, params=fc.SearchParameters()), full))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_filtered_search_world2_equals_a_scan_of_the_selected_ids():
    out = _spawn(_static_worker)
    assert out[0] == out[1]
    bad = [key for key, ok in out[0].items() if not ok]
    assert not bad and len(out[0]) == 2 * (7 * 6 + 1), bad


class _ScriptedTimer:
    """Scoring times for the controller: rank 0's GPU is 'slower' per row than rank 1's."""

    def __init__(self, index, ms_per_row):
        self.index, self.ms_per_row = index, ms_per_row

    def start(self, i):
        pass

    def stop(self, i):
        pass

    def mean_ms(self, lo, hi):
        b = self.index._bounds
        return float(b[self.index.rank + 1] - b[self.index.rank]) * self.ms_per_row


def _elastic_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        from ivr_b200 import faiss_compat as fc
        from ivr_b200.sharded import partition_rows
        n, d, k, margin = 4001, 16, 20, 700
        nominal = partition_rows(n, world)
        cut = int(nominal[1])
        # copies of the rows at every boundary the controller will use: equal scores on both ranks
        xb = _rows(n, d, seed=41, copy_at=[cut, cut - margin, cut - 1024])
        sh = _sharded(d)
        sh.add_global(xb, margin=margin)
        sh.enable_elastic(nominal, margin, period=4, gain=1.0,
                          timer=_ScriptedTimer(sh, 0.003 if rank == 0 else 0.001))
        # selected runs across every boundary the controller can reach: the whole margin band on both sides
        sels = {"band": fc.IDSelectorRange(cut - margin - 40, cut + margin + 40),
                "rand": fc.IDSelectorBatch(np.random.default_rng(5).choice(n, 300, replace=False)),
                "edges": fc.IDSelectorBitmap(np.packbits(np.isin(np.arange(n) % 1024, [0, 1, 1023]),
                                                         bitorder="little"))}
        ok, untouched, windows = True, True, set()
        for s_ in range(14):
            xq = torch.from_numpy(_rows(5, d, seed=300 + s_))
            sh.search(xq, k)                                       # a timed search: the controller may step
            windows.add(tuple(int(v) for v in sh._bounds))
            before = (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
            for name, sel in sels.items():
                p = fc.SearchParameters(sel=sel)
                got = sh.search(xq, k, params=p)
                ok = ok and _same_topk(got, _scan_topk(xb, xq.numpy(), sel, k)) and _no_duplicates(got[1].numpy())
                pend = sh.search_async(xq, k, params=p)
                ok = ok and _same_topk(pend.result(), _scan_topk(xb, xq.numpy(), sel, k))
                radius = float(np.median(np.sort(xq.numpy() @ xb.T, 1)[:, -80]))
                got = sh.range_search(xq, radius, params=p)
                ok = ok and _same_range(got, _scan_range(xb, xq.numpy(), sel, radius))
                ok = ok and _no_duplicate_hits(got[0].numpy(), got[2].numpy())
            untouched = untouched and before == (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
        out[rank] = (ok, untouched, [(i, list(map(int, rows))) for i, _, rows in sh.balance_log], len(windows))
    finally:
        dist.destroy_process_group()


def test_filtered_search_world2_on_moving_elastic_boundaries():
    """Each rank stores 700 rows of its neighbour; the scripted timer's controller steps (searches 4, 8 and 12) move
    the boundary to the edge of the margin.  Filtered searches before and after equal the scan, report no row twice,
    and are not timed searches: the search counter, balance_log and the boundaries are exactly those of the
    unfiltered searches alone."""
    out = _spawn(_elastic_worker)
    for r in (0, 1):
        ok, untouched, log, n_windows = out[r]
        assert ok and untouched, out[r]
        assert [i for i, _ in log] == [4, 8, 12] and log[-1][1] == [2000 - 700, 2001 + 700]
        assert n_windows == 2                                    # nominal, then clipped
    assert out[0][2] == out[1][2]


def _error_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        from ivr_b200 import faiss_compat as fc
        n, d = 601, 16
        xb = _rows(n, d, seed=51)
        xq = torch.from_numpy(_rows(4, d, seed=52))
        sh = _sharded(d)
        sh.add_global(xb)
        res = {}
        try:                                                       # another selector on rank 1: both raise
            sh.range_search(xq, 0.5, params=fc.SearchParameters(sel=fc.IDSelectorRange(0, 300 + rank)))
            res["selector"] = "no error"
        except ValueError as e:
            res["selector"] = str(e)
        for what, call in (("type", lambda: sh.search(xq, 5, params=fc.SearchParameters(sel=[1, 2, 3]))),
                           ("k", lambda: sh.search(xq, 0, params=fc.SearchParameters(sel=fc.IDSelectorBatch([1])))),
                           ("dim", lambda: sh.search(xq[:, :8], 5,
                                                     params=fc.SearchParameters(sel=fc.IDSelectorBatch([1])))),
                           ("nan", lambda: sh.range_search(xq, float("nan"),
                                                           params=fc.SearchParameters(sel=fc.IDSelectorBatch([1]))))):
            try:
                call()
                res[what] = "no error"
            except (TypeError, ValueError) as e:                   # raised before any collective, on every rank
                res[what] = type(e).__name__
        sel = fc.IDSelectorRange(100, 500)
        got = sh.range_search(xq, 0.5, params=fc.SearchParameters(sel=sel))   # the group is still in step
        res["after"] = _same_range(got, _scan_range(xb, xq.numpy(), sel, 0.5))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_filtered_search_world2_errors_are_raised_on_every_rank():
    out = _spawn(_error_worker)
    assert out[0] == out[1], out
    assert "rank 1" in out[0]["selector"] and "selector of 301 ids" in out[0]["selector"], out[0]
    assert (out[0]["type"], out[0]["k"], out[0]["dim"], out[0]["nan"]) == ("TypeError", "ValueError", "ValueError",
                                                                           "ValueError")
    assert out[0]["after"]


def test_single_rank_filtered_search_takes_the_slice_of_its_rows():
    """world 1 (no process group): add_local with an id offset searches the selector's slice of its rows."""
    from ivr_b200 import faiss_compat as fc
    from ivr_b200.sharded import ShardedFlatIP
    n, d, first = 700, 16, 5000
    xb = _rows(n, d, seed=61)
    xq = torch.from_numpy(_rows(3, d, seed=62))
    sh = ShardedFlatIP(d, local_index=_NumpyLocal(d), merge=_merge, range_merge=_range_merge)
    assert sh.world == 1
    sh.add_local(xb, id_offset=first, ntotal_global=first + n + 100)
    sel = fc.IDSelectorRange(first - 50, first + 321)
    D, I = sh.search(xq, 400, params=fc.SearchParameters(sel=sel))
    Dw, Iw = _topk(xq.numpy() @ xb[:321].T, np.arange(321) + first, 400)
    assert np.array_equal(D.numpy(), Dw) and np.array_equal(I.numpy(), Iw)
    got = sh.range_search(xq, 2.0, params=fc.SearchParameters(sel=sel))
    assert _same_range(got, _range(xq.numpy() @ xb[:321].T, np.arange(321) + first, 2.0))
