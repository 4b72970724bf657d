"""CPU: range search across row shards.  The host restatement of the merge (tests/range_merge_ref.py), the argument
checks of the two new C entry points (no device needed), and ShardedFlatIP.range_search at world size 2 over gloo
with a stand-in local index and merge built on the oracle -- the CUDA kernels behind them are covered by
tests/test_sharded_range_gpu.py."""
import ctypes
import os
import socket
import time

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ivr_b200 import _native as nat
from oracle import flat_ip, synth
from oracle import range_search as orr
from range_merge_ref import merge_range_parts


# ---------------------------------------------------------------------------
# merge_range_parts
# ---------------------------------------------------------------------------
def _parts(xb, xq, radius, off):
    """Per-shard oracle range results as (lims, packed keys with global ids)."""
    lims_parts, keys_parts = [], []
    for r in range(len(off) - 1):
        lims, D, I = orr.range_search(xb[off[r]:off[r + 1]], xq, radius)
        lims_parts.append(lims)
        keys_parts.append(flat_ip.pack_keys(D, I + off[r]))
    return lims_parts, keys_parts


def _scan(xb, xq, radius):
    s = xq @ xb.T
    lims, D, I = [0], [], []
    for q in range(xq.shape[0]):
        ids = np.nonzero(s[q] > np.float32(radius))[0]
        order = sorted(ids, key=lambda i: (-s[q, i], i))
        D.extend(s[q, order])
        I.extend(order)
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D, np.float32), np.array(I, np.int64)


def test_merge_range_parts_matches_a_direct_scan():
    rng = np.random.default_rng(3)
    xb = rng.standard_normal((900, 16)).astype(np.float32)
    xb[600:620] = xb[100:120]                                      # equal scores on two parts
    xq = np.concatenate([rng.standard_normal((4, 16)), -xb[:1] * 100]).astype(np.float32)
    for off in ([0, 300, 600, 900], [0, 0, 450, 900], [0, 899, 900]):     # an empty part, a one-row part
        for radius in (-np.inf, 0.0, 3.0, 8.0, np.inf):
            lims_p, keys_p = _parts(xb, xq, radius, off)
            lims, D, I = merge_range_parts(lims_p, keys_p)
            want = _scan(xb, xq, radius)
            np.testing.assert_array_equal(lims, want[0])
            np.testing.assert_array_equal(I, want[2])
            np.testing.assert_allclose(D, want[1], rtol=1e-6, atol=1e-5)
    lims_p, keys_p = _parts(xb, xq, 3.0, [0, 300, 600, 900])
    lims, D, I = merge_range_parts(lims_p, keys_p)
    for q in range(xq.shape[0]):                                   # the copies: lower id first
        i = I[lims[q]:lims[q + 1]]
        for a in range(100, 120):
            if a in i:
                assert np.nonzero(i == a)[0][0] + 1 == np.nonzero(i == a + 500)[0][0]
    lims, D, I = merge_range_parts([np.zeros(5, np.int64)] * 3, [np.zeros(0, np.uint64)] * 3)
    assert lims.tolist() == [0] * 5 and D.size == 0 and I.size == 0


def test_merge_range_parts_keeps_an_equal_key_of_both_parts():
    keys = flat_ip.pack_keys(np.array([0.9, 0.5], np.float32), np.array([7, 3]))
    lims, D, I = merge_range_parts([[0, 2], [0, 1]], [keys, keys[:1]])
    assert lims.tolist() == [0, 3] and I.tolist() == [7, 7, 3] and D.tolist() == [np.float32(0.9)] * 2 + [0.5]


# ---------------------------------------------------------------------------
# C argument checks: no device is touched
# ---------------------------------------------------------------------------
def test_range_search_keys_argument_validation_needs_no_gpu():
    L = (ctypes.c_int64 * 2)()
    K = (ctypes.c_uint64 * 4)()
    q = (ctypes.c_float * 8)()

    def call(idx, nq, radius, capacity, lims=L, keys=K):
        return nat.lib.ivr_index_range_search_keys_device(idx, q, nq, radius, capacity, lims, keys, 0, None)

    assert call(None, 1, 0.5, 4) == nat.IVR_EINVAL                  # NULL handle
    assert "NULL" in nat.last_error()
    assert call(None, 1, float("nan"), 4) == nat.IVR_EINVAL         # NaN radius
    assert "NaN" in nat.last_error()
    assert call(None, 1, 0.5, -1) == nat.IVR_EINVAL                 # negative capacity
    assert call(None, -1, 0.5, 4) == nat.IVR_EINVAL                 # negative nq
    assert call(None, 1, 0.5, 4, lims=None) == nat.IVR_EINVAL


def test_range_merge_argument_validation_needs_no_gpu():
    keys = (ctypes.c_uint64 * 8)()
    lims_p = (ctypes.c_int64 * 8)()
    lims = (ctypes.c_int64 * 4)()
    D = (ctypes.c_float * 8)()
    I = (ctypes.c_int64 * 8)()

    def call(n_parts=2, nq=3, stride=4, keys=keys, lims_p=lims_p, lims=lims, D=D, I=I):
        return nat.lib.ivr_range_merge_keys_device(0, keys, stride, lims_p, n_parts, nq, lims, D, I, None)

    for bad in (dict(n_parts=0), dict(n_parts=65), dict(nq=-1), dict(stride=-1), dict(keys=None), dict(lims_p=None),
                dict(lims=None), dict(D=None), dict(I=None), dict(stride=1 << 62)):
        assert call(**bad) == nat.IVR_EINVAL, bad
        assert "range_merge_keys" in nat.last_error()


# ---------------------------------------------------------------------------
# world size 2 over gloo
# ---------------------------------------------------------------------------
class _OracleLocal:
    """The local index protocol of faiss_compat.IndexFlatIP, restated on the oracle (a search window included)."""

    def __init__(self, d, fail_range=False):
        self.d, self.xb, self.first, self.count, self.fail_range = d, np.zeros((0, d), np.float32), 0, -1, fail_range

    @property
    def ntotal(self):
        return self.xb.shape[0]

    def add(self, x):
        self.xb = np.concatenate([self.xb, np.asarray(x, np.float32)])

    def set_window(self, first=0, count=-1):
        assert count < 0 or 0 <= first and first + count <= self.ntotal
        self.first, self.count = (first, count) if count >= 0 else (0, -1)

    def _rows(self):
        return self.xb if self.count < 0 else self.xb[self.first:self.first + self.count]

    def search_keys_tensor(self, q, k, id_offset=0, out=None):
        ix = flat_ip.IndexFlatIP(self.d)
        ix.add(self._rows())
        D, I = ix.search(q.numpy(), k)
        keys = torch.from_numpy(flat_ip.pack_keys(D, np.where(I >= 0, I + id_offset + self.first, -1)).view(np.int64))
        if out is None:
            return keys
        out.copy_(keys)
        return out

    def range_search_keys_tensor(self, q, radius, id_offset=0):
        if self.fail_range:
            raise RuntimeError("injected local failure")
        lims, D, I = orr.range_search(self._rows(), q.numpy(), radius)
        keys = flat_ip.pack_keys(D, I + id_offset + self.first).view(np.int64)
        return torch.from_numpy(lims), torch.from_numpy(keys)


def _merge(keys_parts, k):
    D_all, I_all = zip(*(flat_ip.unpack_keys(p) for p in keys_parts.numpy().view(np.uint64)))
    D, I = flat_ip.merge_shard_results(list(D_all), list(I_all), k)
    return torch.from_numpy(D), torch.from_numpy(I)


def _range_merge(keys_parts, lims_parts, total):
    lims, D, I = merge_range_parts(lims_parts.numpy(), keys_parts.numpy())
    assert lims[-1] == total
    return torch.from_numpy(lims), torch.from_numpy(D), torch.from_numpy(I)


def _sharded(d, **kw):
    from ivr_b200.sharded import ShardedFlatIP
    return ShardedFlatIP(d, local_index=_OracleLocal(d, **kw), merge=_merge, range_merge=_range_merge)


def _same(got, want):
    return (np.array_equal(got[0].numpy(), want[0]) and np.array_equal(got[2].numpy(), want[2])
            and np.allclose(got[1].numpy(), want[1], atol=1e-6))


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
        from ivr_b200.sharded import partition_rows
        n, d = 1001, 32
        xb = synth.clip_like(n, d, seed=31, n_centres=64)
        xb[520:540] = xb[300:320]                                   # equal scores on both ranks
        xq = np.concatenate([xb[:3], synth.clip_like(6, d, seed=32, n_centres=64)])
        res = []
        for weights in (None, [1.0, 3.0]):
            sh = _sharded(d)
            sh.add_global(xb, weights=weights)
            off = partition_rows(n, world, weights)
            s = xq @ xb.T
            radii = [-np.inf, np.inf, float(np.median(np.sort(s, 1)[:, -30])), float(np.median(np.sort(s, 1)[:, -300]))]
            for radius in radii:
                got = sh.range_search(torch.from_numpy(xq), radius)
                res.append(_same(got, orr.range_search(xb, xq, radius)))
            # rank 1 has no hit at all: the radius is its best score for these rank-0 rows
            lone = xq[:3]
            radius = float((lone @ xb[off[1]:].T).max())
            got = sh.range_search(torch.from_numpy(lone), radius)
            want = orr.range_search(xb, lone, radius)
            res.append(_same(got, want) and want[0][-1] > 0 and np.all(want[2] < off[1]))
            # no queries: no collective, the same empty result everywhere
            got = sh.range_search(torch.zeros((0, d)), 0.5)
            res.append(got[0].tolist() == [0] and got[1].numel() == 0 and got[2].numel() == 0)
            # between search_async calls: the pending searches keep their hits
            full = flat_ip.IndexFlatIP(d)
            full.add(xb)
            h1 = sh.search_async(torch.from_numpy(xq), 10)
            got = sh.range_search(torch.from_numpy(xq), radii[2])
            h2 = sh.search_async(torch.from_numpy(xq), 10)
            Dr, Ir = full.search(xq, 10)
            res.append(_same(got, orr.range_search(xb, xq, radii[2])))
            for h in (h1, h2):
                D, I = h.result()
                res.append(np.array_equal(I.numpy(), Ir) and np.allclose(D.numpy(), Dr, atol=1e-6))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_sharded_range_search_world2_static_partitions():
    out = _spawn(_static_worker)
    assert out[0] == out[1] and all(out[0]) and len(out[0]) == 18, out


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
        from ivr_b200.sharded import partition_rows
        n, d, k, margin = 4001, 32, 10, 700
        xb = synth.clip_like(n, d, seed=41, n_centres=64)
        sh = _sharded(d)
        sh.add_global(xb, margin=margin)
        sh.enable_elastic(partition_rows(n, world), margin, period=4, gain=1.0,
                          timer=_ScriptedTimer(sh, 0.003 if rank == 0 else 0.001))
        ok = True
        for s_ in range(14):
            xq = synth.clip_like(5, d, seed=300 + s_, n_centres=64)
            sh.search(torch.from_numpy(xq), k)
            before = (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
            radius = float(np.median(np.sort(xq @ xb.T, 1)[:, -40]))
            got = sh.range_search(torch.from_numpy(xq), radius)
            ok = ok and _same(got, orr.range_search(xb, xq, radius))
            ok = ok and before == (sh._nsearch, list(sh.balance_log), sh._bounds.tolist())
        out[rank] = (ok, [(i, list(map(int, rows))) for i, _, rows in sh.balance_log])
    finally:
        dist.destroy_process_group()


def test_sharded_range_search_world2_after_the_elastic_boundaries_moved():
    """Range searches between the searches of the elastic-boundary test: still exact on the moved boundaries, and the
    controller steps exactly as without them (at searches 4, 8, 12, up to the margin)."""
    out = _spawn(_elastic_worker)
    assert out[0][0] and out[1][0]
    assert out[0][1] == out[1][1] and [i for i, _ in out[0][1]] == [4, 8, 12]
    assert out[0][1][-1][1] == [2000 - 700, 2001 + 700]


def _error_worker(rank, world, port, out):
    _init(rank, world, port)
    try:
        n, d = 601, 16
        xb = synth.clip_like(n, d, seed=51, n_centres=16)
        xq = torch.from_numpy(synth.clip_like(4, d, seed=52, n_centres=16))
        res = {}
        sh = _sharded(d)
        sh.add_global(xb)
        try:
            sh.range_search(xq, 0.5 if rank == 0 else 0.25)
            res["radius"] = "no error"
        except ValueError as e:
            res["radius"] = str(e)
        bad = _sharded(d, fail_range=(rank == 1))
        bad.add_global(xb)
        try:
            bad.range_search(xq, 0.5)
            res["failure"] = "no error"
        except RuntimeError as e:
            res["failure"] = str(e)
        got = sh.range_search(xq, 0.5)                             # the group is still in step
        res["after"] = _same(got, orr.range_search(xb, xq.numpy(), 0.5))
        out[rank] = res
    finally:
        dist.destroy_process_group()


def test_sharded_range_search_world2_errors_are_raised_on_every_rank():
    out = _spawn(_error_worker)
    for r in (0, 1):
        assert "rank 1" in out[r]["radius"] and "radius=0.25" in out[r]["radius"], out[r]
        assert "failed on rank 1" in out[r]["failure"], out[r]
        assert out[r]["after"]
    assert out[0]["radius"] == out[1]["radius"] and out[0]["failure"] == out[1]["failure"]
