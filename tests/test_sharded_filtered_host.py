"""CPU: the host side of filtered sharded search without a device -- a selector's slice of a shard's stored rows (packing
at unaligned offsets, its cache and ``close``), the selector fingerprint ranks compare, and the argument checks of the
two windowed filtered C entry points."""
import ctypes

import numpy as np
import pytest

from ivr_b200 import _native as nat
from ivr_b200 import faiss_compat as fc


def unpack(words, n):
    """uint32 words -> bool [n] (bit i & 31 of word i >> 5); the bits past n must be clear."""
    bits = np.unpackbits(np.asarray(words, np.uint32).view(np.uint8), bitorder="little").astype(bool)
    assert bits.size >= n and not bits[n:].any()
    return bits[:n]


def selectors(n):
    rng = np.random.default_rng(7)
    m = rng.random(n) < 0.3
    return [fc.IDSelectorRange(97, 1234), fc.IDSelectorBatch(rng.choice(n, 200, replace=False)),
            fc.IDSelectorBitmap(np.packbits(m, bitorder="little")), fc.IDSelectorNot(fc.IDSelectorRange(500, 1500))]


@pytest.mark.parametrize("first,count", [(0, 2000), (1, 31), (31, 33), (33, 1000), (127, 129), (1000, 1000),
                                         (1500, 800), (2000, 5), (0, 0), (640, 128)])
def test_slice_words_match_the_mask(first, count):
    n = 2000
    for sel in selectors(n):
        w = sel.slice_words(n, first, count)
        assert w.dtype == np.uint32 and w.size == (count + 31) // 32
        want = np.zeros(count, bool)
        part = sel._mask(n)[first:first + count]
        want[:part.size] = part                                    # ids at or past ntotal_global: not selected
        assert np.array_equal(unpack(w, count), want)
        view = sel.shard(n, first)                                 # the selector a shard's local index is given
        assert np.array_equal(view._mask(count), want)
        assert np.array_equal(unpack(view.words(count), count), want)


def test_slice_words_reject_negative_bounds():
    with pytest.raises(ValueError):
        fc.IDSelectorRange(0, 10).slice_words(100, -1, 10)
    with pytest.raises(ValueError):
        fc.IDSelectorRange(0, 10).slice_words(100, 0, -1)


class _FakeLib:
    """ivr_selection_create / _destroy / _count without a device: handles are numbers, the words are kept."""

    def __init__(self):
        self.next, self.live, self.created = 100, {}, []

    def ivr_selection_create(self, device, words_ptr, n_rows, out):
        n_words = (n_rows + 31) // 32
        words = np.ctypeslib.as_array(ctypes.cast(words_ptr, ctypes.POINTER(ctypes.c_uint32)), (max(n_words, 1),))
        h = self.next
        self.next += 1
        self.live[h] = (device, n_rows, words[:n_words].copy())
        self.created.append((device, n_rows))
        ctypes.cast(out, ctypes.POINTER(ctypes.c_void_p))[0] = h
        return nat.IVR_OK

    def ivr_selection_destroy(self, h):
        del self.live[h.value]
        return nat.IVR_OK


def test_slice_selection_cache_and_close(monkeypatch):
    fake = _FakeLib()
    monkeypatch.setattr(nat, "lib", fake)
    n = 3000
    sel = fc.IDSelectorRange(1000, 2100)
    a = sel.shard(n, 1200)._selection(0, 1500)                     # a rank storing global ids [1200, 2700)
    b = sel.shard(n, 1200)._selection(0, 1500)                     # a new view per search: the same handle
    assert a.value == b.value and fake.created == [(0, 1500)]
    device, n_rows, words = fake.live[a.value]
    assert n_rows == 1500 and np.array_equal(unpack(words, 1500), np.arange(1200, 2700) < 2100)
    c = sel.shard(n, 1201)._selection(0, 1500)                     # another offset, count, device or ntotal_global
    d = sel.shard(n, 1200)._selection(0, 1499)
    e = sel.shard(n, 1200)._selection(1, 1500)
    f = sel.shard(n + 1, 1200)._selection(0, 1500)
    full = sel._selection(0, n)                                    # the unsharded selection keeps its own entry
    assert len({h.value for h in (a, c, d, e, f, full)}) == 6 and len(fake.live) == 6
    sel.shard(n, 1200).close()                                     # a view owns nothing
    assert len(fake.live) == 6
    sel.close()
    assert fake.live == {}
    g = sel.shard(n, 1200)._selection(0, 1500)                     # rebuilt after close
    assert g.value not in (a.value, c.value) and len(fake.live) == 1
    sel.close()


def test_fingerprint_names_the_selection_not_the_selector_type():
    n = 5000
    rng = np.random.default_rng(3)
    ids = np.sort(rng.choice(n, 300, replace=False))
    m = np.zeros(n, bool)
    m[ids] = True
    a = fc.IDSelectorBatch(ids).fingerprint(n)
    assert a == fc.IDSelectorBitmap(np.packbits(m, bitorder="little")).fingerprint(n)
    assert a[0] == 300 and -(1 << 63) <= a[1] < (1 << 63)
    assert fc.IDSelectorBatch(ids[1:]).fingerprint(n) != a
    assert fc.IDSelectorBatch(ids).fingerprint(n + 64) != a                 # more words
    assert fc.IDSelectorRange(10, 20).fingerprint(n) == (10, fc.IDSelectorRange(10, 20).fingerprint(n)[1])
    assert fc.IDSelectorRange(10, 20).fingerprint(n) != fc.IDSelectorRange(11, 21).fingerprint(n)


def test_windowed_filtered_keys_argument_checks_need_no_device():
    q = np.zeros((1, 8), np.float32)
    keys = np.zeros(4, np.uint64)
    lims = np.zeros(2, np.int64)
    lib = nat.lib

    def topk(idx=None, sel=None, nq=1, k=4, q=q.ctypes.data, keys=keys.ctypes.data, off=0):
        return lib.ivr_index_search_selected_keys_device(idx, sel, q, nq, k, keys, off, None)

    def rng(idx=None, sel=None, nq=1, radius=0.5, cap=4, lims=lims.ctypes.data, keys=keys.ctypes.data, off=0):
        return lib.ivr_index_range_search_selected_keys_device(idx, sel, q.ctypes.data, nq, radius, cap, lims, keys,
                                                               off, None)

    assert topk() == nat.IVR_EINVAL                                # NULL index
    assert topk(nq=-1) == nat.IVR_EINVAL
    assert topk(q=None) == nat.IVR_EINVAL
    assert topk(keys=None) == nat.IVR_EINVAL
    assert "search_selected_keys" in nat.last_error()
    assert rng() == nat.IVR_EINVAL                                 # NULL index
    assert "NULL" in nat.last_error()
    assert rng(radius=float("nan")) == nat.IVR_EINVAL              # the range checks come first
    assert "NaN" in nat.last_error()
    assert rng(cap=-1) == nat.IVR_EINVAL
    assert "capacity" in nat.last_error()
    assert rng(nq=-1) == nat.IVR_EINVAL
    assert rng(lims=None) == nat.IVR_EINVAL
    assert rng(keys=None) == nat.IVR_EINVAL
