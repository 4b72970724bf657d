"""CPU: filtered search without a device -- the id selectors' packed words, the argument checks of the selection and
filtered-search C entry points, and UnifiedIndex's folder -> rows map."""
import ctypes

import numpy as np
import pytest

from ivr_b200 import _native as nat
from ivr_b200 import faiss_compat as fc
from ivr_b200.unified_index import UnifiedIndex


def unpack(words, n):
    """uint32 words -> bool [n] (bit i & 31 of word i >> 5)."""
    w = np.asarray(words, np.uint32)
    bits = np.unpackbits(w.view(np.uint8), bitorder="little").astype(bool)
    assert bits.size >= n and not bits[n:].any()
    return bits[:n]


@pytest.mark.parametrize("ntotal", [0, 1, 31, 32, 33, 128, 1000])
def test_range_words(ntotal):
    for lo, hi in ((0, 0), (0, ntotal), (3, 40), (-5, 7), (50, 20), (ntotal - 1, ntotal + 100)):
        sel = fc.IDSelectorRange(lo, hi)
        w = sel.words(ntotal)
        assert w.dtype == np.uint32 and w.size == (ntotal + 31) // 32
        want = (np.arange(ntotal) >= lo) & (np.arange(ntotal) < hi)
        assert np.array_equal(unpack(w, ntotal), want)
        assert sel.count(ntotal) == int(want.sum())


def test_batch_words_duplicates_and_out_of_range():
    sel = fc.IDSelectorBatch([5, 5, 0, 99, 100, 1000, -1, 64])
    want = np.zeros(100, bool)
    want[[0, 5, 64, 99]] = True
    assert np.array_equal(unpack(sel.words(100), 100), want)
    assert sel.count(100) == 4
    assert fc.IDSelectorBatch([]).count(100) == 0
    assert not unpack(fc.IDSelectorBatch([]).words(100), 100).any()


def test_bitmap_words_follow_faiss_bit_order():
    rng = np.random.default_rng(0)
    bitmap = rng.integers(0, 256, 13, dtype=np.uint8)
    n = 130                                          # past the bitmap's 104 ids: not selected
    want = np.array([(bitmap[i >> 3] >> (i & 7)) & 1 if i < 104 else 0 for i in range(n)], bool)
    assert np.array_equal(unpack(fc.IDSelectorBitmap(bitmap).words(n), n), want)
    assert np.array_equal(unpack(fc.IDSelectorBitmap(bitmap).words(50), 50), want[:50])
    b = np.zeros(2, np.uint8)
    b[0] = 0b00000100                                # id 2
    b[1] = 0b10000000                                # id 15
    assert np.nonzero(unpack(fc.IDSelectorBitmap(b).words(16), 16))[0].tolist() == [2, 15]
    with pytest.raises(TypeError):
        fc.IDSelectorBitmap(np.zeros(4, np.int32))


def test_not_words():
    n = 77
    inner = fc.IDSelectorRange(10, 20)
    got = unpack(fc.IDSelectorNot(inner).words(n), n)
    assert np.array_equal(got, ~((np.arange(n) >= 10) & (np.arange(n) < 20)))
    assert np.array_equal(unpack(fc.IDSelectorNot(fc.IDSelectorNot(inner)).words(n), n), ~got)
    assert fc.IDSelectorNot(fc.IDSelectorBatch([])).count(n) == n


def test_search_parameters_default_is_unfiltered():
    assert fc.SearchParameters().sel is None
    s = fc.IDSelectorRange(0, 1)
    assert fc.SearchParameters(sel=s).sel is s


def test_selection_argument_checks_need_no_device():
    out = ctypes.c_void_p()
    w = np.ones(4, np.uint32)
    assert nat.lib.ivr_selection_create(0, w.ctypes.data, 10, None) == nat.IVR_EINVAL
    assert nat.lib.ivr_selection_create(0, w.ctypes.data, -1, ctypes.byref(out)) == nat.IVR_EINVAL
    assert "n_rows" in nat.last_error()
    assert nat.lib.ivr_selection_create(0, None, 10, ctypes.byref(out)) == nat.IVR_EINVAL
    assert nat.lib.ivr_selection_create(0, w.ctypes.data, (1 << 32) + 1, ctypes.byref(out)) == nat.IVR_EUNSUPPORTED
    assert not out.value
    assert nat.lib.ivr_selection_count(None) == -1
    assert nat.lib.ivr_selection_destroy(None) == nat.IVR_OK


def test_filtered_search_argument_checks_need_no_device():
    q = np.zeros((1, 8), np.float32)
    D = np.zeros(4, np.float32)
    I = np.zeros(4, np.int64)
    lims = np.zeros(2, np.int64)
    lib = nat.lib
    assert lib.ivr_index_search_selected(None, None, q.ctypes.data, 1, 4, D.ctypes.data, I.ctypes.data) == \
        nat.IVR_EINVAL
    assert lib.ivr_index_search_selected_device(None, None, q.ctypes.data, 1, 4, D.ctypes.data, I.ctypes.data, 0,
                                                None) == nat.IVR_EINVAL
    assert lib.ivr_index_range_search_selected(None, None, q.ctypes.data, 1, 0.5, 4, lims.ctypes.data, D.ctypes.data,
                                               I.ctypes.data) == nat.IVR_EINVAL
    assert lib.ivr_index_range_search_selected_device(None, None, q.ctypes.data, 1, 0.5, 4, lims.ctypes.data,
                                                      D.ctypes.data, I.ctypes.data, 0, None) == nat.IVR_EINVAL
    # the range checks come first: a NaN radius and a negative capacity are named
    assert lib.ivr_index_range_search_selected(None, None, q.ctypes.data, 1, float("nan"), 4, lims.ctypes.data,
                                               D.ctypes.data, I.ctypes.data) == nat.IVR_EINVAL
    assert "NaN" in nat.last_error()
    assert lib.ivr_index_range_search_selected_device(None, None, q.ctypes.data, 1, 0.5, -1, lims.ctypes.data,
                                                      D.ctypes.data, I.ctypes.data, 0, None) == nat.IVR_EINVAL
    assert "capacity" in nat.last_error()


def make_unified(folders):
    u = UnifiedIndex()
    u.metadata_list = [{"folder_name": f, "frame_id": i} for i, f in enumerate(folders)]
    u.is_loaded = True
    return u


def test_unified_folder_rows_map():
    folders = ["a", "b", "a", "c", "b", "a"]
    u = make_unified(folders)
    assert u.video_rows(["a"]).tolist() == [0, 2, 5]
    assert u.video_rows("b").tolist() == [1, 4]
    assert u.video_rows(["c", "a", "a"]).tolist() == [0, 2, 3, 5]
    assert u.video_rows(["nope"]).tolist() == []
    assert u.video_rows([]).tolist() == []
    assert u.video_rows(["nope", "c"]).tolist() == [3]
    # the map is built once per load and dropped when the metadata is replaced
    first = u._folder_rows
    u.video_rows(["b"])
    assert u._folder_rows is first
    u.metadata_list.append({"folder_name": "d"})
    u._folder_rows = None                            # what load_unified_index / build_from_embeddings do
    assert u.video_rows(["d"]).tolist() == [6]


def test_unified_rows_skip_metadata_without_folder():
    u = make_unified(["a", "b"])
    u.metadata_list.append({"frame_id": 9})
    u.metadata_list.append(None)
    assert u.video_rows(["a", "b"]).tolist() == [0, 1]
