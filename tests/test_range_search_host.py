"""CPU: range search's argument checks need no device; the range oracle and the band comparator
(oracle/range_search.py)."""
import ctypes

import numpy as np
import pytest

from ivr_b200 import _native as nat
from oracle import range_search as orr


def _host(idx, nq, radius, capacity, lims=True, out=True):
    L = (ctypes.c_int64 * (max(nq, 0) + 1))() if lims else None
    D = (ctypes.c_float * 4)() if out else None
    I = (ctypes.c_int64 * 4)() if out else None
    q = (ctypes.c_float * 8)()
    return nat.lib.ivr_index_range_search(idx, q, nq, radius, capacity, L, D, I)


def _device(idx, nq, radius, capacity):
    L = (ctypes.c_int64 * 2)()
    D = (ctypes.c_float * 4)()
    I = (ctypes.c_int64 * 4)()
    q = (ctypes.c_float * 8)()
    return nat.lib.ivr_index_range_search_device(idx, q, nq, radius, capacity, L, D, I, 0, None)


@pytest.mark.parametrize("call", [_host, _device], ids=["host", "device"])
def test_range_search_argument_validation_needs_no_gpu(call):
    assert call(None, 1, 0.5, 4) == nat.IVR_EINVAL                  # NULL handle
    assert "NULL" in nat.last_error()
    assert call(None, 1, float("nan"), 4) == nat.IVR_EINVAL         # NaN radius
    assert "NaN" in nat.last_error()
    assert call(None, 1, 0.5, -1) == nat.IVR_EINVAL                 # negative capacity
    assert "capacity" in nat.last_error()
    assert call(None, -1, 0.5, 4) == nat.IVR_EINVAL                 # negative nq
    assert "nq" in nat.last_error()


def test_range_search_null_outputs_are_rejected():
    assert _host(None, 1, 0.5, 4, lims=False) == nat.IVR_EINVAL
    assert _host(None, 1, 0.5, 4, out=False) == nat.IVR_EINVAL


def _numpy_range(xb, xq, radius):
    s = xq @ xb.T
    lims, D, I = [0], [], []
    for q in range(xq.shape[0]):
        ids = np.nonzero(s[q] > np.float32(radius))[0]
        order = sorted(ids, key=lambda i: (-s[q, i], i))
        D.extend(s[q, order])
        I.extend(order)
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D, np.float32), np.array(I, np.int64)


def test_oracle_range_search_matches_a_direct_scan():
    rng = np.random.default_rng(0)
    xb = rng.standard_normal((700, 24)).astype(np.float32)
    xq = rng.standard_normal((5, 24)).astype(np.float32)
    for radius in (-np.inf, -1.0, 2.0, 6.0, np.inf):
        lims, D, I = orr.range_search(xb, xq, radius, db_block=128)
        want = _numpy_range(xb, xq, radius)
        np.testing.assert_array_equal(lims, want[0])
        np.testing.assert_array_equal(I, want[2])
        np.testing.assert_array_equal(D, want[1])
    lims, D, I = orr.range_search(xb, np.zeros((0, 24), np.float32), 0.0)
    assert lims.tolist() == [0] and D.size == 0 and I.size == 0


def test_oracle_range_search_is_strict_and_orders_ties_by_id():
    xb = np.array([[1, 0], [0.5, 0], [1, 0], [0.25, 0], [1, 0]], np.float32)
    q = np.array([[1, 0]], np.float32)
    lims, D, I = orr.range_search(xb, q, 0.5)                        # 0.5 is an exact score: not a hit
    assert lims.tolist() == [0, 3] and I.tolist() == [0, 2, 4] and D.tolist() == [1, 1, 1]
    lims, D, I = orr.range_search(xb, q, 0.25)
    assert I.tolist() == [0, 2, 4, 1]
    lims, D, I = orr.range_search(xb, q, 1.0)
    assert lims.tolist() == [0, 0]


def _case():
    xb = np.array([[0.9, 0], [0.8, 0], [0.6, 0], [0.1, 0]], np.float32)
    xq = np.array([[1, 0], [0, 1]], np.float32)
    lims, D, I = orr.range_search(xb, xq, 0.5)
    return xb, xq, lims, D, I


def test_compare_range_accepts_parity_and_band_substitutions():
    xb, xq, lims, D, I = _case()
    score_of = lambda q, ids: xb[ids] @ xq[q]
    assert orr.compare_range(lims, D, I, lims, D, I, score_of, 0.5) == []
    # a row inside the band (0.5 + 5e-4) may be missing or present
    assert orr.compare_range(lims, D, I, lims, D, I, score_of, 0.6 - 5e-4) == []


def test_compare_range_rejects_missing_duplicate_and_misordered_hits():
    xb, xq, lims, D, I = _case()
    score_of = lambda q, ids: xb[ids] @ xq[q]
    assert lims.tolist() == [0, 3, 3]
    bad = orr.compare_range(np.array([0, 2, 2]), D[:2], I[:2], lims, D, I, score_of, 0.5)
    assert any("missing" in b for b in bad)
    dup_D, dup_I = np.array([0.9, 0.8, 0.8], np.float32), np.array([0, 1, 1])
    bad = orr.compare_range(lims, dup_D, dup_I, lims, D, I, score_of, 0.5)
    assert any("duplicate" in b for b in bad)
    bad = orr.compare_range(lims, D[[1, 0, 2]], I[[1, 0, 2]], lims, D, I, score_of, 0.5)
    assert any("non-increasing" in b for b in bad)
    bad = orr.compare_range(np.array([0, 3, 2]), D, I, lims, D, I, score_of, 0.5)
    assert any("monotone" in b for b in bad)
    bad = orr.compare_range(np.array([0, 2, 3]), D, I, lims, D, I, score_of, 0.5)
    assert bad                                                       # hit attributed to the wrong query
    below = np.array([0, 4, 4])
    bad = orr.compare_range(below, np.append(D, 0.1).astype(np.float32), np.append(I, 3), lims, D, I,
                            score_of, 0.5)
    assert any("radius-tol" in b for b in bad)
