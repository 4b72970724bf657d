"""CPU: the self-join's argument checks need no device; the join model and its checker (tests/self_join_ref.py)."""
import ctypes

import numpy as np
import pytest

from ivr_b200 import _native as nat
from oracle import fp16_model as fm

import self_join_ref as sj


def _host(idx, radius, capacity, lims=True, out=True):
    L = (ctypes.c_int64 * 2)() if lims else None
    D = (ctypes.c_float * 4)() if out else None
    I = (ctypes.c_int64 * 4)() if out else None
    return nat.lib.ivr_index_range_self_join(idx, radius, capacity, L, D, I)


def _device(idx, radius, capacity, lims=True, out=True):
    L = (ctypes.c_int64 * 2)() if lims else None
    D = (ctypes.c_float * 4)() if out else None
    I = (ctypes.c_int64 * 4)() if out else None
    return nat.lib.ivr_index_range_self_join_device(idx, radius, capacity, L, D, I, None)


@pytest.mark.parametrize("call", [_host, _device], ids=["host", "device"])
def test_range_self_join_argument_checks_in_header_order(call):
    nan = float("nan")
    # every case below is wrong in all the later ways too: the first check in the header's order must answer
    assert call(None, nan, -1, lims=False, out=False) == nat.IVR_EINVAL
    assert "NaN" in nat.last_error()
    assert call(None, 0.5, -1, lims=False, out=False) == nat.IVR_EINVAL
    assert "capacity" in nat.last_error()
    assert call(None, 0.5, 4) == nat.IVR_EINVAL                     # NULL handle
    assert "NULL" in nat.last_error()
    assert call(None, 0.5, 4, lims=False) == nat.IVR_EINVAL
    assert "NULL" in nat.last_error()
    assert call(None, 0.5, 4, out=False) == nat.IVR_EINVAL          # NULL D / I with capacity > 0
    assert "NULL" in nat.last_error()
    assert call(None, 0.5, 0, out=False) == nat.IVR_EINVAL          # capacity 0 may pass NULL D / I; the handle not
    assert "NULL" in nat.last_error()


def _scan(rows16, radius):
    """The join by a direct double loop over the pairs, in float64."""
    x = rows16.astype(np.float64)
    n = x.shape[0]
    lims, D, I = [0], [], []
    for i in range(n):
        hits = []
        for j in range(n):
            if j == i or np.isnan(x[i]).any() or np.isnan(x[j]).any():
                continue
            s = float(np.dot(x[i], x[j]))
            if s > float(np.float32(radius)):
                hits.append((-s, j))
        hits.sort()
        D += [-s for s, _ in hits]
        I += [j for _, j in hits]
        lims.append(len(I))
    return np.array(lims, np.int64), np.array(D), np.array(I, np.int64)


def test_model_join_matches_a_direct_scan():
    xb, _ = fm.exact_inputs(60, 24, 1, seed=3)
    xb[7, 3] = np.nan
    xb[20] = xb[5]                                                   # duplicated rows: exact ties
    rows16 = fm.store(xb)
    m, _ = sj.model_scores(rows16)
    for radius in (-np.inf, -0.5, 0.0, 0.25, 1.0, np.inf):
        lims, D, I = sj.model_join(rows16, radius)
        want = _scan(rows16, radius)
        np.testing.assert_array_equal(lims, want[0])
        np.testing.assert_array_equal(I, want[2])
        np.testing.assert_array_equal(D, want[1])
    assert np.isnan(m[7]).all() and np.isnan(m[:, 7]).all()
    lims, D, I = sj.model_join(rows16, -np.inf)
    assert lims[-1] == 59 * 58 and lims[8] - lims[7] == 0


def _exact_case():
    xb, _ = fm.exact_inputs(40, 16, 1, seed=11)
    xb[9] = xb[2]
    rows16 = fm.store(xb)
    radius = sj.kth_radius(rows16, 5)
    lims, D, I = sj.model_join(rows16, radius)
    return rows16, radius, lims, D.astype(np.float32), I


def test_check_join_accepts_the_model():
    rows16, radius, lims, D, I = _exact_case()
    assert lims[-1] > 0
    assert sj.check_join(lims, D, I, rows16, radius, exact=True) == []
    assert sj.check_join(lims, D, I + 100, rows16, radius, id_offset=100, exact=True) == []
    assert sj.check_join(lims, D, I, rows16, radius, sample=[0, 2, 9]) == []


def _drop(lims, D, I, pos):
    keep = np.ones(D.size, bool)
    keep[pos] = False
    row = np.searchsorted(lims, pos, side="right") - 1
    lims = lims.copy()
    lims[row + 1:] -= np.size(pos) if np.ndim(pos) else 1
    return lims, D[keep], I[keep]


def test_check_join_rejects_a_missing_pair():
    rows16, radius, lims, D, I = _exact_case()
    i = int(np.argmax(np.diff(lims) > 0))
    j = int(I[lims[i]])
    back = lims[j] + int(np.nonzero(I[lims[j]:lims[j + 1]] == i)[0][0])
    first = int(lims[i])
    a, b = sorted((first, back))
    lims2, D2, I2 = _drop(lims, D, I, b)
    lims2, D2, I2 = _drop(lims2, D2, I2, a)                       # both directions gone: still symmetric
    bad = sj.check_join(lims2, D2, I2, rows16, radius)
    assert any("missing" in x for x in bad)
    assert not any("symmetric" in x for x in bad)


def test_check_join_rejects_an_asymmetric_pair():
    rows16, radius, lims, D, I = _exact_case()
    i = int(np.argmax(np.diff(lims) > 0))
    lims2, D2, I2 = _drop(lims, D, I, int(lims[i]))               # one direction only
    assert any("symmetric" in x for x in sj.check_join(lims2, D2, I2, rows16, radius))
    D3 = D.copy()
    D3[lims[i]] = np.nextafter(D3[lims[i]], np.float32(np.inf))   # both present, score bits differ
    bad = sj.check_join(lims, D3, I, rows16, radius)
    assert any("symmetric" in x for x in bad)


def test_check_join_rejects_a_self_hit_and_a_misordered_row():
    rows16, radius, lims, D, I = _exact_case()
    i = int(np.argmax(np.diff(lims) >= 2))
    assert lims[i + 1] - lims[i] >= 2
    I2 = I.copy()
    I2[lims[i]] = i
    assert any("self-hit" in x for x in sj.check_join(lims, D, I2, rows16, radius))
    a = int(lims[i])
    D3, I3 = D.copy(), I.copy()
    D3[[a, a + 1]], I3[[a, a + 1]] = D[[a + 1, a]], I[[a + 1, a]]
    bad = sj.check_join(lims, D3, I3, rows16, radius)
    assert any("non-increasing" in x or "ascending id" in x for x in bad)
