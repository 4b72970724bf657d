"""CPU: the work schedule of ShardedFlatIP.range_self_join (``join_schedule``) and the argument checks of the new C
calls that need no device (the checks that need an index are in tests/test_sharded_self_join_gpu.py)."""
import ctypes
import itertools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from ivr_b200 import _native as nat
from ivr_b200.sharded import join_schedule, partition_rows


def _pair_owners(bounds):
    """owner[i, j] (i < j): the ranks that score the pair (i, j); also every same-rank pair a cross task scores."""
    n = int(bounds[-1])
    count = np.zeros((n, n), np.int64)
    rank_of = np.searchsorted(bounds, np.arange(n), side="right") - 1
    per_rank = []
    for r in range(len(bounds) - 1):
        tasks = join_schedule(bounds, r)
        a, b, p, c, d = tasks[0]
        assert (a, b, p, c, d) == (bounds[r], bounds[r + 1], r, bounds[r], bounds[r + 1])
        pairs = (b - a) * (b - a - 1) // 2
        for i, j in itertools.combinations(range(a, b), 2):
            count[i, j] += 1
        for a, b, p, c, d in tasks[1:]:
            assert p != r and bounds[r] <= a <= b <= bounds[r + 1] and bounds[p] <= c <= d <= bounds[p + 1]
            pairs += (b - a) * (d - c)
            for i in range(a, b):
                for j in range(c, d):
                    assert rank_of[i] != rank_of[j]
                    count[min(i, j), max(i, j)] += 1
        per_rank.append(pairs)
    return count, per_rank


@pytest.mark.parametrize("world", range(1, 10))
@pytest.mark.parametrize("layout", ["equal", "unequal", "empty"])
def test_schedule_scores_every_pair_once(world, layout):
    n = 6 * world
    if layout == "equal":
        bounds = partition_rows(n, world)
    elif layout == "unequal":
        bounds = partition_rows(n + 5, world, weights=np.arange(1, world + 1))
    else:                                               # every other rank holds no row
        sizes = [0] + [7 + r if r % 2 == 0 else 0 for r in range(world)]
        bounds = np.cumsum(sizes).astype(np.int64)
    count, per_rank = _pair_owners(bounds)
    iu = np.triu_indices(int(bounds[-1]), 1)
    assert np.all(count[iu] == 1)                        # every unordered pair of distinct rows exactly once
    assert np.all(np.tril(count) == 0)
    assert all(len(join_schedule(bounds, r)) == 1 + world // 2 for r in range(world))   # the same rounds everywhere
    if layout == "equal":
        assert len(set(per_rank)) == 1                  # equal shards: equal work
        m = n // world
        assert per_rank[0] * world == n * (n - 1) // 2 and per_rank[0] == m * m * world // 2 - m // 2


def test_schedule_of_a_large_library_balances_the_pairs():
    """Counted, not enumerated: 8 ranks of 12.5 M rows each score n^2 / (2N) pairs up to the diagonal's n / 2."""
    world, m = 8, 12_500_000
    bounds = np.arange(world + 1, dtype=np.int64) * m
    for r in range(world):
        pairs = sum((b - a) * (d - c) if p != r else (b - a) * (b - a - 1) // 2
                    for a, b, p, c, d in join_schedule(bounds, r))
        assert pairs == m * m * world // 2 - m // 2


def _cross(idx=None, other=1, n_other=1, first=0, lower=0, radius=0.5, capacity=4, lims=True, keys=True, off=0):
    L = (ctypes.c_int64 * 4)() if lims else None
    K = (ctypes.c_uint64 * 4)() if keys else None
    return nat.lib.ivr_index_range_cross_join_keys_device(idx, other, n_other, first, lower, radius, capacity, L, K,
                                                          off, None)


def _self_keys(idx=None, radius=0.5, capacity=4, lims=True, keys=True, off=0):
    L = (ctypes.c_int64 * 4)() if lims else None
    K = (ctypes.c_uint64 * 4)() if keys else None
    return nat.lib.ivr_index_range_self_join_keys_device(idx, radius, capacity, L, K, off, None)


def test_cross_join_argument_checks_in_header_order():
    nan = float("nan")
    # every case is also wrong in all the later ways: the first check in the header's order must answer
    assert _cross(radius=nan, capacity=-1, n_other=-1, lims=False, keys=False, other=None) == nat.IVR_EINVAL
    assert "NaN" in nat.last_error()
    assert _cross(capacity=-1, lims=False, keys=False, other=None) == nat.IVR_EINVAL
    assert "n_other" in nat.last_error()
    assert _cross(n_other=-1, lims=False, keys=False, other=None) == nat.IVR_EINVAL
    assert "n_other" in nat.last_error()
    assert _cross() == nat.IVR_EINVAL                                  # NULL index
    assert "NULL" in nat.last_error()
    assert _cross(lims=False) == nat.IVR_EINVAL
    assert _cross(keys=False) == nat.IVR_EINVAL                        # NULL keys with capacity > 0
    assert _cross(other=None) == nat.IVR_EINVAL                        # NULL rows with n_other > 0
    assert "NULL" in nat.last_error()
    assert _cross(capacity=0, keys=False, n_other=0, other=None) == nat.IVR_EINVAL   # may pass those; not the index
    assert "NULL" in nat.last_error()


def test_self_join_keys_and_rows_argument_checks():
    assert _self_keys(radius=float("nan"), capacity=-1, lims=False, keys=False) == nat.IVR_EINVAL
    assert "NaN" in nat.last_error()
    assert _self_keys(capacity=-1, lims=False, keys=False) == nat.IVR_EINVAL
    assert "capacity" in nat.last_error()
    assert _self_keys() == nat.IVR_EINVAL and "NULL" in nat.last_error()
    assert _self_keys(keys=False) == nat.IVR_EINVAL
    buf = (ctypes.c_uint16 * 64)()
    assert nat.lib.ivr_index_rows_f16_device(None, 0, 1, buf, None) == nat.IVR_EINVAL
    assert nat.lib.ivr_index_rows_f16_device(None, 0, 0, None, None) == nat.IVR_EINVAL
    assert nat.lib.ivr_index_dpad(None) == -1


def test_cross_join_kernel_sass():
    """The cross-join kernel runs on tcgen05 (UTCHMMA) fed by TMA (UTMALDG) and keeps its registers (no local
    memory)."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tool = shutil.which("cuobjdump") or os.path.join(os.path.dirname(nvcc), "cuobjdump")
    if not os.access(tool, os.X_OK):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([tool, "-sass", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)
    body = [f for f in funcs if f.startswith("_ZN3ivr34search_mma_small_cross_join_kernel")]
    assert len(body) == 1
    assert "UTCHMMA" in body[0] and "UTMALDG" in body[0]
    assert not re.search(r"\b(LDL|STL)\b", body[0])
