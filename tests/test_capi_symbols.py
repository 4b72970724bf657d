"""CPU: the C-ABI library loads, exports every symbol include/ivr_b200.h declares, and fails
loudly (no CPU fallback) when there is no GPU."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import ivr_b200
from ivr_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "ivr_b200.h")).read()
    return sorted(set(re.findall(r"IVR_API\s+[\w\s\*]+?\b(ivr_\w+)\s*\(", src)))


def test_header_and_library_agree():
    syms = declared_symbols()
    assert len(syms) >= 25
    lib = ctypes.CDLL(nat.LIB_PATH)
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, f"declared in the header but not exported: {missing}"
    assert sorted(nat.PROTOTYPES) == syms, "ctypes PROTOTYPES out of sync with the header"


def _cuobjdump():
    """cuobjdump on PATH, else next to the nvcc the library was built with (NVCC, as in __graft_entry__.build())."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    for cand in (shutil.which("cuobjdump"), os.path.join(os.path.dirname(nvcc), "cuobjdump")):
        if cand and os.access(cand, os.X_OK):
            return cand
    return None


def test_library_is_sm100a_native():
    """The .so carries sm_100a SASS (no PTX-JIT for other archs, no multi-backend)."""
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-lelf", nat.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "sm_100a" in out
    assert not re.search(r"sm_(7|8|9)\d", out)


def test_version_and_error_string():
    assert nat.lib.ivr_version() >= 100
    assert isinstance(nat.last_error(), str)


@pytest.mark.skipif(nat.device_count() > 0, reason="only meaningful without a GPU")
def test_no_cpu_fallback_without_gpu():
    with pytest.raises(nat.NativeError) as e:
        ivr_b200.IndexFlatIP(64)
    assert e.value.code == nat.IVR_ENODEVICE
    x = np.ones((4, 8), np.float32)
    with pytest.raises(nat.NativeError):
        ivr_b200.normalize_L2(x)
    with pytest.raises(nat.NativeError):
        ivr_b200.frame_filter.calculate_similarities(x)
    with pytest.raises(nat.NativeError):
        ivr_b200.FrameFilter().apply_filters(x)


def test_argument_validation_needs_no_gpu():
    assert nat.lib.ivr_index_create(0, 0, ctypes.byref(ctypes.c_void_p())) == nat.IVR_EINVAL
    assert "dim" in nat.last_error()
    assert nat.lib.ivr_index_ntotal(None) == -1
    assert nat.lib.ivr_index_search(None, None, 1, 1, None, None, 0) == nat.IVR_EINVAL
