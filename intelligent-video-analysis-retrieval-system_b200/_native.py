"""ctypes binding of the C ABI in include/ivr_b200.h (libivr_b200.so).

The shared library is built in-tree by ``__graft_entry__.build()`` (or
``make -C csrc``).  There is no CPU fallback: if the library is missing this
module raises at import, and every compute entry point fails with
``IVR_ENODEVICE`` when no sm_100 GPU is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libivr_b200.so")

IVR_OK, IVR_EINVAL, IVR_ENODEVICE, IVR_ECUDA, IVR_ENOMEM, IVR_EUNSUPPORTED = 0, -1, -2, -3, -4, -5
IVR_MAX_K = 2048
IVR_MAX_WINDOW = 32
IVR_IPC_HANDLE_BYTES = 64
PATH_AUTO, PATH_STREAM, PATH_MMA = 0, 1, 2

_c_f32p = C.POINTER(C.c_float)
_c_i64p = C.POINTER(C.c_int64)
_c_u8p = C.POINTER(C.c_uint8)
_c_u32p = C.POINTER(C.c_uint32)
_c_intp = C.POINTER(C.c_int)

# name -> (restype, argtypes); mirrors include/ivr_b200.h one-to-one
PROTOTYPES = {
    "ivr_last_error": (C.c_char_p, []),
    "ivr_version": (C.c_int, []),
    "ivr_device_count": (C.c_int, [_c_intp]),
    "ivr_device_info": (C.c_int, [C.c_int, C.c_char_p, C.c_size_t, _c_intp, _c_intp, _c_intp,
                                  C.POINTER(C.c_size_t)]),
    "ivr_index_create": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "ivr_index_destroy": (C.c_int, [C.c_void_p]),
    "ivr_index_reserve": (C.c_int, [C.c_void_p, C.c_int64]),
    "ivr_index_add": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "ivr_index_add_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ivr_index_reconstruct": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "ivr_index_reset": (C.c_int, [C.c_void_p]),
    "ivr_index_ntotal": (C.c_int64, [C.c_void_p]),
    "ivr_index_dim": (C.c_int, [C.c_void_p]),
    "ivr_index_device": (C.c_int, [C.c_void_p]),
    "ivr_index_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_int]),
    "ivr_index_search_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "ivr_index_search_keys_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                               C.c_int64, C.c_int, C.c_void_p]),
    "ivr_index_range_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_int64, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "ivr_index_range_search_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_int64,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ivr_index_range_search_keys_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_int64,
                                                     C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ivr_index_range_self_join": (C.c_int, [C.c_void_p, C.c_float, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ivr_index_range_self_join_device": (C.c_int, [C.c_void_p, C.c_float, C.c_int64, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p]),
    "ivr_index_dpad": (C.c_int, [C.c_void_p]),
    "ivr_index_rows_f16_device": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "ivr_index_range_self_join_keys_device": (C.c_int, [C.c_void_p, C.c_float, C.c_int64, C.c_void_p, C.c_void_p,
                                                        C.c_int64, C.c_void_p]),
    "ivr_index_range_cross_join_keys_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int,
                                                         C.c_float, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                                         C.c_void_p]),
    "ivr_selection_create": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "ivr_selection_destroy": (C.c_int, [C.c_void_p]),
    "ivr_selection_count": (C.c_int64, [C.c_void_p]),
    "ivr_index_search_selected": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                            C.c_void_p]),
    "ivr_index_search_selected_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                                   C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "ivr_index_range_search_selected": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                                  C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ivr_index_range_search_selected_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                                         C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                                         C.c_void_p]),
    "ivr_index_search_selected_keys_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                                        C.c_void_p, C.c_int64, C.c_void_p]),
    "ivr_index_range_search_selected_keys_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                                              C.c_float, C.c_int64, C.c_void_p, C.c_void_p,
                                                              C.c_int64, C.c_void_p]),
    "ivr_index_set_window": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64]),
    "ivr_index_set_timing": (C.c_int, [C.c_void_p, C.c_int]),
    "ivr_index_last_timing": (C.c_int, [C.c_void_p, _c_f32p, _c_intp]),
    "ivr_index_last_path": (C.c_int, [C.c_void_p]),
    "ivr_index_last_kernel": (C.c_char_p, [C.c_void_p]),
    "ivr_topk_merge_device": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int64,
                                        C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ivr_topk_merge_keys_device": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "ivr_range_merge_keys_device": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int64,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ivr_exchange_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.POINTER(C.c_void_p)]),
    "ivr_exchange_destroy": (C.c_int, [C.c_void_p]),
    "ivr_exchange_base": (C.c_void_p, [C.c_void_p]),
    "ivr_exchange_ipc_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ivr_exchange_connect_ipc": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ivr_exchange_connect_ptrs": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ivr_exchange_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_uint32, C.c_void_p]),
    "ivr_exchange_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_void_p]),
    "ivr_exchange_slot": (C.c_void_p, [C.c_void_p, C.c_int]),
    "ivr_normalize_l2": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int]),
    "ivr_normalize_l2_device": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "ivr_consecutive_cosine": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "ivr_consecutive_cosine_device": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int,
                                                C.c_void_p, C.c_void_p]),
    "ivr_dedup_window": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_int64, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "ivr_dedup_window_device": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "ivr_frame_filter": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int,
                                   C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "ivr_dedup_set_timing": (C.c_int, [C.c_int]),
    "ivr_dedup_last_timing": (C.c_int, [_c_f32p]),
    "ivr_dedup_chain": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_int64, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "ivr_dedup_fifo": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_int64, C.c_int, C.c_float, C.c_void_p]),
    "ivr_sequence_similarity": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_int,
                                          C.c_float, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_int64)]),
    "ivr_cosine_neighbors": (C.c_int, [C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_void_p]),
    "ivr_lzf_decompress": (C.c_int64, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]),
    "ivr_lz4_block_decompress": (C.c_int64, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64]),
    "ivr_unshuffle": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
}


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"ivr_b200 error {code}: {message}")
        self.code = code


def _load():
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)           # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def last_error() -> str:
    return (lib.ivr_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc != IVR_OK:
        raise NativeError(rc, last_error())


def device_count() -> int:
    n = C.c_int(0)
    check(lib.ivr_device_count(C.byref(n)))
    return n.value


def default_device() -> int:
    """Device this process should use: IVR_DEVICE, else LOCAL_RANK, else 0."""
    for var in ("IVR_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(var)
        if v is not None and v.strip() != "":
            return int(v)
    return 0


def device_info(device: int = 0) -> dict:
    name = C.create_string_buffer(256)
    sm, maj, mino = C.c_int(0), C.c_int(0), C.c_int(0)
    tot = C.c_size_t(0)
    check(lib.ivr_device_info(device, name, 256, C.byref(sm), C.byref(maj), C.byref(mino), C.byref(tot)))
    return {"name": name.value.decode(), "sm_count": sm.value, "cc": (maj.value, mino.value),
            "total_bytes": tot.value}
