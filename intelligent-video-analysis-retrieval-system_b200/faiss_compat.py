"""A ``faiss``-shaped module backed by the sm_100a kernels (boundary level B0).

The reference never computes the flat inner-product search itself: it calls
``faiss.IndexFlatIP`` (unified_index.py:503, 1767-1779; core.py:827, 891, 1208;
system.py:1330).  Installing this module as ``faiss``
(``sys.modules['faiss'] = faiss_compat``) makes the reference's own
``UnifiedIndex.search_vectors`` and ``FAISSRetriever.search`` run on the B200
path unchanged; see INTEGRATION.md.

Only the surface the reference touches is provided.  Everything computes on the
GPU through the C ABI (``_native``); there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat

__all__ = ["Index", "IndexFlatIP", "IndexFlatL2", "IndexIVFFlat", "normalize_L2",
           "StandardGpuResources", "index_cpu_to_gpu", "index_gpu_to_cpu", "write_index",
           "read_index", "serialize_index", "deserialize_index", "IO_FLAG_MMAP", "METRIC_INNER_PRODUCT",
           "SearchParameters", "IDSelector", "IDSelectorRange", "IDSelectorBatch", "IDSelectorBitmap",
           "IDSelectorNot"]

IO_FLAG_MMAP = 1
METRIC_INNER_PRODUCT = 0


def _as_f32_2d(x, d=None, what="x"):
    a = np.ascontiguousarray(x, dtype=np.float32)
    if a.ndim != 2:
        raise ValueError(f"{what} must be a 2-D array, got shape {a.shape}")
    if d is not None and a.shape[1] != d:
        raise ValueError(f"{what} has dimension {a.shape[1]}, index has {d}")   # FAISS asserts d == self.d
    return a


# -- filtered search: FAISS's SearchParameters(sel=IDSelector...) ------------------------------------------------
class IDSelector:
    """Base of the id selectors.  ``words(ntotal)`` is the selection over ids [0, ntotal) as packed uint32 words (bit
    ``i & 31`` of word ``i >> 5`` = id i), the layout of ``ivr_selection_create``.  The device selection built from it
    is cached per (device, ntotal) and freed by ``close`` (or when the selector is collected).

    A row shard applies a selector of GLOBAL ids to the rows it stores: ``slice_words`` / ``shard`` give the selection
    of ids [first, first + count) renumbered from 0, cached per (device, ntotal_global, first, count)."""

    def words(self, ntotal: int) -> np.ndarray:
        return _pack_words(self._mask(int(ntotal)))

    def _mask(self, ntotal: int) -> np.ndarray:       # bool [ntotal]
        raise NotImplementedError

    def _selection(self, device: int, ntotal: int):
        cache = self.__dict__.setdefault("_sel_cache", {})
        key = (int(device), int(ntotal))
        h = cache.get(key)
        if h is None:
            w = self.words(ntotal)
            h = C.c_void_p()
            nat.check(nat.lib.ivr_selection_create(int(device), w.ctypes.data, int(ntotal), C.byref(h)))
            cache[key] = h
        return h

    def slice_words(self, ntotal_global: int, first: int, count: int) -> np.ndarray:
        """The ids [first, first + count) of this selection over ``ntotal_global`` ids as packed words over ``count``
        local rows: bit 0 is id ``first``.  Ids at or past ``ntotal_global`` are not selected."""
        first, count = int(first), int(count)
        if first < 0 or count < 0:
            raise ValueError(f"slice_words: first ({first}) and count ({count}) must be >= 0")
        m = self._mask(int(ntotal_global))[first:first + count]
        return _pack_words(np.concatenate([m, np.zeros(count - m.size, bool)]))

    def _slice_selection(self, device: int, ntotal_global: int, first: int, count: int):
        cache = self.__dict__.setdefault("_sel_cache", {})
        key = (int(device), int(ntotal_global), int(first), int(count))
        h = cache.get(key)
        if h is None:
            w = self.slice_words(ntotal_global, first, count)
            h = C.c_void_p()
            nat.check(nat.lib.ivr_selection_create(int(device), w.ctypes.data, int(count), C.byref(h)))
            cache[key] = h
        return h

    def shard(self, ntotal_global: int, first: int) -> "IDSelector":
        """This selector of ids [0, ntotal_global) as seen by a shard whose stored row 0 is global id ``first``: a
        selector of stored rows, for the per-rank filtered searches of ``ShardedFlatIP``."""
        return _ShardSelector(self, int(ntotal_global), int(first))

    def fingerprint(self, ntotal_global: int) -> tuple:
        """(selected ids below ntotal_global, a 64-bit hash of the packed words): ranks compare it to find out that they
        were given different selectors.  Cached per ntotal_global."""
        import hashlib
        cache = self.__dict__.setdefault("_fp_cache", {})
        fp = cache.get(int(ntotal_global))
        if fp is None:
            w = self.words(int(ntotal_global))
            h = hashlib.blake2b(w.astype("<u4").tobytes(), digest_size=8).digest()
            fp = (int(np.unpackbits(w.view(np.uint8)).sum()), int.from_bytes(h, "little", signed=True))
            cache[int(ntotal_global)] = fp
        return fp

    def count(self, ntotal: int, device: int | None = None) -> int:
        """Selected ids below ``ntotal`` (computed by the device selection when ``device`` is given)."""
        if device is None:
            return int(self._mask(int(ntotal)).sum())
        return int(nat.lib.ivr_selection_count(self._selection(device, ntotal)))

    def close(self):
        cache = self.__dict__.pop("_sel_cache", {})
        for h in cache.values():
            nat.lib.ivr_selection_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _pack_words(mask: np.ndarray) -> np.ndarray:
    """bool [n] -> uint32 [ceil(n / 32)], bit i & 31 of word i >> 5 = mask[i]."""
    b = np.packbits(np.asarray(mask, bool), bitorder="little")
    b = np.concatenate([b, np.zeros(-b.size % 4, np.uint8)])
    return b.view("<u4").astype(np.uint32)


class _ShardSelector(IDSelector):
    """``IDSelector.shard``: ids [first, first + ntotal) of ``sel`` over ``ntotal_global`` ids, renumbered from 0.  Its
    device selections are ``sel``'s slice selections (cached and freed there), so a new view per search costs nothing."""

    def __init__(self, sel: IDSelector, ntotal_global: int, first: int):
        self.sel, self.ntotal_global, self.first = sel, ntotal_global, first

    def _mask(self, ntotal):
        m = self.sel._mask(self.ntotal_global)[self.first:self.first + ntotal]
        return np.concatenate([m, np.zeros(ntotal - m.size, bool)])

    def _selection(self, device, ntotal):
        return self.sel._slice_selection(device, self.ntotal_global, self.first, ntotal)

    def close(self):
        pass


class IDSelectorRange(IDSelector):
    """``faiss.IDSelectorRange(imin, imax)``: ids in the half-open range [imin, imax)."""

    def __init__(self, imin: int, imax: int):
        self.imin, self.imax = int(imin), int(imax)

    def _mask(self, ntotal):
        m = np.zeros(ntotal, bool)
        m[max(self.imin, 0):max(min(self.imax, ntotal), 0)] = True
        return m


class IDSelectorBatch(IDSelector):
    """``faiss.IDSelectorBatch(ids)``: the ids listed (duplicates and ids outside [0, ntotal) are ignored)."""

    def __init__(self, ids):
        self.ids = np.asarray(ids, np.int64).reshape(-1)

    def _mask(self, ntotal):
        m = np.zeros(ntotal, bool)
        ids = self.ids[(self.ids >= 0) & (self.ids < ntotal)]
        m[ids] = True
        return m


class IDSelectorBitmap(IDSelector):
    """``faiss.IDSelectorBitmap(bitmap)``: ``bitmap`` is a 1-D uint8 array in FAISS's bit order, id i is selected
    iff ``(bitmap[i >> 3] >> (i & 7)) & 1``; ids past the bitmap are not selected."""

    def __init__(self, bitmap):
        b = np.asarray(bitmap)
        if b.dtype != np.uint8 or b.ndim != 1:
            raise TypeError("IDSelectorBitmap expects a 1-D uint8 array")
        self.bitmap = b.copy()

    def _mask(self, ntotal):
        bits = np.unpackbits(self.bitmap, bitorder="little")[:ntotal].astype(bool)
        return np.concatenate([bits, np.zeros(ntotal - bits.size, bool)])


class IDSelectorNot(IDSelector):
    """``faiss.IDSelectorNot(sel)``: the ids in [0, ntotal) that ``sel`` does not select."""

    def __init__(self, sel: IDSelector):
        self.sel = sel

    def _mask(self, ntotal):
        return ~self.sel._mask(ntotal)


class SearchParameters:
    """``faiss.SearchParameters(sel=...)``: ``sel`` restricts a search to the ids it selects (None = all ids)."""

    def __init__(self, sel: IDSelector | None = None):
        self.sel = sel


class IndexFlatIP:
    """Exact inner-product index; rows live in HBM as fp16, ids are insertion order.

    ``add`` / ``search`` / ``ntotal`` / ``d`` / ``is_trained`` / ``train`` / ``reset`` follow
    ``faiss.IndexFlatIP`` as used by the reference; ``range_search`` follows FAISS's flat-index range query.
    """

    metric_type = METRIC_INNER_PRODUCT

    def __init__(self, d: int, device: int | None = None):
        self.d = int(d)
        self.is_trained = True
        self.device = nat.default_device() if device is None else int(device)
        h = C.c_void_p()
        nat.check(nat.lib.ivr_index_create(self.d, self.device, C.byref(h)))
        self._h = h
        self.search_path = nat.PATH_AUTO
        self._window_count = -1

    # -- lifecycle -------------------------------------------------------
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            nat.lib.ivr_index_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _handle(self):
        if not self._h:
            raise RuntimeError("index is closed")
        return self._h

    @property
    def ntotal(self) -> int:
        return int(nat.lib.ivr_index_ntotal(self._handle()))

    def train(self, x=None):          # flat index: nothing to train (core.py:820-825)
        return None

    def reset(self):
        nat.check(nat.lib.ivr_index_reset(self._handle()))

    def set_window(self, first: int = 0, count: int = -1):
        """Searches score only the stored rows [first, first + count) until cleared (``count < 0``); ids stay
        "stored row + id_offset".  No data moves (``ivr_index_set_window``)."""
        nat.check(nat.lib.ivr_index_set_window(self._handle(), int(first), int(count)))
        self._window_count = int(count)

    def reserve(self, n_rows: int):
        nat.check(nat.lib.ivr_index_reserve(self._handle(), int(n_rows)))

    # -- build -----------------------------------------------------------
    def add(self, x) -> None:
        """Append rows (float32 [n, d] host array, or a CUDA float32 torch tensor)."""
        if _is_cuda_tensor(x):
            return self.add_tensor(x)
        a = _as_f32_2d(x, self.d, "add(x)")
        nat.check(nat.lib.ivr_index_add(self._handle(), a.ctypes.data, a.shape[0]))

    def add_tensor(self, x) -> None:
        import torch
        if x.dim() != 2 or x.shape[1] != self.d:
            raise ValueError(f"add(x): expected [n,{self.d}], got {tuple(x.shape)}")
        x = x.to(dtype=torch.float32).contiguous()
        _check_device(x, self.device)
        st = torch.cuda.current_stream(x.device).cuda_stream
        nat.check(nat.lib.ivr_index_add_device(self._handle(), x.data_ptr(), x.shape[0], st))

    def reconstruct_n(self, first: int = 0, n: int | None = None) -> np.ndarray:
        """``faiss.Index.reconstruct_n``: rows [first, first + n) as float32 (the stored fp16 values, widened)."""
        n = self.ntotal - first if n is None else int(n)
        out = np.empty((n, self.d), np.float32)
        if n:
            nat.check(nat.lib.ivr_index_reconstruct(self._handle(), int(first), n, out.ctypes.data))
        return out

    # -- search ----------------------------------------------------------
    def search(self, x, k: int, *, params: SearchParameters | None = None):
        """D, I = index.search(x, k): float32 [nq,k] descending, int64 [nq,k], -1 padded.  ``params.sel`` restricts
        the search to the ids it selects: the k best selected rows (``ivr_index_search_selected``)."""
        if _is_cuda_tensor(x):
            return self.search_tensor(x, k, params=params)
        q = _as_f32_2d(x, self.d, "search(x)")
        k = int(k)
        if k <= 0:
            raise ValueError("k must be positive")
        nq = q.shape[0]
        D = np.empty((nq, k), np.float32)
        I = np.empty((nq, k), np.int64)
        sel = self._selection(params)
        if nq and sel is None:
            nat.check(nat.lib.ivr_index_search(self._handle(), q.ctypes.data, nq, k,
                                               D.ctypes.data, I.ctypes.data, self.search_path))
        elif nq:
            nat.check(nat.lib.ivr_index_search_selected(self._handle(), sel, q.ctypes.data, nq, k,
                                                        D.ctypes.data, I.ctypes.data))
        return D, I

    def search_tensor(self, q, k: int, id_offset: int = 0, path: int | None = None,
                      params: SearchParameters | None = None):
        """Device-resident search on torch's current stream; returns CUDA tensors (D, I).  ``params.sel``: as in
        ``search`` (``path`` does not apply: filtered search has one kernel)."""
        import torch
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"search(x): expected [nq,{self.d}], got {tuple(q.shape)}")
        q = q.to(dtype=torch.float32).contiguous()
        _check_device(q, self.device)
        nq, k = q.shape[0], int(k)
        if k <= 0:
            raise ValueError("k must be positive")
        D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        sel = self._selection(params)
        if nq and sel is None:
            st = torch.cuda.current_stream(q.device).cuda_stream
            nat.check(nat.lib.ivr_index_search_device(
                self._handle(), q.data_ptr(), nq, k, D.data_ptr(), I.data_ptr(), int(id_offset),
                self.search_path if path is None else path, st))
        elif nq:
            st = torch.cuda.current_stream(q.device).cuda_stream
            nat.check(nat.lib.ivr_index_search_selected_device(
                self._handle(), sel, q.data_ptr(), nq, k, D.data_ptr(), I.data_ptr(), int(id_offset), st))
        return D, I

    def search_keys_tensor(self, q, k: int, id_offset: int = 0, out=None, path: int | None = None,
                           params: SearchParameters | None = None):
        """Device-resident search that leaves the hits as packed 64-bit keys (int64 tensor [nq, k] holding
        ``order_preserving(score) << 32 | ~(row + id_offset)``, 0 = padding): the 8-byte-per-hit payload of the
        cross-shard exchange (``ShardedFlatIP``).  ``out`` may be a preallocated contiguous int64 [nq, k] tensor.
        ``params.sel`` selects stored rows, as in ``search``; unlike ``search`` the filtered call honours the search
        window (``set_window``): only the selected rows inside it are reported (``ivr_index_search_selected_keys_device``;
        ``path`` does not apply)."""
        import torch
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"search(x): expected [nq,{self.d}], got {tuple(q.shape)}")
        q = q.to(dtype=torch.float32).contiguous()
        _check_device(q, self.device)
        nq, k = q.shape[0], int(k)
        if k <= 0:
            raise ValueError("k must be positive")
        if out is None:
            out = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        elif out.shape != (nq, k) or out.dtype != torch.int64 or not out.is_contiguous():
            raise ValueError("out must be a contiguous int64 [nq, k] tensor")
        sel = self._selection(params)
        if nq and sel is None:
            st = torch.cuda.current_stream(q.device).cuda_stream
            nat.check(nat.lib.ivr_index_search_keys_device(
                self._handle(), q.data_ptr(), nq, k, out.data_ptr(), int(id_offset),
                self.search_path if path is None else path, st))
        elif nq:
            st = torch.cuda.current_stream(q.device).cuda_stream
            nat.check(nat.lib.ivr_index_search_selected_keys_device(
                self._handle(), sel, q.data_ptr(), nq, k, out.data_ptr(), int(id_offset), st))
        return out

    def range_search(self, x, radius: float, *, params: SearchParameters | None = None):
        """lims, D, I = index.range_search(x, radius): every stored row whose inner product with the query is
        strictly greater than ``radius``.  Query i's hits are ``D[lims[i]:lims[i+1]]`` (float32, descending, ties ->
        lower id) and ``I[lims[i]:lims[i+1]]`` (int64).  A CUDA tensor ``x`` runs ``range_search_tensor``.
        ``params.sel`` restricts the search to the ids it selects (``ivr_index_range_search_selected``)."""
        if _is_cuda_tensor(x):
            return self.range_search_tensor(x, radius, params=params)
        q = _as_f32_2d(x, self.d, "range_search(x)")
        radius = _radius(radius)
        nq = q.shape[0]
        lims = np.zeros(nq + 1, np.int64)
        cap = _range_capacity(nq, self.ntotal)
        sel = self._selection(params)
        while True:                                     # at most twice: the first call reports the exact total
            D = np.empty(cap, np.float32)
            I = np.empty(cap, np.int64)
            if sel is None:
                nat.check(nat.lib.ivr_index_range_search(self._handle(), q.ctypes.data, nq, radius, cap,
                                                         lims.ctypes.data, D.ctypes.data, I.ctypes.data))
            else:
                nat.check(nat.lib.ivr_index_range_search_selected(self._handle(), sel, q.ctypes.data, nq, radius, cap,
                                                                  lims.ctypes.data, D.ctypes.data, I.ctypes.data))
            total = int(lims[nq])
            if total <= cap:
                return lims, D[:total].copy(), I[:total].copy()
            cap = total

    def range_search_tensor(self, q, radius: float, id_offset: int = 0, params: SearchParameters | None = None):
        """Device-resident range search on torch's current stream; returns CUDA tensors (lims, D, I), ids =
        stored row + ``id_offset``.  Sizing the outputs reads ``lims[nq]`` back to the host once (twice when more
        hits than the first guess of the capacity turn up), so this call waits for the search to finish.
        ``params.sel``: as in ``range_search``."""
        import torch
        sel = self._selection(params)

        def call(q, radius, cap, lims, st):
            D = torch.empty(cap, dtype=torch.float32, device=q.device)
            I = torch.empty(cap, dtype=torch.int64, device=q.device)
            if sel is None:
                nat.check(nat.lib.ivr_index_range_search_device(self._handle(), q.data_ptr(), q.shape[0], radius, cap,
                                                                lims.data_ptr(), D.data_ptr(), I.data_ptr(),
                                                                int(id_offset), st))
            else:
                nat.check(nat.lib.ivr_index_range_search_selected_device(
                    self._handle(), sel, q.data_ptr(), q.shape[0], radius, cap, lims.data_ptr(), D.data_ptr(),
                    I.data_ptr(), int(id_offset), st))
            return D, I
        lims, total, (D, I) = self._range_device(q, radius, call)
        return lims, D[:total], I[:total]

    def range_search_keys_tensor(self, q, radius: float, id_offset: int = 0, params: SearchParameters | None = None):
        """``range_search_tensor`` with the hits left as packed 64-bit keys: returns CUDA int64 tensors (lims, keys),
        query i's hits are ``keys[lims[i]:lims[i+1]]`` holding ``order_preserving(score) << 32 | ~(row + id_offset)``
        in descending unsigned order (score descending, then lower id).  The per-rank step of
        ``ShardedFlatIP.range_search``; global ids must stay below 2^32.  ``params.sel``: as in
        ``search_keys_tensor``, the selected stored rows inside the search window
        (``ivr_index_range_search_selected_keys_device``)."""
        import torch
        sel = self._selection(params)

        def call(q, radius, cap, lims, st):
            keys = torch.empty(cap, dtype=torch.int64, device=q.device)
            if sel is None:
                nat.check(nat.lib.ivr_index_range_search_keys_device(self._handle(), q.data_ptr(), q.shape[0], radius,
                                                                     cap, lims.data_ptr(), keys.data_ptr(),
                                                                     int(id_offset), st))
            else:
                nat.check(nat.lib.ivr_index_range_search_selected_keys_device(
                    self._handle(), sel, q.data_ptr(), q.shape[0], radius, cap, lims.data_ptr(), keys.data_ptr(),
                    int(id_offset), st))
            return (keys,)
        lims, total, (keys,) = self._range_device(q, radius, call)
        return lims, keys[:total]

    def _range_device(self, q, radius, call):
        """Checks, then ``call(q, radius, capacity, lims, stream)`` with the first capacity guess and once more with
        the exact total when that overflowed.  Returns (lims, total hits, the outputs of the last call)."""
        import torch
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"range_search(x): expected [nq,{self.d}], got {tuple(q.shape)}")
        q = q.to(dtype=torch.float32).contiguous()
        _check_device(q, self.device)
        radius = _radius(radius)
        nq = q.shape[0]
        lims = torch.zeros(nq + 1, dtype=torch.int64, device=q.device)
        cap = _range_capacity(nq, self.ntotal)
        st = torch.cuda.current_stream(q.device).cuda_stream
        while True:
            out = call(q, radius, cap, lims, st)
            total = int(lims[nq].item())
            if total <= cap:
                return lims, total, out
            cap = total

    def range_self_join(self, radius: float):
        """lims, D, I = every pair of distinct stored rows whose inner product is strictly greater than ``radius``,
        over the rows of the search window (``set_window``) or all rows; n = their count.  Row i's hits (i = position
        in the window) are ``D[lims[i]:lims[i+1]]`` (float32, descending, ties -> lower id) and ``I[...]`` (int64
        stored row ids).  Each pair is scored once, so j is in row i's list iff i is in row j's, with the same score
        bits.  A row holding a NaN has no hits and is no hit."""
        radius = _radius(radius, "range_self_join")
        n = self._join_rows()
        lims = np.zeros(n + 1, np.int64)
        cap = _join_capacity(n)
        while True:                                     # at most twice: the first call reports the exact total
            D = np.empty(cap, np.float32)
            I = np.empty(cap, np.int64)
            nat.check(nat.lib.ivr_index_range_self_join(self._handle(), radius, cap, lims.ctypes.data,
                                                        D.ctypes.data, I.ctypes.data))
            total = int(lims[n])
            if total <= cap:
                return lims, D[:total].copy(), I[:total].copy()
            cap = total

    def range_self_join_tensor(self, radius: float):
        """Device-resident ``range_self_join`` on torch's current stream; returns CUDA tensors (lims, D, I).  Sizing
        the outputs reads ``lims[n]`` back to the host once (twice when more hits than the first capacity guess turn
        up), so this call waits for the join to finish."""
        import torch
        radius = _radius(radius, "range_self_join")
        n = self._join_rows()
        dev = torch.device("cuda", self.device)
        lims = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        cap = _join_capacity(n)
        st = torch.cuda.current_stream(dev).cuda_stream
        while True:
            D = torch.empty(cap, dtype=torch.float32, device=dev)
            I = torch.empty(cap, dtype=torch.int64, device=dev)
            nat.check(nat.lib.ivr_index_range_self_join_device(self._handle(), radius, cap, lims.data_ptr(),
                                                               D.data_ptr(), I.data_ptr(), st))
            total = int(lims[n].item())
            if total <= cap:
                return lims, D[:total], I[:total]
            cap = total

    @property
    def dpad(self) -> int:
        """The storage dimension: d padded to a multiple of 64 (the row stride of ``rows_f16_tensor``)."""
        return int(nat.lib.ivr_index_dpad(self._handle()))

    def rows_f16_tensor(self, first: int, n: int):
        """The stored fp16 rows [first, first + n) (whatever the search window) as a new CUDA float16 tensor
        [n, dpad], copied on torch's current stream: the rows ``ShardedFlatIP.range_self_join`` sends to a peer."""
        import torch
        dev = torch.device("cuda", self.device)
        out = torch.empty((int(n), self.dpad), dtype=torch.float16, device=dev)
        nat.check(nat.lib.ivr_index_rows_f16_device(self._handle(), int(first), int(n), out.data_ptr(),
                                                    torch.cuda.current_stream(dev).cuda_stream))
        return out

    def range_self_join_keys_tensor(self, radius: float, id_offset: int = 0):
        """``range_self_join_tensor`` with the hits left as packed 64-bit keys: CUDA int64 tensors (lims, keys), row
        i's hits are ``keys[lims[i]:lims[i+1]]`` holding ``order_preserving(score) << 32 | ~(partner + id_offset)``
        (partner = stored row), unsigned descending.  The diagonal step of ``ShardedFlatIP.range_self_join``; global
        ids must stay below 2^32."""
        import torch
        radius = _radius(radius, "range_self_join")
        n = self._join_rows()
        dev = torch.device("cuda", self.device)
        lims = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        cap = _join_capacity(n)
        st = torch.cuda.current_stream(dev).cuda_stream
        while True:                                     # at most twice: the first call reports the exact total
            keys = torch.empty(cap, dtype=torch.int64, device=dev)
            nat.check(nat.lib.ivr_index_range_self_join_keys_device(self._handle(), radius, cap, lims.data_ptr(),
                                                                    keys.data_ptr(), int(id_offset), st))
            total = int(lims[n].item())
            if total <= cap:
                return lims, keys[:total]
            cap = total

    def range_cross_join_keys_tensor(self, other_rows, other_first_id: int, radius: float, other_is_lower: bool,
                                     id_offset: int = 0):
        """Every pair (row i of the search window, row j of ``other_rows``) whose inner product is strictly greater
        than ``radius``, each pair scored once, as packed keys of GLOBAL ids: a window row's id is its stored row +
        ``id_offset``, other row j's is ``other_first_id + j``.  ``other_rows``: CUDA float16 [n_other, dpad] on this
        index's device (``rows_f16_tensor`` of another index).  ``other_is_lower``: the other rows' ids are below the
        window's.  Returns (lims_self [n_self + 1], keys_self, lims_other [n_other + 1], keys_other), each row's hits
        unsigned descending.  More than 2^31-1 hits in one call raise ``OverflowError``: split the other rows."""
        import torch
        radius = _radius(radius, "range_cross_join")
        if other_rows.dim() != 2 or other_rows.dtype != torch.float16 or other_rows.shape[1] != self.dpad:
            raise ValueError(f"other_rows: expected a float16 [n, {self.dpad}] tensor, got {other_rows.dtype} "
                             f"{tuple(other_rows.shape)}")
        other_rows = other_rows.contiguous()
        _check_device(other_rows, self.device)
        n, m = self._join_rows(), other_rows.shape[0]
        dev = other_rows.device
        lims = torch.zeros(n + m + 1, dtype=torch.int64, device=dev)
        cap = _cross_capacity(n, m)
        st = torch.cuda.current_stream(dev).cuda_stream
        while True:                                     # at most twice: the first call reports the exact total
            keys = torch.empty(cap, dtype=torch.int64, device=dev)
            nat.check(nat.lib.ivr_index_range_cross_join_keys_device(
                self._handle(), other_rows.data_ptr(), m, int(other_first_id), int(bool(other_is_lower)), radius, cap,
                lims.data_ptr(), keys.data_ptr(), int(id_offset), st))
            total = int(lims[n + m].item())
            if total <= cap:
                break
            if total > (1 << 31) - 1:
                raise OverflowError(f"range_cross_join: {total} hits, more than one call holds (2^31-1)")
            cap = total
        mid = int(lims[n].item())
        return lims[:n + 1], keys[:mid], lims[n:] - mid, keys[mid:total]

    def _selection(self, params):
        """The device selection of ``params.sel`` for this index's device and row count; None = unfiltered."""
        sel = getattr(params, "sel", None) if params is not None else None
        return None if sel is None else sel._selection(self.device, self.ntotal)

    def _join_rows(self) -> int:
        return self._window_count if self._window_count >= 0 else self.ntotal

    # -- instrumentation ---------------------------------------------------
    def set_timing(self, enable: bool = True):
        nat.check(nat.lib.ivr_index_set_timing(self._handle(), int(bool(enable))))

    def last_timing(self) -> dict:
        ms = (C.c_float * 3)()
        ln = (C.c_int * 3)()
        nat.check(nat.lib.ivr_index_last_timing(self._handle(), ms, ln))
        return {"score_ms": ms[0], "merge_ms": ms[1], "prep_ms": ms[2],
                "score_launches": ln[0], "merge_launches": ln[1], "prep_launches": ln[2],
                "path": {0: "empty", 1: "stream", 2: "mma"}.get(
                    nat.lib.ivr_index_last_path(self._handle()), "?"),
                "kernel": (nat.lib.ivr_index_last_kernel(self._handle()) or b"").decode()}


Index = IndexFlatIP


def IndexFlatL2(d):      # core.py:1204 offers it; the hot path in scope is inner product only
    raise NotImplementedError("ivr_b200 implements IndexFlatIP only (exact inner-product search)")


def IndexIVFFlat(*a, **k):   # unified_index.py:897-926 is dead code; the reference forces FlatIP (core.py:1209-1219)
    raise NotImplementedError("approximate IVF indexes are out of scope; use IndexFlatIP")


def normalize_L2(x) -> None:
    """In-place row L2 normalisation of a float32 [n,d] array (unified_index.py:1776)."""
    if not isinstance(x, np.ndarray) or x.dtype != np.float32 or x.ndim != 2:
        raise TypeError("normalize_L2 expects a 2-D float32 numpy array")
    if not x.flags.c_contiguous:
        raise ValueError("normalize_L2 expects a C-contiguous array")
    if x.shape[0]:
        nat.check(nat.lib.ivr_normalize_l2(nat.default_device(), x.ctypes.data, x.shape[0], x.shape[1]))


# -- no-op GPU plumbing the reference probes for (core.py:1057-1066, 1222-1228) --
class StandardGpuResources:
    pass


def index_cpu_to_gpu(res, device, index):
    return index


def index_gpu_to_cpu(index):
    return index


# -- persistence in the FAISS on-disk layout -------------------------------------------------
# The reference stores its index with ``faiss.write_index`` (unified_index.py:1811 -> the 'faiss_index' dataset of
# a .rvdb; core.py:987 -> index.faiss) and restores it with ``faiss.deserialize_index`` / ``read_index``
# (unified_index.py:1182-1188; core.py:1057, 4274-4278; system.py:2387).  For an ``IndexFlatIP`` the published
# FAISS layout (faiss/impl/index_write.cpp: fourcc, write_index_header, WRITEXBVECTOR) is, little-endian:
#
#     offset  size  field
#          0     4  fourcc "IxFI"  (inner product; "IxF2" = L2, "IxFl" = legacy flat)
#          4     4  int32  d
#          8     8  int64  ntotal
#         16    16  int64  dummy, dummy   (FAISS writes 1 << 20 twice)
#         32     1  bool   is_trained
#         33     4  int32  metric_type    (0 = METRIC_INNER_PRODUCT, 1 = METRIC_L2)
#         37     8  uint64 number of float32 values that follow (= ntotal * d)
#         45   4*n  float32 rows, row-major
#
# FAISS itself is absent from this image, so the layout is pinned by a hand-built buffer in the tests, not by a
# file FAISS wrote -- stated in DESIGN.md.
_FLAT_HEADER = 45
_FOURCC_IP, _FOURCC_L2, _FOURCC_LEGACY = b"IxFI", b"IxF2", b"IxFl"
_IO_CHUNK_ROWS = 1 << 16


def _flat_header(d: int, ntotal: int) -> bytes:
    import struct
    return (_FOURCC_IP + struct.pack("<iqqq?i", int(d), int(ntotal), 1 << 20, 1 << 20, True, METRIC_INNER_PRODUCT) +
            struct.pack("<Q", int(ntotal) * int(d)))


def _parse_flat_header(buf) -> tuple:
    import struct
    head = bytes(buf[:_FLAT_HEADER])
    if len(head) < _FLAT_HEADER:
        raise ValueError("not a FAISS index: shorter than a flat-index header")
    fourcc = head[:4]
    if fourcc == _FOURCC_L2:
        raise NotImplementedError("the stored index is an IndexFlatL2; ivr_b200 implements inner product only")
    if fourcc not in (_FOURCC_IP, _FOURCC_LEGACY):
        raise NotImplementedError(f"unsupported FAISS index type {fourcc!r}: only IndexFlatIP ('IxFI') is read "
                                  "(the reference forces every index type to FlatIP: core.py:1209-1219)")
    d, ntotal, _d1, _d2, _trained, metric = struct.unpack("<iqqq?i", head[4:37])
    (count,) = struct.unpack("<Q", head[37:45])
    if metric != METRIC_INNER_PRODUCT:
        raise NotImplementedError(f"metric_type {metric}: only METRIC_INNER_PRODUCT (0) is supported")
    if d <= 0 or ntotal < 0 or count != ntotal * d:
        raise ValueError(f"corrupt flat-index header: d={d} ntotal={ntotal} payload={count} floats")
    return d, ntotal


def _add_payload(index: "IndexFlatIP", payload: np.ndarray, ntotal: int, d: int) -> None:
    rows = payload.reshape(ntotal, d)
    index.reserve(ntotal)
    for s in range(0, ntotal, 1 << 20):              # ivr_index_add streams each block through pinned double buffers
        index.add(rows[s:s + (1 << 20)])


def serialize_index(index: IndexFlatIP) -> np.ndarray:
    """``faiss.serialize_index``: the index as a uint8 array in the FAISS IndexFlatIP layout (see above).  The
    payload is what the index holds: the added rows after their one rounding to fp16."""
    n, d = index.ntotal, index.d
    out = np.empty(_FLAT_HEADER + 4 * n * d, np.uint8)
    out[:_FLAT_HEADER] = np.frombuffer(_flat_header(d, n), np.uint8)
    if n:
        rows = out[_FLAT_HEADER:].view(np.float32).reshape(n, d)
        nat.check(nat.lib.ivr_index_reconstruct(index._handle(), 0, n, rows.ctypes.data))
    return out


def deserialize_index(buf, device: int | None = None) -> IndexFlatIP:
    """``faiss.deserialize_index`` for the IndexFlatIP layout: uint8 array / bytes -> index on the GPU."""
    a = np.frombuffer(buf, np.uint8) if isinstance(buf, (bytes, bytearray, memoryview)) else np.asarray(buf)
    if a.dtype != np.uint8 or a.ndim != 1:
        raise TypeError("deserialize_index expects a 1-D uint8 array (or bytes)")
    d, ntotal = _parse_flat_header(a)
    if a.size < _FLAT_HEADER + 4 * ntotal * d:
        raise ValueError("truncated FAISS index: payload shorter than the header announces")
    index = IndexFlatIP(d, device=device)
    if ntotal:
        payload = np.frombuffer(a, np.float32, count=ntotal * d, offset=_FLAT_HEADER) if a.flags.c_contiguous \
            else np.ascontiguousarray(a[_FLAT_HEADER:_FLAT_HEADER + 4 * ntotal * d]).view(np.float32)
        _add_payload(index, payload, ntotal, d)
    return index


def write_index(index: IndexFlatIP, path) -> None:
    """``faiss.write_index``: same bytes as ``serialize_index``, streamed to ``path`` in 64 k-row blocks."""
    n, d = index.ntotal, index.d
    with open(path, "wb") as f:
        f.write(_flat_header(d, n))
        blk = np.empty((min(_IO_CHUNK_ROWS, max(n, 1)), d), np.float32)
        for s in range(0, n, _IO_CHUNK_ROWS):
            m = min(_IO_CHUNK_ROWS, n - s)
            nat.check(nat.lib.ivr_index_reconstruct(index._handle(), s, m, blk.ctypes.data))
            f.write(memoryview(blk[:m]).cast("B"))


def read_index(path, flags: int = 0, device: int | None = None) -> IndexFlatIP:
    """``faiss.read_index`` for an IndexFlatIP file.  The float32 payload is memory-mapped (whatever ``flags`` says:
    ``IO_FLAG_MMAP`` is how core.py:4274 asks for it) and streamed page cache -> pinned double buffer -> HBM by
    ``ivr_index_add``, converted to fp16 rows on the device: no second host copy of the matrix is ever made."""
    with open(path, "rb") as f:
        d, ntotal = _parse_flat_header(f.read(_FLAT_HEADER))
    index = IndexFlatIP(d, device=device)
    if ntotal:
        payload = np.memmap(path, dtype=np.float32, mode="r", offset=_FLAT_HEADER, shape=(ntotal * d,))
        _add_payload(index, payload, ntotal, d)
        del payload
    return index


def _radius(radius, who: str = "range_search") -> float:
    r = float(radius)
    if r != r:
        raise ValueError(f"{who}: radius is NaN")
    return r


def _range_capacity(nq: int, ntotal: int) -> int:
    """First guess of a range search's hit count: 1024 per query (at least 1 M), never more than nq * ntotal."""
    return min(nq * ntotal, max(nq * 1024, 1 << 20), (1 << 31) - 1)


def _join_capacity(n: int) -> int:
    """First guess of a self-join's pool size: 64 entries per row (at least 1 M), never more than the n(n-1) ordered
    pairs.  A near-duplicate radius finds a handful of copies per row, so one call usually suffices; a radius that
    finds more costs one retry with the exact total, not a pool sized for range search's 1024 hits per row."""
    return min(n * (n - 1), max(64 * n, 1 << 20), (1 << 31) - 1)


def _cross_capacity(n: int, m: int) -> int:
    """First guess of a cross join's pool size: 64 entries per row of either side (at least 1 M), never more than
    the 2nm entries of every pair."""
    return min(2 * n * m, max(64 * (n + m), 1 << 20), (1 << 31) - 1)


def _is_cuda_tensor(x) -> bool:
    return type(x).__module__.startswith("torch") and getattr(x, "is_cuda", False)


def _check_device(t, device: int):
    if t.device.index != device:
        raise ValueError(f"tensor lives on cuda:{t.device.index}, index on cuda:{device}")
