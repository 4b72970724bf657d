"""Row-sharded exact search across the GPUs of one box (SURVEY.md section 8e).

One process per GPU (``torch.distributed``, NCCL over NVLink/NVSwitch).  The
embedding matrix is partitioned into contiguous row blocks at ``add`` time:
rank r owns global ids ``[offsets[r], offsets[r+1])``.  A search replicates the
queries, runs the local exact top-k on every GPU with GLOBAL ids
(``id_offset``) and leaves the hits as PACKED 64-bit keys (score and id in one
word, 8 bytes per hit -- the form the local search already holds before its
final unpack), exchanges the ``[nq, k]`` key lists and folds them with the
on-device k-way merge kernel (``ivr_topk_merge_keys_device``: one launch, no
scratch, no allocation).  Exactness: the global top-k is a subset of the union
of the local top-k lists.  The key holds a 32-bit id, so a sharded index is
limited to 2^32 - 1 rows in total (checked at ``add``).

The exchange (``exchange="peer"``, the default on GPUs with peer access) is our
own kernel over NVLink peer memory: every rank PUSHES its keys into a mailbox
in each peer's HBM and raises a flag; the receiver waits with a stream memory
operation, not with a spinning kernel (``csrc/exchange.cu``).  Push, wait and
merge run on a side stream, so ``search_async`` lets the scoring of batch i+1
start while slower peers still finish batch i -- the per-batch straggler wait
of a collective disappears from the throughput.  ``exchange="nccl"`` keeps the
ONE ``all_gather_into_tensor`` path (and is what injected CPU back-ends use).

Reference precedent for the semantics: ``_search_with_remote_index``
concatenates the per-shard hit lists, sorts and truncates (system.py:1721-1746;
api.py:1661-1694).  The merge here runs on raw inner products (descending); the
``1 - ip`` mapping of ``search_vectors`` is applied only at that facade.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import numpy as np


def partition_rows(n_total: int, world_size: int, weights=None, align: int = 1) -> np.ndarray:
    """Contiguous partition.  Balanced by default: offsets[r] = floor(r * n / world).  With ``weights`` (one
    positive number per rank, e.g. the scoring rates ``ShardedFlatIP.scoring_rate`` measured: GPUs under the same
    power cap differ by a few per cent, and with the pipelined exchange throughput is set by the SLOWEST rank's own
    work) rank r receives a share proportional to its weight; inner boundaries are rounded to ``align`` rows."""
    if weights is None:
        return np.array([(r * n_total) // world_size for r in range(world_size + 1)], dtype=np.int64)
    w = np.asarray(weights, dtype=np.float64)
    if w.shape != (world_size,) or not np.all(np.isfinite(w)) or np.any(w <= 0):
        raise ValueError("weights: one positive finite number per rank")
    cum = np.concatenate([[0.0], np.cumsum(w)]) / w.sum()
    off = np.rint(cum * n_total / align).astype(np.int64) * align
    off[0], off[-1] = 0, n_total
    return np.minimum(np.maximum.accumulate(off), n_total)


MAX_SHARDED_ROWS = (1 << 32) - 1          # the exchange key holds a 32-bit global row id
MAX_MERGE_PARTS = 64                      # runs one ivr_range_merge_keys_device call merges


def join_schedule(bounds, rank: int) -> list:
    """The work of rank ``rank`` in ``ShardedFlatIP.range_self_join`` (pure, the same answer on every rank).
    ``bounds`` [world + 1]: the windows ``W_r = [bounds[r], bounds[r+1])``.  Returns tasks ``(a, b, peer, c, d)``:
    score every pair of the rows ``[a, b)`` of this rank's window against the rows ``[c, d)`` of ``peer``'s.  Task 0 is
    the diagonal (``peer == rank``, the self-join of ``W_rank``); then, for every step 1 <= delta with 2 delta < N,
    the full block ``W_rank x W_(rank + delta) mod N``; and for an even N the block of the ranks r and r + N/2 split at
    ``m = bounds[r] + n_r // 2``: rank r scores ``[bounds[r], m) x W_(r + N/2)``, rank r + N/2 scores
    ``W_(r + N/2) x [m, bounds[r+1])``.  Every unordered pair of distinct rows is scored by exactly one rank, every
    rank has N // 2 cross tasks, and with equal windows every rank scores the same number of pairs."""
    b = [int(v) for v in np.asarray(bounds, dtype=np.int64)]
    N = len(b) - 1
    lo, hi = b[rank], b[rank + 1]
    tasks = [(lo, hi, rank, lo, hi)]
    for delta in range(1, (N + 1) // 2):
        p = (rank + delta) % N
        tasks.append((lo, hi, p, b[p], b[p + 1]))
    if N % 2 == 0:
        h = N // 2
        if rank < h:
            tasks.append((lo, lo + (hi - lo) // 2, rank + h, b[rank + h], b[rank + h + 1]))
        else:
            r = rank - h
            tasks.append((lo, hi, r, b[r] + (b[r + 1] - b[r]) // 2, b[r + 1]))
    return tasks


def rebalance_bounds(bounds, times_ms, nominal, margin: int, gain: float = 0.7, align: int = 1024) -> np.ndarray:
    """One step of the elastic-boundary controller (pure, deterministic: every rank computes the same answer from
    the same all-gathered times).  ``bounds`` [world + 1]: the boundaries the timed searches ran with; ``times_ms``
    [world]: every rank's mean local scoring time.  Rank r's rate is rows / time; its target share is proportional to
    its rate; the shares move ``gain`` of the way there.  Inner boundaries are rounded to ``align`` rows and stay
    within ``margin`` rows of the ``nominal`` partition -- the rows both neighbours hold."""
    bounds = np.asarray(bounds, dtype=np.int64)
    nominal = np.asarray(nominal, dtype=np.int64)
    t = np.asarray(times_ms, dtype=np.float64)
    n = np.diff(bounds).astype(np.float64)
    if len(t) != len(n) or np.any(n <= 0) or not np.all(np.isfinite(t)) or np.any(t <= 0):
        return bounds.copy()
    rate = n / t
    share = n + gain * (n.sum() * rate / rate.sum() - n)
    inner = bounds[0] + np.cumsum(share)[:-1]
    inner = np.rint(inner / align).astype(np.int64) * align
    inner = np.clip(inner, nominal[1:-1] - margin, nominal[1:-1] + margin)
    out = bounds.copy()
    out[1:-1] = inner
    return np.maximum.accumulate(out)


class _EventTimer:
    """Local scoring time of the last searches from CUDA events on the scoring stream (no host sync at record time)."""

    def __init__(self, depth: int):
        self.depth, self.ring = depth, {}

    def start(self, i):
        import torch
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ring[i] = [e, None]

    def stop(self, i):
        import torch
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ring[i][1] = e
        self.ring.pop(i - self.depth, None)

    def mean_ms(self, lo: int, hi: int) -> float:
        """Mean over searches [lo, hi); blocks the host until search hi - 1 has been scored."""
        self.ring[hi - 1][1].synchronize()
        return sum(self.ring[i][0].elapsed_time(self.ring[i][1]) for i in range(lo, hi)) / (hi - lo)


class _WallTimer(_EventTimer):
    """The same for host back-ends (CPU tests): the local search is synchronous."""

    def start(self, i):
        import time
        self.ring[i] = [time.perf_counter(), None]

    def stop(self, i):
        import time
        self.ring[i][1] = time.perf_counter()
        self.ring.pop(i - self.depth, None)

    def mean_ms(self, lo: int, hi: int) -> float:
        return 1e3 * sum(self.ring[i][1] - self.ring[i][0] for i in range(lo, hi)) / (hi - lo)


def _cuda_merge(device: int):
    from . import _native as nat

    def merge(keys_parts, k):
        import torch
        n_parts, nq, kk = keys_parts.shape
        D = torch.empty((nq, k), dtype=torch.float32, device=keys_parts.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=keys_parts.device)
        st = torch.cuda.current_stream(keys_parts.device).cuda_stream
        nat.check(nat.lib.ivr_topk_merge_keys_device(device, keys_parts.data_ptr(), n_parts, nq, k,
                                                     D.data_ptr(), I.data_ptr(), st))
        return D, I
    return merge


def _cuda_range_merge(keys_parts, lims_parts, total: int):
    """ivr_range_merge_keys_device on the current stream: keys_parts int64 [world, stride] (the all-gathered padded
    runs), lims_parts int64 [world, nq + 1], total = the sum of lims_parts[:, nq].  Returns (lims, D, I)."""
    import torch
    from . import _native as nat
    dev = lims_parts.device
    n_parts, stride = keys_parts.shape
    nq = lims_parts.shape[1] - 1
    lims = torch.empty(nq + 1, dtype=torch.int64, device=dev)
    D = torch.empty(total, dtype=torch.float32, device=dev)
    I = torch.empty(total, dtype=torch.int64, device=dev)
    nat.check(nat.lib.ivr_range_merge_keys_device(dev.index, keys_parts.data_ptr(), stride, lims_parts.data_ptr(),
                                                  n_parts, nq, lims.data_ptr(), D.data_ptr(), I.data_ptr(),
                                                  torch.cuda.current_stream(dev).cuda_stream))
    return lims, D, I


class _PeerExchange:
    """The mailbox of ``csrc/exchange.cu`` for one rank (ctypes over ``ivr_exchange_*``)."""

    SLOTS = 2

    def __init__(self, device: int, rank: int, world: int, capacity: int):
        from . import _native as nat
        self.nat, self.device, self.rank, self.world, self.capacity = nat, device, rank, world, int(capacity)
        h = C.c_void_p()
        nat.check(nat.lib.ivr_exchange_create(device, rank, world, self.SLOTS, self.capacity, C.byref(h)))
        self.h = h

    def ipc_handle(self) -> bytes:
        buf = (C.c_uint8 * self.nat.IVR_IPC_HANDLE_BYTES)()
        self.nat.check(self.nat.lib.ivr_exchange_ipc_handle(self.h, buf))
        return bytes(buf)

    def base(self) -> int:
        return int(self.nat.lib.ivr_exchange_base(self.h))

    def connect_ipc(self, handles: bytes) -> None:
        buf = (C.c_uint8 * len(handles)).from_buffer_copy(handles)
        self.nat.check(self.nat.lib.ivr_exchange_connect_ipc(self.h, buf))

    def connect_ptrs(self, bases) -> None:
        arr = (C.c_void_p * self.world)(*[C.c_void_p(int(b)) for b in bases])
        self.nat.check(self.nat.lib.ivr_exchange_connect_ptrs(self.h, arr))

    def push(self, keys_ptr: int, n: int, slot: int, epoch: int, stream: int) -> None:
        self.nat.check(self.nat.lib.ivr_exchange_push(self.h, keys_ptr, n, slot, epoch, stream))

    def wait(self, slot: int, epoch: int, stream: int) -> None:
        self.nat.check(self.nat.lib.ivr_exchange_wait(self.h, slot, epoch, stream))

    def slot_ptr(self, slot: int) -> int:
        return int(self.nat.lib.ivr_exchange_slot(self.h, slot))

    def close(self) -> None:
        if self.h:
            self.nat.lib.ivr_exchange_destroy(self.h)
            self.h = None


class PendingSearch:
    """Result of ``ShardedFlatIP.search_async``: the hits exist once the side stream has merged them.
    ``result()`` orders the CURRENT stream behind that and returns ``(D, I)``; with ``copy=False`` these are the
    index's own per-slot buffers, valid until two further searches have been issued.  ``to_host`` queues the
    device-to-host copies behind the merge (no wait on the scoring stream); ``synchronize`` blocks the host."""

    def __init__(self, D, I, done, stream):
        self.D, self.I, self._done, self._stream = D, I, done, stream

    def result(self, copy: bool = True):
        import torch
        if self._done is not None:
            torch.cuda.current_stream(self.D.device).wait_event(self._done)
        return (self.D.clone(), self.I.clone()) if copy else (self.D, self.I)

    def to_host(self, D_host, I_host) -> "PendingSearch":
        import torch
        if self._stream is None:
            D_host.copy_(self.D, non_blocking=True); I_host.copy_(self.I, non_blocking=True)
            self._done = torch.cuda.Event(); self._done.record()
            return self
        with torch.cuda.stream(self._stream):
            D_host.copy_(self.D, non_blocking=True); I_host.copy_(self.I, non_blocking=True)
            self._done = torch.cuda.Event(); self._done.record(self._stream)
        return self

    def synchronize(self) -> None:
        if self._done is not None:
            self._done.synchronize()


class ShardedFlatIP:
    """Exact inner-product index row-sharded over the ranks of a process group.

    ``local_index`` / ``merge`` can be injected (the CPU ``gloo`` tests exercise the
    partition / offset / gather logic with a stand-in backend that speaks the same packed-key
    protocol: ``search_keys_tensor(q, k, id_offset, out)`` and ``merge(keys [world, nq, k], k)``; for
    ``range_search`` also ``range_search_tensor`` / ``range_search_keys_tensor(q, radius, id_offset)`` and
    ``range_merge(keys [world, stride], lims [world, nq + 1], total)``; for filtered searches the same calls with
    ``params=`` holding a selector of stored rows, which must honour ``set_window``; for ``range_self_join``
    ``dpad``, ``rows_f16_tensor(first, n)``, ``range_self_join_tensor(radius)``,
    ``range_self_join_keys_tensor(radius, id_offset)`` and ``range_cross_join_keys_tensor(other_rows, other_first_id,
    radius, other_is_lower, id_offset)``, the last two over the rows of the window); by default they are the CUDA
    index and the CUDA merge kernels and fail loudly without a GPU.

    FILTERED SEARCH (``params=SearchParameters(sel=...)``): ``sel`` selects GLOBAL ids.  Each rank searches the
    selector's slice of the rows it stores (``IDSelector.shard``: one device selection per selector, built once and
    kept across boundary moves) under its current window, so the rows two ranks both store are reported by exactly
    one of them; the keys take the unfiltered exchange and merge unchanged.  A filtered search streams only the
    selected row tiles, so its time says nothing about a rank's row count: it sets the window but is not a timed
    search of the elastic controller (no ``balance_log`` entry, no step of the search counter).
    """

    def __init__(self, d: int, group=None, device: Optional[int] = None,
                 local_index=None, merge: Optional[Callable] = None, exchange: Optional[str] = None,
                 range_merge: Optional[Callable] = None):
        import os
        import torch.distributed as dist
        self.d = int(d)
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        cuda_backend = local_index is None
        if cuda_backend:
            from . import _native as nat
            from .faiss_compat import IndexFlatIP
            self.device = nat.default_device() if device is None else device
            local_index = IndexFlatIP(self.d, device=self.device)
            merge = merge or _cuda_merge(self.device)
        else:
            self.device = device
        self.local = local_index
        self._merge = merge
        self._range_merge = range_merge or _cuda_range_merge
        self.id_offset = 0
        self.ntotal_global = 0
        self._keys = None          # [nq, k] local keys and [world, nq, k] gathered keys, reused across searches
        self._gathered = None
        # exchange transport: "peer" (mailboxes over NVLink peer memory, pipelined) or "nccl" (one all-gather);
        # None = IVR_EXCHANGE, else peer for the CUDA back-end (falling back to nccl, on every rank together, when the
        # mailboxes cannot be mapped) and nccl for injected back-ends
        want = exchange or (os.environ.get("IVR_EXCHANGE") if cuda_backend else None) or ("peer" if cuda_backend else "nccl")
        if want not in ("peer", "nccl"):
            raise ValueError(f"exchange must be 'peer' or 'nccl', got {want!r}")
        self.exchange = want
        self._auto_exchange = exchange is None and "IVR_EXCHANGE" not in os.environ
        self._mail = None          # _PeerExchange, created at the first search (capacity = nq * k, regrown collectively)
        self._comm = None          # side stream: push -> wait -> merge of consecutive searches, in order
        self._step = 0
        self._slots = None         # per slot: keys, D, I, pushed-event
        # elastic shard boundaries (enabled by add_global / add_local with margin > 0)
        self._nominal = None       # [world + 1] partition the shards were built for
        self._bounds = None        # [world + 1] boundaries the NEXT search runs with (identical on every rank)
        self._margin = 0           # rows of each neighbour this rank also stores on either side
        self._period, self._gain = 8, 0.7
        self._nsearch = 0
        self._timer = None
        self._ctl, self._ctl_ready = None, False   # host-side (gloo) group the controller all-gathers the times on
        self.balance_log = []      # (search number, times_ms, rows per rank) of every controller step

    # ---- build ---------------------------------------------------------
    def add_global(self, x, weights=None, margin: int = 0) -> None:
        """Every rank passes the same [n, d] matrix (or a view of it); each keeps its block (``weights``: see
        ``partition_rows``; the same on every rank).  ``margin`` > 0 also keeps that many rows of either neighbour and
        turns on the elastic boundaries (``enable_elastic``)."""
        n = x.shape[0]
        off = partition_rows(n, self.world, weights)
        if self.ntotal_global != 0:
            raise RuntimeError("add_global supports one contiguous build; use add_local to append")
        if n > MAX_SHARDED_ROWS:
            raise ValueError(f"a sharded index holds at most 2^32 - 1 rows in total (got {n})")
        lo = max(0, int(off[self.rank]) - int(margin))
        hi = min(n, int(off[self.rank + 1]) + int(margin))
        self.id_offset = lo
        self.local.add(x[lo:hi])
        self.ntotal_global = n
        if margin > 0 and self.world > 1:
            self.enable_elastic(off, margin)

    def add_local(self, x_local, id_offset: int, ntotal_global: int) -> None:
        """This rank's pre-partitioned block (e.g. generated on device), with its global offset."""
        if int(ntotal_global) > MAX_SHARDED_ROWS:
            raise ValueError(f"a sharded index holds at most 2^32 - 1 rows in total (got {ntotal_global})")
        if self.local.ntotal == 0:
            self.id_offset = int(id_offset)
        self.local.add(x_local)
        self.ntotal_global = int(ntotal_global)

    def enable_elastic(self, nominal, margin: int, period: int = 8, gain: float = 0.7, ctl_group=None,
                       timer=None) -> None:
        """ELASTIC SHARD BOUNDARIES.  GPUs under the same power cap differ by a few per cent and drift with
        temperature; with the pipelined exchange the job runs at the pace of the slowest rank's own work.  Every rank
        therefore also stores ``margin`` rows of either neighbour (HBM is plentiful: + 2 * margin rows), which lets
        the boundary between two ranks move between two searches WITHOUT moving data: each search scores the rows
        ``[bounds[r], bounds[r+1])`` through ``ivr_index_set_window``.  Every ``period`` searches the ranks
        all-gather their mean local scoring times on a host-side group and apply ``rebalance_bounds`` -- the same
        deterministic step on every rank, so every row is scored by exactly one rank in every search and the hits
        stay exactly those of the static partition.

        ``nominal`` [world + 1]: the partition (the same on every rank); this rank must hold the rows
        ``[nominal[r] - margin, nominal[r+1] + margin)`` clipped to the index, starting at ``id_offset``.
        ``ctl_group``: a gloo group for the controller (created on first use otherwise -- collective)."""
        nominal = np.asarray(nominal, dtype=np.int64)
        if nominal.shape != (self.world + 1,) or nominal[0] != 0 or nominal[-1] != self.ntotal_global:
            raise ValueError("nominal: offsets [world + 1] from 0 to ntotal")
        lo = max(0, int(nominal[self.rank]) - int(margin))
        hi = min(self.ntotal_global, int(nominal[self.rank + 1]) + int(margin))
        if self.id_offset != lo or self.local.ntotal != hi - lo:
            raise ValueError(f"rank {self.rank} must hold rows [{lo}, {hi}) for margin {margin}: it holds "
                             f"[{self.id_offset}, {self.id_offset + self.local.ntotal})")
        self._nominal, self._bounds, self._margin = nominal, nominal.copy(), int(margin)
        self._period, self._gain = max(4, int(period)), float(gain)
        self._ctl, self._ctl_ready, self._nsearch = ctl_group, ctl_group is not None, 0
        self._timer = timer
        self.balance_log = []

    def _elastic_begin(self, q) -> int:
        """Controller step (every ``period`` searches) + the row window of this search.  Returns the search number."""
        import torch
        import torch.distributed as dist
        i, P = self._nsearch, self._period
        self._nsearch += 1
        if self._timer is None:
            self._timer = _EventTimer(2 * P) if getattr(q, "is_cuda", False) else _WallTimer(2 * P)
        if i >= P and i % P == 0:
            # the two latest searches may still be in flight: use the P - 2 before them (all run with these bounds)
            mine = torch.tensor([self._timer.mean_ms(i - P, i - 2)], dtype=torch.float64)
            if not self._ctl_ready:                      # the controller talks on a HOST-side group: a GPU collective
                try:                                     # would hold SMs the scoring kernels need while it waits
                    if dist.get_backend(self.group) != "gloo":
                        ranks = dist.get_process_group_ranks(self.group) if self.group is not None else None
                        self._ctl = dist.new_group(ranks=ranks, backend="gloo")
                    else:
                        self._ctl = self.group
                except Exception as e:                   # no host-side transport on this box (every rank alike):
                    import warnings                      # keep the boundaries where they are
                    warnings.warn(f"elastic shard boundaries disabled: cannot create the gloo control group ({e})")
                    self._period = 1 << 62
                    self._ctl_ready = True
                    return self._elastic_window(i)
                self._ctl_ready = True
            times = [torch.empty_like(mine) for _ in range(self.world)]
            dist.all_gather(times, mine, group=self._ctl)
            times = [float(t.item()) for t in times]
            self._bounds = rebalance_bounds(self._bounds, times, self._nominal, self._margin, self._gain)
            self.balance_log.append((i, times, np.diff(self._bounds).tolist()))
        return self._elastic_window(i)

    def _elastic_window(self, i: int) -> int:
        self._set_window()
        self._timer.start(i)
        return i

    def _set_window(self) -> None:
        """The local index scores the rows [bounds[r], bounds[r+1]) of the current elastic boundaries."""
        first = int(self._bounds[self.rank]) - self.id_offset
        self.local.set_window(first, int(self._bounds[self.rank + 1] - self._bounds[self.rank]))

    @property
    def ntotal(self) -> int:
        return self.ntotal_global

    @property
    def rows_per_rank(self):
        """Rows every rank scores in the NEXT search (elastic boundaries), or None for a static partition."""
        return None if self._bounds is None else [int(v) for v in np.diff(self._bounds)]

    def scoring_rate(self, q, k: int, reps: int = 8, warm: int = 3) -> float:
        """Rows per millisecond THIS rank's GPU scores for the batch ``q`` on its current shard (device-timed, local
        search only, no exchange).  All-gather the rates and pass them to ``partition_rows`` / ``add_global`` as
        ``weights`` to size the shards by measured speed."""
        self.local.set_timing(True)
        ms = []
        for i in range(warm + reps):
            self.local.search_keys_tensor(q, int(k), id_offset=self.id_offset)
            t = self.local.last_timing()
            if i >= warm:
                ms.append(t["score_ms"] + t["merge_ms"] + t["prep_ms"])
        self.local.set_timing(False)
        return float(self.local.ntotal) / (sum(ms) / len(ms))

    # ---- search --------------------------------------------------------
    def search(self, q, k: int, params=None):
        """q: [nq, d] tensor (CUDA for the product path), replicated on every rank.
        Returns (D [nq,k] float32 descending, I [nq,k] int64 global ids) on every rank.  ``params``: see
        ``search_async``."""
        return self.search_async(q, k, params=params).result(copy=True)

    def search_async(self, q, k: int, params=None) -> PendingSearch:
        """Queue one search and return at once.  The local scoring runs on the current stream; with the peer
        exchange the push / arrival wait / merge run on the index's side stream, so the NEXT ``search_async`` starts
        scoring while this one's exchange is still waiting for slower ranks.  Searches complete in issue order.

        ``params=SearchParameters(sel=...)`` restricts the search to the global ids ``sel`` selects: the k best of
        them, padded with -1 / -FLT_MAX (see the class docstring).  Like ``q``, ``params`` must be the same on every
        rank.  A filtered search takes a mailbox slot in issue order like any other, so filtered and unfiltered
        ``search_async`` calls may be mixed; it is not a timed search of the elastic controller."""
        import torch
        import torch.distributed as dist
        k = int(k)
        lp = self._local_params(q, params, k=k)
        kw = {} if lp is None else {"params": lp}
        if self.world == 1:
            D, I = self.local.search_tensor(q, k, id_offset=self.id_offset, **kw)
            return PendingSearch(D, I, None, None)
        nq = q.shape[0]
        if self.exchange == "peer" and nq > 0 and self._ensure_mailbox(nq * k, q.device):
            return self._search_peer(q, nq, k, kw)
        if self._keys is None or self._keys.shape != (nq, k) or self._keys.device != q.device:
            self._keys = torch.empty((nq, k), dtype=torch.int64, device=q.device)
            self._gathered = torch.empty((self.world, nq, k), dtype=torch.int64, device=q.device)
        i = self._local_begin(q, lp)
        self.local.search_keys_tensor(q, k, id_offset=self.id_offset, out=self._keys, **kw)
        if i >= 0:
            self._timer.stop(i)
        dist.all_gather_into_tensor(self._gathered.view(self.world * nq, k), self._keys, group=self.group)
        D, I = self._merge(self._gathered, k)
        return PendingSearch(D, I, None, None)

    def _local_params(self, q, params, k=None, radius=None):
        """The local index's ``params`` for a search with ``params`` (None = unfiltered): the selector's slice of the
        rows this rank stores.  The argument checks of a filtered search run here, before any collective or mailbox
        push; they depend only on arguments that are the same on every rank, so every rank raises alike."""
        sel = getattr(params, "sel", None) if params is not None else None
        if sel is None:
            return None
        from ._native import IVR_MAX_K
        from .faiss_compat import IDSelector, SearchParameters
        if not isinstance(sel, IDSelector):
            raise TypeError(f"params.sel must be an IDSelector, got {type(sel).__name__}")
        if q.dim() != 2 or q.shape[1] != self.d:
            raise ValueError(f"search(x): expected [nq,{self.d}], got {tuple(q.shape)}")
        if k is not None and not 1 <= k <= IVR_MAX_K:
            raise ValueError(f"k must be in 1..{IVR_MAX_K} (got {k})")
        if radius is not None and float(radius) != float(radius):
            raise ValueError("range_search: radius is NaN")
        return SearchParameters(sel=sel.shard(self.ntotal_global, self.id_offset))

    def _local_begin(self, q, lp) -> int:
        """Before a search's local scoring: the window of the current boundaries.  An unfiltered search is also a
        timed search of the elastic controller (returns its number, -1 without elastic boundaries); a filtered one
        (``lp`` not None) streams only its selected tiles and is not timed (returns -1)."""
        if self._bounds is None:
            return -1
        if lp is not None:
            self._set_window()
            return -1
        return self._elastic_begin(q)

    def range_search(self, q, radius: float, params=None):
        """Exact range search over the rows of every rank: every row whose inner product with a query is strictly
        greater than ``radius``.  q: [nq, d] tensor, the same on every rank (as for ``search``).  Returns tensors
        (lims int64 [nq + 1], D float32, I int64 global ids) on q's device, identical on every rank; query i's hits
        are ``D[lims[i]:lims[i+1]]``, descending, ties -> lower id.  Collective: every rank must call it.

        Each rank scores the rows it would score in a search (the current elastic boundaries, or its block) and keeps
        its hits as sorted packed keys (``range_search_keys_tensor``).  One all-gather carries every rank's ``lims``
        with a status, nq and the radius, so every rank learns every run length -- and raises the same error when any
        rank failed or was called with a different radius.  A second all-gather carries the runs, padded to the
        longest; ``ivr_range_merge_keys_device`` merges them on the current stream.  A range search is not a timed
        search: it leaves the elastic controller and ``balance_log`` alone.

        The exchange always uses these collectives over ``group``, never the peer mailboxes (their slots are sized
        for nq * k and pipelined).  So ``range_search`` may be called between ``search_async`` calls: its scoring
        queues on the current stream behind theirs, it blocks the host until its run lengths are known, it takes no
        mailbox slot, and the pending searches still complete in issue order.

        ``params=SearchParameters(sel=...)``: only the global ids ``sel`` selects (see the class docstring).  The
        status row then also carries the selector's fingerprint (its selected count and a hash of its words), so ranks
        called with different selectors all raise the same ``ValueError``.  ``params`` must be given on every rank or
        on none."""
        import torch
        import torch.distributed as dist
        lp = self._local_params(q, params, radius=radius)
        kw = {} if lp is None else {"params": lp}
        if self._bounds is not None:
            self._set_window()
        if self.world == 1:
            return self.local.range_search_tensor(q, radius, id_offset=self.id_offset, **kw)
        nq, dev = q.shape[0], q.device
        if nq == 0:                                      # replicated queries: every rank takes this branch
            return (torch.zeros(1, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.float32, device=dev),
                    torch.empty(0, dtype=torch.int64, device=dev))
        # every rank reaches both collectives whatever happens locally: a local failure travels as a status
        err, rbits = None, 0
        try:
            rbits = int(np.float32(radius).view(np.int32))
            lims, keys = self.local.range_search_keys_tensor(q, radius, id_offset=self.id_offset, **kw)
        except Exception as e:
            err = e
            lims, keys = torch.zeros(nq + 1, dtype=torch.int64, device=dev), None
        # a batch of another size would also change the row length: queries must be replicated, as for search
        fp = [] if lp is None else list(params.sel.fingerprint(self.ntotal_global))
        row = torch.cat([lims, torch.tensor([0 if err is None else 1, nq, rbits] + fp, dtype=torch.int64, device=dev)])
        rows = torch.empty((self.world, nq + 4 + len(fp)), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(rows.view(-1), row, group=self.group)
        host = rows.cpu().numpy()
        failed = np.nonzero(host[:, nq + 1])[0]
        if failed.size:
            raise RuntimeError(f"range_search failed on rank {int(failed[0])}") from err
        differ = np.nonzero((host[:, nq + 2] != host[0, nq + 2]) | (host[:, nq + 3] != host[0, nq + 3]))[0]
        if differ.size:
            def call(r):
                return f"nq={int(host[r, nq + 2])} radius={float(np.int32(host[r, nq + 3]).view(np.float32))}"
            raise ValueError(f"range_search: rank {int(differ[0])} was called with {call(int(differ[0]))}, "
                             f"rank 0 with {call(0)}")
        if fp:
            differ = np.nonzero(np.any(host[:, nq + 4:] != host[0, nq + 4:], axis=1))[0]
            if differ.size:
                def call(r):
                    return f"a selector of {int(host[r, nq + 4])} ids (hash {int(host[r, nq + 5]) & ((1 << 64) - 1):016x})"
                raise ValueError(f"range_search: rank {int(differ[0])} was called with {call(int(differ[0]))}, "
                                 f"rank 0 with {call(0)}")
        totals = host[:, nq]
        stride = int(totals.max())
        gathered = torch.empty((self.world, 0), dtype=torch.int64, device=dev)
        if stride > 0:                                   # every rank knows stride: all skip or all gather
            fail = self.world
            try:
                gathered = torch.empty((self.world, stride), dtype=torch.int64, device=dev)
                mine = torch.empty(stride, dtype=torch.int64, device=dev)
                mine[:keys.numel()] = keys
            except RuntimeError:                         # torch.OutOfMemoryError included
                fail = self.rank
            flag = torch.tensor([fail], dtype=torch.int64, device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
            if int(flag.item()) < self.world:
                raise RuntimeError(f"range_search: rank {int(flag.item())} cannot allocate the exchange buffers "
                                   f"({self.world} x {stride} keys)")
            dist.all_gather_into_tensor(gathered.view(-1), mine, group=self.group)
        return self._range_merge(gathered, rows[:, :nq + 1].contiguous(), int(totals.sum()))

    def range_self_join(self, radius: float, gather: bool = False):
        """Exact range self-join over the rows of every rank: for every row, the other rows whose inner product with it
        is strictly greater than ``radius``.  Returns tensors (lims int64 [n_local + 1], D float32, I int64 global ids)
        for the rows of this rank's window (the current elastic boundaries, or its block), on the local index's
        device: row i's hits are ``D[lims[i]:lims[i+1]]``, descending, ties -> lower id; the rows equal those of the
        single-index ``range_self_join`` over all rows, bit for bit.  ``gather=True`` returns the whole result, every
        row in global order, on every rank.  Collective: every rank must call it, with the same radius.

        Each rank scores the tasks of ``join_schedule``: the self-join of its window, then one block of another rank's
        rows per round, received through ``batch_isend_irecv`` and scored by the local cross join (the window's rows
        against the received ones, each pair once).  The hits of the other side go back to their owner; every rank
        merges the runs over its rows with ``range_merge``.  One all-gather before any row moves carries the radius and
        the windows, one before any hit moves every run length and a status, so all ranks raise the same error when
        one was called with another radius or one failed.  The join is not a timed search: ``balance_log``, the
        search counter and the peer mailboxes are left alone; the window of the current boundaries is restored."""
        import torch
        import torch.distributed as dist
        from .faiss_compat import _radius
        radius = _radius(radius, "range_self_join")
        if 1 + 2 * (self.world // 2) > MAX_MERGE_PARTS:  # the window's own join, then two runs per round
            raise ValueError(f"range_self_join: {self.world} ranks give each rank {1 + 2 * (self.world // 2)} runs "
                             f"to merge, more than the merge takes ({MAX_MERGE_PARTS})")
        if self._bounds is not None:
            self._set_window()
        if self.world == 1:
            lims, D, I = self.local.range_self_join_tensor(radius)
            return lims, D, I + self.id_offset
        dev = torch.device("cpu") if self.device is None else torch.device("cuda", self.device)
        if self._bounds is not None:
            lo, hi = int(self._bounds[self.rank]), int(self._bounds[self.rank + 1])
        else:
            lo, hi = self.id_offset, self.id_offset + self.local.ntotal
        rbits = int(np.float32(radius).view(np.int32))
        agree = torch.empty((self.world, 3), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(agree.view(-1), torch.tensor([rbits, lo, hi], dtype=torch.int64, device=dev),
                                    group=self.group)
        host = agree.cpu().numpy()
        differ = np.nonzero(host[:, 0] != host[0, 0])[0]
        if differ.size:
            def rad(r):
                return float(np.int32(host[r, 0]).view(np.float32))
            raise ValueError(f"range_self_join: rank {int(differ[0])} was called with radius={rad(int(differ[0]))}, "
                             f"rank 0 with radius={rad(0)}")
        bounds = np.concatenate([host[:, 1], host[-1:, 2]])
        if bounds[0] != 0 or bounds[-1] != self.ntotal_global or np.any(host[1:, 1] != host[:-1, 2]):
            raise ValueError(f"range_self_join: the ranks' windows {host[:, 1:].tolist()} do not tile "
                             f"[0, {self.ntotal_global})")
        sched = [join_schedule(bounds, r) for r in range(self.world)]
        mine, n_rounds = sched[self.rank], len(sched[self.rank]) - 1
        parts, back, err = [], [], None                 # parts: runs (a, b, lims, keys) over this rank's rows [a, b)
        try:
            try:
                self.local.set_window(lo - self.id_offset, hi - lo)
                parts.append((lo, hi) + tuple(self.local.range_self_join_keys_tensor(radius, id_offset=self.id_offset)))
            except Exception as e:                      # reported in the run-length all-gather
                err = e
            for k in range(n_rounds):
                a, b, p, c, d = mine[k + 1]
                needs = [(q,) + sched[q][k + 1][3:] for q in range(self.world) if sched[q][k + 1][2] == self.rank]
                fail = self.world
                try:
                    recv = torch.empty((d - c, self.local.dpad), dtype=torch.float16, device=dev)
                    sends = [(q, self.local.rows_f16_tensor(s - self.id_offset, e - s)) for q, s, e in needs]
                except RuntimeError:                    # torch.OutOfMemoryError and the native errors included
                    fail = self.rank
                self._agree(fail, dev, "cannot allocate the row exchange buffers")
                self._p2p([(dist.irecv, recv, p)] + [(dist.isend, t, q) for q, t in sends])
                if err is not None:
                    back.append((p, c, d, None, None))
                    continue
                try:
                    self.local.set_window(a - self.id_offset, b - a)
                    runs, lims_o, keys_o = self._cross_runs(recv, c, radius, c < a)
                    parts += [(a, b, L, K) for L, K in runs]
                    back.append((p, c, d, lims_o, keys_o))
                except Exception as e:
                    err = e
                    back.append((p, c, d, None, None))
                del recv, sends
        finally:
            if self._bounds is not None:
                self._set_window()
            else:
                self.local.set_window()
        # every run length before any hit moves: status, then the hits this rank sends back in each round
        counts = [0 if err is None else 1] + [0 if L is None else int(K.numel()) for _, _, _, L, K in back]
        allc = torch.empty((self.world, 1 + n_rounds), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allc.view(-1), torch.tensor(counts, dtype=torch.int64, device=dev),
                                    group=self.group)
        allc = allc.cpu().numpy()
        failed = np.nonzero(allc[:, 0])[0]
        if failed.size:
            raise RuntimeError(f"range_self_join failed on rank {int(failed[0])}") from err
        for k in range(n_rounds):                       # the other side's runs go back to their owner
            p, c, d, L, K = back[k]
            needs = [(q,) + sched[q][k + 1][3:] for q in range(self.world) if sched[q][k + 1][2] == self.rank]
            fail, recvs = self.world, []
            try:
                recvs = [(q, s, e, torch.empty(e - s + 1 + int(allc[q, 1 + k]), dtype=torch.int64, device=dev))
                         for q, s, e in needs]
                payload = torch.cat([L, K])
            except RuntimeError:
                fail = self.rank
            self._agree(fail, dev, "cannot allocate the hit exchange buffers")
            self._p2p([(dist.isend, payload, p)] + [(dist.irecv, t, q) for q, _, _, t in recvs])
            parts += [(s, e, t[:e - s + 1], t[e - s + 1:]) for _, s, e, t in recvs]
        # the merge can fail on one rank only (memory, or more runs than the merge takes after overflow splits):
        # every rank learns it before any rank leaves or enters the gather
        fail, err = self.world, None
        try:
            if len(parts) > MAX_MERGE_PARTS:
                raise RuntimeError(f"{len(parts)} runs, more than the merge takes ({MAX_MERGE_PARTS})")
            lims, D, I = self._merge_runs(parts, lo, hi, dev)
        except RuntimeError as e:                       # torch.OutOfMemoryError and the native errors included
            fail, err = self.rank, e
        self._agree(fail, dev, "could not merge its runs", err)
        return self._gather_join(lims, D, I, dev) if gather else (lims, D, I)

    def _cross_runs(self, other, first: int, radius: float, lower: bool):
        """The local cross join of the window against ``other`` (rows of global ids ``first + j``): (runs over the
        window, lims over the other rows, their keys).  A call that would hold more than 2^31-1 hits is split over
        halves of the other rows; each half adds one run over the window, and the halves' runs over the other rows
        concatenate into one."""
        try:
            ls, ks, lo_, ko = self.local.range_cross_join_keys_tensor(other, first, radius, lower,
                                                                      id_offset=self.id_offset)
            return [(ls, ks)], lo_, ko
        except OverflowError:
            m = other.shape[0]
            if m < 2:
                raise
            h = m // 2
            r1, l1, k1 = self._cross_runs(other[:h], first, radius, lower)
            r2, l2, k2 = self._cross_runs(other[h:], first + h, radius, lower)
            import torch
            return r1 + r2, torch.cat([l1[:-1], l2 + l1[-1]]), torch.cat([k1, k2])

    def _agree(self, fail: int, dev, what: str, err=None) -> None:
        """All ranks learn whether any failed a local step (``fail`` = this rank, else ``world``) and raise together,
        naming the lowest such rank."""
        import torch
        import torch.distributed as dist
        flag = torch.tensor([fail], dtype=torch.int64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) < self.world:
            raise RuntimeError(f"range_self_join: rank {int(flag.item())} {what}") from err

    def _p2p(self, ops) -> None:
        """One batch of point-to-point transfers (op, tensor, group rank); empty tensors are skipped (both sides
        know every size)."""
        import torch.distributed as dist
        ops = [dist.P2POp(op, t, p if self.group is None else dist.get_global_rank(self.group, p), self.group)
               for op, t, p in ops if t.numel() > 0]
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    def _merge_runs(self, parts, lo: int, hi: int, dev):
        """``range_merge`` of runs over sub-ranges of the rows [lo, hi): each run's lims embedded in [n + 1] entries,
        zeros before its rows and its total after them, its keys padded to the longest run."""
        import torch
        n = hi - lo
        stride = max([int(K.numel()) for _, _, _, K in parts] + [0])
        keys_parts = torch.zeros((len(parts), stride), dtype=torch.int64, device=dev)
        lims_parts = torch.zeros((len(parts), n + 1), dtype=torch.int64, device=dev)
        total = 0
        for i, (a, b, L, K) in enumerate(parts):
            keys_parts[i, :K.numel()] = K
            lims_parts[i, a - lo:b - lo + 1] = L
            lims_parts[i, b - lo + 1:] = int(K.numel())
            total += int(K.numel())
        return self._range_merge(keys_parts, lims_parts, total)

    def _gather_join(self, lims, D, I, dev):
        """Every rank's (lims, D, I) on every rank, in rank (= global row) order."""
        import torch
        import torch.distributed as dist
        sizes = torch.empty((self.world, 2), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sizes.view(-1), torch.tensor([lims.numel() - 1, D.numel()], dtype=torch.int64,
                                                                 device=dev), group=self.group)
        sizes = sizes.cpu().numpy()
        rmax, hmax = int(sizes[:, 0].max()) + 1, int(sizes[:, 1].max())
        out = []
        for t, m in ((lims, rmax), (D, hmax), (I, hmax)):
            buf = torch.zeros(m, dtype=t.dtype, device=dev)
            buf[:t.numel()] = t
            allb = torch.empty((self.world, m), dtype=t.dtype, device=dev)
            dist.all_gather_into_tensor(allb.view(-1), buf, group=self.group)
            out.append(allb)
        L_all, D_all, I_all = out
        base = np.concatenate([[0], np.cumsum(sizes[:, 1])])
        lims_g = torch.cat([L_all[r, :int(sizes[r, 0])] + int(base[r]) for r in range(self.world)] +
                           [torch.tensor([int(base[-1])], dtype=torch.int64, device=dev)])
        D_g = torch.cat([D_all[r, :int(sizes[r, 1])] for r in range(self.world)])
        I_g = torch.cat([I_all[r, :int(sizes[r, 1])] for r in range(self.world)])
        return lims_g, D_g, I_g

    # ---- peer-memory exchange (csrc/exchange.cu) ---------------------------
    def _ensure_mailbox(self, n_entries: int, device) -> bool:
        """Collective: (re)creates the mailboxes when the payload outgrows them and maps the peers' through CUDA
        IPC.  Every rank calls it with the same size (queries are replicated).  Returns False -- on every rank --
        when some rank cannot map a peer and the transport was chosen automatically (then NCCL takes over)."""
        import torch
        import torch.distributed as dist
        if self._mail is not None and n_entries <= self._mail.capacity:
            return True
        from . import _native as nat
        if self._mail is not None:                      # nobody may still be writing into the old mailboxes
            torch.cuda.synchronize(device)
            dist.barrier(group=self.group)
            self._mail.close()
            self._mail = None
        # every rank reaches both collectives below whatever happens locally: a rank that cannot create or map a
        # mailbox reports it through the all-reduce instead of leaving the others waiting
        mail, err = None, None
        try:
            mail = _PeerExchange(self.device, self.rank, self.world, n_entries)
            handle = mail.ipc_handle()
        except nat.NativeError as e:
            err, handle = e, bytes(nat.IVR_IPC_HANDLE_BYTES)
        mine = torch.frombuffer(bytearray(handle), dtype=torch.uint8).to(device)
        allh = torch.empty((self.world, nat.IVR_IPC_HANDLE_BYTES), dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(allh, mine, group=self.group)
        if err is None:
            try:
                mail.connect_ipc(allh.cpu().numpy().tobytes())
            except nat.NativeError as e:
                err = e
        flag = torch.tensor([0 if err else 1], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            if mail is not None:
                mail.close()
            if not self._auto_exchange:
                raise RuntimeError(f"exchange='peer' is not available on every rank (rank {self.rank}: {err or 'ok'})")
            self.exchange = "nccl"
            return False
        self._mail = mail
        self._step = 0
        self._slots = None
        if self._comm is None:
            self._comm = torch.cuda.Stream(device=device)
        return True

    def _search_peer(self, q, nq: int, k: int, kw) -> PendingSearch:
        import torch
        S = _PeerExchange.SLOTS
        if self._slots is None or self._slots[0]["keys"].shape != (nq, k) or self._slots[0]["keys"].device != q.device:
            if self._slots is not None:
                self._comm.synchronize()
            self._slots = [{"keys": torch.empty((nq, k), dtype=torch.int64, device=q.device),
                            "D": torch.empty((nq, k), dtype=torch.float32, device=q.device),
                            "I": torch.empty((nq, k), dtype=torch.int64, device=q.device),
                            "pushed": None} for _ in range(S)]
        slot, epoch = self._step % S, self._step // S + 1
        self._step += 1
        b = self._slots[slot]
        cur = torch.cuda.current_stream(q.device)
        if b["pushed"] is not None:                     # the push of search (step - S) has read this keys buffer
            cur.wait_event(b["pushed"])
        i = self._local_begin(q, kw.get("params"))
        self.local.search_keys_tensor(q, k, id_offset=self.id_offset, out=b["keys"], **kw)
        if i >= 0:
            self._timer.stop(i)
        scored = torch.cuda.Event()
        scored.record(cur)
        comm = self._comm
        comm.wait_event(scored)                          # also orders the merge behind every consumer of D / I[slot]
        cs = comm.cuda_stream                            # that was queued on the current stream before this search
        self._mail.push(b["keys"].data_ptr(), nq * k, slot, epoch, cs)
        b["pushed"] = torch.cuda.Event()
        b["pushed"].record(comm)
        self._mail.wait(slot, epoch, cs)
        from . import _native as nat
        nat.check(nat.lib.ivr_topk_merge_keys_device(self.device, self._mail.slot_ptr(slot), self.world, nq, k,
                                                     b["D"].data_ptr(), b["I"].data_ptr(), cs))
        done = torch.cuda.Event()
        done.record(comm)
        return PendingSearch(b["D"], b["I"], done, comm)

    def close(self) -> None:
        """Collective: waits for every rank's outstanding exchanges, then frees the mailbox."""
        if self._mail is not None:
            import torch
            import torch.distributed as dist
            torch.cuda.synchronize()
            dist.barrier(group=self.group)
            self._mail.close()
            self._mail = None


# ---------------------------------------------------------------------------
# Dedup across GPUs: whole videos per rank, no data-path collective (SURVEY.md section 8e)
# ---------------------------------------------------------------------------
def partition_units(lengths, world_size: int) -> np.ndarray:
    """Contiguous assignment of indivisible units (videos) to ranks, balanced by frame count:
    unit u goes to the rank whose ideal frame range contains the unit's midpoint.  Returns unit
    offsets [world_size + 1]; rank r owns units [off[r], off[r+1])."""
    lengths = np.asarray(lengths, dtype=np.int64)
    total = int(lengths.sum())
    off = np.zeros(world_size + 1, dtype=np.int64)
    if total == 0 or len(lengths) == 0:
        off[1:] = len(lengths)
        return off
    mid = np.cumsum(lengths) - lengths / 2.0
    owner = np.minimum((mid * world_size / total).astype(np.int64), world_size - 1)
    for r in range(world_size):
        off[r + 1] = int(np.searchsorted(owner, r, side="right"))
    return off


class ShardedFrameFilter:
    """Near-duplicate pruning of many videos on several GPUs: every rank prunes ITS videos (scene split on
    the consecutive cosine inside each video, then the windowed rule inside each scene -- filter.py:142-315)
    with one fused ``ivr_frame_filter`` call per video; videos are never split, so no halo and no
    collective on the data path.  ``gather`` (optional, control plane) collects the kept indices.

    ``ops`` is the module providing ``calculate_similarities``, ``detect_scene_transitions``,
    ``group_into_scenes`` and ``apply_similarity_filtering_to_scenes`` (default: ``frame_filter``, the
    CUDA path; the world-size-2 gloo test injects the oracle)."""

    def __init__(self, window: int = 8, threshold: float = 0.95, transition_threshold: float = 0.75,
                 min_scene_length: int = 2, group=None, ops=None):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.transition_threshold, self.min_scene_length = float(transition_threshold), int(min_scene_length)
        self.config = {"enable_similarity_filtering": True, "similarity_threshold": float(threshold),
                       "similarity_window_size": int(window), "use_advanced_similarity_filtering": True,
                       "min_frame_distance": 1}
        if ops is None:
            from . import frame_filter as ops
        self.ops = ops

    def my_units(self, video_bounds):
        off = partition_units([e - s + 1 for s, e in video_bounds], self.world)
        return int(off[self.rank]), int(off[self.rank + 1])

    def filter_videos(self, embeddings, video_bounds) -> list:
        """Kept GLOBAL frame indices of this rank's videos.  ``video_bounds``: inclusive (start, end) per video,
        ascending and non-overlapping; ``embeddings`` may be the whole matrix (only this rank's range is read)."""
        lo, hi = self.my_units(video_bounds)
        if lo >= hi:
            return []
        if hasattr(self.ops, "FrameFilter"):                        # CUDA path: one fused call per video -- the frames cross
            f = self.ops.FrameFilter(window=self.config["similarity_window_size"],     # PCIe once, scene split and greedy
                                     threshold=self.config["similarity_threshold"],    # rule run on the device, and a scene
                                     transition_threshold=self.transition_threshold,   # can never cross a video boundary
                                     min_scene_length=self.min_scene_length)
            kept: list = []
            for vs, ve in video_bounds[lo:hi]:
                kept.extend((f.apply_filters(embeddings[vs:ve + 1]) + vs).tolist())
            return kept
        s0, e1 = video_bounds[lo][0], video_bounds[hi - 1][1]
        x = embeddings[s0:e1 + 1]
        sims = self.ops.calculate_similarities(x)                   # one pass over the rank's frames
        scenes = []
        for vs, ve in video_bounds[lo:hi]:
            inside = sims[vs - s0:ve - s0]                          # cosines between frames of THIS video only
            cuts = self.ops.detect_scene_transitions(inside, self.transition_threshold)
            for a, b in self.ops.group_into_scenes(cuts, ve - vs + 1, self.min_scene_length):
                scenes.append((a + vs - s0, b + vs - s0))
        rows = list(range(s0, e1 + 1))
        return list(self.ops.apply_similarity_filtering_to_scenes(x, rows, scenes, self.config)[1])

    def gather(self, kept_local: list) -> list:
        """All ranks' kept indices in video order (control plane: a Python-object all-gather)."""
        if self.world == 1:
            return list(kept_local)
        import torch.distributed as dist
        parts = [None] * self.world
        dist.all_gather_object(parts, list(kept_local), group=self.group)
        return [i for p in parts for i in p]
