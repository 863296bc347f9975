"""Row-sharded flat index over several GPUs of one box (one process per GPU).

New relative to the reference (which is single-process, SURVEY.md section 2.2): the database is
split by rows, every rank scores ALL queries against its shard with the single-GPU engine,
the per-shard (D, I) are exchanged with one NCCL all-gather over NVLink and merged per query
on the device (knn_merge_topk_dev).  Ids stay global row numbers, so (D, I) is still a
drop-in for the reference's consumers.  Tie rule is shard-count invariant: equal score ->
lower global id.

``index_factory`` / ``merge_fn`` exist so that the host logic (row split, id mapping,
collective, merge call) can be exercised under gloo on CPU in tests.
"""
from __future__ import annotations

import numpy as np


class _DeviceBytes:
    """A raw device allocation presented to torch through the CUDA array interface (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


class PeerExchange:
    """Exchange buffers of all ranks of one box, mapped into every rank with CUDA IPC (NVLink peer memory).

    Each rank owns one cudaMalloc'ed buffer laid out [I_local | I_merged | D_local | D_merged] for the current
    (nq, k); ``tables`` gives, per region, a host array with the address of that region in every rank's buffer
    as seen from THIS rank.  All methods are collective over ``group``."""

    def __init__(self, dist, group, rank: int, world: int, device: int):
        import torch

        from . import _lib

        self._dist, self.group, self.rank, self.world, self.device = dist, group, rank, world, device
        self._lib = _lib.load()
        self._check = _lib.check
        self.capacity = 0
        self.own = None          # ctypes.c_void_p
        self.bases = []          # address of every rank's buffer in this process
        self._own_tensor = None
        backend = dist.get_backend(group)
        self._stream_ordered = backend == "nccl"
        self._token = torch.zeros(1, device=torch.device("cuda", device)) if self._stream_ordered else None

    def barrier(self) -> None:
        """Everything enqueued before it on every rank happens before anything enqueued after it on any rank."""
        import torch

        if self._stream_ordered:
            self._dist.all_reduce(self._token, group=self.group)  # on the current stream, no host sync
        else:
            torch.cuda.synchronize(self.device)
            self._dist.barrier(group=self.group)

    def _release(self) -> None:
        import ctypes

        if self.own is None:
            return
        self.barrier()
        import torch

        torch.cuda.synchronize(self.device)
        for r, b in enumerate(self.bases):
            if r != self.rank:
                self._check(self._lib.knn_peer_handle_close(ctypes.c_void_p(b)))
        self._dist.barrier(group=self.group)  # nobody maps the buffer any more
        self._check(self._lib.knn_peer_buffer_free(self.own))
        self.own, self.bases, self._own_tensor, self.capacity = None, [], None, 0

    def ensure(self, nbytes: int) -> None:
        import ctypes

        import torch

        if nbytes <= self.capacity:
            return
        self._release()
        cap = 1 << 20
        while cap < nbytes:
            cap *= 2
        own = ctypes.c_void_p()
        self._check(self._lib.knn_peer_buffer_alloc(ctypes.byref(own), cap, self.device))
        handle = (ctypes.c_ubyte * 64)()
        self._check(self._lib.knn_peer_handle_get(own, handle))
        handles = [None] * self.world
        self._dist.all_gather_object(handles, bytes(handle), group=self.group)
        bases = []
        for r, h in enumerate(handles):
            if r == self.rank:
                bases.append(own.value)
            else:
                p = ctypes.c_void_p()
                buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
                self._check(self._lib.knn_peer_handle_open(buf, self.device, ctypes.byref(p)))
                bases.append(p.value)
        self.own, self.bases, self.capacity = own, bases, cap
        self._own_tensor = torch.as_tensor(_DeviceBytes(own.value, cap), device=torch.device("cuda", self.device))

    @staticmethod
    def layout(nq: int, k: int):
        n = nq * k
        return {"I_local": 0, "I_merged": 8 * n, "D_local": 16 * n, "D_merged": 20 * n, "bytes": 24 * n}

    def views(self, nq: int, k: int):
        """torch views of this rank's own regions."""
        import torch

        lay = self.layout(nq, k)
        n = nq * k
        t = self._own_tensor

        def region(name, dtype, size):
            return t[lay[name]:lay[name] + n * size].view(dtype).view(nq, k)

        return (region("D_local", torch.float32, 4), region("I_local", torch.int64, 8),
                region("D_merged", torch.float32, 4), region("I_merged", torch.int64, 8))

    def tables(self, nq: int, k: int):
        import ctypes

        lay = self.layout(nq, k)
        arr = lambda name: (ctypes.c_void_p * self.world)(*[b + lay[name] for b in self.bases])  # noqa: E731
        return arr("D_local"), arr("I_local"), arr("D_merged"), arr("I_merged")

    def close(self) -> None:
        self._release()


class BoundsExchange:
    """Per-batch MAX-reduction of the two-phase search's bounds over peer memory (knn_bounds_push_peer_dev /
    knn_bounds_wait_max_dev).  Every rank owns slots [batch][rank][2 * rows] floats and flags [batch][rank]; a search is
    one epoch.  Two searches are separated by the barriers of the result merge, so slots are never overwritten while a
    slower rank still reads them.  All methods are collective in the sense that every rank calls them in the same order.
    ``exchange``: an object with PeerExchange's ``bases``, ``_own_tensor``, ``ensure``, ``barrier`` and ``close`` to use
    instead of a new PeerExchange (tests run G ranks in one process over shared buffers)."""

    MAX_QUERY_ROWS = 131072 + 16384  # two-phase limit + one padded batch

    def __init__(self, dist, group, rank: int, world: int, device: int, exchange=None):
        import torch

        from . import _lib

        self._lib, self._check = _lib.load(), _lib.check
        self.rank, self.world, self.device = rank, world, device
        self.max_batches = 1024
        self.flags_off = 0
        self.slots_off = self.max_batches * world * 4
        nbytes = self.slots_off + self.MAX_QUERY_ROWS * 2 * world * 4
        self.ex = exchange if exchange is not None else PeerExchange(dist, group, rank, world, device)
        self.ex.ensure(nbytes)
        self.ex._own_tensor.zero_()
        self.ex.barrier()  # nobody pushes into a buffer that is not zeroed yet
        dev = torch.device("cuda", device)
        self.counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.timeout = torch.zeros(1, dtype=torch.int32, device=dev)
        self.epoch = 0
        self.n = 0

    def begin(self, nbatches: int, rows: int) -> None:
        if nbatches > self.max_batches or nbatches * rows > self.MAX_QUERY_ROWS:
            raise ValueError("too many query batches for the peer bound exchange")
        self.epoch += 1
        self.n = 2 * rows

    def _offsets(self, b: int):
        """Byte offsets of batch b's slots [rank][2 * rows] and flags [rank] in every rank's buffer."""
        return self.slots_off + b * self.world * self.n * 4, self.flags_off + b * self.world * 4

    def push(self, b: int, bounds_b) -> None:
        """Stores bounds_b (2 * rows floats, contiguous) into slot [rank] of batch b on every rank, then raises this
        rank's flag there to the epoch; on the current stream."""
        import ctypes

        from .index import _torch_stream

        slot_b, flag_b = self._offsets(b)
        slots = (ctypes.c_void_p * self.world)(*[base + slot_b for base in self.ex.bases])
        flags = (ctypes.c_void_p * self.world)(*[base + flag_b for base in self.ex.bases])
        self._check(self._lib.knn_bounds_push_peer_dev(self.world, self.rank, self.n, bounds_b.data_ptr(), slots, flags,
                                                       self.epoch, self.counter.data_ptr(), _torch_stream(self.device)))

    def wait_max(self, b: int, bounds_b) -> None:
        """bounds_b <- element-wise MAX over the slots of batch b in this rank's buffer, once every rank has pushed
        them; on the current stream."""
        from .index import _torch_stream

        slot_b, flag_b = self._offsets(b)
        own = self.ex.bases[self.rank]
        self._check(self._lib.knn_bounds_wait_max_dev(self.world, self.n, own + slot_b, own + flag_b, self.epoch,
                                                      bounds_b.data_ptr(), self.timeout.data_ptr(), _torch_stream(self.device)))

    def max_over_ranks(self, b: int, bounds_b) -> None:
        """bounds_b (2 * rows floats, contiguous) <- element-wise MAX over the ranks, on the current stream."""
        self.push(b, bounds_b)
        self.wait_max(b, bounds_b)

    def check(self) -> None:
        if int(self.timeout.item()):
            self.timeout.zero_()
            raise RuntimeError("bound exchange: a peer rank did not deliver its bounds within the spin limit")

    def close(self) -> None:
        self.ex.close()


def _to_numpy(t):
    """Result tensor -> numpy.  CUDA results travel straight into page-locked memory (ordinary numpy arrays to the
    caller, see index._result_arrays) instead of through the driver's pageable bounce buffers."""
    if not t.is_cuda:
        return t.numpy()
    import torch

    if 0 < t.numel() * t.element_size() <= (1 << 30):
        try:
            out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            out.copy_(t, non_blocking=True)
            torch.cuda.current_stream(t.device).synchronize()
            return out.numpy()
        except RuntimeError:
            pass
    return t.cpu().numpy()


def shard_bounds(n: int, world: int, weights=None):
    """Contiguous row ranges: rank r owns [b[r], b[r+1]).  Near-equal by default; with ``weights`` (one positive
    number per rank, e.g. measured_rank_speeds) rank r gets a share of the rows proportional to weights[r]."""
    if weights is None:
        return [(n * r) // world for r in range(world + 1)]
    w = [float(v) for v in weights]
    if len(w) != world or min(w) <= 0:
        raise ValueError("weights: one positive number per rank")
    total, acc, b = sum(w), 0.0, [0]
    for r in range(world - 1):
        acc += w[r]
        b.append(max(b[-1], min(n, int(round(n * acc / total)))))
    b.append(n)
    return b


def measured_rank_speeds(d: int, device: int, group=None, seconds: float = 1.5, rows: int = 1 << 20, queries: int = 16384,
                         spread: float = 0.15):
    """Relative speed of every rank's GPU on the engine's own dominant kernel, for speed-proportional sharding.

    A search step ends when the SLOWEST shard is done (the bound exchange and the merge are collectives), and under a
    board power cap the chips of one box do not run the tensor cores at the same clock.  All ranks run the same
    synthetic search (``rows`` x ``queries``, k = 100) simultaneously for ``seconds`` - long enough for the clocks to
    settle under the cap - and the pairs/s of the second half are all-gathered.  Returns one weight per rank with mean
    1, clipped to 1 +- ``spread``.  Collective over ``group``; every rank gets the same list."""
    import time

    import torch
    import torch.distributed as dist

    from .index import IndexFlat, normalize_L2

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return [1.0]
    dev = torch.device("cuda", device)
    g = torch.Generator(device=dev).manual_seed(99)
    idx = IndexFlat(d, 0, device=device)
    idx.set_param("path", 2)
    idx.reserve(rows)
    for i in range(0, rows, 1 << 18):
        x = torch.randn(min(1 << 18, rows - i), d, device=dev, generator=g)
        normalize_L2(x)
        idx.add(x)
    xq = torch.randn(queries, d, device=dev, generator=g)
    normalize_L2(xq)
    idx.search(xq, 100)
    torch.cuda.synchronize(dev)
    dist.barrier(group=group)
    t0 = time.perf_counter()
    done, half_t, half_n = 0, None, 0
    while True:
        idx.search(xq, 100)
        torch.cuda.synchronize(dev)
        done += 1
        t = time.perf_counter() - t0
        if half_t is None and t >= seconds / 2:
            half_t, half_n = t, done
        if t >= seconds and half_t is not None and done > half_n:
            break
    rate = (done - half_n) / (t - half_t)
    rates = torch.zeros(world, device=dev, dtype=torch.float64)
    dist.all_gather_into_tensor(rates, torch.tensor([rate], device=dev, dtype=torch.float64), group=group)
    del idx
    r = rates.tolist()
    mean = sum(r) / world
    return [min(1.0 + spread, max(1.0 - spread, v / mean)) for v in r]


class ShardedIndexFlat:
    TWO_PHASE_MAX_QUERIES = 131072  # limit of knn_index_search_filter_dev (candidate lists stay resident)
    MAX_TOTAL_ROWS = 2 ** 32 - 1

    def __init__(self, d: int, metric: int, group=None, device=None, index_factory=None, merge_fn=None,
                 exchange_bounds: bool = True, peer_merge: bool = True, shard_weights=None, **index_kw):
        import torch.distributed as dist

        self._dist = dist
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.d = int(d)
        self.metric_type = int(metric)
        self.is_trained = True
        if index_factory is None:
            from .index import IndexFlat

            index_factory = lambda: IndexFlat(d, metric, device=device, **index_kw)  # noqa: E731
        if merge_fn is None:
            from .index import merge_topk

            merge_fn = merge_topk
        self.exchange_bounds = exchange_bounds
        self.peer_merge = peer_merge  # exchange + merge in one kernel over NVLink peer memory (CUDA results only)
        self._exchange = None
        self._side_stream = None
        self._main_stream = None
        self._bounds = None
        # bound exchange of the pipelined two-phase search over NVLink peer memory instead of NCCL (CUDA + NCCL groups)
        self.peer_bounds = peer_merge and self.world <= 16 and dist.is_initialized() and dist.get_backend(group) == "nccl"
        self.pipeline_batches = True  # exchange + finish of query batch b on a side stream under the filter of batch b + 1
        self.profile_phases = False
        self.last_phases_ms = None
        self.last_stats = None
        self.local = index_factory()
        self._merge = merge_fn
        # share of the rows every rank keeps (None: equal shares; see measured_rank_speeds)
        self.shard_weights = list(shard_weights) if shard_weights is not None else None
        # one (global_start, local_start, count) triple per add() call
        self._segments = []
        self._ntotal = 0
        self._nlocal = 0

    @property
    def ntotal(self) -> int:
        return self._ntotal

    def train(self, x) -> None:
        pass

    def add(self, x) -> None:
        """Every rank passes the same rows (as the reference's drivers would); rank r keeps its
        contiguous slice.  Global id of a row = its position in the concatenation of all adds."""
        n = x.shape[0]
        b = shard_bounds(n, self.world, self.shard_weights)
        lo, hi = b[self.rank], b[self.rank + 1]
        self.add_local(x[lo:hi], global_start=self._ntotal + lo, n_global=n)

    def add_local(self, x_local, global_start: int, n_global: int) -> None:
        """For data generated per shard: this rank's rows are x_local, their global ids start at
        global_start; n_global rows are being added across all ranks."""
        cnt = x_local.shape[0]
        self._check_total(int(n_global))
        if cnt:
            self.local.add(x_local)
        self._segments.append((int(global_start), self._nlocal, cnt))
        self._nlocal += cnt
        self._ntotal += int(n_global)

    def _check_total(self, n_more: int) -> None:
        # the cross-shard merges build their keys from 32-bit ids (csrc/select.cu, csrc/peer.cu)
        if self._ntotal + n_more >= self.MAX_TOTAL_ROWS:
            raise ValueError("a sharded index holds at most 2^32-2 rows in total (global ids are merged as 32-bit keys)")

    def close(self) -> None:
        """Releases the NVLink exchange buffer and the peers' IPC mappings.  Collective over the group."""
        if self._exchange is not None:
            self._exchange.close()
            self._exchange = None
        if self._bounds is not None:
            self._bounds.close()
            self._bounds = None

    def adopt_local(self, global_start: int, n_global: int) -> None:
        """Book-keeping for rows that were added straight into ``self.local`` (e.g. generated
        block by block on the device): they become one segment starting at global_start."""
        cnt = self.local.ntotal - self._nlocal
        self._check_total(int(n_global))
        self._segments.append((int(global_start), self._nlocal, cnt))
        self._nlocal += cnt
        self._ntotal += int(n_global)

    def _to_global(self, I):
        """local row numbers -> global row numbers, -1 kept."""
        import torch

        if not self._segments:  # searched before any add: all padding
            return I
        if len(self._segments) == 1:
            g0 = self._segments[0][0]
            return torch.where(I >= 0, I + g0, I) if g0 else I
        starts = torch.tensor([s[1] for s in self._segments], device=I.device, dtype=I.dtype)
        offs = torch.tensor([s[0] - s[1] for s in self._segments], device=I.device, dtype=I.dtype)
        seg = torch.bucketize(I.clamp(min=0), starts, right=True) - 1
        return torch.where(I >= 0, I + offs[seg], I)

    def upload_queries(self, x_host):
        """Host queries that EVERY rank holds (the reference's drivers load the same file in every process) -> the full
        (n, d) float32 matrix on this rank's device, crossing PCIe once in total instead of once per rank: rank r
        uploads rows [r n/G, (r+1) n/G) and one all-gather over NVLink hands every rank the rest (C4 on 8 GPUs: 51 MB
        instead of 410 MB over each rank's PCIe link).  x_host: CPU torch tensor (pinned for an asynchronous copy) or
        numpy array.  float16 / bfloat16 rows keep their dtype (half the PCIe and NVLink bytes; the index reads them as
        they are), anything else becomes float32.  Collective."""
        import torch

        from .index import _h16_code

        if isinstance(x_host, np.ndarray):
            x_host = torch.from_numpy(np.ascontiguousarray(x_host, dtype=None if x_host.dtype == np.float16 else np.float32))
        elif _h16_code(x_host.dtype) is None:
            x_host = x_host.to(torch.float32)
        n, d = x_host.shape
        dev = torch.device("cuda", self.local.device) if self._dist.is_initialized() and self._dist.get_backend(self.group) == "nccl" \
            else x_host.device
        if self.world == 1:
            return x_host.to(dev, non_blocking=True).contiguous()
        chunk = -(-n // self.world)  # equal chunks (all_gather_into_tensor); the tail of the last one is padding
        buf = torch.empty((self.world * chunk, d), dtype=x_host.dtype, device=dev)
        lo, hi = min(n, self.rank * chunk), min(n, (self.rank + 1) * chunk)
        mine = buf[self.rank * chunk:(self.rank + 1) * chunk]
        if hi > lo:
            mine[:hi - lo].copy_(x_host[lo:hi], non_blocking=True)
        self._dist.all_gather_into_tensor(buf, mine, group=self.group)
        return buf[:n]

    def search(self, x, k: int, *, params=None, exclude=None):
        """Returns the merged (D, I) on every rank (torch tensors on the local index's device, or
        numpy arrays when x is numpy).  Calls with more queries than the two-phase search keeps resident
        (TWO_PHASE_MAX_QUERIES) are processed in chunks of that size (config C5: 1M queries).

        params (faiss.SearchParameters(sel=...)) selects global rows and exclude (an (nq,) array of global ids, -1:
        none) removes one row per query; a filtered search always runs the pipelined two-phase search, every shard
        reading the one global bitmap from its first global row on."""
        n = x.shape[0]
        if (getattr(params, "sel", None) is not None or exclude is not None) and n > 0:
            return self._search_filtered(x, k, params, exclude)
        if n == 0:  # nothing to search (every rank of the group sees the same empty call: no collective is entered)
            if isinstance(x, np.ndarray):
                return np.empty((0, k), np.float32), np.empty((0, k), np.int64)
            import torch

            return (torch.empty((0, k), dtype=torch.float32, device=x.device), torch.empty((0, k), dtype=torch.int64, device=x.device))
        if n > self.TWO_PHASE_MAX_QUERIES and self.world > 1:
            step = self.TWO_PHASE_MAX_QUERIES
            parts, acc = [], {"gemm_ms": 0.0, "gemm_launches": 0.0}
            for i in range(0, n, step):
                parts.append(self._search_chunk(x[i:i + step], k))
                if hasattr(self.local, "stat"):  # per-call statistics of the shard engine, summed over the chunks
                    for name in acc:
                        acc[name] += self.local.stat(name)
            self.last_stats = acc
            if isinstance(x, np.ndarray):
                return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
            import torch

            return torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])
        out = self._search_chunk(x, k)
        self.last_stats = ({name: self.local.stat(name) for name in ("gemm_ms", "gemm_launches")}
                           if hasattr(self.local, "stat") else None)
        return out

    def _search_chunk(self, x, k: int):
        import torch

        as_numpy = isinstance(x, np.ndarray)
        on_cuda = self._dist.is_initialized() and self._dist.get_backend(self.group) == "nccl"
        if on_cuda and (as_numpy or not x.is_cuda):
            # host queries that every rank holds: each rank uploads 1/G of them, one all-gather over NVLink does the rest
            x = self.upload_queries(x)
        marks = []

        def mark(name, stream=None):
            if self.profile_phases:
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream) if stream is not None else e.record()
                marks.append((name, e))

        mark("start")
        two_phase = (self.world > 1 and self.exchange_bounds and hasattr(self.local, "search_filter")
                     and x.shape[0] <= self.TWO_PHASE_MAX_QUERIES)
        globalised = False
        if two_phase and self.pipeline_batches and hasattr(self.local, "search_begin"):
            xd = torch.from_numpy(x).to(torch.device("cuda", self.local.device)) if isinstance(x, np.ndarray) else x
            D, I = self._two_phase_pipelined(xd, k, mark)
            globalised = len(self._segments) == 1
        elif two_phase:
            # filter on every shard -> all-reduce(MAX) of the per-query lower bounds of the k-th best score ->
            # each shard rescoring only what can still be in the global top-k (DESIGN.md section 6)
            xd = torch.from_numpy(x).to(torch.device("cuda", self.local.device)) if isinstance(x, np.ndarray) else x
            # two bounds on the global k-th best true score: the best shard's own k-th, and - every shard holding
            # j = ceil(k/G) rows at or above its own j-th - the smallest j-th over the shards
            j = -(-k // self.world)
            lower, lower_j = self.local.search_filter(xd, k, j)
            mark("filter")
            # one collective for both: MAX over the shards of lower, MIN of lower_j = -MAX(-lower_j)
            both = torch.stack([lower, -lower_j])
            self._dist.all_reduce(both, op=self._dist.ReduceOp.MAX, group=self.group)
            lower = torch.maximum(both[0], -both[1])
            mark("all_reduce_bounds")
            D, I = self.local.search_finish(lower, k)
            mark("finish")
        else:
            D, I = self.local.search(x, k)
            if isinstance(D, np.ndarray):
                D, I = torch.from_numpy(D), torch.from_numpy(I)
                if on_cuda:
                    dev = torch.device("cuda", self.local.device)
                    D, I = D.to(dev), I.to(dev)
        if not globalised:
            I = self._to_global(I)
        mark("to_global")
        if self.world > 1 and self.peer_merge and D.is_cuda and self.world <= 16 and (self.world + 1) * k * 8 <= 200 * 1024:
            D, I = self._merge_over_peer_memory(D, I)
            mark("peer_merge")
        elif self.world > 1:
            nq, kk = D.shape
            Dg = torch.empty((self.world * nq, kk), dtype=D.dtype, device=D.device)
            Ig = torch.empty((self.world * nq, kk), dtype=I.dtype, device=I.device)
            self._dist.all_gather_into_tensor(Dg, D.contiguous(), group=self.group)
            self._dist.all_gather_into_tensor(Ig, I.contiguous(), group=self.group)
            mark("all_gather")
            D, I = self._merge(Dg.view(self.world, nq, kk), Ig.view(self.world, nq, kk), self.metric_type)
            mark("merge")
        if marks:
            torch.cuda.synchronize()
            self.last_phases_ms = {b[0]: a[1].elapsed_time(b[1]) for a, b in zip(marks[:-1], marks[1:])}
        if as_numpy:
            return _to_numpy(D), _to_numpy(I)
        return D, I

    def _search_filtered(self, x, k: int, params, exclude):
        import torch

        if len(self._segments) > 1:
            raise NotImplementedError("a filtered search of a ShardedIndexFlat needs its rows from a single add()")
        as_numpy = isinstance(x, np.ndarray)
        dev = torch.device("cuda", self.local.device) if torch.cuda.is_available() else torch.device("cpu")
        on_cuda = self._dist.is_initialized() and self._dist.get_backend(self.group) == "nccl"
        xd = self.upload_queries(x) if on_cuda and (as_numpy or not x.is_cuda) else torch.as_tensor(x).to(dev)
        g0 = self._segments[0][0] if self._segments else 0
        if exclude is not None:
            exclude = torch.as_tensor(exclude, dtype=torch.int64).to(dev)
        flt = {"params": params, "exclude": exclude, "id_base": g0, "allow_bit0": g0, "allow_nbits": self._ntotal}
        parts = []
        for i in range(0, xd.shape[0], self.TWO_PHASE_MAX_QUERIES):
            sl = slice(i, i + self.TWO_PHASE_MAX_QUERIES)
            chunk = dict(flt, exclude=exclude[sl] if exclude is not None else None)
            D, I = self._two_phase_pipelined(xd[sl], k, lambda *a: None, chunk)
            if self.world > 1 and self.peer_merge and D.is_cuda and self.world <= 16 and (self.world + 1) * k * 8 <= 200 * 1024:
                D, I = self._merge_over_peer_memory(D, I)
            elif self.world > 1:
                nq, kk = D.shape
                Dg = torch.empty((self.world * nq, kk), dtype=D.dtype, device=D.device)
                Ig = torch.empty((self.world * nq, kk), dtype=I.dtype, device=I.device)
                self._dist.all_gather_into_tensor(Dg, D.contiguous(), group=self.group)
                self._dist.all_gather_into_tensor(Ig, I.contiguous(), group=self.group)
                D, I = self._merge(Dg.view(self.world, nq, kk), Ig.view(self.world, nq, kk), self.metric_type)
            parts.append((D, I))
        D, I = (torch.cat([p[0] for p in parts]), torch.cat([p[1] for p in parts])) if len(parts) > 1 else parts[0]
        if as_numpy:
            return _to_numpy(D), _to_numpy(I)
        return D, I

    def _two_phase_pipelined(self, xd, k: int, mark, flt=None):
        """The two-phase search, one query batch at a time over two streams.  Main stream: tensor-core filter of
        batch 0, 1, 2 ...  Side stream, per batch as soon as its filter is done: ONE all-reduce(MAX) of the batch's two
        bounds (a few hundred KB over NVLink), then the finish phase (exact rescoring of what can still be in the
        global top-k, final select).  The finish phase is HBM gathers and shared-memory sorts, the filter is tensor-core
        work that leaves HBM idle, so the two share the SMs; the collective's wait for the slowest shard of batch b is
        hidden under this rank's own filter of batch b + 1.  Only the last batch's exchange + finish is exposed.
        With a single add() segment the global id base goes into the kernels (id_base), sparing a pass over I."""
        import torch

        dev = torch.device("cuda", self.local.device)
        caller = torch.cuda.current_stream(dev)
        if self._side_stream is None:
            # priorities: a GEMM CTA of the filter takes the first SM slot that frees up, the thousands of short
            # rescoring CTAs of the finish phase fill what the resident GEMM CTAs leave (see csrc/index.cu search_tensor)
            self._side_stream = torch.cuda.Stream(device=dev, priority=0)
            self._main_stream = torch.cuda.Stream(device=dev, priority=-1)
        side, main = self._side_stream, self._main_stream
        nq = xd.shape[0]
        main.wait_stream(caller)
        with torch.cuda.stream(main):
            nbatches, rows = self.local.search_begin(xd, k, **flt) if flt else self.local.search_begin(xd, k)
            bx = self._bounds_exchange(nbatches, rows) if self.peer_bounds else None
            bounds = torch.zeros((nbatches, 2, rows), dtype=torch.float32, device=dev)
            D = torch.empty((nq, k), dtype=torch.float32, device=dev)
            I = torch.empty((nq, k), dtype=torch.int64, device=dev)
            id_base = self._segments[0][0] if len(self._segments) == 1 else 0
            if flt:
                id_base = flt["id_base"]
            j = -(-k // self.world)
            side.wait_stream(main)  # bounds / D / I exist before the side stream touches them
            for b in range(nbatches):
                self.local.search_filter_batch(b, j, bounds)
                filtered = torch.cuda.Event()
                filtered.record(main)
                with torch.cuda.stream(side):
                    side.wait_event(filtered)
                    if bx is not None:   # two tiny kernels over NVLink peer memory (csrc/peer.cu): fit next to the GEMM
                        bx.max_over_ranks(b, bounds[b])
                    else:                # NCCL: its kernel waits for a panel boundary of the GEMM on the main stream
                        self._dist.all_reduce(bounds[b], op=self._dist.ReduceOp.MAX, group=self.group)
                    self.local.search_finish_batch(b, bounds, D, I, id_base)
            mark("filter", main)
            main.wait_stream(side)
            mark("exchange_finish_exposed", main)
            self.local.search_end(D, I, id_base)
        caller.wait_stream(main)
        for t in (bounds, D, I, xd):
            t.record_stream(side)
            t.record_stream(main)
            t.record_stream(caller)
        if bx is not None:
            bx.check()
        return D, I

    def _bounds_exchange(self, nbatches: int, rows: int):
        if self._bounds is None:
            self._bounds = BoundsExchange(self._dist, self.group, self.rank, self.world, self.local.device)
        self._bounds.begin(nbatches, rows)
        return self._bounds

    def _merge_over_peer_memory(self, D, I):
        """This rank merges its slice of the queries out of the peers' memory and stores the merged rows into every
        rank's buffer (knn_merge_topk_peer_dev); two barriers order it against the per-shard searches and the readers."""
        from . import _lib
        from .index import _torch_stream

        nq, k = D.shape
        if self._exchange is None:
            self._exchange = PeerExchange(self._dist, self.group, self.rank, self.world, D.device.index)
        ex = self._exchange
        ex.ensure(ex.layout(nq, k)["bytes"])
        D_loc, I_loc, D_out, I_out = ex.views(nq, k)
        D_loc.copy_(D)
        I_loc.copy_(I)
        ex.barrier()  # every shard's results are in place
        b = shard_bounds(nq, self.world)
        tD, tI, tDo, tIo = ex.tables(nq, k)
        _lib.check(_lib.load().knn_merge_topk_peer_dev(self.metric_type, nq, k, self.world, b[self.rank], b[self.rank + 1],
                                                       tD, tI, tDo, tIo, _torch_stream(D.device.index)))
        ex.barrier()  # every rank's slice has landed in this rank's buffer
        return D_out.clone(), I_out.clone()


def choose_query_groups(world: int, n_rows: int, d: int, bytes_per_element: int, device: int | None = None,
                        memory_fraction: float = 0.6) -> int:
    """How many query groups Q (Q divides world; R = world / Q row shards per group) for a database of n_rows x d:
    the LARGEST Q whose per-rank share of the rows, (n_rows / R) * d * bytes_per_element, fits memory_fraction of the
    GPU's memory (the rest is for query batches, candidate lists and the caller).  bytes_per_element: 6 for the default
    storage (fp32 master rows + 16-bit tensor-core rows), 2 for bf16 storage.

    Why larger Q is faster (measured on 8 B200, C4; profiles/r02_bench_c4_8gpu_*.json): row sharding replicates the
    per-QUERY work of a search - query preparation, threshold tightening after every panel, the exact rescoring and
    the final select - on every rank of a group, and under the board power cap that work costs its energy whether or
    not it is overlapped with the GEMM: 8 x 1 row shards 519k queries/s, 2 groups x 4 shards 530k, 4 groups x 2 shards
    541k.  With 180 GB of HBM per GPU a 10M x 1024 database (61 GB) fits every GPU, so C4 runs as pure query sharding;
    the 100M-row database of C5 (205 GB in bf16) needs at least two row shards."""
    total = None
    try:
        import torch

        total = torch.cuda.get_device_properties(torch.cuda.current_device() if device is None else device).total_memory
    except Exception:
        pass
    if not total:
        total = 180 << 30
    budget = memory_fraction * total
    best = 1
    for q in range(1, world + 1):
        if world % q:
            continue
        r = world // q
        if (n_rows / r) * d * bytes_per_element <= budget:
            best = q
    return best


class GridIndexFlat:
    """Rows x query-groups grid of ranks (world = R x Q, rank = g * R + r).

    Row sharding replicates the per-QUERY work of a search (query preparation, threshold tightening after every panel,
    the finish phase) on every rank: at 8 GPUs that is ~14 ms of a 196 ms C4 step (DESIGN.md section 6).  Here the Q
    query groups each hold the WHOLE database, row-sharded over their R ranks (a ShardedIndexFlat on a sub-group), and
    take 1/Q of the queries of a call; the ranks with the same row position then all-gather their result slices, so
    every rank still returns the full (D, I).  Per-rank GEMM work is unchanged (Q x more rows, Q x fewer queries than
    with plain row sharding), the per-query work drops by Q, the database costs Q x the memory (C4: 2 x 15 GB per rank).

    Status: the host logic is covered by a world-size-4 gloo test (tests/test_sharded_cpu.py); on GPUs it has run as
    2 groups x 1 shard (profiles/r01_bench_c4_2gpu_query_groups2.json), the 2 x 4 shape it is meant for is unmeasured
    (opt-in: bench.py --query-groups Q)."""

    def __init__(self, d: int, metric: int, query_groups: int, device=None, shard_weights=None, **kw):
        import torch.distributed as dist

        self._dist = dist
        world, rank = dist.get_world_size(), dist.get_rank()
        if query_groups < 1 or world % query_groups:
            raise ValueError("query_groups must divide the world size")
        self.Q, self.R = int(query_groups), world // int(query_groups)
        self.g, self.r = rank // self.R, rank % self.R
        # every rank creates every sub-group, in the same order (torch.distributed requirement)
        row_groups = [dist.new_group([g * self.R + r for r in range(self.R)]) for g in range(self.Q)]
        col_groups = [dist.new_group([g * self.R + r for g in range(self.Q)]) for r in range(self.R)]
        self.col_group = col_groups[self.r]
        self.group_weights = None  # share of the queries every group takes (None: equal shares)
        # Large searches re-balance the query slices from the groups' own measured times: a call ends when the slowest
        # group is done, the chips of one box do not clock alike under the board power cap, and a 2 s calibration on a
        # small database (measured_rank_speeds) leaves ~2 % of spread on the real workload (8 B200, C4: GEMM 171.5-175.9
        # ms per rank).  Every large call is bracketed by two CUDA events (no synchronisation); at call numbers 2, 4, 8,
        # 16, ... the PREVIOUS call's time - taken back to back with its neighbours, i.e. in the power state the chips
        # really run in; a first version that tuned on synchronised calls measured the wrong (cool) state and left the
        # spread where it was - is all-gathered and the shares move towards the measured rates.  That costs one host
        # synchronisation per tuning point; results never depend on the slices (ids are global, every query is answered
        # by one whole group).
        self.autotune = True
        self.autotune_min_queries = 8192
        self._calls = 0
        self._last = None  # (t0, t1, per-group query counts) of the previous large call
        if shard_weights is not None:  # one weight per rank of the world
            w = list(shard_weights)
            # a group is as fast as its ranks together (its row shards are already sized by their weights)
            self.group_weights = [sum(w[g * self.R:(g + 1) * self.R]) for g in range(self.Q)]
            shard_weights = w[self.g * self.R:(self.g + 1) * self.R]
        self.inner = ShardedIndexFlat(d, metric, group=row_groups[self.g], device=device, shard_weights=shard_weights, **kw)
        self.d, self.metric_type, self.is_trained = self.inner.d, self.inner.metric_type, True

    local = property(lambda self: self.inner.local)
    ntotal = property(lambda self: self.inner.ntotal)
    last_stats = property(lambda self: self.inner.last_stats)
    last_phases_ms = property(lambda self: self.inner.last_phases_ms)

    @property
    def profile_phases(self):
        return self.inner.profile_phases

    @profile_phases.setter
    def profile_phases(self, on):
        self.inner.profile_phases = on

    def train(self, x) -> None:
        pass

    def add(self, x) -> None:
        self.inner.add(x)

    def add_local(self, x_local, global_start: int, n_global: int) -> None:
        self.inner.add_local(x_local, global_start, n_global)

    def adopt_local(self, global_start: int, n_global: int) -> None:
        self.inner.adopt_local(global_start, n_global)

    def query_bounds(self, n: int):
        return shard_bounds(n, self.Q, self.group_weights)

    def query_slice(self, n: int):
        b = self.query_bounds(n)
        return b[self.g], b[self.g + 1]

    def search(self, x, k: int, *, params=None, exclude=None):
        """Every rank passes ALL queries and gets the full (D, I); its group searches rows [lo, hi) of them."""
        import torch

        if getattr(params, "sel", None) is not None or exclude is not None:
            raise NotImplementedError("GridIndexFlat has no filtered search; use ShardedIndexFlat (row shards only)")

        as_numpy = isinstance(x, np.ndarray)
        n = x.shape[0]
        on_cuda = self._dist.get_backend(self.col_group) == "nccl"
        timed_call = on_cuda and self.Q > 1 and self.autotune and n >= self.autotune_min_queries
        if timed_call:
            self._calls += 1
            if self._last is not None and self._calls >= 2 and (self._calls & (self._calls - 1)) == 0:
                self._retune(*self._last)  # the shares move before this call is sliced
        lo, hi = self.query_slice(n)
        xs = x[lo:hi]
        if on_cuda and (as_numpy or not xs.is_cuda):
            # host queries: only this group's slice crosses PCIe (its ranks share the upload), results stay on the device
            xs = self.inner.upload_queries(xs)
        if timed_call:
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
        D, I = self.inner.search(xs, k)
        if timed_call:
            t1.record()
            b_now = self.query_bounds(n)
            self._last = (t0, t1, [b_now[g + 1] - b_now[g] for g in range(self.Q)])
        if self.Q == 1:
            return (_to_numpy(D), _to_numpy(I)) if as_numpy and not isinstance(D, np.ndarray) else (D, I)
        if isinstance(D, np.ndarray):
            D, I = torch.from_numpy(D), torch.from_numpy(I)
        b = self.query_bounds(n)
        chunk = max(b[g + 1] - b[g] for g in range(self.Q))  # equal chunks for all_gather_into_tensor; tails are padding
        bufD = torch.empty((self.Q * chunk, k), dtype=D.dtype, device=D.device)
        bufI = torch.empty((self.Q * chunk, k), dtype=I.dtype, device=I.device)
        mineD, mineI = bufD[self.g * chunk:(self.g + 1) * chunk], bufI[self.g * chunk:(self.g + 1) * chunk]
        mineD[:hi - lo].copy_(D)
        mineI[:hi - lo].copy_(I)
        self._dist.all_gather_into_tensor(bufD, mineD, group=self.col_group)
        self._dist.all_gather_into_tensor(bufI, mineI, group=self.col_group)
        D = torch.cat([bufD[g * chunk:g * chunk + (b[g + 1] - b[g])] for g in range(self.Q)])
        I = torch.cat([bufI[g * chunk:g * chunk + (b[g + 1] - b[g])] for g in range(self.Q)])
        if as_numpy:
            return _to_numpy(D), _to_numpy(I)
        return D, I

    def _retune(self, t0, t1, counts) -> None:
        """Collective over the world: every group's time for its slice of the measured call -> new query shares,
        moved towards the measured rates (damped), identical on every rank."""
        import torch

        t1.synchronize()
        mine = torch.tensor([t0.elapsed_time(t1)], dtype=torch.float64, device=torch.device("cuda", self.inner.local.device))
        world = self.Q * self.R
        times = torch.zeros(world, dtype=torch.float64, device=mine.device)
        self._dist.all_gather_into_tensor(times, mine)
        times = times.tolist()
        group_ms = [max(times[g * self.R:(g + 1) * self.R]) for g in range(self.Q)]
        if min(group_ms) <= 0 or min(counts) <= 0:
            return
        rates = [c / t for c, t in zip(counts, group_ms)]          # queries per ms, as measured on this workload
        old = self.group_weights or [1.0] * self.Q
        so, sr = sum(old), sum(rates)
        new = [0.3 * o / so + 0.7 * r / sr for o, r in zip(old, rates)]  # damped: one noisy call cannot swing the split
        self.group_weights = [w * self.Q / sum(new) for w in new]

    def close(self) -> None:
        self.inner.close()
