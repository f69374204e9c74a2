"""NCCL data plane: the search fan-out of IndexClient.search over GPUs instead of sockets.

The reference sends the same pickled query to every IndexServer over TCP and merges the
pickled replies on the client's CPU (distributed_faiss/client.py:200-210, 265-310;
rpc.py:120-131).  Inside one 8xB200 box this module replaces that with:

    query  --(ncclBroadcast from the client rank)-->  every rank
    every rank: libdfx search of its resident shards (+ local id -> caller / exchange id on device)
    results --(ONE ncclAllGather over NVLink/NVSwitch of the packed (D, I) blocks)--> every rank
    merge kernel K6 (float_maxheap_array_t semantics)  -> (D, I) on device

One process per GPU (`IndexServer(rank=r)` <-> GPU r), `torch.distributed` for the plumbing.
A rank may hold several shards (the 1/2/4-GPU points of the scaling curve hold 8/4/2 shards
each); shards are numbered rank-major so the merge's "earlier shard wins ties" rule is the
same for every GPU count.  The path has exactly one exchange step, as in the reference.

Two layers:

* `ShardGroup`  -- the collective itself over engine objects (what bench.py's device-resident
  `value` times, and what the plane runs underneath);
* `SearchPlane` -- `IndexClient.search` over that collective: the client lives in the process of
  plane rank 0, the other ranks sit in `serve_forever()`; a search is announced by a 256-byte
  header broadcast (op, nq, k, flags, index id), followed by the query broadcast.  The servers'
  `Index` objects keep their lock / state rules; the socket RPC stays for the control plane
  (create / add / train / save / set_nprobe) and for metadata OBJECTS of the winners.

`backend` abstracts the device operations so that the world_size>1 host logic can be exercised
on CPU with gloo (tests inject an oracle-backed backend); the default backend is CUDA-only and
has no fallback.
"""
from __future__ import annotations

import os
import pickle
import threading
from typing import List, Optional, Sequence

# NOTE for deployments that mix the two transports: a process that serves the plane also answers
# control-plane and socket RPCs from other threads.  With CUDA's default LAZY module loading the
# first launch of any kernel needs a context-wide synchronisation, which cannot complete while a
# NCCL kernel of this process waits for its peer (every rank sitting in serve_forever() has one
# pending).  Control-plane RPCs launch nothing; a socket SEARCH against such a process can hang on a
# first-use kernel.  Either send searches through the plane only (what IndexClient does once
# attached), or start the processes with CUDA_MODULE_LOADING=EAGER (minutes of extra start-up: every
# torch kernel is loaded).

import numpy as np
import torch
import torch.distributed as dist

FLT_MAX = float(np.finfo(np.float32).max)
LOCAL_BITS = 40                    # exchange id = (global shard << 40) | shard-local id
LOCAL_MASK = (1 << LOCAL_BITS) - 1
DROP_FLAG = 1 << 62                # entries search_with_filter's post-filter drops


def _align8(n: int) -> int:
    return (n + 7) & ~7


class CudaBackend:
    """The product backend: everything runs in libdfx kernels on torch's current stream."""

    name = "cuda"

    def search_local(self, shard, x_t, k, D_out, I_out):
        shard.search_dev(x_t, k, D_out, I_out)

    def map_ids(self, ids_t, table_t, out_t=None):
        from . import engine

        return engine.map_ids_dev(ids_t, table_t, out_t)

    def encode_ids(self, ids_t, tag, out_t, col_t=None, drop_code=-1):
        from . import engine

        return engine.encode_ids_dev(ids_t, tag, out_t, col_t, drop_code)

    def merge_packed(self, packed_t, R, S_loc, nq, k, stride, off_I, negate):
        from . import engine

        return engine.merge_packed_dev(packed_t, R, S_loc, nq, k, stride, off_I, negate)

    def filter_compact(self, D_t, I_t, k_out):
        from . import engine

        return engine.filter_compact_dev(D_t, I_t, k_out)

    def reconstruct_owned(self, shard, I_t, R_t, tag):
        shard.reconstruct_dev(I_t, R_t, tag)

    # kept for callers of the round-1 interface
    def merge(self, D_t, I_t, negate):
        from . import engine

        return engine.merge_dev(D_t, I_t, negate=negate)


class SearchOut:
    """What one collective search leaves on the device of every rank."""

    __slots__ = ("D", "I", "count", "embs", "meta_int", "status")

    def __init__(self, D, I, count=None, embs=None, meta_int=None, status=None):
        self.D, self.I, self.count, self.embs, self.meta_int, self.status = D, I, count, embs, meta_int, status


class ShardGroup:
    """The set of shards of one index spread over the ranks of a process group.

    shards     : this rank's engine objects (engine.GpuIndex), in global shard order
    id_tables  : per local shard, int64 device tensor mapping shard-local id -> caller id
                 (the integer-metadata convention of scripts/load_data.py:120-124), or None
                 to return shard-local ids
    Every rank must own the same number of shards.
    """

    def __init__(self, shards: Sequence, id_tables: Optional[Sequence] = None, group=None,
                 backend=None, device=None):
        self.shards = list(shards)
        self.id_tables = list(id_tables) if id_tables is not None else [None] * len(self.shards)
        assert len(self.id_tables) == len(self.shards)
        self.group = group
        self.backend = backend or CudaBackend()
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.device = device if device is not None else (
            torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu"))
        self._pin_q = None
        self._pin_out = None
        # side streams for intra-rank shard overlap (CUDA backend only)
        self._streams = []
        self._stream_max_nq = 0
        if self.device.type == "cuda" and isinstance(self.backend, CudaBackend) and len(self.shards) > 1:
            # latency-bound batches gain ~1.8x from overlapping the shards; large batches already
            # fill the machine and are run back to back (also keeps per-kernel timing clean)
            self._stream_max_nq = int(os.environ.get("DFX_SHARD_STREAMS_MAX_NQ", "1024"))
            n_side = int(os.environ.get("DFX_SHARD_STREAMS", "4"))
            self._streams = [torch.cuda.Stream(device=self.device) for _ in range(max(0, n_side))]
        # latency-bound batches (a batch-1 search over 8 shards is ~50 short launches whose issue
        # cost dominates: 0.39 -> 0.15 ms on a B200, profiles/r02_*) are replayed from a CUDA graph
        # captured per (shape, options, shard generations); single rank only (DFX_GRAPHS=0 disables)
        self.last_error = None
        self._graphs = {}
        self._graph_gens = None
        self._graph_max_nq = 0
        if self.device.type == "cuda" and isinstance(self.backend, CudaBackend) and self.world == 1:
            if os.environ.get("DFX_GRAPHS", "1") != "0":
                self._graph_max_nq = int(os.environ.get("DFX_GRAPHS_MAX_NQ", "256"))

    @property
    def num_shards(self) -> int:
        return len(self.shards) * self.world

    def set_nprobe(self, nprobe: int):
        for s in self.shards:
            s.nprobe = nprobe
        self._graphs.clear()

    def get_ntotal(self) -> int:
        n = torch.tensor([sum(s.ntotal for s in self.shards)], dtype=torch.int64, device=self.device)
        if self.world > 1:
            dist.all_reduce(n, group=self.group)
        return int(n.item())

    # ------------------------------------------------------------------ the hot path
    def search(self, x_t: torch.Tensor, k: int, maximize: bool = False, src: Optional[int] = 0):
        """Collective.  x_t: float32 [nq, d] on this rank's device; the contents of rank `src`
        are used (broadcast) -- the other ranks only need to pass a tensor of the same shape;
        `src=None` says every rank already holds the batch (no broadcast).
        Returns (D [nq,k] float32 ascending -- negated scores when `maximize`, as the reference
        returns them for metric "dot" --, I [nq,k] int64 caller ids, -1 = no result), on device,
        identical on every rank."""
        out = self.search_ex(x_t, k, maximize, src)
        return out.D, out.I

    def search_ex(self, x_t: torch.Tensor, k: int, maximize: bool = False, src: Optional[int] = 0, *,
                  ids: str = "table", shard_ok: Optional[Sequence[bool]] = None, status: int = 0,
                  cols: Optional[Sequence] = None, drop_codes: Optional[Sequence[int]] = None,
                  k_out: Optional[int] = None, return_embeddings: bool = False,
                  meta_tables: Optional[Sequence] = None, dst: int = 0) -> SearchOut:
        """The collective with every option of the client API (see _search_ex_eager).  Small
        batches of the plain form are replayed from a captured CUDA graph."""
        if (self._graph_max_nq and x_t.is_cuda and x_t.shape[0] <= self._graph_max_nq and cols is None
                and not return_embeddings and (shard_ok is None or all(shard_ok))):
            out = self._search_ex_graphed(x_t, k, maximize, ids, status)
            if out is not None:
                return out
        return self._search_ex_eager(x_t, k, maximize, src, ids=ids, shard_ok=shard_ok, status=status, cols=cols,
                                     drop_codes=drop_codes, k_out=k_out, return_embeddings=return_embeddings,
                                     meta_tables=meta_tables, dst=dst)

    def _search_ex_graphed(self, x_t, k, maximize, ids, status):
        gens = tuple(s.generation for s in self.shards)
        if gens != self._graph_gens:      # a shard changed (add / nprobe / ...): every capture is stale
            self._graphs.clear()
            self._graph_gens = gens
        key = (tuple(x_t.shape), int(k), bool(maximize), ids, int(status),
               tuple(0 if t is None else t.data_ptr() for t in self.id_tables))
        ent = self._graphs.get(key)
        if ent is None:
            static_x = x_t.clone()
            cur = torch.cuda.current_stream(x_t.device)
            side = torch.cuda.Stream(device=x_t.device)
            side.wait_stream(cur)
            with torch.cuda.stream(side):  # two eager passes: workspaces reach their final size
                for _ in range(2):
                    self._search_ex_eager(static_x, k, maximize, None, ids=ids, status=status)
            cur.wait_stream(side)
            torch.cuda.synchronize(x_t.device)
            graph = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(graph):
                    out = self._search_ex_eager(static_x, k, maximize, None, ids=ids, status=status)
            except RuntimeError as e:  # something in the path is not capturable: stay eager
                import logging

                logging.getLogger("distributed_faiss_b200").warning("CUDA-graph capture failed, disabled: %s", e)
                self._graph_max_nq = 0
                self._graphs.clear()
                torch.cuda.synchronize(x_t.device)
                return None
            ent = (graph, static_x, out)
            self._graphs[key] = ent
        graph, static_x, out = ent
        static_x.copy_(x_t)
        graph.replay()
        return SearchOut(out.D.clone(), out.I.clone(), status=out.status.clone())

    def _search_ex_eager(self, x_t: torch.Tensor, k: int, maximize: bool = False, src: Optional[int] = 0, *,
                         ids: str = "table", shard_ok: Optional[Sequence[bool]] = None, status: int = 0,
                         cols: Optional[Sequence] = None, drop_codes: Optional[Sequence[int]] = None,
                         k_out: Optional[int] = None, return_embeddings: bool = False,
                         meta_tables: Optional[Sequence] = None, dst: int = 0) -> SearchOut:
        """The collective with every option of the client API.

        ids          "table": I = id_tables[j][local id] (or the local id when the table is None);
                     "exchange": I = (global shard << 40) | local id
        shard_ok     per local shard, False = do not search it (not TRAINED): its block is empty
        status       this rank's status word, gathered to every rank in `SearchOut.status`
        cols / drop_codes / k_out
                     search_with_filter: per local shard an int32 device column of metadata codes
                     and the code to drop; the merged k slots are compacted to k_out kept entries
        return_embeddings
                     winners are decoded by the shard that owns them and summed to rank `dst`
                     (requires ids="exchange"); with `meta_tables` the winners' integer metadata
                     is collected the same way
        """
        be = self.backend
        if self.world > 1 and src is not None:
            dist.broadcast(x_t, src=src, group=self.group)
        nq = x_t.shape[0]
        S_loc = len(self.shards)
        n = S_loc * nq * k
        off_I = _align8(4 * n)
        stride = off_I + 8 * n + 8                      # D | I | status word
        dev = x_t.device
        all_packed = torch.empty((self.world * stride,), dtype=torch.uint8, device=dev)
        packed = all_packed[self.rank * stride:(self.rank + 1) * stride]
        D_loc = packed[:4 * n].view(torch.float32).view(S_loc, nq, k)
        I_loc = packed[off_I:off_I + 8 * n].view(torch.int64).view(S_loc, nq, k)
        exchange = ids == "exchange"
        assert exchange or not (return_embeddings or cols), "embeddings / filter need exchange ids"
        failed = []

        def one(j, shard):
            if shard_ok is not None and not shard_ok[j]:
                D_loc[j].fill_(FLT_MAX)
                I_loc[j].fill_(-1)
                return
            try:
                one_checked(j, shard)
            except RuntimeError as e:   # e.g. k beyond the engine's limit: an empty block + status,
                failed.append(str(e))   # never a rank that skips the collective
                D_loc[j].fill_(FLT_MAX)
                I_loc[j].fill_(-1)

        def one_checked(j, shard):
            tag = self.rank * S_loc + j
            table = None if exchange else self.id_tables[j]
            if not exchange and table is None:
                be.search_local(shard, x_t, k, D_loc[j], I_loc[j])
                return
            I_tmp = torch.empty((nq, k), dtype=torch.int64, device=dev)
            be.search_local(shard, x_t, k, D_loc[j], I_tmp)
            if exchange:
                be.encode_ids(I_tmp, tag, I_loc[j], cols[j] if cols else None, drop_codes[j] if cols else -1)
            else:
                be.map_ids(I_tmp, table, I_loc[j])

        if self._streams and S_loc > 1 and nq <= self._stream_max_nq:
            # shards of one rank are independent: alternate them over a few side streams so the
            # short kernels of one shard (table build, re-rank, selection) fill the tail of
            # another shard's list scan
            main = torch.cuda.current_stream(dev)
            ready = torch.cuda.Event()
            ready.record(main)
            for j, shard in enumerate(self.shards):
                st = self._streams[j % len(self._streams)]
                if j < len(self._streams):
                    st.wait_event(ready)
                with torch.cuda.stream(st):
                    one(j, shard)
            for st in self._streams[:min(len(self._streams), S_loc)]:
                done = torch.cuda.Event()
                done.record(st)
                main.wait_event(done)
            # (no record_stream: main waits for every side stream before anything reuses the buffer)
        else:
            for j, shard in enumerate(self.shards):
                one(j, shard)
        if failed:
            import logging

            logging.getLogger("distributed_faiss_b200").error("shard search failed: %s", failed[0])
            status = max(int(status), 4)
        packed[off_I + 8 * n:].view(torch.int64).fill_(int(status))
        self.last_error = failed[0] if failed else None
        if self.world > 1:
            dist.all_gather_into_tensor(all_packed, packed, group=self.group)
        D, I = be.merge_packed(all_packed, self.world, S_loc, nq, k, stride, off_I, maximize)
        out = SearchOut(D, I)
        out.status = all_packed.view(self.world, stride)[:, off_I + 8 * n:].reshape(-1).view(torch.int64)
        if k_out is not None:
            out.D, out.I, out.count = be.filter_compact(D, I, k_out)
        if return_embeddings:
            d = x_t.shape[1]
            kk = out.I.shape[1]
            R = torch.zeros((nq, kk, d), dtype=torch.float32, device=dev)
            for j, shard in enumerate(self.shards):
                if shard_ok is None or shard_ok[j]:
                    be.reconstruct_owned(shard, out.I, R, self.rank * S_loc + j)
            if self.world > 1:
                dist.reduce(R, dst=dst, group=self.group)
            out.embs = R
            if meta_tables is not None:
                Mi = torch.zeros((nq, kk), dtype=torch.int64, device=dev)
                for j in range(S_loc):
                    if meta_tables[j] is None:
                        continue
                    own = (out.I >= 0) & (((out.I >> LOCAL_BITS) & 0xFFFFF) == self.rank * S_loc + j)
                    loc = torch.where(own, out.I & LOCAL_MASK, torch.zeros_like(out.I))
                    Mi += torch.where(own, meta_tables[j][loc], torch.zeros_like(out.I))
                if self.world > 1:
                    dist.reduce(Mi, dst=dst, group=self.group)
                out.meta_int = Mi
        return out

    def search_host(self, x: np.ndarray, k: int, maximize: bool = False, src: Optional[int] = 0):
        """End-to-end form with HOST buffers: pinned staging, H2D of the query batch, the
        collective search, ONE D2H of (D, I).  Returns fresh arrays."""
        nq, d = x.shape
        if self.device.type != "cuda":
            D, I = self.search(torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)), k, maximize, src)
            return D.numpy(), I.numpy()
        if self._pin_q is None or self._pin_q.shape != (nq, d):
            self._pin_q = torch.empty((nq, d), dtype=torch.float32, pin_memory=True)
        off_I = _align8(4 * nq * k)
        nb = off_I + 8 * nq * k
        if self._pin_out is None or self._pin_out.numel() != nb:
            self._pin_out = torch.empty((nb,), dtype=torch.uint8, pin_memory=True)
        self._pin_q.numpy()[...] = x
        x_t = self._pin_q.to(self.device, non_blocking=True)
        D, I = self.search(x_t, k, maximize, src)
        self._pin_out[:4 * nq * k].view(torch.float32).copy_(D.view(-1), non_blocking=True)
        self._pin_out[off_I:].view(torch.int64).copy_(I.view(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        o = self._pin_out.numpy()
        return (o[:4 * nq * k].view(np.float32).reshape(nq, k).copy(),
                o[off_I:].view(np.int64).reshape(nq, k).copy())


# =================================================================================================
# IndexClient.search over the collective
# =================================================================================================
OP_STOP, OP_SEARCH, OP_TIMER_START, OP_TIMER_STOP = 0, 1, 2, 3
F_MAXIMIZE, F_EMBS, F_INT_META, F_FILTER, F_HAVE_QUERY = 1, 2, 4, 8, 16
HDR_WORDS = 32                      # int64 words: 8 scalars + 128 bytes of index id + spare
HDR_RING = 64                       # pinned header buffers in flight (see SearchPlane.__init__)
ST_OK, ST_NOT_TRAINED, ST_META_KIND, ST_NO_INDEX, ST_ERROR = 0, 1, 2, 3, 4

_plane_lock = threading.Lock()
_current_plane = None


def current_plane():
    """The SearchPlane of this process, if one was constructed (IndexClient attaches to it)."""
    return _current_plane


class PlaneError(RuntimeError):
    pass


class SearchPlane:
    """`IndexClient.search` as a collective over the IndexServers of one box.

    servers : this process's IndexServer objects (server rank = plane_rank * len(servers) + j;
              every process hosts the same number).  The client must live in plane rank 0's
              process; the other ranks call `serve_forever()`.
    """

    def __init__(self, servers: Sequence, group=None, backend=None, device=None, register: bool = True):
        global _current_plane
        self.servers = list(servers)
        self.group = group
        self.backend = backend or CudaBackend()
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        self.device = device if device is not None else (
            torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu"))
        self.S_loc = len(self.servers)
        for j, s in enumerate(self.servers):
            assert s.rank == self.rank * self.S_loc + j, "server ranks must be rank-major over the plane"
        self._groups = {}
        self._lock = threading.Lock()          # one search at a time through the plane
        # headers go out through a RING of pinned buffers: the host-to-device copy of a header is
        # asynchronous, and a caller that enqueues device-resident searches back to back (no sync)
        # must not overwrite a header the copy engine has not read yet
        self._hdr_ring = [self._pin((HDR_WORDS,), torch.int64) for _ in range(HDR_RING)]
        self._hdr_done = [None] * HDR_RING
        self._hdr_next = 0
        self._pin_q = None
        self._pin_out = None
        self._t0 = None
        self._stream = torch.cuda.Stream(device=self.device) if self.device.type == "cuda" else None
        if register:
            with _plane_lock:
                _current_plane = self

    # ------------------------------------------------------------ helpers
    def _pin(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, pin_memory=self.device.type == "cuda")

    @property
    def num_servers(self) -> int:
        return self.S_loc * self.world

    def owner_of(self, server_rank: int):
        """local IndexServer for a global server rank, or None when another process hosts it"""
        r, j = divmod(server_rank, self.S_loc)
        return self.servers[j] if r == self.rank else None

    def _stream_ctx(self):
        import contextlib

        return torch.cuda.stream(self._stream) if self._stream is not None else contextlib.nullcontext()

    def _group_for(self, index_id, engines):
        g = self._groups.get(index_id)
        if g is None or any(a is not b for a, b in zip(g.shards, engines)):
            g = ShardGroup(engines, None, group=self.group, backend=self.backend, device=self.device)
            self._groups[index_id] = g
        return g

    # ------------------------------------------------------------ protocol
    def _send_header(self, words: List[int], index_id: str = "", blob: bytes = b""):
        h = np.zeros(HDR_WORDS, dtype=np.int64)
        h[:len(words)] = words
        raw = index_id.encode("utf-8")
        assert len(raw) <= 128, "index id too long for the plane header (128 bytes)"
        h[7] = len(raw)
        h[8:24].view(np.uint8)[:len(raw)] = np.frombuffer(raw, dtype=np.uint8)
        h[24] = len(blob)
        if self.world > 1:
            slot = self._hdr_next
            self._hdr_next = (slot + 1) % HDR_RING
            if self._hdr_done[slot] is not None:
                self._hdr_done[slot].synchronize()   # the copy that last used this buffer has read it
            pin = self._hdr_ring[slot]
            pin.numpy()[...] = h
            h_dev = pin.to(self.device, non_blocking=True)
            if self.device.type == "cuda":
                ev = torch.cuda.Event()
                ev.record()
                self._hdr_done[slot] = ev
            dist.broadcast(h_dev, src=0, group=self.group)
            if blob:
                b_dev = torch.from_numpy(np.frombuffer(blob, dtype=np.uint8).copy()).to(self.device)
                dist.broadcast(b_dev, src=0, group=self.group)
        return h

    def _recv_header(self):
        h_dev = torch.empty((HDR_WORDS,), dtype=torch.int64, device=self.device)
        dist.broadcast(h_dev, src=0, group=self.group)
        h = h_dev.cpu().numpy()
        blob = b""
        if h[24] > 0:
            b_dev = torch.empty((int(h[24]),), dtype=torch.uint8, device=self.device)
            dist.broadcast(b_dev, src=0, group=self.group)
            blob = b_dev.cpu().numpy().tobytes()
        index_id = h[8:24].view(np.uint8)[:int(h[7])].tobytes().decode("utf-8")
        return h, index_id, blob

    def serve_forever(self):
        """Ranks != 0: execute the collectives the client rank announces, until `stop()`."""
        assert self.rank != 0
        with self._stream_ctx():
            while True:
                h, index_id, blob = self._recv_header()
                op = int(h[0])
                if op == OP_STOP:
                    return
                if op == OP_TIMER_START:
                    self._timer_start()
                elif op == OP_TIMER_STOP:
                    self._timer_stop()
                elif op == OP_SEARCH:
                    self._run_search(h, index_id, blob, None)

    def stop(self):
        global _current_plane
        with _plane_lock:   # an IndexClient created from now on must not attach to a stopped plane
            if _current_plane is self:
                _current_plane = None
        if self.rank == 0 and self.world > 1:
            with self._lock, self._stream_ctx():
                self._send_header([OP_STOP])
                if self._stream is not None:
                    self._stream.synchronize()

    # device timing, max over ranks (bench): every rank brackets the same collectives
    def _timer_start(self):
        if self.device.type == "cuda":
            self._t0 = torch.cuda.Event(enable_timing=True)
            self._t0.record()
        else:
            import time

            self._t0 = time.perf_counter()

    def _timer_stop(self):
        if self.device.type == "cuda":
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            e1.synchronize()
            ms = self._t0.elapsed_time(e1)
        else:
            import time

            ms = 1e3 * (time.perf_counter() - self._t0)
        t = torch.tensor([ms], dtype=torch.float64, device=self.device)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return float(t.item())

    def timer_start(self):
        with self._lock, self._stream_ctx():
            self._send_header([OP_TIMER_START])
            self._timer_start()

    def timer_stop(self) -> float:
        with self._lock, self._stream_ctx():
            self._send_header([OP_TIMER_STOP])
            return self._timer_stop()

    # ------------------------------------------------------------ the collective, every rank
    def _run_search(self, h, index_id, blob, x_t) -> SearchOut:
        nq, k, flags, d = int(h[1]), int(h[2]), int(h[3]), int(h[4])
        k_out = int(h[6]) if flags & F_FILTER else None
        if x_t is None:
            x_t = torch.empty((nq, d), dtype=torch.float32, device=self.device)
        indexes = [s.indexes.get(index_id) for s in self.servers]
        status = ST_OK if all(ix is not None for ix in indexes) else ST_NO_INDEX
        embs = bool(flags & F_EMBS)
        exchange = embs or not (flags & F_INT_META)
        # metadata tables / filter columns first (they take buffer_lock; never under index_lock).
        # Nothing before the collectives may raise on one rank only: failures become status words.
        tables = cols = drops = None
        try:
            if flags & F_INT_META:
                tables = [ix.meta_int_table(self.device) if ix is not None else None for ix in indexes]
                if any(t is None and ix is not None for t, ix in zip(tables, indexes)):
                    status = max(status, ST_META_KIND)
            if flags & F_FILTER:
                fpos, fval = pickle.loads(blob)
                cd = [ix.filter_column(fpos, fval, self.device) if ix is not None else (None, -1) for ix in indexes]
                cols, drops = [c for c, _ in cd], [v for _, v in cd]
        except Exception:
            import logging

            logging.getLogger("distributed_faiss_b200").exception("plane rank %d: metadata tables failed", self.rank)
            status = max(status, ST_ERROR)
        locked = []
        try:
            engines, ok = [], []
            for ix in indexes:
                if ix is None:
                    engines.append(None)
                    ok.append(False)
                    continue
                ix.index_lock.acquire()   # one search at a time per shard (reference index.py:246-252)
                locked.append(ix)
                trained = ix.is_searchable()
                if not trained:
                    status = max(status, ST_NOT_TRAINED)
                engines.append(ix.faiss_index)
                ok.append(trained and status in (ST_OK, ST_NOT_TRAINED))
            grp = self._group_for(index_id, engines)
            grp.id_tables = tables if (tables is not None and not exchange) else [None] * len(engines)
            return grp.search_ex(x_t, k, bool(flags & F_MAXIMIZE), 0 if (flags & F_HAVE_QUERY) else None,
                                 ids="exchange" if exchange else "table", shard_ok=ok, status=status,
                                 cols=cols, drop_codes=drops, k_out=k_out, return_embeddings=embs,
                                 meta_tables=tables if embs else None)
        finally:
            for ix in locked:
                ix.index_lock.release()

    # ------------------------------------------------------------ client side (plane rank 0)
    def search(self, index_id: str, query, k: int, *, maximize: bool, return_embeddings: bool = False,
               int_meta: bool = False, filter_pos: int = -1, filter_value=None, k_out: Optional[int] = None):
        """Returns host arrays (D [nq,kk] f32, I [nq,kk] i64, count [nq] i32 | None,
        embs [nq,kk,d] f32 | None, meta_int [nq,kk] i64 | None).  I holds caller integers in
        int_meta mode (no embeddings) and exchange ids otherwise."""
        assert self.rank == 0, "the client lives in the process of plane rank 0"
        on_dev = isinstance(query, torch.Tensor)
        nq, d = query.shape
        flags = (F_MAXIMIZE if maximize else 0) | (F_EMBS if return_embeddings else 0) | \
                (F_INT_META if int_meta else 0) | (F_FILTER if filter_pos >= 0 else 0) | F_HAVE_QUERY
        blob = pickle.dumps((filter_pos, filter_value)) if filter_pos >= 0 else b""
        if self._stream is not None:   # the caller's stream produced the query (device form)
            self._stream.wait_stream(torch.cuda.current_stream(self.device))
        with self._lock, self._stream_ctx():
            h = self._send_header([OP_SEARCH, nq, k, flags, d, filter_pos, k_out or 0], index_id, blob)
            if on_dev:
                x_t = query
            elif self.device.type == "cuda":
                if self._pin_q is None or self._pin_q.shape != (nq, d):
                    self._pin_q = self._pin((nq, d), torch.float32)
                self._pin_q.numpy()[...] = query
                x_t = self._pin_q.to(self.device, non_blocking=True)
            else:
                x_t = torch.from_numpy(np.ascontiguousarray(query, dtype=np.float32))
            out = self._run_search(h, index_id, blob, x_t)
            if not on_dev:
                return self._to_host(out)
        if self._stream is not None:   # device form: results are ordered after the caller's stream
            torch.cuda.current_stream(self.device).wait_stream(self._stream)
        return out

    def _to_host(self, out: SearchOut):
        parts = [out.D.reshape(-1).view(torch.uint8), out.I.reshape(-1).view(torch.uint8),
                 out.status.reshape(-1).view(torch.uint8)]
        if out.count is not None:
            parts.append(out.count.reshape(-1).view(torch.uint8))
        if out.meta_int is not None:
            parts.append(out.meta_int.reshape(-1).view(torch.uint8))
        sizes = [p.numel() for p in parts]
        total = sum(sizes)
        if self.device.type == "cuda":
            if self._pin_out is None or self._pin_out.numel() < total:
                self._pin_out = self._pin((max(total, 1 << 16),), torch.uint8)
            off = 0
            for p, s in zip(parts, sizes):
                self._pin_out[off:off + s].copy_(p, non_blocking=True)
                off += s
            embs = None
            if out.embs is not None:
                embs_pin = self._pin(tuple(out.embs.shape), torch.float32)
                embs_pin.copy_(out.embs, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            host = self._pin_out.numpy()[:total].copy()
            if out.embs is not None:
                embs = embs_pin.numpy()
        else:
            host = np.concatenate([p.numpy() for p in parts])
            embs = out.embs.numpy() if out.embs is not None else None
        nq, kk = out.D.shape
        off = 0
        D = host[off:off + sizes[0]].view(np.float32).reshape(nq, kk)
        off += sizes[0]
        I = host[off:off + sizes[1]].view(np.int64).reshape(nq, kk)
        off += sizes[1]
        status = host[off:off + sizes[2]].view(np.int64)
        off += sizes[2]
        count = meta_int = None
        i = 3
        if out.count is not None:
            count = host[off:off + sizes[i]].view(np.int32)
            off += sizes[i]
            i += 1
        if out.meta_int is not None:
            meta_int = host[off:off + sizes[i]].view(np.int64).reshape(nq, kk)
        st = int(status.max()) if status.size else ST_OK
        if st == ST_NOT_TRAINED:
            raise PlaneError("Server index is not trained. (reported by plane rank(s) "
                             f"{np.nonzero(status == ST_NOT_TRAINED)[0].tolist()})")
        if st == ST_NO_INDEX:
            raise PlaneError("Server has no index with this id (plane rank(s) "
                             f"{np.nonzero(status == ST_NO_INDEX)[0].tolist()})")
        if st == ST_META_KIND:
            raise MetaKindChanged()
        if st == ST_ERROR:
            local = [g.last_error for g in self._groups.values() if g.last_error]
            raise PlaneError(f"shard search failed on plane rank(s) {np.nonzero(status == ST_ERROR)[0].tolist()}"
                             + (f": {local[0]}" if local else " (see that rank's log)"))
        return D, I, count, embs, meta_int


class MetaKindChanged(PlaneError):
    """a shard's metadata stopped being all-integer since the client last asked"""


def init_process_group_from_env(backend: Optional[str] = None):
    """One process per GPU launched by torchrun: RANK / LOCAL_RANK / WORLD_SIZE / MASTER_*."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if torch.cuda.is_available():
        torch.cuda.set_device(local_rank % torch.cuda.device_count())
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        kw = {}
        if torch.cuda.is_available():
            kw["device_id"] = torch.device("cuda", torch.cuda.current_device())
        dist.init_process_group(backend or ("nccl" if torch.cuda.is_available() else "gloo"),
                                rank=rank, world_size=world, **kw)
    return rank, local_rank, world
