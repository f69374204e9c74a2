"""One shard: RAM buffer -> train -> add -> search, over a GPU-resident engine.

Behavioural mirror of the reference's `Index` (distributed_faiss/index.py:111-508):
same public methods, same state machine (NOT_TRAINED -> TRAINING -> TRAINED -> ADD ->
TRAINED), same `train_num` / `train_ratio` / `buffer_bsz` semantics, same id -> metadata
convention (local id = arrival order on this shard, index.py:155,264).  What changes is
the object behind `self.faiss_index`: instead of a CPU faiss index it is a
`engine.GpuIndex` whose vectors live in the HBM of one B200 and whose `.search` runs the
hand-written sm_100a kernels of libdfx.so.  There is no CPU fallback.

Builders (reference index.py:93-100):
  "flat"       -> IndexFlatIP            (always inner product, quirk B1 of SURVEY.md)
  "ivf_simple" -> IndexIVFFlat(metric)   nprobe = cfg.nprobe
  "knnlm"      -> IndexIVFPQ             always L2 / by_residual; M = extra["code_size"] (64),
                                          nbits = extra["bits_per_vector"] (8; 4 halves the
                                          code bytes, needs M % 8 == 0); cfg.nprobe is
                                          overwritten by the index default 1 (quirk B3)
  "ivfsq"      -> IndexIVFScalarQuantizer(QT_fp16), always L2, nprobe = cfg.nprobe
"hnswsq", "ivf_gpu" and free-form `faiss_factory` strings are outside the hot path this
package rebuilds (SURVEY.md section 8) and raise.
"""
import _thread
import logging
import math
import os
import pickle
import threading
import time
from typing import Callable, List, Optional, Tuple, Union

import numpy as np

from .index_cfg import IndexCfg, METRIC_INNER_PRODUCT
from .index_state import IndexState

logger = logging.getLogger("distributed_faiss_b200")

INDEX_FILE = "index.dfx.npz"
# the reference's file name (index.py:104); written instead of INDEX_FILE when the cfg carries
# index_format="faiss", and read when no INDEX_FILE is present (see faiss_io.py)
FAISS_INDEX_FILE = "index.faiss"


def default_engine_factory(cfg: IndexCfg, device: Optional[int] = None):
    """cfg -> GPU engine object (the CUDA library is loaded here; fails loudly without it).
    `device`: the GPU ordinal of the owning IndexServer rank; None = the calling thread's current
    device (only safe on the thread that was pinned, see Index._bind_device)."""
    from . import engine

    btype = cfg.index_builder_type
    if btype == "flat":
        return engine.GpuIndex(engine.KIND_FLAT, cfg.dim, METRIC_INNER_PRODUCT, device=device)
    if btype == "ivf_simple":
        idx = engine.GpuIndex(engine.KIND_IVF_FLAT, cfg.dim, cfg.get_metric(), nlist=int(cfg.centroids),
                              device=device)
        idx.nprobe = cfg.nprobe
        return idx
    if btype == "knnlm":
        idx = engine.GpuIndex(engine.KIND_IVF_PQ, cfg.dim, cfg.get_metric(), nlist=int(cfg.centroids),
                              pq_m=int(cfg.extra.get("code_size", 64)),
                              pq_nbits=int(cfg.extra.get("bits_per_vector", 8)), device=device)
        cfg.nprobe = idx.nprobe  # the reference copies the index default back into cfg (index.py:47)
        return idx
    if btype == "ivfsq":
        idx = engine.GpuIndex(engine.KIND_IVF_SQ16, cfg.dim, cfg.get_metric(), nlist=int(cfg.centroids),
                              device=device)
        idx.nprobe = cfg.nprobe
        return idx
    if btype in ("hnswsq", "ivf_gpu") or cfg.faiss_factory:
        raise RuntimeError(
            f"index_builder_type={btype!r} / faiss_factory={cfg.faiss_factory!r} is not part of the "
            "B200 search path (supported builders: flat, ivf_simple, knnlm, ivfsq)")
    raise RuntimeError("Either faiss_factory or valid index_builder_type should be specified to initialize index")


class IntMetadata:
    """`id_to_metadata` of a shard adopted from the device: local id -> integer, kept as an int64
    tensor (1 B vectors worth of Python ints would not fit a host).  Read-only sequence."""

    def __init__(self, table):
        self.table = table
        self._host = None

    def __len__(self):
        return int(self.table.shape[0])

    def __getitem__(self, i):
        return int(self.table[i])

    def lookup(self, ids: np.ndarray):
        import torch

        ids = np.asarray(ids, dtype=np.int64)
        t = torch.from_numpy(np.where(ids < 0, 0, ids).reshape(-1)).to(self.table.device)
        vals = self.table[t].cpu().numpy().reshape(ids.shape)
        out = vals.astype(object)
        out[ids < 0] = None
        return out.tolist()


def get_index_files(index_storage_dir: str) -> Tuple[str, str, str, str]:
    return tuple(os.path.join(index_storage_dir, f) for f in (INDEX_FILE, "meta.pkl", "buffer.pkl", "cfg.json"))


class Index:
    def __init__(self, cfg: IndexCfg, engine_factory: Optional[Callable] = None, device: Optional[int] = None):
        self.cfg = cfg
        # the GPU of the owning server rank, resolved ONCE here: training and adds run on threads
        # started with _thread.start_new_thread, whose current CUDA device would be 0
        self.device = device
        if engine_factory is None:
            if device is None:
                try:
                    import torch

                    if torch.cuda.is_available():
                        self.device = torch.cuda.current_device()
                except Exception:
                    pass
            dev = self.device
            self._engine_factory = lambda c: default_engine_factory(c, dev)
        else:
            self._engine_factory = engine_factory
        self._stop_watcher = threading.Event()
        self.embeddings_buffer: List[np.ndarray] = []
        self.total_data = 0
        self.id_to_metadata: List[object] = []
        self._meta_arr = None  # object-array view of id_to_metadata, rebuilt lazily
        self._meta_int_cache = None  # (len(id_to_metadata), int64 device table | None), see meta_int_table
        self._filter_cols = {}  # filter_pos -> (len(id_to_metadata), int32 device codes, {value: code})
        self.buffer_lock = threading.Lock()
        self.index_lock = threading.Lock()
        self.state = IndexState.NOT_TRAINED
        self.faiss_index = None  # the engine object; the name is part of the reference surface
        self.index_save_time = time.time()
        self.index_saved_size = 0
        if cfg.save_interval_sec > 0:
            self._run_save_watcher()

    # ------------------------------------------------------------ ingest
    def _bind_device(self):
        """pin the calling thread to this shard's GPU (no-op for injected engines / no GPU)"""
        if self.device is None:
            return
        import torch

        if torch.cuda.is_available():
            torch.cuda.set_device(self.device)

    def drop_index(self):
        self._stop_watcher.set()
        with self.buffer_lock:
            self.embeddings_buffer, self.total_data, self.id_to_metadata = [], 0, []
            self._meta_arr = None
        with self.index_lock:
            self.faiss_index = None
            self.state = IndexState.NOT_TRAINED

    def add_batch(self, embeddings: np.ndarray, metadata: Optional[List[object]],
                  train_async_if_triggered: bool = True):
        n = embeddings.shape[0]
        if not metadata:
            metadata = [None] * n
        if n != len(metadata):
            raise RuntimeError("metadata length should match the batch size of the embeddings")
        embeddings = np.ascontiguousarray(embeddings, dtype=np.float32)
        with self.buffer_lock:
            self.embeddings_buffer.append(embeddings)
            self.id_to_metadata.extend(metadata)
            self._meta_arr = None
            self.total_data += n
            buffered = self.total_data
        state = self.get_state()
        if state == IndexState.TRAINED:
            self.add_buffer_to_index()
        elif state == IndexState.NOT_TRAINED and 0 < self.cfg.train_num <= buffered:
            if train_async_if_triggered:
                _thread.start_new_thread(self.train, ())
            else:
                self.train()

    def get_idx_data_num(self) -> Tuple[int, int]:
        with self.buffer_lock:
            buffered = self.total_data
        with self.index_lock:
            indexed = self.faiss_index.ntotal if self.faiss_index else 0
        return buffered, indexed

    def train(self) -> None:
        self._bind_device()
        with self.index_lock:
            if self.state != IndexState.NOT_TRAINED:
                return
            self.state = IndexState.TRAINING
        cfg = self.cfg
        try:
            with self.buffer_lock:
                if cfg.dim == 0:
                    cfg.dim = self.embeddings_buffer[0].shape[1]
                if cfg.train_num > 0:
                    train_num = cfg.train_num
                elif cfg.train_ratio >= 1.0:
                    train_num = self.total_data
                else:
                    train_num = int(cfg.train_ratio * self.total_data)
                everything = np.concatenate(self.embeddings_buffer, axis=0)
            # the reference trains on the FIRST train_num buffered rows, shuffled (index.py:202-211)
            train_data = everything[:train_num].copy()
            np.random.shuffle(train_data)
            engine = self._init_engine(everything.shape[0])
            engine.train(train_data)
        except BaseException:
            with self.index_lock:
                self.state = IndexState.NOT_TRAINED
            raise
        with self.index_lock:
            self.faiss_index = engine
            self.state = IndexState.TRAINED
        self.add_buffer_to_index()

    def add_buffer_to_index(self) -> None:
        with self.index_lock:
            start = self.state == IndexState.TRAINED
            if start:
                self.state = IndexState.ADD
        if start:
            # background thread, so that the client's next batch can go to the next shard
            _thread.start_new_thread(self._add_buffer_to_idx, ())

    def _add_buffer_to_idx(self):
        self._bind_device()
        try:
            while True:
                with self.buffer_lock:
                    take, rows = [], 0
                    for chunk in self.embeddings_buffer:
                        take.append(chunk)
                        rows += chunk.shape[0]
                        if rows >= self.cfg.buffer_bsz:
                            break
                    if rows == 0:
                        break
                    self.embeddings_buffer = self.embeddings_buffer[len(take):]
                    self.total_data -= rows
                self.faiss_index.add(np.concatenate(take, axis=0) if len(take) > 1 else take[0])
                self._maybe_save(ignore_time=False)
        finally:
            with self.index_lock:
                self.state = IndexState.TRAINED

    # ------------------------------------------------------------ search (the hot path)
    def search(self, query_batch: np.ndarray, top_k: int = 100, return_embeddings: bool = False
               ) -> Tuple[np.ndarray, List[List[object]], Optional[np.ndarray]]:
        with self.index_lock:
            if self.state != IndexState.TRAINED:
                raise RuntimeError(f"Server index is not trained. state: {self.state}")
            # one search at a time per shard, as in the reference (index.py:246-252)
            if return_embeddings:
                scores, ids, embs = self.faiss_index.search_and_reconstruct(query_batch, top_k)
            else:
                scores, ids = self.faiss_index.search(query_batch, top_k)
                embs = None
        return scores, self._ids_to_meta(ids), embs

    # ---- the NCCL data plane (spmd.SearchPlane) drives the engine directly, under the same rules
    def is_searchable(self) -> bool:
        """caller holds index_lock; same condition as search() (reference index.py:247)"""
        return self.state == IndexState.TRAINED and self.faiss_index is not None

    def adopt_engine(self, engine, meta_table=None) -> None:
        """Install a shard that was built directly on the device (bench / bulk loaders that cannot
        afford host round trips): the engine becomes `faiss_index`, state TRAINED.  `meta_table`
        (int64 device tensor, local id -> integer metadata) stands in for `id_to_metadata`."""
        with self.buffer_lock, self.index_lock:
            self.faiss_index = engine
            self.state = IndexState.TRAINED
            if meta_table is not None:
                self.id_to_metadata = IntMetadata(meta_table)
            self._meta_arr = None
            self._meta_int_cache = None
            self._filter_cols = {}

    def meta_int_table(self, device):
        """int64 device tensor `local id -> metadata` when EVERY metadata entry of this shard is a
        non-negative integer (the convention of scripts/load_data.py:120-124), else None.  This is
        the device form of the id -> metadata loop of the reference (index.py:260-268)."""
        import torch

        with self.buffer_lock:
            n = len(self.id_to_metadata)
            c = self._meta_int_cache
            if c is not None and c[0] == n:
                return c[1]
            tab = None
            if isinstance(self.id_to_metadata, IntMetadata):
                tab = self.id_to_metadata.table.to(device)
            else:
                try:
                    arr = np.asarray(self.id_to_metadata)
                except ValueError:  # ragged tuples
                    arr = None
                if arr is not None and arr.ndim == 1 and arr.dtype.kind in "iu" and (n == 0 or arr.min() >= 0):
                    tab = torch.from_numpy(arr.astype(np.int64)).to(device)
            self._meta_int_cache = (n, tab)
            return tab

    def filter_column(self, filter_pos: int, filter_value, device):
        """(int32 device codes of metadata[filter_pos] per local id, code of filter_value).
        Code -2 = what the reference's post-filter skips outright (no metadata, or a tuple too short,
        client.py:235-241); entries whose code equals the returned drop code are the ones with
        metadata[filter_pos] == filter_value."""
        import torch

        with self.buffer_lock:
            n = len(self.id_to_metadata)
            c = self._filter_cols.get(filter_pos)
            if c is None or c[0] != n:
                codes = np.full(n, -2, dtype=np.int32)
                vocab = c[2] if c is not None else {}
                start = 0
                if c is not None and c[0] < n:      # metadata only grows: extend the old column
                    codes[:c[0]] = c[3]
                    start = c[0]
                for i in range(start, n):
                    m = self.id_to_metadata[i]
                    try:
                        if m and len(m) > filter_pos:
                            codes[i] = vocab.setdefault(m[filter_pos], len(vocab))
                    except TypeError:               # no len() / unhashable value: never kept, never matched
                        pass
                c = (n, torch.from_numpy(codes).to(device), vocab, codes)
                self._filter_cols[filter_pos] = c
            try:
                drop = c[2].get(filter_value, -1)
            except TypeError:
                drop = -1
            return c[1], drop

    def lookup_meta(self, local_ids) -> List[object]:
        """metadata objects of shard-local ids (flat list; -1 -> None)"""
        return self._ids_to_meta(np.asarray(local_ids, dtype=np.int64).reshape(-1))

    def get_meta_kind(self) -> str:
        """"int" when the integer fast path applies to this shard, else "object" """
        with self.buffer_lock:
            if isinstance(self.id_to_metadata, IntMetadata):
                return "int"
            try:
                arr = np.asarray(self.id_to_metadata)
            except ValueError:
                return "object"
            ok = arr.ndim == 1 and arr.dtype.kind in "iu" and (arr.size == 0 or arr.min() >= 0)
            return "int" if ok else "object"

    def search_ids(self, query_batch: np.ndarray, top_k: int) -> Tuple[np.ndarray, np.ndarray]:
        """Same as search() but returns shard-local ids (used by the NCCL data plane)."""
        with self.index_lock:
            if self.state != IndexState.TRAINED:
                raise RuntimeError(f"Server index is not trained. state: {self.state}")
            return self.faiss_index.search(query_batch, top_k)

    def _ids_to_meta(self, ids: np.ndarray) -> List[List[object]]:
        # vectorised form of the reference's O(nq*k) double loop (index.py:260-268): -1 -> None
        with self.buffer_lock:
            if isinstance(self.id_to_metadata, IntMetadata):
                return self.id_to_metadata.lookup(ids)
            if self._meta_arr is None or self._meta_arr.shape[0] != len(self.id_to_metadata) + 1:
                arr = np.empty(len(self.id_to_metadata) + 1, dtype=object)
                arr[:-1] = self.id_to_metadata
                arr[-1] = None
                self._meta_arr = arr
            return self._meta_arr[ids].tolist()  # index -1 hits the trailing None

    # ------------------------------------------------------------ accessors
    def get_centroids(self):
        with self.index_lock:
            if self.state != IndexState.TRAINED:
                raise RuntimeError("Server index is not trained")
            return self.faiss_index.quantizer.reconstruct_n(0, self.faiss_index.nlist)

    def set_nprobe(self, nprobe: int):
        self.cfg.nprobe = nprobe
        with self.index_lock:
            if self.faiss_index:
                self.faiss_index.nprobe = nprobe

    def get_state(self):
        with self.index_lock:
            return self.state

    def get_ids(self):
        pos = self.cfg.custom_meta_id_idx
        return {meta[pos] for meta in self.id_to_metadata if meta}

    def upd_cfg(self, cfg: IndexCfg):
        self.cfg = cfg
        self._override_nprobe(cfg)

    def _override_nprobe(self, cfg: IndexCfg):
        if self.faiss_index is not None and hasattr(self.faiss_index, "nprobe"):
            self.faiss_index.nprobe = cfg.nprobe

    def _init_engine(self, total_data_size: int):
        cfg = self.cfg
        if not cfg.index_builder_type and cfg.faiss_factory:
            cfg.centroids = int(cfg.centroids)
            if cfg.centroids == 0 or cfg.infer_centroids:
                cfg.centroids = self.infer_n_centroids(total_data_size)
        return self._engine_factory(cfg)

    @staticmethod
    def infer_n_centroids(total_data_size):
        # reference tiers (index.py:497-508)
        if total_data_size < 10e5:
            return int(2 * math.sqrt(total_data_size))
        if total_data_size < 10e6:
            return 65536
        if total_data_size < 10e7:
            return 262144
        return 1048576

    # ------------------------------------------------------------ persistence
    def save(self) -> bool:
        state = self.get_state()
        if state == IndexState.TRAINED:
            return self._maybe_save(ignore_time=True)
        if state == IndexState.ADD:
            self.index_save_time = 0  # save as soon as the running add finishes
        return False

    def _maybe_save(self, ignore_time: bool = False) -> bool:
        if not ignore_time:
            if self.cfg.save_interval_sec <= 0:
                return False
            if time.time() - self.index_save_time < self.cfg.save_interval_sec:
                return False
        with self.buffer_lock, self.index_lock:
            if self.faiss_index is None or self.faiss_index.ntotal == self.index_saved_size:
                return False
            index_file, meta_file, buffer_file, cfg_file = get_index_files(self.cfg.index_storage_dir)
            state = self.faiss_index.get_state()
            if self.cfg.extra.get("index_format", "dfx") == "faiss":
                from . import faiss_io

                index_file = os.path.join(self.cfg.index_storage_dir, FAISS_INDEX_FILE)
                tmp = index_file + ".tmp"
                faiss_io.write_index(state, tmp, nprobe=int(getattr(self.faiss_index, "nprobe", 1)))
            else:
                tmp = index_file + ".tmp.npz"
                np.savez(tmp, **{k: np.asarray(v) for k, v in state.items()})
            os.replace(tmp, index_file)
            with open(meta_file, "wb") as fh:
                pickle.dump(self.id_to_metadata, fh)
            with open(buffer_file, "wb") as fh:
                pickle.dump(self.embeddings_buffer, fh)
            with open(cfg_file, "w") as fh:
                fh.write(self.cfg.to_json_string() + "\n")
            self.index_saved_size = self.faiss_index.ntotal
            self.index_save_time = time.time()
            return True

    def _run_save_watcher(self):
        import weakref

        # the watcher must not keep a dropped shard (and its HBM) alive: weak reference + stop flag
        ref, stop, period = weakref.ref(self), self._stop_watcher, self.cfg.save_interval_sec

        def loop():
            while not stop.wait(period):
                idx = ref()
                if idx is None:
                    return
                idx._bind_device()
                idx._maybe_save(ignore_time=False)
                del idx

        _thread.start_new_thread(loop, ())

    @classmethod
    def from_storage_dir(cls, index_storage_dir: str, cfg: IndexCfg = None, ignore_buffer: bool = True,
                         engine_factory: Optional[Callable] = None, device: Optional[int] = None
                         ) -> Union[None, "Index"]:
        index_file, meta_file, buffer_file, cfg_file = get_index_files(index_storage_dir)
        faiss_file = os.path.join(index_storage_dir, FAISS_INDEX_FILE)
        if not os.path.exists(index_file) and not os.path.exists(faiss_file):
            return None
        if not os.path.exists(meta_file):
            raise RuntimeError("no meta file found. Can't use index.")
        with open(meta_file, "rb") as fh:
            meta = pickle.load(fh)
        buffer = []
        if (not ignore_buffer) and os.path.exists(buffer_file):
            with open(buffer_file, "rb") as fh:
                buffer = pickle.load(fh)
        if cfg is None:
            cfg = IndexCfg.from_json(cfg_file) if os.path.isfile(cfg_file) else IndexCfg()
        result = cls(cfg, engine_factory=engine_factory, device=device)
        # builder type / sizes come from the cfg stored next to the index when the caller's cfg lacks them
        build_cfg = cfg
        if not cfg.index_builder_type and os.path.isfile(cfg_file):
            build_cfg = IndexCfg.from_json(cfg_file)
        if os.path.exists(index_file):
            with np.load(index_file, allow_pickle=False) as z:
                state = {k: (z[k].item() if z[k].ndim == 0 else z[k]) for k in z.files}
        else:  # a shard saved by the reference (faiss.write_index) or with index_format="faiss"
            from . import faiss_io

            state, _ = faiss_io.read_index(faiss_file)
        saved_nprobe = cfg.nprobe
        engine = result._engine_factory(build_cfg)
        cfg.nprobe = saved_nprobe
        engine.set_state(state)
        assert len(meta) >= engine.ntotal, "Deserialized meta list should be at least of index size"
        result.faiss_index = engine
        result.state = IndexState.TRAINED
        result.upd_cfg(cfg)
        buffered = sum(v.shape[0] for v in buffer)
        if len(meta) == engine.ntotal + buffered:
            result.id_to_metadata = meta
            result.embeddings_buffer = buffer
            result.total_data = buffered
            if buffered > 0:
                result.add_buffer_to_index()
        else:
            result.id_to_metadata = meta[: engine.ntotal]
        result.index_saved_size = engine.ntotal
        return result
