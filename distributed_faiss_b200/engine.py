"""ctypes binding of libdfx.so (include/dfx.h) and the engine objects that replace
`Index.faiss_index` of the reference.

The reference keeps a SWIG-wrapped faiss object in `Index.faiss_index`
(distributed_faiss/index.py:120) and touches exactly this surface:
`.train(x)` (index.py:217), `.add(x)` (index.py:425), `.search(x, k)` (index.py:257),
`.search_and_reconstruct(x, k)` (index.py:255), `.ntotal` (index.py:184),
`.nprobe` (index.py:356, 495), `.nlist` / `.quantizer.reconstruct_n(0, nlist)`
(index.py:350), and the absence of `.hnsw` (index.py:491).  `GpuIndex` exposes the
same names over the C-ABI; all arithmetic happens in the CUDA library.

There is NO CPU fallback: if libdfx.so is missing or no sm_100 device is
present every computing call raises RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdfx.so")

KIND_FLAT, KIND_IVF_FLAT, KIND_IVF_PQ, KIND_IVF_SQ16 = 0, 1, 2, 3
METRIC_INNER_PRODUCT, METRIC_L2 = 0, 1  # faiss enum values (reference index_cfg.py:44-52)
KIND_NAMES = {KIND_FLAT: "flat", KIND_IVF_FLAT: "ivf_flat", KIND_IVF_PQ: "ivf_pq", KIND_IVF_SQ16: "ivf_sq"}

# every symbol include/dfx.h declares (tests check that the library exports each one)
EXPORTED_SYMBOLS = [
    "dfx_create", "dfx_destroy", "dfx_train", "dfx_add", "dfx_train_dev", "dfx_add_dev", "dfx_set_param", "dfx_get_param",
    "dfx_reserve", "dfx_finalize", "dfx_search", "dfx_search_dev", "dfx_reconstruct", "dfx_set_nprobe",
    "dfx_get_nprobe", "dfx_generation", "dfx_ntotal", "dfx_nlist", "dfx_is_trained", "dfx_get_centroids", "dfx_merge",
    "dfx_merge_dev", "dfx_merge_packed_dev", "dfx_encode_ids_dev", "dfx_filter_compact_dev",
    "dfx_reconstruct_dev", "dfx_map_ids_dev", "dfx_get_array", "dfx_set_array", "dfx_import_done",
    "dfx_last_stats", "dfx_profile_enable", "dfx_profile_read", "dfx_launch_count", "dfx_synth_init", "dfx_synth_rows_dev", "dfx_free",
    "dfx_last_error", "dfx_version", "dfx_debug_il_byte",
]


class DfxCfg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("metric", C.c_int32), ("d", C.c_int32), ("pq_m", C.c_int32),
                ("pq_nbits", C.c_int32), ("device", C.c_int32), ("nlist", C.c_int64)]


class DfxSynth(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("d", C.c_int32), ("r", C.c_int32), ("nclusters", C.c_int64),
                ("ngroups", C.c_int64), ("sigma", C.c_float), ("eps", C.c_float), ("sigma_q", C.c_float),
                ("delta", C.c_float)]


_lib = None
_lib_lock = threading.Lock()


def lib():
    """Load libdfx.so (fails loudly -- there is no fallback implementation)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -m distributed_faiss_b200.build` "
                    "(or __graft_entry__.build()). There is no CPU fallback for the search path.")
            if LIB_PATH == os.path.join(_HERE, "libdfx.so") and os.path.isdir(os.path.join(_HERE, "csrc")):
                # a binary that does not match the sources next to it is rebuilt, never used silently
                from . import build as _build
                if not _build.is_current():
                    _build.build()
            L = C.CDLL(LIB_PATH)
            L.dfx_last_error.restype = C.c_char_p
            L.dfx_version.restype = C.c_char_p
            for f in ("dfx_get_nprobe", "dfx_generation", "dfx_ntotal", "dfx_nlist", "dfx_launch_count"):
                getattr(L, f).restype = C.c_int64
            L.dfx_destroy.restype = None
            _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise RuntimeError(lib().dfx_last_error().decode("utf-8", "replace"))


def _np_ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _as_f32(x):
    x = np.asarray(x)
    if x.dtype != np.float32 or not x.flags["C_CONTIGUOUS"]:
        x = np.ascontiguousarray(x, dtype=np.float32)
    return x


def launch_count() -> int:
    return int(lib().dfx_launch_count())


class _Quantizer:
    """`.quantizer.reconstruct_n(0, nlist)` as used by Index.get_centroids (index.py:350)."""

    def __init__(self, owner):
        self._o = owner

    def reconstruct_n(self, i0, n):
        return self._o.get_centroids()[i0:i0 + n]


class GpuIndex:
    """One shard resident in the HBM of one B200, behind the faiss-object surface."""

    def __init__(self, kind, d, metric=METRIC_INNER_PRODUCT, nlist=0, pq_m=0, pq_nbits=8, device=None):
        import torch  # device bookkeeping only

        if device is None:
            device = torch.cuda.current_device() if torch.cuda.is_available() else 0
        self.kind, self.d, self.metric = int(kind), int(d), int(metric)
        self.device = int(device)
        self._cfg = DfxCfg(self.kind, self.metric, self.d, int(pq_m), int(pq_nbits), self.device, int(nlist))
        self._h = C.c_void_p()
        _check(lib().dfx_create(C.byref(self._cfg), C.byref(self._h)))
        if self.kind != KIND_FLAT:
            self.quantizer = _Quantizer(self)
        self.pq_m = int(pq_m)
        self.pq_nbits = int(pq_nbits)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value and _lib is not None:
            _lib.dfx_destroy(h)
            self._h = C.c_void_p()

    # ---- attributes
    @property
    def ntotal(self):
        return int(lib().dfx_ntotal(self._h))

    @property
    def nlist(self):
        return int(lib().dfx_nlist(self._h))

    @property
    def nprobe(self):
        return int(lib().dfx_get_nprobe(self._h))

    @nprobe.setter
    def nprobe(self, v):
        _check(lib().dfx_set_nprobe(self._h, C.c_int64(int(v))))

    @property
    def generation(self):
        return int(lib().dfx_generation(self._h))

    @property
    def is_trained(self):
        return bool(lib().dfx_is_trained(self._h))

    def set_param(self, name, value):
        _check(lib().dfx_set_param(self._h, name.encode(), C.c_double(float(value))))

    def get_param(self, name):
        v = C.c_double(0.0)
        _check(lib().dfx_get_param(self._h, name.encode(), C.byref(v)))
        return v.value

    def reserve(self, n_total):
        _check(lib().dfx_reserve(self._h, C.c_int64(int(n_total))))

    # ---- build
    def train(self, x):
        x = _as_f32(x)
        assert x.ndim == 2 and x.shape[1] == self.d
        _check(lib().dfx_train(self._h, C.c_int64(x.shape[0]), _np_ptr(x)))

    def add(self, x):
        x = _as_f32(x)
        assert x.ndim == 2 and x.shape[1] == self.d
        _check(lib().dfx_add(self._h, C.c_int64(x.shape[0]), _np_ptr(x)))

    def train_dev(self, x_t):
        """x_t: torch.float32 CUDA tensor [n, d] on this shard's device."""
        import torch

        assert x_t.is_cuda and x_t.dtype == torch.float32 and x_t.is_contiguous()
        st = torch.cuda.current_stream(x_t.device).cuda_stream
        _check(lib().dfx_train_dev(self._h, C.c_int64(x_t.shape[0]), C.c_void_p(x_t.data_ptr()), C.c_void_p(st)))

    def add_dev(self, x_t):
        import torch

        assert x_t.is_cuda and x_t.dtype == torch.float32 and x_t.is_contiguous()
        st = torch.cuda.current_stream(x_t.device).cuda_stream
        _check(lib().dfx_add_dev(self._h, C.c_int64(x_t.shape[0]), C.c_void_p(x_t.data_ptr()), C.c_void_p(st)))

    def finalize(self):
        _check(lib().dfx_finalize(self._h, C.c_void_p(0)))

    # ---- search (host buffers: the reference-facing call, index.py:257)
    def search(self, x, k):
        x = _as_f32(x)
        assert x.ndim == 2 and x.shape[1] == self.d, f"query must be [nq, {self.d}] float32"
        nq = x.shape[0]
        D = np.empty((nq, k), dtype=np.float32)
        I = np.empty((nq, k), dtype=np.int64)
        _check(lib().dfx_search(self._h, C.c_int64(nq), _np_ptr(x), C.c_int64(k), _np_ptr(D), _np_ptr(I)))
        return D, I

    def search_dev(self, x_t, k, D_t=None, I_t=None):
        """Device-resident search: torch CUDA tensors in, torch CUDA tensors out, enqueued on
        torch's current stream, no synchronisation."""
        import torch

        assert x_t.is_cuda and x_t.dtype == torch.float32 and x_t.is_contiguous()
        nq = x_t.shape[0]
        if D_t is None:
            D_t = torch.empty((nq, k), dtype=torch.float32, device=x_t.device)
        if I_t is None:
            I_t = torch.empty((nq, k), dtype=torch.int64, device=x_t.device)
        st = torch.cuda.current_stream(x_t.device).cuda_stream
        _check(lib().dfx_search_dev(self._h, C.c_int64(nq), C.c_void_p(x_t.data_ptr()), C.c_int64(k),
                                    C.c_void_p(D_t.data_ptr()), C.c_void_p(I_t.data_ptr()), C.c_void_p(st)))
        return D_t, I_t

    def reconstruct_rows(self, ids):
        ids = np.ascontiguousarray(ids, dtype=np.int64).reshape(-1)
        out = np.empty((ids.shape[0], self.d), dtype=np.float32)
        _check(lib().dfx_reconstruct(self._h, C.c_int64(ids.shape[0]), _np_ptr(ids), _np_ptr(out)))
        return out

    def reconstruct_dev(self, ids_t, out_t, shard_tag=-1):
        """Decode on device.  shard_tag < 0: ids_t are shard-local ids; shard_tag >= 0: ids_t are
        exchange ids (encode_ids_dev) and only the rows this shard owns are written into out_t."""
        import torch

        assert ids_t.is_cuda and ids_t.dtype == torch.int64 and ids_t.is_contiguous()
        assert out_t.is_cuda and out_t.dtype == torch.float32 and out_t.is_contiguous()
        n = ids_t.numel()
        assert out_t.numel() == n * self.d
        st = torch.cuda.current_stream(ids_t.device).cuda_stream
        _check(lib().dfx_reconstruct_dev(self._h, C.c_int64(n), C.c_void_p(ids_t.data_ptr()),
                                         C.c_int64(int(shard_tag)), C.c_void_p(out_t.data_ptr()), C.c_void_p(st)))
        return out_t

    def search_and_reconstruct(self, x, k):
        D, I = self.search(x, k)
        R = self.reconstruct_rows(I).reshape(I.shape[0], I.shape[1], self.d)
        return D, I, R

    def get_centroids(self):
        out = np.empty((self.nlist, self.d), dtype=np.float32)
        _check(lib().dfx_get_centroids(self._h, _np_ptr(out)))
        return out

    def last_stats(self):
        ndis, nq, npb = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        _check(lib().dfx_last_stats(self._h, C.byref(ndis), C.byref(nq), C.byref(npb)))
        return {"ndis": ndis.value, "nq": nq.value, "nprobe": npb.value}

    def profile(self, on=True):
        _check(lib().dfx_profile_enable(self._h, C.c_int(1 if on else 0)))

    def profile_read(self, reset=True):
        ms, n = C.c_double(0), C.c_int64(0)
        _check(lib().dfx_profile_read(self._h, C.byref(ms), C.byref(n), C.c_int(1 if reset else 0)))
        return ms.value, n.value

    # ---- state exchange (tests / persistence)
    _DTYPES = {"centroids": np.float32, "codebooks": np.float32, "list_off": np.int64, "ids": np.int64,
               "codes": np.uint8, "tvals": np.float32, "vecs": np.float32, "codes16": np.uint16,
               "xb": np.float32}

    def get_array(self, name):
        nb = C.c_int64(0)
        _check(lib().dfx_get_array(self._h, name.encode(), None, C.c_int64(0), C.byref(nb)))
        dt = np.dtype(self._DTYPES[name])
        out = np.empty((nb.value // dt.itemsize,), dtype=dt)
        _check(lib().dfx_get_array(self._h, name.encode(), _np_ptr(out), C.c_int64(nb.value), C.byref(nb)))
        return out

    def set_array(self, name, arr):
        arr = np.ascontiguousarray(arr, dtype=self._DTYPES[name])
        _check(lib().dfx_set_array(self._h, name.encode(), _np_ptr(arr), C.c_int64(arr.nbytes)))

    def payload_name(self):
        return {KIND_FLAT: "xb", KIND_IVF_FLAT: "vecs", KIND_IVF_PQ: "codes", KIND_IVF_SQ16: "codes16"}[self.kind]

    def get_state(self):
        """Same dict layout as oracle.get_state() (list-sorted storage order)."""
        d = self.d
        if self.kind == KIND_FLAT:
            return {"kind": "flat", "d": d, "metric": self.metric, "xb": self.get_array("xb").reshape(-1, d)}
        st = {"kind": KIND_NAMES[self.kind], "d": d, "nlist": self.nlist,
              "centroids": self.get_array("centroids").reshape(-1, d),
              "list_off": self.get_array("list_off"), "ids": self.get_array("ids")}
        if self.kind == KIND_IVF_FLAT:
            st["metric"] = self.metric
            st["vecs"] = self.get_array("vecs").reshape(-1, d)
        else:
            st["coarse_metric"] = self.metric
        if self.kind == KIND_IVF_PQ:
            # codes: M * nbits / 8 bytes per vector in faiss bit order (include/dfx.h "codes")
            ksub = 1 << self.pq_nbits
            st["M"], st["ksub"] = self.pq_m, ksub
            st["codebooks"] = self.get_array("codebooks").reshape(self.pq_m, ksub, d // self.pq_m)
            st["codes"] = self.get_array("codes").reshape(-1, self.pq_m * self.pq_nbits // 8)
            st["tvals"] = self.get_array("tvals")
        if self.kind == KIND_IVF_SQ16:
            st["codes16"] = self.get_array("codes16").reshape(-1, d)
        return st

    def set_state(self, st):
        if self.kind == KIND_FLAT:
            self.set_array("xb", st["xb"])
        else:
            self.set_array("centroids", st["centroids"])
            if self.kind == KIND_IVF_PQ:
                self.set_array("codebooks", st["codebooks"])
            self.set_array("list_off", st["list_off"])
            self.set_array("ids", st["ids"])
            self.set_array(self.payload_name(), st[self.payload_name()])
        _check(lib().dfx_import_done(self._h))


# ---------------------------------------------------------------- cross-shard merge (K6)
def merge(Dall, Iall, negate=False):
    """ResultHeap / float_maxheap_array_t semantics on device (reference client.py:29-54).
    Dall float32 [S, nq, k], Iall int64 [S, nq, k] host arrays."""
    Dall = np.ascontiguousarray(Dall, dtype=np.float32)
    Iall = np.ascontiguousarray(Iall, dtype=np.int64)
    S, nq, k = Dall.shape
    outD = np.empty((nq, k), dtype=np.float32)
    outI = np.empty((nq, k), dtype=np.int64)
    _check(lib().dfx_merge(C.c_int64(S), C.c_int64(nq), C.c_int64(k), _np_ptr(Dall), _np_ptr(Iall),
                           C.c_int(1 if negate else 0), _np_ptr(outD), _np_ptr(outI)))
    return outD, outI


def merge_dev(D_t, I_t, negate=False, outD=None, outI=None):
    """Device form: D_t [S, nq, k] float32, I_t [S, nq, k] int64 CUDA tensors."""
    import torch

    S, nq, k = D_t.shape
    assert D_t.is_contiguous() and I_t.is_contiguous()
    if outD is None:
        outD = torch.empty((nq, k), dtype=torch.float32, device=D_t.device)
    if outI is None:
        outI = torch.empty((nq, k), dtype=torch.int64, device=D_t.device)
    st = torch.cuda.current_stream(D_t.device).cuda_stream
    _check(lib().dfx_merge_dev(C.c_int64(S), C.c_int64(nq), C.c_int64(k), C.c_void_p(D_t.data_ptr()),
                               C.c_void_p(I_t.data_ptr()), C.c_int(1 if negate else 0),
                               C.c_void_p(outD.data_ptr()), C.c_void_p(outI.data_ptr()), C.c_void_p(st)))
    return outD, outI


def merge_packed_dev(packed_t, R, S_loc, nq, k, rank_stride, off_I, negate=False, outD=None, outI=None):
    """K6 over the buffer ONE all-gather delivers (layout: include/dfx.h dfx_merge_packed_dev)."""
    import torch

    assert packed_t.is_cuda and packed_t.is_contiguous() and packed_t.dtype == torch.uint8
    assert packed_t.numel() >= R * rank_stride
    if outD is None:
        outD = torch.empty((nq, k), dtype=torch.float32, device=packed_t.device)
    if outI is None:
        outI = torch.empty((nq, k), dtype=torch.int64, device=packed_t.device)
    st = torch.cuda.current_stream(packed_t.device).cuda_stream
    _check(lib().dfx_merge_packed_dev(C.c_int64(R), C.c_int64(S_loc), C.c_int64(nq), C.c_int64(k),
                                      C.c_void_p(packed_t.data_ptr()), C.c_int64(rank_stride), C.c_int64(off_I),
                                      C.c_int(1 if negate else 0), C.c_void_p(outD.data_ptr()),
                                      C.c_void_p(outI.data_ptr()), C.c_void_p(st)))
    return outD, outI


EXCHANGE_LOCAL_BITS = 40            # exchange id = (shard tag << 40) | shard-local id
EXCHANGE_DROP_FLAG = 1 << 62        # set on entries search_with_filter's post-filter drops


def encode_ids_dev(ids_t, shard_tag, out_t=None, col_t=None, drop_code=-1):
    import torch

    if out_t is None:
        out_t = torch.empty_like(ids_t)
    assert ids_t.dtype == torch.int64 and out_t.dtype == torch.int64
    assert col_t is None or (col_t.dtype == torch.int32 and col_t.is_cuda)
    st = torch.cuda.current_stream(ids_t.device).cuda_stream
    _check(lib().dfx_encode_ids_dev(C.c_int64(ids_t.numel()), C.c_void_p(ids_t.data_ptr()), C.c_int64(int(shard_tag)),
                                    C.c_void_p(col_t.data_ptr()) if col_t is not None else None,
                                    C.c_int32(int(drop_code)), C.c_void_p(out_t.data_ptr()), C.c_void_p(st)))
    return out_t


def filter_compact_dev(D_t, I_t, k_out):
    """search_with_filter's post-filter on device: (D, I) [nq, k_in] merged -> the first k_out kept
    entries per query, padded with (FLT_MAX, -1), and the number kept per query."""
    import torch

    nq, k_in = D_t.shape
    assert D_t.is_contiguous() and I_t.is_contiguous()
    outD = torch.empty((nq, k_out), dtype=torch.float32, device=D_t.device)
    outI = torch.empty((nq, k_out), dtype=torch.int64, device=D_t.device)
    cnt = torch.empty((nq,), dtype=torch.int32, device=D_t.device)
    st = torch.cuda.current_stream(D_t.device).cuda_stream
    _check(lib().dfx_filter_compact_dev(C.c_int64(nq), C.c_int64(k_in), C.c_int64(k_out), C.c_void_p(D_t.data_ptr()),
                                        C.c_void_p(I_t.data_ptr()), C.c_void_p(outD.data_ptr()),
                                        C.c_void_p(outI.data_ptr()), C.c_void_p(cnt.data_ptr()), C.c_void_p(st)))
    return outD, outI, cnt


def map_ids_dev(ids_t, table_t, out_t=None):
    import torch

    if out_t is None:
        out_t = torch.empty_like(ids_t)
    st = torch.cuda.current_stream(ids_t.device).cuda_stream
    _check(lib().dfx_map_ids_dev(C.c_int64(ids_t.numel()), C.c_void_p(ids_t.data_ptr()),
                                 C.c_void_p(table_t.data_ptr()), C.c_void_p(out_t.data_ptr()), C.c_void_p(st)))
    return out_t


# ---------------------------------------------------------------- synthetic data (bench harness)
class Synth:
    """Device-side generator of SURVEY.md 8(d): clustered, low intrinsic dimension, counter based."""

    def __init__(self, seed, d, r, nclusters, sigma, sigma_q=0.0, ngroups=0, eps=0.0, delta=0.0):
        import torch

        self.p = DfxSynth(int(seed), int(d), int(r), int(nclusters), int(ngroups), float(sigma), float(eps),
                          float(sigma_q), float(delta))
        self._A = C.c_void_p()
        st = torch.cuda.current_stream().cuda_stream
        _check(lib().dfx_synth_init(C.byref(self.p), C.byref(self._A), C.c_void_p(st)))

    def rows(self, row0, n, out_t=None, rows_t=None, noise_stream=0):
        import torch

        if out_t is None:
            out_t = torch.empty((n, self.p.d), dtype=torch.float32, device="cuda")
        st = torch.cuda.current_stream().cuda_stream
        rp = C.c_void_p(rows_t.data_ptr()) if rows_t is not None else None
        _check(lib().dfx_synth_rows_dev(C.byref(self.p), self._A, C.c_int64(int(row0)), rp, C.c_int64(int(n)),
                                        C.c_uint64(int(noise_stream)), C.c_void_p(out_t.data_ptr()), C.c_void_p(st)))
        return out_t

    def __del__(self):
        if getattr(self, "_A", None) is not None and self._A.value and _lib is not None:
            _lib.dfx_free(self._A)
            self._A = C.c_void_p()
