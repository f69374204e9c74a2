"""Reader / writer for the faiss on-disk index format, for the four index types the reference's
builders create (reference index.py:94 IndexFlatIP, :36-40 IndexIVFFlat, :43-48 IndexIVFPQ,
:63-68 IndexIVFScalarQuantizer(QT_fp16)); the reference saves shards with
`faiss.write_index(self.faiss_index, index_file)` (index.py:459) and loads them with
`faiss.read_index` (index.py:303).  SURVEY.md section 8(f) next-3.

The engine state dict (engine.GpuIndex.get_state / set_state: centroids, codebooks, list-sorted
codes + shard-local ids + list offsets) maps one-to-one onto what faiss serialises, so a shard
saved by the reference can be loaded straight into HBM and vice versa.  The per-vector IVF-PQ
term `tvals` is not part of the faiss format; the engine recomputes it on import.

STATUS: written from the layout of faiss 1.7.x `impl/index_write.cpp` / `index_read.cpp`; faiss
itself is not available in this environment (SURVEY.md section 8c), so the format is checked for
self-consistency only (tests/test_faiss_io.py), never against a file written by faiss.

Layout (little endian, no padding; `vec<T>` = u64 count + raw elements):
  header   : i32 d, i64 ntotal, i64 1<<20, i64 1<<20, u8 is_trained, i32 metric (0 IP, 1 L2)
  flat     : fourcc "IxFI" | "IxF2", header, vec<f32> xb
  ivf hdr  : header, u64 nlist, u64 nprobe, <quantizer: flat index of the centroids>,
             u8 direct-map type (0), vec<i64> direct map (empty)
  invlists : fourcc "ilar", u64 nlist, u64 code_size, fourcc "full" + vec<u64> sizes  (or "sprs" +
             vec<u64> (list, size) pairs when at most half of the lists are non-empty), then for
             every non-empty list: codes (size * code_size bytes), ids (size * i64)
  IVFFlat  : "IwFl", ivf hdr, invlists (code = raw f32 vector)
  IVFPQ    : "IwPQ", ivf hdr, u8 by_residual, u64 code_size, PQ (u64 d, u64 M, u64 nbits,
             vec<f32> centroids [M][ksub][dsub]), invlists (code = M * nbits / 8 bytes; nbits 8
             or 4, 4-bit codes packed LSB first: code m in the low nibble of byte m >> 1 when m is
             even, in the high nibble when odd -- faiss PQEncoderGeneric order, which is also the
             order of the engine state dict)
  IVFSQ    : "IwSq", ivf hdr, SQ (i32 qtype = 4 (fp16), i32 rangestat, f32 rangestat_arg, u64 d,
             u64 code_size, vec<f32> trained (empty)), u64 code_size, u8 by_residual, invlists
             (code = d little-endian fp16 of the residual)
"""
import struct
from typing import BinaryIO, Dict, Tuple

import numpy as np

METRIC_IP, METRIC_L2 = 0, 1
QT_FP16 = 4


class FaissFormatError(RuntimeError):
    pass


# ------------------------------------------------------------------ primitives
def _w(f: BinaryIO, fmt: str, *vals):
    f.write(struct.pack("<" + fmt, *vals))


def _r(f: BinaryIO, fmt: str):
    size = struct.calcsize("<" + fmt)
    raw = f.read(size)
    if len(raw) != size:
        raise FaissFormatError("unexpected end of file")
    return struct.unpack("<" + fmt, raw)


def _wvec(f: BinaryIO, arr: np.ndarray, dtype):
    arr = np.ascontiguousarray(arr, dtype=dtype).reshape(-1)
    _w(f, "Q", arr.size)
    f.write(arr.tobytes())


def _rvec(f: BinaryIO, dtype) -> np.ndarray:
    (n,) = _r(f, "Q")
    return _rraw(f, n, dtype)


def _rraw(f: BinaryIO, n: int, dtype) -> np.ndarray:
    nbytes = int(n) * np.dtype(dtype).itemsize
    raw = f.read(nbytes)
    if len(raw) != nbytes:
        raise FaissFormatError("unexpected end of file")
    return np.frombuffer(raw, dtype=dtype).copy()


def _fourcc(f: BinaryIO) -> str:
    raw = f.read(4)
    if len(raw) != 4:
        raise FaissFormatError("unexpected end of file")
    return raw.decode("ascii", errors="replace")


def _wheader(f, d, ntotal, metric, is_trained=True):
    _w(f, "iqqqBi", int(d), int(ntotal), 1 << 20, 1 << 20, 1 if is_trained else 0, int(metric))


def _rheader(f):
    d, ntotal, _, _, trained, metric = _r(f, "iqqqBi")
    if metric > 1:
        _r(f, "f")  # metric_arg of the exotic metrics
    return d, ntotal, bool(trained), metric


# ------------------------------------------------------------------ pieces
def _write_flat(f, xb: np.ndarray, metric: int):
    xb = np.ascontiguousarray(xb, dtype=np.float32)
    f.write(b"IxFI" if metric == METRIC_IP else b"IxF2")
    _wheader(f, xb.shape[1], xb.shape[0], metric)
    _wvec(f, xb, np.float32)


def _read_flat_body(f, cc):
    d, ntotal, _, metric = _rheader(f)
    xb = _rvec(f, np.float32)
    if xb.size != d * ntotal:
        raise FaissFormatError(f"flat index: {xb.size} floats for ntotal={ntotal}, d={d}")
    return {"kind": "flat", "d": d, "metric": metric, "xb": xb.reshape(ntotal, d)}


def _write_ivf_header(f, st, metric, coarse_metric, nprobe):
    _wheader(f, st["d"], len(st["ids"]), metric)
    _w(f, "QQ", int(st["nlist"]), int(nprobe))
    _write_flat(f, st["centroids"], coarse_metric)
    _w(f, "B", 0)  # DirectMap::NoMap
    _w(f, "Q", 0)


def _read_ivf_header(f):
    d, ntotal, _, metric = _rheader(f)
    nlist, nprobe = _r(f, "QQ")
    cc = _fourcc(f)
    if cc not in ("IxFI", "IxF2", "IxFl"):
        raise FaissFormatError(f"coarse quantizer {cc!r} is not a flat index")
    q = _read_flat_body(f, cc)
    if q["xb"].shape != (nlist, d):
        raise FaissFormatError("coarse quantizer does not hold nlist centroids")
    (dm_type,) = _r(f, "B")
    _rvec(f, np.int64)
    if dm_type == 2:  # DirectMap::Hashtable: vec of (i64, i64) pairs
        (n,) = _r(f, "Q")
        _rraw(f, 2 * n, np.int64)
    return d, ntotal, metric, nlist, nprobe, q["xb"], q["metric"]


def _write_invlists(f, list_off, ids, rows_u8: np.ndarray, code_size: int):
    list_off = np.asarray(list_off, dtype=np.int64)
    nlist = len(list_off) - 1
    sizes = np.diff(list_off).astype(np.uint64)
    f.write(b"ilar")
    _w(f, "QQ", nlist, int(code_size))
    if int((sizes > 0).sum()) > nlist // 2:
        f.write(b"full")
        _wvec(f, sizes, np.uint64)
    else:
        f.write(b"sprs")
        nz = np.nonzero(sizes)[0]
        _wvec(f, np.stack([nz.astype(np.uint64), sizes[nz]], axis=1), np.uint64)
    ids = np.ascontiguousarray(ids, dtype=np.int64)
    rows_u8 = np.ascontiguousarray(rows_u8).view(np.uint8).reshape(len(ids), code_size)
    for l in range(nlist):
        a, b = int(list_off[l]), int(list_off[l + 1])
        if b > a:
            f.write(rows_u8[a:b].tobytes())
            f.write(ids[a:b].tobytes())


def _read_invlists(f, nlist_expected):
    cc = _fourcc(f)
    if cc == "il00":  # no inverted lists stored
        raise FaissFormatError("index file holds no inverted lists")
    if cc != "ilar":
        raise FaissFormatError(f"inverted lists of type {cc!r} are not supported")
    nlist, code_size = _r(f, "QQ")
    if nlist != nlist_expected:
        raise FaissFormatError("inverted lists / header nlist mismatch")
    lt = _fourcc(f)
    sizes = np.zeros(nlist, dtype=np.int64)
    if lt == "full":
        v = _rvec(f, np.uint64)
        if v.size != nlist:
            raise FaissFormatError("list size table has the wrong length")
        sizes[:] = v
    elif lt == "sprs":
        v = _rvec(f, np.uint64).reshape(-1, 2)
        sizes[v[:, 0].astype(np.int64)] = v[:, 1]
    else:
        raise FaissFormatError(f"unknown list size encoding {lt!r}")
    list_off = np.zeros(nlist + 1, dtype=np.int64)
    np.cumsum(sizes, out=list_off[1:])
    n = int(list_off[-1])
    rows = np.empty((n, code_size), dtype=np.uint8)
    ids = np.empty(n, dtype=np.int64)
    for l in range(nlist):
        a, b = int(list_off[l]), int(list_off[l + 1])
        if b > a:
            rows[a:b] = _rraw(f, (b - a) * code_size, np.uint8).reshape(b - a, code_size)
            ids[a:b] = _rraw(f, b - a, np.int64)
    return list_off, ids, rows, code_size


# ------------------------------------------------------------------ PQ code packing
def pack_codes(codes: np.ndarray, nbits: int) -> np.ndarray:
    """codes [n, M] (one code per byte) -> rows of M * nbits / 8 bytes in faiss bit order."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    if nbits == 8:
        return codes
    if nbits != 4 or codes.shape[1] % 2:
        raise FaissFormatError(f"cannot pack {codes.shape[1]} codes of {nbits} bits")
    return (codes[:, 0::2] & 15) | ((codes[:, 1::2] & 15) << 4)


def unpack_codes(rows: np.ndarray, M: int, nbits: int) -> np.ndarray:
    """rows of M * nbits / 8 bytes in faiss bit order -> codes [n, M], one code per byte."""
    rows = np.ascontiguousarray(rows, dtype=np.uint8).reshape(-1, M * nbits // 8)
    if nbits == 8:
        return rows
    if nbits != 4:
        raise FaissFormatError(f"cannot unpack codes of {nbits} bits")
    out = np.empty((rows.shape[0], M), dtype=np.uint8)
    out[:, 0::2] = rows & 15
    out[:, 1::2] = rows >> 4
    return out


# ------------------------------------------------------------------ public
def write_index(state: Dict, path: str, nprobe: int = 1) -> None:
    """state: engine / oracle `get_state()` dict.  Writes a faiss index file."""
    kind = state["kind"]
    with open(path, "wb") as f:
        if kind == "flat":
            _write_flat(f, state["xb"], int(state["metric"]))
        elif kind == "ivf_flat":
            f.write(b"IwFl")
            _write_ivf_header(f, state, int(state["metric"]), int(state["metric"]), nprobe)
            vecs = np.ascontiguousarray(state["vecs"], dtype=np.float32)
            _write_invlists(f, state["list_off"], state["ids"], vecs, 4 * int(state["d"]))
        elif kind == "ivf_pq":
            M, ksub = int(state["M"]), int(state["ksub"])
            nbits = {256: 8, 16: 4}.get(ksub)
            if nbits is None:
                raise FaissFormatError("only 8-bit and 4-bit product quantizers are supported")
            code_size = M * nbits // 8
            f.write(b"IwPQ")
            _write_ivf_header(f, state, METRIC_L2, int(state["coarse_metric"]), nprobe)
            _w(f, "B", 1)  # by_residual
            _w(f, "Q", code_size)
            _w(f, "QQQ", int(state["d"]), M, nbits)
            _wvec(f, state["codebooks"], np.float32)
            codes = np.ascontiguousarray(state["codes"], dtype=np.uint8)
            if codes.ndim != 2 or codes.shape[1] != code_size:
                raise FaissFormatError(f"IndexIVFPQ: codes must be [ntotal, {code_size}] bytes (M * nbits / 8)")
            _write_invlists(f, state["list_off"], state["ids"], codes, code_size)
        elif kind == "ivf_sq":
            d = int(state["d"])
            f.write(b"IwSq")
            _write_ivf_header(f, state, METRIC_L2, int(state["coarse_metric"]), nprobe)
            _w(f, "iif", QT_FP16, 0, 0.0)
            _w(f, "QQ", d, 2 * d)
            _w(f, "Q", 0)  # trained: empty for fp16
            _w(f, "Q", 2 * d)
            _w(f, "B", 1)  # by_residual
            c16 = np.ascontiguousarray(state["codes16"], dtype="<u2")
            _write_invlists(f, state["list_off"], state["ids"], c16, 2 * d)
        else:
            raise FaissFormatError(f"unknown index kind {kind!r}")


def read_index(path: str) -> Tuple[Dict, int]:
    """Returns (state dict for `set_state`, nprobe stored in the file)."""
    with open(path, "rb") as f:
        cc = _fourcc(f)
        if cc in ("IxFI", "IxF2", "IxFl"):
            st = _read_flat_body(f, cc)
            return st, 1
        if cc not in ("IwFl", "IwPQ", "IwSq"):
            raise FaissFormatError(
                f"faiss index type {cc!r} is not one of the types the B200 search path serves "
                "(IndexFlat, IndexIVFFlat, IndexIVFPQ, IndexIVFScalarQuantizer fp16)")
        d, ntotal, metric, nlist, nprobe, cent, cmetric = _read_ivf_header(f)
        st = {"d": d, "nlist": nlist, "centroids": cent}
        if cc == "IwFl":
            list_off, ids, rows, cs = _read_invlists(f, nlist)
            if cs != 4 * d:
                raise FaissFormatError("IndexIVFFlat code size is not 4 * d")
            st.update(kind="ivf_flat", metric=metric, vecs=rows.view(np.float32).reshape(-1, d))
        elif cc == "IwPQ":
            (by_res,) = _r(f, "B")
            (code_size,) = _r(f, "Q")
            pd, M, nbits = _r(f, "QQQ")
            cb = _rvec(f, np.float32)
            if not by_res or nbits not in (4, 8) or pd != d or code_size != M * nbits // 8:
                raise FaissFormatError("IndexIVFPQ: only by_residual, 4 or 8 bits per sub-quantizer is supported")
            if metric != METRIC_L2:
                raise FaissFormatError("IndexIVFPQ: only METRIC_L2 is supported")
            list_off, ids, rows, cs = _read_invlists(f, nlist)
            ksub = 1 << nbits
            st.update(kind="ivf_pq", coarse_metric=cmetric, M=M, ksub=ksub,
                      codebooks=cb.reshape(M, ksub, d // M), codes=rows.reshape(-1, code_size))
        else:
            qtype, _, _ = _r(f, "iif")
            sd, scs = _r(f, "QQ")
            _rvec(f, np.float32)
            (code_size,) = _r(f, "Q")
            (by_res,) = _r(f, "B")
            if qtype != QT_FP16 or not by_res or code_size != 2 * d:
                raise FaissFormatError("IndexIVFScalarQuantizer: only QT_fp16, by_residual is supported")
            list_off, ids, rows, cs = _read_invlists(f, nlist)
            st.update(kind="ivf_sq", coarse_metric=cmetric, codes16=rows.view("<u2").reshape(-1, d))
        if len(ids) != ntotal:
            raise FaissFormatError("inverted lists do not hold ntotal vectors")
        st.update(list_off=list_off, ids=ids)
        return st, int(nprobe)
