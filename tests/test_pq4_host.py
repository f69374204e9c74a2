"""IVF-PQ with 4-bit codes (knnlm `bits_per_vector=4`), host side: the code format, the oracle
restatement, faiss files and the API pipeline with the oracle engine.  The same scenarios on the
CUDA engine are in tests/test_gpu_pq4.py; `test_gpu_pq4_on_the_emulated_library` runs them, at
reduced sizes, against the library built for the CPU emulator (tests/emu/)."""
import os
import platform
import shutil
import subprocess
import sys
import tempfile
import threading

import numpy as np
import pytest

from distributed_faiss_b200 import faiss_io
from tests.conftest import clustered
from tests.pq4_oracle import PackedOracleIVFPQ, packed_oracle_engine_factory

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L2, IP = 1, 0


def test_packing_is_faiss_bit_order():
    """sub-quantizer m in byte m >> 1, low nibble for even m, high nibble for odd m"""
    packed = faiss_io.pack_codes(np.array([[1, 2, 3, 4]], dtype=np.uint8), 4)
    assert packed.tolist() == [[0x21, 0x43]]
    assert faiss_io.unpack_codes(packed, 4, 4).tolist() == [[1, 2, 3, 4]]
    rs = np.random.RandomState(0)
    c = rs.randint(0, 16, (50, 24)).astype(np.uint8)
    assert np.array_equal(faiss_io.unpack_codes(faiss_io.pack_codes(c, 4), 24, 4), c)
    c8 = rs.randint(0, 256, (5, 8)).astype(np.uint8)
    assert np.array_equal(faiss_io.pack_codes(c8, 8), c8)


def _oracle_shard(d, M, nlist, n, metric=L2, seed=0):
    rs = np.random.RandomState(seed)
    xb = clustered(rs, n, d, ncl=max(8, nlist // 2))
    o = PackedOracleIVFPQ(d, nlist, M, 4, coarse_metric=metric)
    o.train_niter = 8
    o.train(xb[: n // 2])
    o.add(xb)
    return o, xb, rs


@pytest.mark.parametrize("d,M,metric", [(64, 32, L2), (128, 64, L2), (96, 24, IP)])
def test_oracle_4bit_matches_float64_restatement(oracle_lib, d, M, metric):
    from oracle import ref_numpy as R

    nlist = 16
    o, xb, rs = _oracle_shard(d, M, nlist, 3000, metric)
    assert o.ksub == 16 and o.codes.max() < 16
    xq = clustered(rs, 12, d, ncl=8)
    o.nprobe = nlist
    D, I = o.search(xq, 10)
    st = o.get_state()
    st["codes"] = faiss_io.unpack_codes(st["codes"], M, 4)  # the restatement reads one code per byte
    D64, I64 = R.ivf_search(st, xq, nlist, 10)
    scale = (xq.astype(np.float64) ** 2).sum(1, keepdims=True) + (xb.astype(np.float64) ** 2).sum(1).max()
    assert (np.abs(D - D64) <= 1e-4 * scale).all()
    # ids equal wherever the float64 distances are separated by more than the fp32 rounding
    gap = np.abs(np.diff(np.concatenate([D64, D64[:, -1:] + 1], axis=1), axis=1))
    sep = (gap > 1e-4 * scale) & np.concatenate([np.ones((len(xq), 1), bool), gap[:, :-1] > 1e-4 * scale], axis=1)
    assert (I[sep] == I64[sep]).all()


def test_faiss_file_roundtrip_4bit(oracle_lib):
    d, M, nlist = 64, 32, 16
    o, xb, rs = _oracle_shard(d, M, nlist, 2000)
    st = o.get_state()
    assert st["codes"].shape == (2000, M // 2)
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "index.faiss")
        faiss_io.write_index(st, path, nprobe=3)
        with open(path, "rb") as f:
            raw = f.read()
        # by_residual, code_size, then the PQ header (d, M, nbits), right before the codebooks
        cb_bytes = np.ascontiguousarray(st["codebooks"], dtype=np.float32).tobytes()
        at = raw.index(np.array([M * 16 * (d // M)], dtype="<u8").tobytes() + cb_bytes[:64])
        by_res, code_size, pd, pm, nbits = (raw[at - 33],) + tuple(np.frombuffer(raw[at - 32:at], dtype="<u8"))
        assert (by_res, code_size, pd, pm, nbits) == (1, M // 2, d, M, 4)
        st2, nprobe = faiss_io.read_index(path)
        # a state whose codes are not M * nbits / 8 bytes wide is refused
        bad = dict(st, codes=faiss_io.unpack_codes(st["codes"], M, 4))
        with pytest.raises(faiss_io.FaissFormatError):
            faiss_io.write_index(bad, os.path.join(tmp, "bad.faiss"))
    assert nprobe == 3 and st2["ksub"] == 16 and st2["M"] == M
    for key in ("centroids", "codebooks", "list_off", "ids", "codes"):
        assert np.array_equal(np.asarray(st2[key]), np.asarray(st[key])), key
    o2 = PackedOracleIVFPQ(d, nlist, M, 4)
    o2.set_state(st2)
    xq = xb[:7]
    o.nprobe = o2.nprobe = 4
    assert all(np.array_equal(a, b) for a, b in zip(o.search(xq, 10), o2.search(xq, 10)))


@pytest.fixture(scope="module")
def servers():
    from distributed_faiss_b200.client import ResultHeap
    from distributed_faiss_b200.server import IndexServer
    from tests.oracle_engine import oracle_merge
    from tests.test_host_logic import free_ports, wait_listening

    ResultHeap.merge_backend = staticmethod(oracle_merge)
    tmp = tempfile.TemporaryDirectory()
    ports = free_ports(1)
    srv = IndexServer(0, tmp.name, engine_factory=packed_oracle_engine_factory)
    threading.Thread(target=srv.start_blocking, args=(ports[0],), daemon=True).start()
    wait_listening(ports)
    yield {"port": ports[0], "dir": tmp.name}
    srv.stop()


@pytest.mark.parametrize("fmt", ["dfx", "faiss"])
def test_knnlm_4bit_pipeline_save_load(oracle_lib, servers, fmt):
    """knnlm bits_per_vector=4 through IndexServer / IndexClient: train, add, search, save, reload"""
    from distributed_faiss_b200.index_cfg import IndexCfg
    from tests.test_host_logic import make_client, wait_trained

    rs = np.random.RandomState(2)
    d, index_id = 64, f"pq4_{fmt}"
    cfg = IndexCfg(index_builder_type="knnlm", dim=d, centroids=16, metric="l2", train_num=1500, code_size=32,
                   bits_per_vector=4, index_format=fmt)
    client = make_client([servers["port"]])
    client.create_index(index_id, cfg)
    x = clustered(rs, 3000, d, ncl=20, sigma=0.2)
    for b in range(3):
        client.add_index_data(index_id, x[b * 1000:(b + 1) * 1000], list(range(b * 1000, (b + 1) * 1000)), False)
    wait_trained(client, index_id)
    assert client.get_ntotal(index_id) == 3000
    client.set_nprobe(index_id, 16)
    D, meta = client.search(x[:10], 5, index_id)
    assert sum(row[0] == i for i, row in enumerate(meta)) >= 8  # a 4-bit code still finds its own vector
    client.save_index(index_id)
    saved = os.listdir(os.path.join(servers["dir"], index_id, "0"))
    assert ("index.faiss" in saved) == (fmt == "faiss")
    client.close()
    c2 = make_client([servers["port"]])
    assert c2.load_index(index_id, cfg)
    c2.set_nprobe(index_id, 16)
    D2, meta2 = c2.search(x[:10], 5, index_id)
    assert np.array_equal(D, D2) and meta == meta2
    c2.close()


def test_gpu_pq4_on_the_emulated_library():
    """tests/test_gpu_pq4.py (reduced sizes) against the library built for the CPU emulator"""
    if shutil.which("g++") is None or platform.machine() != "x86_64":
        pytest.skip("the emulator needs g++ on x86-64")
    sys.path.insert(0, os.path.join(ROOT, "tests", "emu"))
    try:
        import build_emu_lib
    finally:
        sys.path.pop(0)
    env = dict(os.environ, DFX_EMU_LIB=build_emu_lib.build())
    run = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-p", "no:cacheprovider",
                          "tests/test_gpu_pq4.py"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (run.stdout + run.stderr)[-3000:]
    assert run.returncode == 0 and " passed" in run.stdout and "failed" not in run.stdout, tail
