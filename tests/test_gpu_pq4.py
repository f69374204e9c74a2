"""IVF-PQ with 4-bit codes on the CUDA engine against the CPU oracle: every comparison is bit-exact on
D and I, ndis and the per-vector terms (t-values) equal the oracle's.  M = 64 x 4 bit runs the fused
block scan (pair table, dfx_scan_il2_dev.cuh); every other M, and interleaved=0, the row-major scan.

DFX_EMU_LIB: the same tests against the library built for the CPU emulator (tests/emu/), with the
shards shrunk (tests/test_pq4_host.py runs them that way)."""
import os
import tempfile
import threading

import numpy as np
import pytest

from tests.conftest import clustered
from tests.pq4_oracle import PackedOracleIVFPQ

pytestmark = pytest.mark.gpu

IP, L2 = 0, 1
EMU = bool(os.environ.get("DFX_EMU_LIB"))


def _sz(full, emu):
    return emu if EMU else full


def _E():
    from distributed_faiss_b200 import engine

    return engine


def _assert_same(Dg, Ig, Do, Io, what):
    if not (np.array_equal(Ig, Io) and np.array_equal(Dg, Do)):
        bad = np.argwhere((Ig != Io) | (Dg != Do))
        q, j = bad[0]
        raise AssertionError(f"{what}: {len(bad)} mismatching slots of {Ig.size}; first at q={q} j={j}: "
                             f"gpu=({Dg[q, j]!r},{Ig[q, j]}) oracle=({Do[q, j]!r},{Io[q, j]})")


def _pair(d, metric, nlist, M):
    E = _E()
    g = E.GpuIndex(E.KIND_IVF_PQ, d, metric, nlist=nlist, pq_m=M, pq_nbits=4)
    o = PackedOracleIVFPQ(d, nlist, M, 4, coarse_metric=metric)
    if EMU:
        g.set_param("kmeans_niter", 2)
        o.train_niter = 2
    return g, o


def _build(d, metric, nlist, M, n, rs, via="gpu", xb=None):
    """train + add on one side, ship the state to the other: both hold the SAME shard"""
    if xb is None:
        xb = clustered(rs, n, d, ncl=max(8, nlist // 2))
    g, o = _pair(d, metric, nlist, M)
    if via == "gpu":
        g.train(xb[: n // 2])
        g.add(xb[: n // 3]); g.add(xb[n // 3:])
        st = g.get_state()
        assert st["ksub"] == 16 and st["codes"].shape == (n, M // 2)
        o.set_state(st)
        assert np.array_equal(st["tvals"], o.tvals)
    else:
        o.train(xb[: n // 2])
        o.add(xb)
        g.set_state(o.get_state())
        assert np.array_equal(g.get_array("tvals"), o.tvals)
    assert g.ntotal == n == o.ntotal
    return g, o, xb


def _queries(rs, xb, d, n1=12, n2=4):
    return np.concatenate([clustered(rs, n1, d, ncl=8), xb[:n2] + 0.01 * rs.randn(n2, d).astype(np.float32)])


def _check(g, o, xq, nprobes, ks, what):
    for nprobe in nprobes:
        g.nprobe = nprobe; o.nprobe = nprobe
        for k in ks:
            _assert_same(*g.search(xq, k), *o.search(xq, k), f"{what} nprobe={nprobe} k={k}")
        assert g.last_stats()["ndis"] == o.last_ndis


# (d, M): (128, 64) fused, (256, 64) fused dsub 4, (768, 64) fused generic dsub, (64, 32) and (96, 24)
# row-major (24: the halving tree padded to 32)
CASES = [(128, 64), (256, 64), (768, 64), (64, 32), (96, 24)]


@pytest.mark.parametrize("d,M", CASES)
@pytest.mark.parametrize("metric", [L2, IP])
@pytest.mark.parametrize("via", ["gpu", "oracle"])
def test_pq4_matches_oracle(d, M, metric, via):
    if EMU and (d, M) in ((256, 64), (768, 64)) and (metric == IP or via == "gpu"):
        pytest.skip("emulator run: one case per extra dsub")
    rs = np.random.RandomState(3)
    nlist = 16
    g, o, xb = _build(d, metric, nlist, M, _sz(6000, 1500), rs, via=via)
    assert g.get_param("interleaved") == 1
    xq = _queries(rs, xb, d, *((20, 5) if not EMU else (6, 2)))
    _check(g, o, xq, (nlist, 1, 5), (10, 1, 100, 300) if not EMU else (10, 1, 100),
           f"pq4 d={d} M={M} metric={metric} via={via}")


def _m64(rs, n=None, via="oracle", xb=None):
    return _build(128, L2, 16, 64, n or _sz(6000, 1500), rs, via=via, xb=xb)


def test_pq4_m64_interleaved_and_row_major_agree():
    rs = np.random.RandomState(4)
    g, o, xb = _m64(rs)
    xq = _queries(rs, xb, 128, 10, 4)
    codes = g.get_array("codes")
    for il in (0, 1, 0, 1):
        g.set_param("interleaved", il)
        assert g.get_param("interleaved") == il
        assert np.array_equal(g.get_array("codes"), codes)  # export is faiss order in both layouts
        _check(g, o, xq, (16, 3), (10, 64), f"interleaved={il}")


def test_pq4_m64_encoding_and_incremental_adds():
    """adds on top of existing blocks: the GPU encodes, assigns and merges exactly like the oracle"""
    rs = np.random.RandomState(5)
    n = _sz(6000, 1500)
    xb = clustered(rs, n, 128, ncl=8)
    o = PackedOracleIVFPQ(128, 16, 64, 4)
    o.train_niter = 2 if EMU else 25
    o.train(xb[: n // 2]); o.add(xb[: n // 2])
    g, _ = _pair(128, L2, 16, 64)
    g.set_state(o.get_state())
    xq = _queries(rs, xb, 128, 8, 4)
    _check(g, o, xq, (16,), (10,), "before adds")
    for a, b in ((n // 2, n // 2 + 37), (n // 2 + 37, n)):  # a partial block, then the rest
        g.add(xb[a:b]); o.add(xb[a:b])
        sg, so = g.get_state(), o.get_state()
        for key in ("list_off", "ids", "codes", "tvals"):
            assert np.array_equal(sg[key], so[key]), key
        _check(g, o, xq, (16, 2), (10, 50), f"after add [{a}, {b})")


def test_pq4_m64_export_import():
    rs = np.random.RandomState(6)
    g, o, xb = _m64(rs, via="gpu")
    st = g.get_state()
    E = _E()
    g2 = E.GpuIndex(E.KIND_IVF_PQ, 128, L2, nlist=16, pq_m=64, pq_nbits=4)
    g2.set_state(st)
    st2 = g2.get_state()
    for key in ("centroids", "codebooks", "list_off", "ids", "codes", "tvals"):
        assert np.array_equal(st[key], st2[key]), key
    xq = _queries(rs, xb, 128, 8, 4)
    g.nprobe = g2.nprobe = 16
    for k in (10, 100):
        _assert_same(*g2.search(xq, k), *g.search(xq, k), f"export/import k={k}")


def test_pq4_m64_duplicates_tie_by_id():
    rs = np.random.RandomState(7)
    n = _sz(4000, 1200)
    xb = clustered(rs, n, 128, ncl=8)
    xb[100:160] = xb[0]      # exact duplicates: equal codes, equal distances, order by id
    xb[500:540] = xb[1]
    g, o, xb = _m64(rs, n=n, xb=xb)
    _check(g, o, np.stack([xb[0], xb[1], xb[0] + 1e-3]), (1, 16), (1, 10, 32, 100), "duplicates")


@pytest.mark.parametrize("k", [10, 32, 33, 300])
def test_pq4_m64_one_and_several_ctas_per_query(k):
    """few queries x many probes: several CTAs per query + the per-query reduction; a batch large
    enough that one CTA owns all probes of its query: (k <= 32) it writes the final rows itself"""
    rs = np.random.RandomState(8)
    g, o, xb = _m64(rs, n=_sz(6000, 2000))
    few = _queries(rs, xb, 128, 6, 2)
    many = xb[rs.randint(0, xb.shape[0], 1184 if EMU else 2400)] + 0.02 * rs.randn(1184 if EMU else 2400, 128).astype(np.float32)
    _check(g, o, few, (16, 5), (k,), "several CTAs per query")
    for nprobe in (4,) if EMU else (8, 1):
        g.nprobe = nprobe; o.nprobe = nprobe
        _assert_same(*g.search(many, k), *o.search(many, k), f"one CTA per query nprobe={nprobe} k={k}")


def test_pq4_reconstruct_both_layouts():
    rs = np.random.RandomState(9)
    for M, d in ((64, 128), (32, 64)):
        g, o, xb = _build(d, L2, 16, M, _sz(3000, 800), rs, via="oracle")
        ids = np.concatenate([rs.randint(0, xb.shape[0], 50), [-1, xb.shape[0] + 5]]).astype(np.int64)
        ok = (ids >= 0) & (ids < xb.shape[0])
        Ro = o.reconstruct_rows(ids[ok])
        for il in (1, 0):
            g.set_param("interleaved", il)
            Rg = g.reconstruct_rows(ids)
            assert np.allclose(Rg[ok], Ro, rtol=0, atol=1e-6), (M, il)
            assert np.isnan(Rg[~ok]).all()


def test_pq4_training_quality():
    """GPU-trained 4-bit codebooks quantise about as well as the oracle's"""
    rs = np.random.RandomState(10)
    d, nlist, n = 128, 16, _sz(20000, 3000)
    xb = clustered(rs, n, d, ncl=40, sigma=0.2)
    for M in (64, 32):
        g, o = _pair(d, L2, nlist, M)
        g.train(xb); g.add(xb)
        o.train(xb); o.add(xb)

        def recon_err(ix):
            R = ix.reconstruct_rows(np.arange(0, n, 7, dtype=np.int64))
            return float(((R - xb[::7]) ** 2).sum(1).mean())

        eg, eo = recon_err(g), recon_err(o)
        assert eg < 1.25 * eo + 1e-6, (M, eg, eo)


@pytest.mark.parametrize("nbits,M", [(1, 32), (2, 32), (3, 32), (5, 32), (6, 32), (7, 32), (9, 32), (16, 32),
                                     (4, 12), (4, 20)])
def test_rejected_pq_configurations(nbits, M):
    E = _E()
    with pytest.raises(RuntimeError, match="IVF-PQ"):
        E.GpuIndex(E.KIND_IVF_PQ, 120 if M != 32 else 128, L2, nlist=8, pq_m=M, pq_nbits=nbits)


# ------------------------------------------------------------------ public API
@pytest.fixture(scope="module")
def cluster():
    from distributed_faiss_b200.server import IndexServer
    from tests.test_gpu_api import free_ports, wait_listening

    dirs = [tempfile.TemporaryDirectory(), tempfile.TemporaryDirectory()]
    ports = free_ports(4)
    ports, sp = ports[:3], ports[3]
    servers = []
    for rank, port in enumerate(ports):
        s = IndexServer(rank, dirs[0].name)
        threading.Thread(target=s.start_blocking, args=(port,), daemon=True).start()
        servers.append(s)
    single = IndexServer(0, dirs[1].name)
    threading.Thread(target=single.start_blocking, args=(sp,), daemon=True).start()
    wait_listening(ports + [sp])
    yield {"ports": ports, "single": sp, "dirs": dirs}
    for s in servers + [single]:
        s.stop()


def test_knnlm_4bit_through_the_api(cluster):
    """bits_per_vector=4 through IndexServer / IndexClient: one shard and three shards answer, embeddings
    decode, save / load in the dfx and faiss formats (exact sharded == unsharded, which needs the same
    codebooks on every shard: test_sharded_equals_unsharded_pq4)"""
    if EMU:
        pytest.skip("the servers train at full k-means length: too slow for the emulator "
                    "(tests/test_pq4_host.py runs this pipeline with the oracle engine)")
    from distributed_faiss_b200.index_cfg import IndexCfg
    from tests.test_gpu_api import make_client, wait_trained

    rs = np.random.RandomState(11)
    d = 128
    n = _sz(6000, 1500)
    x = clustered(rs, n, d, ncl=20, sigma=0.2)
    for fmt in ("dfx", "faiss"):
        index_id = f"pq4_api_{fmt}"
        cfg = IndexCfg(index_builder_type="knnlm", dim=d, centroids=16, metric="l2", train_num=n // 6, code_size=64,
                       bits_per_vector=4, index_format=fmt)
        single = make_client([cluster["single"]])
        multi = make_client(cluster["ports"])
        single.create_index(index_id, cfg)
        multi.create_index(index_id, cfg)
        step = n // 6
        for b in range(6):
            xb, meta = x[b * step:(b + 1) * step], list(range(b * step, (b + 1) * step))
            single.add_index_data(index_id, xb, meta, False)
            multi.add_index_data(index_id, xb, meta, False)
        wait_trained(single, index_id)
        wait_trained(multi, index_id)
        assert single.get_ntotal(index_id) == multi.get_ntotal(index_id) == n
        single.set_nprobe(index_id, 16)
        multi.set_nprobe(index_id, 16)
        q = x[:10]
        D, meta = single.search(q, 5, index_id)
        assert sum(row[0] == i * 1 for i, row in enumerate(meta)) >= 8
        D2, meta2, embs = single.search(q, 5, index_id, return_embeddings=True)
        assert np.array_equal(D, D2) and meta == meta2
        embs = np.asarray(embs)
        # the decoded vectors are the PQ reconstructions: their distance to the query is D
        d2 = ((embs.astype(np.float64) - q[:, None, :]) ** 2).sum(-1)
        assert np.allclose(d2, D, rtol=1e-3, atol=1e-3)
        Dm, mm = multi.search(q, 5, index_id)
        assert Dm.shape == D.shape and all(len(r) == 5 for r in mm)
        single.save_index(index_id)
        single.close()
        c2 = make_client([cluster["single"]])
        assert c2.load_index(index_id, cfg)
        c2.set_nprobe(index_id, 16)
        D3, meta3 = c2.search(q, 5, index_id)
        assert np.array_equal(D, D3) and meta == meta3
        c2.close(); multi.close()


def test_sharded_equals_unsharded_pq4():
    """shards built from one trained 4-bit shard: merging S shard answers == one shard holding all"""
    from distributed_faiss_b200 import engine as E

    rs = np.random.RandomState(12)
    g, o, xb = _m64(rs)
    st = g.get_state()
    n = xb.shape[0]
    owner = np.arange(n) % 3
    xq = _queries(rs, xb, 128, 8, 4)
    g.nprobe = 16
    D1, I1 = g.search(xq, 10)
    Ds, Is = [], []
    for s in range(3):
        keep = owner[st["ids"]] == s
        gid = st["ids"][keep]
        table = np.sort(gid)  # shard-local id = rank of the global id: ties keep their order
        sub = dict(st, ids=np.searchsorted(table, gid).astype(np.int64), codes=st["codes"][keep],
                   list_off=np.concatenate([[0], np.cumsum(np.bincount(
                       np.repeat(np.arange(16), np.diff(st["list_off"]))[keep], minlength=16))]).astype(np.int64))
        sh = E.GpuIndex(E.KIND_IVF_PQ, 128, L2, nlist=16, pq_m=64, pq_nbits=4)
        sh.set_state(sub)
        sh.nprobe = 16
        D, I = sh.search(xq, 10)
        Ds.append(D); Is.append(np.where(I >= 0, table[np.maximum(I, 0)], -1))
    Dm, Im = E.merge(np.stack(Ds), np.stack(Is))
    _assert_same(Dm, Im, D1, I1, "sharded vs unsharded")
