"""CPU checks of bench.py's pure helpers (sharding rule, tiers, recall arithmetic)."""
import numpy as np
import torch

import bench


def test_shard_rows_partition_the_database():
    """row block b of 50 000 rows -> shard b mod 8 (the client's round-robin, client.py:186-192);
    every row belongs to exactly one shard, in arrival order."""
    nvec = 1_234_567
    seen = np.zeros(nvec, dtype=np.int32)
    total = 0
    for s in range(bench.NSHARDS):
        prev_end = -1
        for r0, n in bench.shard_rows(nvec, s):
            assert (r0 // bench.BLOCK) % bench.NSHARDS == s
            assert r0 > prev_end
            prev_end = r0 + n - 1
            seen[r0:r0 + n] += 1
            total += n
    assert total == nvec and (seen == 1).all()
    # the last block is the only short one
    sizes = [n for s in range(bench.NSHARDS) for _, n in bench.shard_rows(nvec, s)]
    assert sorted(sizes)[0] == nvec % bench.BLOCK and sizes.count(bench.BLOCK) == nvec // bench.BLOCK


def test_nlist_tiers_and_names():
    assert bench.nlist_for(125_000_000) == 65536      # 1 B vectors / 8 shards
    assert bench.nlist_for(12_500_000) == 16384       # 100 M / 8
    assert bench.nlist_for(2_500_000) == 4096
    assert bench.nlist_for(100_000) == 1024
    assert "1B synthetic vectors" in bench.workload_name(1_000_000_000)


def test_recall_at_k():
    K = bench.K
    gt = torch.arange(2 * K).reshape(2, K)
    I = gt.clone()
    assert bench.recall_at_k(I, gt) == 1.0
    I[0, :5] = 10_000 + torch.arange(5)                # half of query 0 wrong
    assert abs(bench.recall_at_k(I, gt) - 0.75) < 1e-6
    ok = torch.tensor([False, True])                   # uncertified queries are excluded
    assert bench.recall_at_k(I, gt, ok) == 1.0
    gt2 = gt.clone()
    gt2[1, -2:] = -1                                   # a group with only K-2 members
    assert abs(bench.recall_at_k(gt.clone(), gt2) - 1.0) < 1e-6


def test_dump_outputs(tmp_path, monkeypatch):
    """--dump-outputs: float32 distances, float64 ids, every row while it fits; above the size
    limit the same seeded sample of rows every time."""
    rs = np.random.RandomState(0)
    D = rs.rand(100, bench.K).astype(np.float32)
    I = rs.randint(0, 1 << 40, size=(100, bench.K)).astype(np.int64)
    bench.dump_outputs(str(tmp_path / "all"), D, I)
    d, i, r = (np.load(tmp_path / "all" / f) for f in ("distances.npy", "ids.npy", "rows.npy"))
    assert d.dtype == np.float32 and i.dtype == np.float64 and r.dtype == np.float64
    assert np.array_equal(d, D) and np.array_equal(i.astype(np.int64), I) and np.array_equal(r, np.arange(100))

    monkeypatch.setattr(bench, "DUMP_BYTES", 30 * (bench.K * 12 + 8))
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), D, I)
    ra, rb = np.load(tmp_path / "a" / "rows.npy"), np.load(tmp_path / "b" / "rows.npy")
    assert len(ra) == 30 and np.array_equal(ra, rb) and (np.diff(ra) > 0).all()
    rows = ra.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "distances.npy"), D[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "ids.npy").astype(np.int64), I[rows])
