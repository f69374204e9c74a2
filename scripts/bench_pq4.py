#!/usr/bin/env python
"""bench_pq4.py -- 4-bit vs 8-bit product quantizers on one bench-sized IVF-PQ shard.

One shard of the bench workload (bench.py: same generator, same queries, d = 128): 125 M vectors
(1 B / 8 shards), nlist 65 536, built three times on one GPU:

  PQ32x8  M = 32 x 8 bit, 32 B / vector   fused block scan (the bench index)
  PQ64x4  M = 64 x 4 bit, 32 B / vector   fused block scan, pair table
  PQ32x4  M = 32 x 4 bit, 16 B / vector   row-major scan

For each configuration, batch 4096, k = 10, nprobe in {8, 16, 32}: scan time per launch (the scan
kernel alone, dfx_profile_*), QPS of the whole shard search with device-resident queries, the
algorithmic scan bandwidth ndis * row_bytes / scan time against the HBM peak, recall@10 over the
certified and over all evaluation queries, and a bit-exact check of a 64-query sample against the
CPU oracle (D, I, ndis and the t-values of every probed row).  Writes one JSON file.

    python scripts/bench_pq4.py --out profiles/r03_pq4_vs_pq8.json
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import D, K, GroundTruth, log, nlist_for, recall_at_k  # noqa: E402

CONFIGS = {"PQ32x8": (32, 8), "PQ64x4": (64, 4), "PQ32x4": (32, 4)}


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        pl, clk = [v.strip() for v in out.stdout.strip().splitlines()[0].split(",")]
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(pl), float(clk)
    except Exception as e:  # noqa: BLE001 -- reported, not fatal
        info["power_limit_error"] = repr(e)
    return info


def build(engine, synth, torch, nvec, nlist, M, nbits, args, gt=None):
    idx = engine.GpuIndex(engine.KIND_IVF_PQ, D, engine.METRIC_L2, nlist=nlist, pq_m=M, pq_nbits=nbits)
    idx.set_param("kmeans_niter", args.kmeans_niter)
    idx.set_param("max_points_per_centroid", args.train_pts)
    idx.reserve(nvec)
    t0 = time.time()
    idx.train_dev(synth.rows(0, min(nvec, args.train_pts * nlist)))
    torch.cuda.synchronize()
    t_train = time.time() - t0
    t0 = time.time()
    chunk = 1 << 20
    buf = torch.empty((chunk, D), dtype=torch.float32, device="cuda")
    for r0 in range(0, nvec, chunk):
        n = min(chunk, nvec - r0)
        synth.rows(r0, n, out_t=buf[:n])
        idx.add_dev(buf[:n])
        if gt is not None:
            gt.update(buf[:n])
    idx.finalize()
    torch.cuda.synchronize()
    return idx, {"train_s": t_train, "add_s": time.time() - t0}


def oracle_check(idx, st, xq_np, nprobe, M, nbits):
    """bit-exact D, I, ndis and t-values of a query sample against the CPU oracle, on the lists the
    sample probes (the oracle holds only those: the other lists are never scanned)"""
    from oracle import oracle as O
    from tests.pq4_oracle import PackedOracleIVFPQ

    nlist = st["list_off"].shape[0] - 1
    keys, _ = O.coarse(O.METRIC_L2, st["centroids"], xq_np, nprobe)
    lists = np.unique(keys[keys >= 0])
    off = st["list_off"]
    rows = np.concatenate([np.arange(off[l], off[l + 1]) for l in lists]).astype(np.int64)
    sizes = np.zeros(nlist, dtype=np.int64)
    sizes[lists] = off[lists + 1] - off[lists]
    sub = {"centroids": st["centroids"], "codebooks": st["codebooks"], "ids": st["ids"][rows],
           "codes": st["codes"][rows], "list_off": np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)}
    o = PackedOracleIVFPQ(D, nlist, M, nbits)
    o.set_state(sub)  # recomputes the t-values on the CPU
    o.nprobe = idx.nprobe = nprobe
    Dg, Ig = idx.search(xq_np, K)
    ndis_g = idx.last_stats()["ndis"]
    Do, Io = o.search(xq_np, K)
    return {"queries": int(xq_np.shape[0]), "nprobe": nprobe, "D_equal": bool(np.array_equal(Dg, Do)),
            "I_equal": bool(np.array_equal(Ig, Io)), "ndis_equal": bool(ndis_g == o.last_ndis),
            "tvals_equal": bool(np.array_equal(st["tvals"][rows], o.tvals)), "rows_checked": int(rows.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nvec", type=int, default=125_000_000)
    ap.add_argument("--nlist", type=int, default=0, help="0 = bench.py's tier for the shard size")
    ap.add_argument("--configs", default="PQ32x8,PQ64x4,PQ32x4")
    ap.add_argument("--nprobes", default="8,16,32")
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--nq-pool", type=int, default=12288)
    ap.add_argument("--nq-eval", type=int, default=1000)
    ap.add_argument("--nq-check", type=int, default=64)
    ap.add_argument("--kmeans-niter", type=int, default=10)
    ap.add_argument("--train-pts", type=int, default=64)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch

    from distributed_faiss_b200 import engine

    nvec = args.nvec
    nlist = args.nlist or nlist_for(nvec)
    nprobes = [int(v) for v in args.nprobes.split(",")]
    # bench.py's generator and queries (its defaults), rows 0 .. nvec-1 form the shard
    G = max(1, nvec // 10)
    synth = engine.Synth(1234, D, 16, 1, 1.0, 0.02, ngroups=G, eps=0.01, delta=0.1)
    g = torch.Generator(device="cpu").manual_seed(1236)
    q_rows = torch.randint(0, nvec, (args.nq_pool,), generator=g, dtype=torch.int64).cuda()
    xq = synth.rows(0, args.nq_pool, rows_t=q_rows, noise_stream=7)
    n_eval = min(args.nq_eval, args.nq_pool)
    gtc = GroundTruth(synth, nvec, q_rows[:n_eval], xq[:n_eval], torch)
    xq_check = xq[:args.nq_check].cpu().numpy()
    batches = [xq[i * args.batch:(i + 1) * args.batch].contiguous() for i in range(max(1, args.nq_pool // args.batch))]

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    out = {"what": "IVF-PQ scan, 4-bit vs 8-bit product quantizers, one bench-sized shard",
           "gpu": gpu_info(torch), "nvec": nvec, "nlist": nlist, "d": D, "k": K, "batch": args.batch,
           "steps": args.steps, "warmup": args.warmup,
           "hbm_peak_gbs": peak, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
           "configs": {}}
    gt = None
    for name in args.configs.split(","):
        M, nbits = CONFIGS[name]
        rb = M * nbits // 8
        log(f"{name}: building {nvec} vectors, nlist {nlist}")
        idx, binfo = build(engine, synth, torch, nvec, nlist, M, nbits, args, gtc if gt is None else None)
        if gt is None:
            nbad = gtc.finish(1, None)
            gt, gt_ok = gtc.gt, gtc.certified
            out["ground_truth"] = {"queries": n_eval, "uncertified": nbad}
        cfg = {"M": M, "nbits": nbits, "row_bytes": rb, "interleaved": bool(idx.get_param("interleaved")),
               "build": binfo, "nprobe": {}}
        st = idx.get_state()
        for nprobe in nprobes:
            idx.nprobe = nprobe
            _, I = idx.search_dev(xq[:n_eval].contiguous(), K)
            rec, rec_all = recall_at_k(I, gt, gt_ok), recall_at_k(I, gt, None)
            ndis = []
            for b in batches:
                idx.search_dev(b, K)
                torch.cuda.synchronize()
                ndis.append(idx.last_stats()["ndis"])
            for it in range(args.warmup):
                idx.search_dev(batches[it % len(batches)], K)
            torch.cuda.synchronize()
            idx.profile(True)
            idx.profile_read(reset=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for it in range(args.steps):
                idx.search_dev(batches[it % len(batches)], K)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            scan_ms, launches = idx.profile_read(reset=True)
            idx.profile(False)
            per_launch = scan_ms / max(launches, 1)
            ndis_step = float(np.mean([ndis[it % len(batches)] for it in range(args.steps)]))
            bytes_per_launch = ndis_step / max(launches / args.steps, 1.0) * rb  # algorithmic: codes read once
            gbs = bytes_per_launch / (per_launch * 1e-3) / 1e9 if per_launch > 0 else 0.0
            chk = oracle_check(idx, st, xq_check, nprobe, M, nbits)
            r = {"scan_ms_per_launch": per_launch, "scan_launches_per_search": launches / args.steps,
                 "ms_per_search": ms / args.steps, "qps": args.steps * args.batch / (ms / 1e3),
                 "ndis_per_search": ndis_step, "scan_gbs": gbs, "scan_frac_of_hbm_peak": gbs / peak,
                 "recall_at_10_certified": rec, "recall_at_10_all": rec_all, "oracle_check": chk}
            cfg["nprobe"][str(nprobe)] = r
            log(f"{name} nprobe {nprobe}: {json.dumps(r)}")
        out["configs"][name] = cfg
        del idx, st
        gc.collect()
        torch.cuda.empty_cache()
    if "PQ32x8" in out["configs"] and "PQ64x4" in out["configs"]:
        out["pq64x4_over_pq32x8_scan_time"] = {
            p: out["configs"]["PQ64x4"]["nprobe"][p]["scan_ms_per_launch"] / out["configs"]["PQ32x8"]["nprobe"][p]["scan_ms_per_launch"]
            for p in out["configs"]["PQ32x8"]["nprobe"]}
    out["all_bit_exact"] = all(all(v for k_, v in r["oracle_check"].items() if k_.endswith("_equal"))
                               for c in out["configs"].values() for r in c["nprobe"].values())
    text = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)
    return 0 if out["all_bit_exact"] else 1


if __name__ == "__main__":
    sys.exit(main())
