#!/usr/bin/env python
"""bench.py -- QPS at recall@10 >= 0.95, IVF-PQ d=128, 1B synthetic vectors, 8 shards.

Usage: `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line from rank 0.  A
"step" is one pass of the hot path (IndexClient.search fan-out -> coarse quantizer -> PQ table ->
inverted-list scan -> cross-shard merge) over one batch of `--batch` synthetic queries; every
timed region runs K steps after W warm-up steps.  N>1 is launched by torchrun (one rank per GPU,
NCCL).  `--dump-outputs DIR` writes what the last timed step returned (see dump_outputs), so
that two builds can be compared output for output on the same seeded inputs.

Workload (BASELINE.json configs[4], SURVEY.md 8d): N vectors, d=128, 8 shards (row block b of
50 000 rows -> shard b mod 8, mimicking the client's round-robin), every shard its own IVF-PQ
(M=32 x 8 bit, nlist per shard by size tier), k=10, nprobe = smallest power of two whose
recall@10 (|top10 ∩ exact top10| / 10) on held-out queries is >= 0.95.  With N GPUs each rank
holds 8/N shards (total work fixed -> "strong" scaling).

`--impl reference` times the CPU restatement of the reference's FAISS path (oracle/, all host
threads) on a bounded sample of the same workload; see cpu_baseline.sample in the output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: keep NCCL's banner / debug output on stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

BLOCK = 50_000   # rows per round-robin block (reference buffer_bsz default, index_cfg.py:23)
NSHARDS = 8
D = 128
K = 10
PQ_M = 32


_T0 = time.time()


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.time() - _T0:7.1f}s]", *a, file=sys.stderr, flush=True)


def nlist_for(n_shard: int) -> int:
    if n_shard >= 50_000_000:
        return 65536
    if n_shard >= 5_000_000:
        return 16384
    if n_shard >= 500_000:
        return 4096
    return 1024


# ---------------------------------------------------------------------------------------------
def shard_rows(nvec: int, shard: int):
    """(first_row, n_rows) of every block owned by `shard`, in arrival order."""
    nblocks = (nvec + BLOCK - 1) // BLOCK
    out = []
    for b in range(shard, nblocks, NSHARDS):
        r0 = b * BLOCK
        out.append((r0, min(BLOCK, nvec - r0)))
    return out


def build_shard(engine, synth, nvec, shard, args, torch, gt=None):
    """generate -> train -> add, all on device.  Returns (GpuIndex, id_table int64 [n_shard])."""
    blocks = shard_rows(nvec, shard)
    n_shard = sum(n for _, n in blocks)
    nlist = args.nlist or nlist_for(n_shard)
    idx = engine.GpuIndex(engine.KIND_IVF_PQ, D, engine.METRIC_L2, nlist=nlist, pq_m=PQ_M)
    idx.set_param("kmeans_niter", args.kmeans_niter)
    idx.set_param("max_points_per_centroid", args.train_pts)
    idx.reserve(n_shard)
    # training set = the first rows of the shard (reference trains on the first train_num rows)
    n_train = min(n_shard, args.train_pts * nlist)
    xs, got = [], 0
    for r0, n in blocks:
        take = min(n, n_train - got)
        xs.append(synth.rows(r0, take))
        got += take
        if got >= n_train:
            break
    xt = torch.cat(xs) if len(xs) > 1 else xs[0]
    t0 = time.time()
    idx.train_dev(xt)
    torch.cuda.synchronize()
    t_train = time.time() - t0
    del xt, xs
    t0 = time.time()
    ids = []
    group = max(1, (1 << 20) // BLOCK)  # add ~1M rows per call
    buf = torch.empty((group * BLOCK, D), dtype=torch.float32, device="cuda")
    for g0 in range(0, len(blocks), group):
        part = blocks[g0:g0 + group]
        off = 0
        for r0, n in part:
            synth.rows(r0, n, out_t=buf[off:off + n])
            ids.append(torch.arange(r0, r0 + n, dtype=torch.int64, device="cuda"))
            off += n
        idx.add_dev(buf[:off])
        if gt is not None:
            gt.update(buf[:off])
    idx.finalize()
    torch.cuda.synchronize()
    t_add = time.time() - t0
    del buf
    return idx, torch.cat(ids), {"nlist": nlist, "n": n_shard, "train_s": t_train, "add_s": t_add}


class GroundTruth:
    """Exact top-K of the evaluation queries, certified by brute force over ALL rows.

    The generator gives every row 9 near neighbours (its group: rows g, g+G, g+2G, ...), so the
    candidate answer of a query drawn from row i is the K closest members of i's group, found by
    generating those ~10 rows and measuring them directly.  It is then CERTIFIED against the
    whole database: while the build pass streams every generated chunk through `update`, the
    number of rows closer than the candidate's K-th distance (plus a rounding margin) is counted
    with one fp32 GEMM per chunk (torch/cuBLAS -- checker code, not the product path).  A query
    whose count exceeds what its own group explains is 'uncertified' and excluded (reported)."""

    def __init__(self, synth, nvec, q_rows, xq, torch):
        self.torch = torch
        G = synth.p.ngroups
        assert G > 0, "ground truth needs the grouped generator"
        nq = xq.shape[0]
        per = (nvec + G - 1) // G
        g = q_rows % G
        j = torch.arange(per, device="cuda", dtype=torch.int64)
        rows = g[:, None] + j[None, :] * G
        valid = rows < nvec
        rows_c = torch.where(valid, rows, g[:, None].expand_as(rows))
        x = synth.rows(0, rows_c.numel(), rows_t=rows_c.reshape(-1).contiguous()).view(nq, per, D)
        d2 = ((x - xq[:, None, :]) ** 2).sum(-1)
        d2 = torch.where(valid, d2, torch.full_like(d2, float("inf")))
        dv, di = torch.sort(d2, dim=1, stable=True)
        self.gt = torch.gather(rows, 1, di[:, :K])
        self.gt[~torch.isfinite(dv[:, :K])] = -1
        self.q = xq
        self.qn = (xq ** 2).sum(1)
        self.margin = 1e-4 * (self.qn + 1.0)
        self.tau = dv[:, K - 1] + self.margin                      # threshold in true squared distance
        # how many group members the GEMM-form test will count (same formula as update())
        xm = x.reshape(-1, D)
        gem = ((xm ** 2).sum(1).view(nq, per) - 2 * (x @ xq[:, :, None]).squeeze(-1)) + self.qn[:, None]
        gem = torch.where(valid, gem, torch.full_like(gem, float("inf")))
        self.expected = (gem < self.tau[:, None]).sum(1)
        self.count = torch.zeros(nq, dtype=torch.int64, device="cuda")

    def update(self, x):
        torch = self.torch
        for r0 in range(0, x.shape[0], 262144):
            xs = x[r0:r0 + 262144]
            v = (xs ** 2).sum(1)[None, :] - 2 * (self.q @ xs.T)      # + qn on the other side
            self.count += (v < (self.tau - self.qn)[:, None]).sum(1)

    def finish(self, world, dist):
        if world > 1:
            dist.all_reduce(self.count)
        self.certified = self.count <= self.expected
        return int((~self.certified).sum().item())


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, D, I):
    """One step's answer -- D [nq,k] float32 distances, I [nq,k] int64 row ids -- as
    out_dir/distances.npy (float32) and out_dir/ids.npy (float64, exact for ids < 2**53), with the
    query rows they belong to in out_dir/rows.npy.  Above DUMP_BYTES a fixed, seeded sample of the
    query rows is kept."""
    nq, k = D.shape
    per_row = k * (4 + 8) + 8
    rows = np.arange(nq)
    if nq * per_row > DUMP_BYTES:
        rows = np.sort(np.random.RandomState(0).choice(nq, DUMP_BYTES // per_row, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "distances.npy"), np.asarray(D, dtype=np.float32)[rows])
    np.save(os.path.join(out_dir, "ids.npy"), np.asarray(I, dtype=np.float64)[rows])
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


def recall_at_k(I, gt, ok=None):
    hits = ((I[:, :, None] == gt[:, None, :]) & (gt[:, None, :] >= 0)).any(-1).sum(-1).float()
    denom = (gt >= 0).sum(-1).clamp(min=1).float()
    r = hits / denom
    if ok is not None:
        r = r[ok]
    return float(r.mean().item())


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed regions (B200_PROFILING.md): an
    in-process NVML thread (5 ms period; the timed region of the default run is ~0.15 s, too short
    for an `nvidia-smi -lms` child to even start), `nvidia-smi` as the fallback.  `start()` returns
    once the first sample is in."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.sm, self.mx, self.mask = [], [], 0
        self._stop = threading.Event()
        self.t = None
        self.source = None

    def _handle(self):
        import pynvml
        import torch

        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.gpu).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)

    def _loop_nvml(self, nv, h):
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while not self._stop.is_set():
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
            self.mx.append(float(mx))
            try:
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            time.sleep(0.005)

    def _loop_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        bits = [0x8, 0x40, 0x20, 0x4]
        self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            if r and r[0].replace(".", "").isdigit():
                self.sm.append(float(r[0]))
                if len(r) > 1 and r[1].replace(".", "").isdigit():
                    self.mx.append(float(r[1]))
                for i, b in enumerate(bits):
                    if len(r) > 2 + i and r[2 + i] == "Active":
                        self.mask |= b
            if self._stop.is_set():
                break
        self.proc.terminate()

    def start(self):
        try:
            nv, h = self._handle()
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            self.source = "nvml"
            self.t = threading.Thread(target=self._loop_nvml, args=(nv, h), daemon=True)
        except Exception:
            self.source = "nvidia-smi"
            self.t = threading.Thread(target=self._loop_smi, daemon=True)
        self.t.start()
        t0 = time.time()
        while not self.sm and time.time() - t0 < 10.0:   # first sample before the timed region starts
            time.sleep(0.005)

    def stop(self):
        self._stop.set()
        if self.t is not None:
            self.t.join(timeout=2.0)
        reasons = [n for b, n in self.REASONS.items() if self.mask & b]
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": reasons, "samples": len(self.sm),
                "source": self.source}


# ---------------------------------------------------------------------------------------------
def make_cpu_baseline(shard_idx_obj, threads):
    """ship ONE shard (codes, ids, centroids, codebooks) to the host: the timed CPU baseline
    (oracle/cpu_baseline.py: sgemm coarse + threaded scan) and the bit-exact checker share the state"""
    from oracle import cpu_baseline as CB

    st = shard_idx_obj.get_state()
    return CB.CpuIVFPQ(st, threads=threads), st


def check_against_oracle(st, shard, xq_np, nprobe, nq_check):
    """bit-exact parity of one GPU shard against the CHECKER oracle on a query sample"""
    from oracle import oracle as O

    o = O.OracleIVFPQ(D, st["nlist"], PQ_M, 8, coarse_metric=O.METRIC_L2)
    o.set_state(st, recompute_tvals=False)
    o.nprobe = nprobe
    q = xq_np[:nq_check]
    Do, Io = o.search(q, K)
    shard.nprobe = nprobe
    Dg, Ig = shard.search(q, K)
    return bool(np.array_equal(Dg, Do) and np.array_equal(Ig, Io))


def time_cpu(cb, xq_np, nprobe, batch, min_seconds, n_shards_total, offset=0):
    """one timed sample of the CPU baseline: whole batches of `batch` queries against ONE shard of
    the workload until `min_seconds` have passed; system QPS = shard QPS / n_shards (the same host
    serves every shard, SURVEY 8d)"""
    nb = max(1, (xq_np.shape[0] - batch) // batch + 1)
    done, t0, it = 0, time.perf_counter(), 0
    while True:
        off = ((offset + it) % nb) * batch
        cb.search(xq_np[off:off + batch], K, nprobe)
        done += batch
        it += 1
        dt = time.perf_counter() - t0
        if dt >= min_seconds:
            break
    return (done / dt) / n_shards_total, dt, done


def free_ports(n):
    import socket

    socks = [socket.socket() for _ in range(n)]
    try:
        for s_ in socks:
            s_.bind(("127.0.0.1", 0))
        return [s_.getsockname()[1] for s_ in socks]
    finally:
        for s_ in socks:
            s_.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nvec", type=int, default=int(os.environ.get("DFX_BENCH_NVEC", 1_000_000_000)))
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--nprobe", type=int, default=0, help="0 = smallest power of two reaching the recall gate")
    ap.add_argument("--nlist", type=int, default=0)
    ap.add_argument("--nq-pool", type=int, default=12288)
    ap.add_argument("--kmeans-niter", type=int, default=10)
    ap.add_argument("--train-pts", type=int, default=64, help="training points per centroid")
    ap.add_argument("--clusters", type=int, default=1, help="generator cluster centres (1 = one smooth distribution)")
    ap.add_argument("--group-size", type=int, default=10, help="rows per near-neighbour group")
    ap.add_argument("--eps", type=float, default=0.01, help="per-row isotropic noise")
    ap.add_argument("--delta", type=float, default=0.1, help="per-row latent spread inside a group")
    ap.add_argument("--nq-eval", type=int, default=1000, help="queries with certified exact ground truth")
    ap.add_argument("--rank-dim", type=int, default=16)
    ap.add_argument("--sigma", type=float, default=1.0)
    ap.add_argument("--sigma-q", type=float, default=0.02)
    ap.add_argument("--cpu-seconds", type=float, default=2.0, help="minimum CPU time of one timed CPU sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the query-batch sweep 1/8/64/512/4096")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the answer of the last timed step into DIR (.npy)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the answer of the GPU path (--impl b200)")

    import torch

    from distributed_faiss_b200 import engine, spmd

    log("imports done")

    if args.impl == "reference":
        # CPU arm: rank 0 alone runs and prints; no process group is needed
        if int(os.environ.get("RANK", "0")) != 0:
            return 0
        rank, local_rank, world = 0, int(os.environ.get("LOCAL_RANK", "0")), 1
        torch.cuda.set_device(local_rank % max(torch.cuda.device_count(), 1))
    else:
        rank, local_rank, world = spmd.init_process_group_from_env()
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    assert NSHARDS % world == 0, "--gpus must divide 8"
    dist = torch.distributed
    nvec = args.nvec
    C = max(1, args.clusters)
    G = max(C, (nvec // args.group_size) // C * C)      # rows i, i+G, i+2G, ... form a group
    synth = engine.Synth(1234, D, args.rank_dim, C, args.sigma, args.sigma_q, ngroups=G, eps=args.eps,
                         delta=args.delta)

    # ---------------- queries (perturbed database rows) and their candidate ground truth
    g = torch.Generator(device="cpu").manual_seed(1236)
    q_rows = torch.randint(0, nvec, (args.nq_pool,), generator=g, dtype=torch.int64).cuda()
    xq = synth.rows(0, args.nq_pool, rows_t=q_rows, noise_stream=7)
    n_eval = min(args.nq_eval, args.nq_pool)
    gtc = None if args.impl == "reference" else GroundTruth(synth, nvec, q_rows[:n_eval], xq[:n_eval], torch)

    # ---------------- build this rank's shards (the GT certification rides on the same pass)
    s_loc = NSHARDS // world
    my_shards = list(range(rank * s_loc, (rank + 1) * s_loc))
    if args.impl == "reference":
        my_shards = [0]
    t_build0 = time.time()
    shards, tables, infos = [], [], []
    for s in my_shards:
        idx, tab, info = build_shard(engine, synth, nvec, s, args, torch, gtc)
        shards.append(idx)
        tables.append(tab)
        infos.append(info)
        log(f"shard {s}: {info}")
    build_s = time.time() - t_build0

    # ---------------- reference arm: the CPU baseline alone (the shard was built on the GPU and
    # exported to the host; nothing of libdfx runs inside the timed region)
    if args.impl == "reference":
        from oracle import cpu_baseline as CB

        nprobe = args.nprobe or (8 if nvec >= 500_000_000 else 4)
        threads = CB.host_threads()
        xq_np = xq.cpu().numpy()
        cb, st = make_cpu_baseline(shards[0], threads)
        log(f"shard 0 exported to the host; CPU baseline on {cb.threads} threads ({CB._lib_kind} build)")
        B = args.batch
        # agreement with the GPU / checker on this shard (the GPU arm measures recall with this nprobe)
        shards[0].nprobe = nprobe
        Dg, Ig = shards[0].search(xq_np[:512], K)
        Dc, Ic = cb.search(xq_np[:512], K, nprobe)
        agree = float((Ic == Ig).mean())
        vals = []
        for it in range(args.warmup + args.steps):
            v, dt, done = time_cpu(cb, xq_np, nprobe, B, args.cpu_seconds, NSHARDS, offset=it)
            if it >= args.warmup:
                vals.append(v)
        v = float(np.median(vals))
        cbj = {"value": v, "unit": "QPS", "cores": cb.threads, "kind": "port",
               "sample": f"shard 0 of {NSHARDS} ({cb.ntotal} vectors, nlist {cb.nlist}), batches of {B} queries, nprobe "
                         f"{nprobe}, >= {args.cpu_seconds:g} s per timed sample, median of {len(vals)}; "
                         f"system QPS = shard QPS / {NSHARDS}",
               "implementation": "oracle/cpu_ivfpq.c: MKL sgemm coarse quantizer + OpenMP table build / list scan "
                                 f"({CB._lib_kind} build); NOT the scalar bit-exact checker",
               "spread": float((max(vals) - min(vals)) / v) if v else None,
               "ids_equal_gpu_shard": agree, "setup": "shard 0 built by libdfx on GPU 0 and exported; timed region is CPU only"}
        out = {"impl": "reference", "metric": "QPS at recall@10>=0.95, IVF-PQ d=128", "value": v, "unit": "QPS",
               "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": 1e3 * B / v if v else None,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": workload_name(nvec), "nvec": nvec, "shards": NSHARDS, "nprobe": nprobe, "batch": B,
                          "k": K, "nprobe_source": "the recall gate of the GPU arm on the same index (config.nprobe there)"},
               "cpu_baseline": cbj,
               "e2e": {"value": v, "unit": "QPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out), flush=True)
        return 0

    gt, gt_viol, gt_ok = None, 0, None
    gt_viol = gtc.finish(world, dist)
    gt, gt_ok = gtc.gt, gtc.certified
    log(f"ground truth: {n_eval} queries, {gt_viol} uncertified")

    # ---------------- the reference's process model on this box: one IndexServer per shard (rank r
    # hosts servers r*s_loc ...), their control sockets, the NCCL search plane over them, and ONE
    # IndexClient in the process of rank 0.  Ranks != 0 serve until rank 0 stops the plane.
    import tempfile
    import threading

    from distributed_faiss_b200.client import IndexClient
    from distributed_faiss_b200.index_cfg import IndexCfg
    from distributed_faiss_b200.server import IndexServer

    store = tempfile.mkdtemp(prefix="dfx_bench_")
    ports = free_ports(s_loc)
    servers = []
    for j, s in enumerate(my_shards):
        srv = IndexServer(s, store, device=torch.cuda.current_device())
        cfg = IndexCfg(index_builder_type="knnlm", dim=D, metric="l2", centroids=infos[j]["nlist"], code_size=PQ_M)
        srv.adopt_index("bench", cfg, shards[j], tables[j])
        threading.Thread(target=srv.start_blocking, args=(ports[j],), daemon=True).start()
        servers.append(srv)
    plane = spmd.SearchPlane(servers)
    all_ports = [None] * world
    if world > 1:
        dist.all_gather_object(all_ports, ports)
    else:
        all_ports = [ports]
    if rank != 0:
        plane.serve_forever()
        dist.barrier()
        dist.destroy_process_group()
        return 0

    disc = os.path.join(store, "servers.txt")
    with open(disc, "w") as fh:
        flat = [p_ for pr in all_ports for p_ in pr]
        fh.write(f"{len(flat)}\n" + "".join(f"127.0.0.1,{p_}\n" for p_ in flat))
    client = IndexClient(disc)
    client.cfg = IndexCfg(index_builder_type="knnlm", dim=D, metric="l2")
    assert client.plane is plane, "IndexClient did not attach to the NCCL search plane"

    def search_dev(x_t):
        """device-resident form of IndexClient.search (inputs already in HBM): the collective only"""
        o = plane.search("bench", x_t, K, maximize=False, int_meta=True)
        return o.D, o.I

    # ---------------- nprobe: smallest power of two meeting the recall gate
    recalls = {}
    nprobe = args.nprobe
    if not nprobe:
        for cand in (1, 2, 4, 8, 16, 32, 64, 128, 256, 512):
            if cand > shards[0].nlist:
                break
            client.set_nprobe("bench", cand)
            _, I = search_dev(xq[:n_eval].contiguous())
            recalls[cand] = recall_at_k(I, gt, gt_ok)
            log(f"nprobe {cand}: recall@10 = {recalls[cand]:.4f}")
            nprobe = cand
            if recalls[cand] >= 0.95:
                break
    client.set_nprobe("bench", nprobe)
    _, I = search_dev(xq[:n_eval].contiguous())
    log(f"nprobe = {nprobe}")
    recall = recall_at_k(I, gt, gt_ok)
    recall_all = recall_at_k(I, gt, None)
    r1 = float((I[:, :1] == gt[:, :1])[gt_ok].float().mean().item())

    # ---------------- timed regions
    def batches_of(b):
        nb = max(1, args.nq_pool // b)
        if b <= args.nq_pool:
            return [xq[i * b:(i + 1) * b].contiguous() for i in range(min(nb, 64))]
        return [xq.repeat((b // args.nq_pool) + 1, 1)[:b].contiguous()]

    def timed(batches_, steps, warmup, host=False):
        """K steps bracketed by device events on EVERY rank (plane.timer_*), max over ranks.
        Returns (ms, what the last step returned)."""
        host_batches = [b.cpu().numpy() for b in batches_] if host else None
        run = (lambda i: client.search(host_batches[i % len(batches_)], K, "bench")) if host else \
              (lambda i: search_dev(batches_[i % len(batches_)]))
        for it in range(warmup):
            run(it)
        torch.cuda.synchronize()
        plane.timer_start()
        for it in range(steps):
            last = run(it)
        return plane.timer_stop(), last

    B = args.batch
    batches = batches_of(B)
    # ndis per batch (untimed) for the roofline's algorithmic bytes: this rank's shards
    ndis_per_batch = []
    for b in batches:
        search_dev(b)
        torch.cuda.synchronize()
        ndis_per_batch.append(sum(s.last_stats()["ndis"] for s in shards))
    for s in shards:
        s.profile(True)
        s.profile_read(reset=True)
    clocks = ClockSampler(local_rank)
    clocks.start()
    launches0 = engine.launch_count()
    torch.cuda.profiler.start()   # for `ncu --profile-from-start off`; a no-op otherwise
    ms, (D_last, I_last) = timed(batches, args.steps, args.warmup)
    torch.cuda.profiler.stop()
    launches = engine.launch_count() - launches0
    if args.dump_outputs:
        # copied now: later searches may reuse the plane's result buffers
        dump_outputs(args.dump_outputs, D_last.cpu().numpy(), I_last.cpu().numpy())
    scan_ms, scan_launches = 0.0, 0
    for s in shards:
        m, n = s.profile_read(reset=True)
        scan_ms += m
        scan_launches += n
        s.profile(False)
    qps = args.steps * B / (ms / 1e3)
    ndis_step = float(np.mean([ndis_per_batch[it % len(batches)] for it in range(args.steps)]))
    launches_timed = launches * args.steps // (args.steps + args.warmup)
    log(f"timed region done: {ms / args.steps:.3f} ms/step")

    # e2e: IndexClient.search with HOST buffers -- pinned staging, H2D, the collective, one D2H,
    # integer metadata rows -- i.e. the call a user of the reference makes
    ms_e2e, _ = timed(batches, args.steps, args.warmup, host=True)
    clk = clocks.stop()
    qps_e2e = args.steps * B / (ms_e2e / 1e3)
    log(f"e2e done: {ms_e2e / args.steps:.3f} ms/step")

    # the same client through the reference's socket fan-out returns the same answer
    # (at N = 1, where all 8 servers live in this process.  At N > 1 the socket path would be served
    # by threads of processes whose main thread waits in a NCCL broadcast: the first launch of a
    # not-yet-used kernel there needs a context-wide synchronisation under CUDA's lazy module
    # loading, which cannot complete while that NCCL kernel waits for its peer -- the 2-GPU run of
    # round 2 hung exactly there.  CUDA_MODULE_LOADING=EAGER avoids it at the price of minutes of
    # start-up (every torch kernel is loaded); tests/test_plane.py covers plane == socket at world
    # size 2 on gloo, DFX_BENCH_SOCKET_CHECK=1 forces the check here.)
    plane_equals_socket = None
    if world == 1 or os.environ.get("DFX_BENCH_SOCKET_CHECK") == "1":
        hb = batches[0][:64].cpu().numpy()
        Dp, Mp = client.search(hb, K, "bench")
        client.detach_plane()
        Ds, Ms = client.search(hb, K, "bench")
        client.plane = plane
        plane_equals_socket = bool(np.array_equal(Dp, Ds) and Mp == Ms)

    sweep, sweep_e2e = {}, {}
    if not args.no_sweep:
        for b in (1, 8, 64, 512, 4096):
            bb = batches_of(b)
            t, _ = timed(bb, args.steps, args.warmup)
            sweep[str(b)] = args.steps * b / (t / 1e3)
            t, _ = timed(bb, args.steps, args.warmup, host=True)
            sweep_e2e[str(b)] = args.steps * b / (t / 1e3)
        log(f"sweep: {sweep}")

    # roofline of the dominant kernel: algorithmic bytes = ndis * code_bytes (SURVEY 8d)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    per_launch_ms = scan_ms / max(scan_launches, 1)
    # this rank's launches cover its local shards; bytes per launch = ndis of one shard-search
    bytes_per_launch = (ndis_step / max(len(shards), 1)) * PQ_M
    launches_per_search = max(1, round(scan_launches / max((args.steps + args.warmup) * len(shards), 1)))
    bytes_per_launch /= launches_per_search
    achieved = bytes_per_launch / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else 0.0
    scan_ms_per_step = scan_ms / (args.steps + args.warmup)
    # DRAM traffic of the same kernel from the committed ncu --set full capture (same command)
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_scan_traffic.json")))
        if tr["when"] == {"nvec": nvec, "batch": B, "nprobe": nprobe} and world == 1:
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
    except Exception:
        pass
    roofline = {"kernel": "scan_pq_il2_kernel (IVF-PQ table build + list scan, block-interleaved M=32)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_launch": bytes_per_launch, "ms_per_launch": per_launch_ms,
                "launches_per_step": scan_launches / (args.steps + args.warmup),
                "scan_share_of_step": scan_ms_per_step / (ms / args.steps) if ms else None}

    cb = None
    if world == 1 and not args.no_cpu:
        from oracle import cpu_baseline as CB

        xq_np = xq.cpu().numpy()
        cbo, st = make_cpu_baseline(shards[0], CB.host_threads())
        cbo.search(xq_np[:256], K, nprobe)   # warm
        vals = [time_cpu(cbo, xq_np, nprobe, B, args.cpu_seconds, NSHARDS, offset=i)[0] for i in range(5)]
        v = float(np.median(vals))
        cb = {"value": v, "unit": "QPS", "cores": cbo.threads, "kind": "port",
              "sample": f"shard 0 of {NSHARDS} ({cbo.ntotal} vectors, nlist {cbo.nlist}), batches of {B} queries, "
                        f"nprobe {nprobe}, >= {args.cpu_seconds:g} s per timed sample, median of 5; "
                        f"system QPS = shard QPS / {NSHARDS}",
              "implementation": "oracle/cpu_ivfpq.c: MKL sgemm coarse quantizer + OpenMP table build / list scan "
                                f"({CB._lib_kind} build); NOT the scalar bit-exact checker",
              "spread": float((max(vals) - min(vals)) / v) if v else None}
        # cross-check on the way: the GPU shard and the CHECKER oracle agree bit for bit on a sample
        cb["gpu_equals_oracle"] = check_against_oracle(st, shards[0], xq_np, nprobe, 256)
        del cbo, st
        log("cpu baseline done")

    out = {
        "metric": "QPS at recall@10>=0.95, IVF-PQ d=128", "value": qps, "unit": "QPS", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32 (u8 PQ codes, f32 tables/accumulate)",
        "data": "synthetic",
        "config": {"workload": workload_name(nvec), "nvec": nvec, "shards": NSHARDS, "shards_per_gpu": s_loc,
                   "nlist_per_shard": infos[0]["nlist"], "pq": "M=32 x 8 bit", "k": K, "nprobe": nprobe,
                   "batch": B, "recall_at_10": recall, "recall_at_10_all_queries": recall_all, "recall_1_at_1": r1,
                   "recall_by_nprobe": recalls,
                   "gt_uncertified_queries": gt_viol, "l2_flush": "working set (PQ codes) >> 126 MB L2",
                   "generator": {"clusters": C, "groups": G, "group_size": args.group_size, "rank": args.rank_dim,
                                 "sigma": args.sigma, "delta": args.delta, "eps": args.eps, "sigma_q": args.sigma_q},
                   "train": {"kmeans_niter": args.kmeans_niter, "points_per_centroid": args.train_pts},
                   "build_seconds": build_s, "ndis_per_step": ndis_step,
                   "api": "value: SearchPlane collective with device-resident queries; e2e: "
                          "distributed_faiss.client.IndexClient.search(host ndarray) over the NCCL search plane, "
                          "8 IndexServer shards, integer metadata"},
        "e2e": {"value": qps_e2e, "unit": "QPS", "h2d_bytes_per_step": B * D * 4, "d2h_bytes_per_step": B * K * 12 + 8 * world,
                "ms_per_step": ms_e2e / args.steps, "through": "IndexClient.search", "plane_equals_socket": plane_equals_socket},
        "gpu_launches": int(launches_timed),
        "clocks": clk,
        "roofline": roofline,
        "cpu_baseline": cb,
    }
    if sweep:
        out["config"]["qps_by_batch"] = sweep
        out["config"]["e2e_qps_by_batch"] = sweep_e2e
    print(json.dumps(out), flush=True)
    client.close()
    plane.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def workload_name(nvec):
    return f"IVF-PQ d=128, {nvec / 1e9:g}B synthetic vectors, 8 shards, k=10 (BASELINE configs[4])"


if __name__ == "__main__":
    sys.exit(main())
