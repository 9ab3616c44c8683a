#!/usr/bin/env python
"""bench.py — QPS of batched IVF search (BASELINE.json configs[1]: 1M x 384, nlist=1024,
nprobe=32, 1024-query batches, k=10) on N B200s, with recall@10, the HBM roofline of the
posting-list scan kernel, an end-to-end number through the host-buffer C-ABI call and the CPU
baseline (the oracle port of the Rust reference) timed on this box's host cores.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 (torchrun, one rank per GPU): weak scaling — every GPU holds 1M rows / 1024 lists of an
N-times larger index (list l on rank l % N), the batch is 1024*N queries, each rank scans the
probed lists it owns, one NCCL all-gather of the per-rank top-k feeds the final merge.
A "step" = one query batch.  The index (1.5 GB per GPU) is 12x larger than L2, so successive
steps cannot be served from cache; query batches rotate through distinct pre-generated sets.
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

DIM = 384
ROWS_PER_GPU = int(os.environ.get("FVDB_BENCH_ROWS", 1_000_000))
NLIST_PER_GPU = int(os.environ.get("FVDB_BENCH_NLIST", 1024))
NQ_PER_GPU = int(os.environ.get("FVDB_BENCH_NQ", 1024))
NPROBE = int(os.environ.get("FVDB_BENCH_NPROBE", 32))
# weak scaling multiplies the number of lists by the world size while nprobe stays 32: recall@10 sinks from 0.999
# (1 GPU) to 0.976 (8 GPUs, 32 of 8192 lists) with 20 training iterations — it was 0.9555 with the 8 iterations of
# round 1, close to the metric's 0.95 floor; probing more lists instead (48: 0.963, 64: 0.970 on the 8-iteration
# index) costs the per-GPU work the scaling run is meant to hold constant.  FVDB_BENCH_NPROBE overrides.
NPROBE_BY_WORLD = {1: 32, 2: 32, 4: 32, 8: 32}


def nprobe_for(world):
    if "FVDB_BENCH_NPROBE" in os.environ:
        return NPROBE
    return NPROBE_BY_WORLD.get(world, 32)
K = 10
SIGMA = float(os.environ.get("FVDB_BENCH_SIGMA", 1.0))
SEED = 1234
SEED_Q = 5678
TRAIN_ITERS = int(os.environ.get("FVDB_BENCH_TRAIN_ITERS", 20))   # SURVEY §8d: cfg-3-style training (20 iterations)
TRAIN_ROWS_PER_LIST = 64
N_QUERY_SETS = 4
RECALL_QUERIES = 256
# CPU legs: the reference arm times this many queries of every step's batch (30 steps x 256 = ~10 s of work on 16
# threads); the cpu_baseline / parity leg of the product arm takes 4x as many (a whole 1024-query batch).
CPU_SAMPLE_QUERIES = int(os.environ.get("FVDB_BENCH_CPU_QUERIES", 256))


def n_comp_for(nlist):  # SURVEY §8(d): 4 mixture components per list
    return 4 * nlist


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
            except ValueError:
                continue
            for n, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def scan_source_digest():
    """sha256 over the sources of the scan kernels (what profiles/scan_traffic.json is stamped with)."""
    import hashlib
    h = hashlib.sha256()
    for f in ("tc_scan.cu", "tc_scan_wide.cuh", "tc_ptx.cuh", "tc_scan.cuh"):
        with open(os.path.join(ROOT, "fabstir_vectordb_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def workload_name(world):
    return (f"IVF search {ROWS_PER_GPU * world}x{DIM} nlist={NLIST_PER_GPU * world} nprobe={nprobe_for(world)} "
            f"nq={NQ_PER_GPU * world}/batch k={K}")


# ---------------------------------------------------------------------------------------------
# index construction (shared by both arms so they search the identical index)
# ---------------------------------------------------------------------------------------------
def train_sample_rows(n_total, n_train):
    """Database rows of the training sample: blocks of 64 consecutive rows every 64*stride rows."""
    stride = max(1, n_total // n_train)
    i = np.arange(n_train, dtype=np.uint64)
    return (i // np.uint64(64)) * np.uint64(64 * stride) + (i % np.uint64(64))


def init_rows_of_sample(nlist, n_train):
    """Which rows of the training sample seed k-means: one per list, each from a different mixture component."""
    blk = np.arange(nlist, dtype=np.int64)
    per = n_train // nlist
    if os.environ.get("FVDB_BENCH_CLUMPED_INIT") or per != 64:
        return blk * per
    return blk * 64 + (blk // max(1, nlist // 16)) % 64


def build_index(torch, eng, rank, world, log, sh=None, scale=None):
    """Generate the synthetic database on the device, train centroids, load this rank's lists
    (size-balanced placement when a ShardedIndex is given, SURVEY §8e).  `scale` = how many times the
    single-GPU workload (default: the world size).  Returns (n_total, nlist, n_comp)."""
    from fabstir_vectordb_b200 import _lib as L
    lib = L.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    scale = world if scale is None else scale
    n_total = ROWS_PER_GPU * scale
    nlist = NLIST_PER_GPU * scale
    n_comp = n_comp_for(nlist)
    stream = torch.cuda.current_stream().cuda_stream
    t0 = time.time()
    # training sample: TRAIN_ROWS_PER_LIST rows per list, strided through the database
    n_train = min(n_total, TRAIN_ROWS_PER_LIST * nlist)
    train = torch.empty((n_train, DIM), dtype=torch.float32, device=dev)
    CH = 1 << 18
    stride = max(1, n_total // n_train)
    # blocks of 64 consecutive rows every 64*stride rows, one launch
    rc = lib.fvdb_synth_rows_strided_device(train.data_ptr(), 0, n_train, DIM, n_comp, SIGMA, SEED, 64, stride,
                                            stream)
    assert rc == 0
    torch.cuda.synchronize()
    # initial centroids: one training row per list, each from a DIFFERENT mixture component.  (Taking
    # the first row of every 64-row block picks rows 64*stride*j, whose components (row mod n_comp)
    # collapse onto n_comp/64 values: 16 seeds per component, a clumped k-means — FVDB_BENCH_CLUMPED_INIT=1
    # reproduces that earlier set-up.)
    init = train[torch.from_numpy(init_rows_of_sample(nlist, n_train)).to(dev)].contiguous()
    res = eng.train_device(train.data_ptr(), n_train, nlist, TRAIN_ITERS, init.data_ptr(), SEED)
    torch.cuda.synchronize()
    t1 = time.time()
    log(f"trained nlist={nlist} on {n_train} rows: {res} in {t1 - t0:.1f}s")
    del train
    buf = torch.empty((CH, DIM), dtype=torch.float32, device=dev)
    ids = torch.empty((CH,), dtype=torch.int32, device=dev)
    if sh is not None and world > 1 and os.environ.get("FVDB_SHARD_PLACEMENT", "balanced") == "balanced":
        # pass 1: list histogram of the whole database (every rank computes the same one), then greedy
        # size-balanced placement of the lists (l % world leaves the shards 12 % apart at 8 GPUs)
        from fabstir_vectordb_b200.shard import place_lists
        hist = torch.zeros((nlist,), dtype=torch.int64, device=dev)
        for r0 in range(0, n_total, CH):
            n = min(CH, n_total - r0)
            assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, DIM, n_comp, SIGMA, SEED, stream) == 0
            sh.list_histogram_device(buf[:n], hist)
        torch.cuda.synchronize()
        sh.set_placement(place_lists(hist.cpu().numpy(), world))
    kept = 0
    for r0 in range(0, n_total, CH):
        n = min(CH, n_total - r0)
        rc = lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, DIM, n_comp, SIGMA, SEED, stream)
        assert rc == 0
        ids[:n] = torch.arange(r0, r0 + n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        if sh is not None:
            kept += sh.add_rows_device(buf[:n], ids[:n])
        else:
            kept += eng.ivf_add_device(buf.data_ptr(), ids.data_ptr(), n, world, rank)
    log(f"rank {rank}: loaded {kept} of {n_total} rows in {time.time() - t1:.1f}s")
    return n_total, nlist, n_comp


def make_queries(torch, lib, nq, n_total, n_comp, set_idx):
    from fabstir_vectordb_b200 import synth
    dev = torch.device("cuda", torch.cuda.current_device())
    q = torch.empty((nq, DIM), dtype=torch.float32, device=dev)
    rc = lib.fvdb_synth_queries_device(q.data_ptr(), set_idx * nq, nq, DIM, n_total, n_comp, SIGMA, SEED,
                                       synth.default_qnoise(DIM, SIGMA), SEED_Q,
                                       torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    return q


def ground_truth(torch, lib, q, n_total, n_comp, rank, world, k):
    """Exact top-k over ALL rows: each rank flat-scans the rows r % world == rank of the
    database (exact fp32 scan), partial results are all-gathered and merged."""
    from fabstir_vectordb_b200 import Engine, _lib as L
    from fabstir_vectordb_b200.shard import ShardedIndex
    dev = q.device
    eng = Engine(DIM, k_max=max(16, k), device=torch.cuda.current_device())
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    CH = 1 << 18
    buf = torch.empty((CH, DIM), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    # contiguous slab per rank
    per = (n_total + world - 1) // world
    lo, hi = rank * per, min(n_total, (rank + 1) * per)
    for r0 in range(lo, hi, CH):
        n = min(CH, hi - r0)
        rc = lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, DIM, n_comp, SIGMA, SEED, stream)
        assert rc == 0
        ids = torch.arange(r0, r0 + n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        eng.flat_add_device(buf.data_ptr(), ids.data_ptr(), n)
    sh = ShardedIndex(eng, rank, world)
    ids, dist, cnt = sh.search(q, k, 0, tiers=L.TIER_RECENT)
    torch.cuda.synchronize()
    out = ids.cpu().numpy().view(np.uint32).copy(), dist.cpu().numpy().copy(), cnt.cpu().numpy().view(np.uint32).copy()
    eng.close()
    return out


def recall_of(found_ids, found_cnt, truth_ids, truth_cnt, k):
    acc = 0.0
    for i in range(found_ids.shape[0]):
        t = set(truth_ids[i, :truth_cnt[i]].tolist())
        f = set(found_ids[i, :found_cnt[i]].tolist())
        acc += len(t & f) / max(1, len(t))
    return acc / found_ids.shape[0]


def dump_outputs(out_dir, ids, dist, cnt):
    """--dump-outputs: the results of the last timed step as a caller of the search receives them (ids and
    distances [nq x k], counts [nq]), one DIR/<name>.npy each, so that two builds can be compared output for
    output.  Ids and counts are stored as float64 (every u32, the 0xFFFFFFFF of an empty slot included, is
    exact), distances in their own float32.  At most 10 K queries x k = 10: well under 64 MB, no sampling."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"ids": ids.cpu().numpy().view(np.uint32).astype(np.float64),
              "distances": dist.cpu().numpy().astype(np.float32),
              "counts": cnt.cpu().numpy().view(np.uint32).astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference (the Rust reference cannot be built in this image)
# ---------------------------------------------------------------------------------------------
def host_index_from_device(torch, lib, eng, n_total, n_comp):
    """Copy the database to the host and build the oracle's IVF over the same centroids and the
    same (parity-tested) list assignment."""
    import oracle as O
    dev = torch.device("cuda", torch.cuda.current_device())
    CH = 1 << 18
    buf = torch.empty((CH, DIM), dtype=torch.float32, device=dev)
    x = np.empty((n_total, DIM), dtype=np.float32)
    stream = torch.cuda.current_stream().cuda_stream
    for r0 in range(0, n_total, CH):
        n = min(CH, n_total - r0)
        rc = lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, DIM, n_comp, SIGMA, SEED, stream)
        assert rc == 0
        torch.cuda.synchronize()
        x[r0:r0 + n] = buf[:n].cpu().numpy()
    cents = eng.get_centroids()
    assign = eng.assign(x)
    return O.IVF(cents, x, np.arange(n_total, dtype=np.uint32), assign_=assign), x


def cpu_search_qps(ivf, q_host, k, nprobe, threads=0):
    import oracle as O
    t0 = time.perf_counter()
    ids, dist, cnt = O.hybrid_batch_search(ivf, None, None, q_host, k, nprobe, tiers=2, threads=threads)
    dt = time.perf_counter() - t0
    return q_host.shape[0] / dt, dt, (ids, dist, cnt)


def host_index(n_total, nlist, n_comp, log):
    """The bench index built WITHOUT the product library: numpy twin of the data generator (bit-identical
    to the device generator), the oracle's Lloyd loop from the same seeds (bit-identical to the engine's,
    tests/test_gpu_parity.py), the oracle's own assignment."""
    import oracle as O
    from concurrent.futures import ThreadPoolExecutor
    from fabstir_vectordb_b200 import synth
    t0 = time.time()
    x = np.empty((n_total, DIM), dtype=np.float32)
    CH = 1 << 15

    def fill(r0):
        n = min(CH, n_total - r0)
        x[r0:r0 + n] = synth.rows(r0, n, DIM, n_comp, SIGMA, SEED)

    with ThreadPoolExecutor(max_workers=max(1, (os.cpu_count() or 2) - 1)) as ex:
        list(ex.map(fill, range(0, n_total, CH)))
    n_train = min(n_total, TRAIN_ROWS_PER_LIST * nlist)
    tr_rows = train_sample_rows(n_total, n_train).astype(np.int64)
    train = x[tr_rows]
    init = train[init_rows_of_sample(nlist, n_train)].copy()
    cents, _, res = O.train_lloyd(train, init, TRAIN_ITERS)
    log(f"host index: generated {n_total} rows, trained nlist={nlist}: {res} in {time.time() - t0:.1f}s")
    ivf = O.IVF(cents, x, np.arange(n_total, dtype=np.uint32))
    log(f"host index: assigned and grouped in {time.time() - t0:.1f}s total")
    return ivf, x


def host_queries(nq, n_total, n_comp, set_idx):
    from fabstir_vectordb_b200 import synth
    return synth.queries(set_idx * nq, nq, DIM, n_total, n_comp, SIGMA, SEED, synth.default_qnoise(DIM, SIGMA), SEED_Q)


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU search path (oracle port, all host threads) on the same
    index / metric / config as the product arm.  Rank 0 only; a step = a bounded sample of one batch.
    One GPU's workload: the index is built on the host (no product library is loaded).  N > 1: the same
    N-times larger workload as the product arm; its 1M x N rows cannot be assigned on the host inside a
    bench run (N^2 x 1e9 distances), so there — and only there — the engine generates and assigns them;
    the timed region is pure host code either way."""
    if rank != 0:
        return
    import oracle as O
    log = lambda m: print(f"[reference] {m}", file=sys.stderr, flush=True)
    nprobe = nprobe_for(world)
    nq = NQ_PER_GPU * world
    sample = CPU_SAMPLE_QUERIES
    if world == 1:
        n_total, nlist = ROWS_PER_GPU, NLIST_PER_GPU
        n_comp = n_comp_for(nlist)
        ivf, _ = host_index(n_total, nlist, n_comp, log)
        qsets = [host_queries(sample, n_total, n_comp, s * (nq // sample)) for s in range(N_QUERY_SETS)]
        built = "host (numpy generator + oracle k-means / assignment)"
    else:
        import torch
        from fabstir_vectordb_b200 import Engine, _lib as L
        lib = L.load()
        torch.cuda.set_device(0)
        eng = Engine(DIM, k_max=16)
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
        n_total, nlist, n_comp = build_index(torch, eng, 0, 1, log, scale=world)
        ivf, _ = host_index_from_device(torch, lib, eng, n_total, n_comp)
        qsets = [make_queries(torch, lib, nq, n_total, n_comp, s).cpu().numpy()[:sample] for s in range(N_QUERY_SETS)]
        eng.close()
        built = "device generator + engine assignment (host build infeasible at this size); timed region is host-only"
    threads = O.num_threads()
    for w in range(args.warmup):
        cpu_search_qps(ivf, qsets[w % N_QUERY_SETS][:16], K, nprobe)
    t0 = time.perf_counter()
    for s in range(args.steps):
        cpu_search_qps(ivf, qsets[s % N_QUERY_SETS], K, nprobe)
    dt = time.perf_counter() - t0
    qps = args.steps * sample / dt
    line = {
        "impl": "reference", "metric": "QPS @ recall@10>=0.95, 1M x 384 IVF", "value": qps,
        "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(world), "note": "oracle C port of the Rust reference "
                   "(rustc/cargo absent), tight mode, OpenMP over queries", "index_built_by": built},
        "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} of {nq} queries per step, full {n_total}-row index"},
        "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def measured_peak_tf32():
    """TF32 dense peak: not in MEASURED_PEAKS.json — half the measured bf16 throughput (SURVEY §8d says so)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            d = json.load(fh)
        return 0.5 * float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "0.5 x measured bf16 sustained (MEASURED_PEAKS.json)"
    except Exception:
        return 0.5 * 2250.0, "0.5 x nominal bf16 (B200_PROFILING.md)"


def run_cfg3(args):
    """BASELINE.json configs[2]: IVF k-means training on 1M x 384, nlist = 4096, 20 iterations, shared initial
    centroids, one GPU.  A secondary line: the assignment (2 N k D flops per iteration, TF32 tensor cores +
    exact verification) is the dominant step; `achieved` divides its flops by the WHOLE iteration time
    (assignment + order-faithful centroid update + the f32 error fold), so it understates the kernel."""
    import torch
    import oracle as O
    from fabstir_vectordb_b200 import Engine, _lib as L
    torch.cuda.set_device(0)
    lib = L.load()
    n, nlist, iters = int(os.environ.get("FVDB_KM_ROWS", 1_000_000)), int(os.environ.get("FVDB_KM_NLIST", 4096)), 20
    n_comp = n_comp_for(nlist)
    data = torch.empty((n, DIM), dtype=torch.float32, device="cuda")
    assert lib.fvdb_synth_rows_device(data.data_ptr(), 0, n, DIM, n_comp, SIGMA, SEED, torch.cuda.current_stream().cuda_stream) == 0
    init = data[torch.arange(nlist, device="cuda") * (n // nlist)].contiguous()
    eng = Engine(DIM, k_max=16)
    eng.train_device(data.data_ptr(), n, nlist, 1, init.data_ptr(), SEED)   # warm-up: allocations, descriptors
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    t0 = time.perf_counter()
    res = eng.train_device(data.data_ptr(), n, nlist, iters, init.data_ptr(), SEED)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    cents = eng.get_centroids()
    rows = np.linspace(0, n - 1, 2048).astype(np.int64)
    xs = data[torch.from_numpy(rows).cuda()].cpu().numpy()
    same = int((eng.assign(xs) == O.assign(xs, cents)).sum())
    t1 = time.perf_counter()
    O.assign(xs, cents)
    cpu_rows_s = len(rows) / (time.perf_counter() - t1)
    flops = 2.0 * n * nlist * DIM * res["iterations"]
    peak, src = measured_peak_tf32()
    line = {"metric": "k-means seconds per Lloyd iteration, 1M x 384, nlist=4096", "value": dt / res["iterations"], "unit": "s/iteration",
            "n_gpus": 1, "steps": res["iterations"], "warmup": 1, "ms_per_step": dt / res["iterations"] * 1e3,
            "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (tf32 assignment, exact verify)",
            "data": "synthetic", "config": {"workload": f"k-means {n}x{DIM} nlist={nlist} max_iter={iters} shared init"},
            "train_result": res, "seconds_total": dt, "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": flops / dt / 1e12, "peak": peak, "unit": "TFLOP/s",
                         "frac": flops / dt / 1e12 / peak, "traffic": None, "kernel": "nearest-centroid assignment (kernel W, identity items)",
                         "peak_source": src, "note": "assignment flops / whole iteration time"},
            "cpu_baseline": {"value": n / cpu_rows_s, "unit": "s/iteration (assignment only, extrapolated from 2048 rows)",
                             "cores": O.num_threads(), "kind": "port", "sample": "2048 of 1M rows against the final centroids"},
            "parity_vs_oracle": {"rows": int(len(rows)), "identical_assignments": same}}
    print(json.dumps(line), flush=True)
    eng.close()


def run_cfg4(args):
    """BASELINE.json configs[3]: 1M x 384 filtered search, hybrid tiers: 300K rows in the recent (flat) tier,
    700K in the IVF tier, filter bitmap with 10 % selectivity, 1 % tombstones, 1024-query batches."""
    import torch
    import oracle as O
    from fabstir_vectordb_b200 import Engine, _lib as L, synth
    torch.cuda.set_device(0)
    lib = L.load()
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream().cuda_stream
    n_total, n_recent, nlist, nq, k, nprobe = 1_000_000, 300_000, 1024, 1024, K, 32
    n_ivf = n_total - n_recent
    n_comp = n_comp_for(nlist)
    eng = Engine(DIM, k_max=16)
    n_train = TRAIN_ROWS_PER_LIST * nlist
    train = torch.empty((n_train, DIM), dtype=torch.float32, device=dev)
    assert lib.fvdb_synth_rows_strided_device(train.data_ptr(), 0, n_train, DIM, n_comp, SIGMA, SEED, 64,
                                              max(1, n_total // n_train), stream) == 0
    init = train[torch.from_numpy(init_rows_of_sample(nlist, n_train)).to(dev)].contiguous()
    eng.train_device(train.data_ptr(), n_train, nlist, TRAIN_ITERS, init.data_ptr(), SEED)
    CH = 1 << 18
    x_host = np.empty((n_total, DIM), dtype=np.float32)
    buf = torch.empty((CH, DIM), dtype=torch.float32, device=dev)
    for r0 in range(0, n_total, CH):
        n = min(CH, n_total - r0)
        assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, DIM, n_comp, SIGMA, SEED, stream) == 0
        ids = torch.arange(r0, r0 + n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        a = max(0, min(n, n_ivf - r0))
        if a > 0:
            eng.ivf_add_device(buf.data_ptr(), ids.data_ptr(), a)
        if a < n:
            eng.flat_add_device(buf[a:].data_ptr(), ids[a:].data_ptr(), n - a)
        x_host[r0:r0 + n] = buf[:n].cpu().numpy()
    fbits = synth.filter_bitmap((n_total + 63) // 64 * 64, 10, 99)
    dele = np.arange(7, n_total, 100, dtype=np.uint32)
    eng.set_deleted(dele, True)
    qs = [make_queries(torch, lib, nq, n_total, n_comp, s) for s in range(N_QUERY_SETS)]
    d_f = torch.from_numpy(fbits.view(np.int64)).to(dev)
    o_ids = torch.empty((nq, k), dtype=torch.int32, device=dev)
    o_dst = torch.empty((nq, k), dtype=torch.float32, device=dev)
    o_cnt = torch.empty((nq,), dtype=torch.int32, device=dev)

    def step(i):
        eng.search_device(qs[i % N_QUERY_SETS].data_ptr(), nq, k, nprobe, L.TIER_BOTH, d_f.data_ptr(), fbits.size * 64,
                          o_ids.data_ptr(), o_dst.data_ptr(), o_cnt.data_ptr(), stream)

    for i in range(max(3, args.warmup)):
        step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        step(i)
    ev1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1) / args.steps
    st = eng.stats()
    step(0)
    torch.cuda.synchronize()
    ns = 32
    cents = eng.get_centroids()
    ivf = O.IVF(cents, x_host[:n_ivf], np.arange(n_ivf, dtype=np.uint32), assign_=eng.assign(x_host[:n_ivf]))
    q0 = qs[0][:ns].cpu().numpy()
    t0 = time.perf_counter()
    want = O.hybrid_batch_search(ivf, x_host[n_ivf:], np.arange(n_ivf, n_total, dtype=np.uint32), q0, k, nprobe, tiers=3,
                                 deleted=O.make_bitmap(n_total, dele), filter_bits=fbits)
    cpu_qps = ns / (time.perf_counter() - t0)
    g_ids = o_ids[:ns].cpu().numpy().view(np.uint32)
    g_dst = o_dst[:ns].cpu().numpy()
    peak, src = measured_peak_hbm()
    alg = int(st.last_algorithmic_bytes)
    line = {"metric": "QPS, 1M x 384 filtered hybrid search (10 % bitmap, 1 % tombstones)", "value": nq / (ms * 1e-3), "unit": "queries/s",
            "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "300K recent (flat) + 700K IVF rows, nlist=1024 nprobe=32 nq=1024/batch k=10, filter bitmap "
                                   "10 % pass, 1 % tombstones", "cache": "index 1.5 GB >> L2; 4 rotating query sets"},
            "fallback_queries": int(st.last_fallback_queries), "gpu_launches": int(st.last_launches) * args.steps, "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                         "kernel": "whole batch (IVF scan + flat-tier scan): rows are streamed, then masked",
                         "algorithmic_bytes_per_launch": alg, "peak_source": src,
                         "note": "the flat tier scores 1024 x 300K pairs: that scan is tensor-bound, not HBM-bound"},
            "cpu_baseline": {"value": cpu_qps, "unit": "queries/s", "cores": O.num_threads(), "kind": "port",
                             "sample": f"{ns} of {nq} queries of one batch"},
            "parity_vs_oracle": {"queries": ns, "identical_id_lists": int((g_ids == want[0]).all(axis=1).sum()),
                                 "identical_distance_bits": int((g_dst.view(np.uint32) == want[1].view(np.uint32)).all(axis=1).sum())}}
    print(json.dumps(line), flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 (default): the headline line, BASELINE.json configs[1].  cfg3 / cfg4: secondary lines for "
                         "configs[2] (k-means) and configs[3] (filtered hybrid), one GPU.  cfg5: configs[4], 100M x 384 "
                         "over 8 GPUs (12.5M rows, 2048 lists, 1250 queries per GPU; run under torchrun with --gpus 8)")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default=os.environ.get("FVDB_BENCH_MODE", "auto"), choices=["auto", "exact", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (ids, distances, counts) to DIR/<name>.npy; "
                         "the inputs are seeded, so runs with the same arguments compare output for output "
                         "(cfg2 / cfg5)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.config in ("cfg3", "cfg4")):
        ap.error("--dump-outputs covers the IVF search of cfg2 / cfg5 (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    if args.config == "cfg5":
        # BASELINE.json configs[4]: 100M x 384 sharded by list over 8 GPUs, nlist 16384, nprobe 64, 10 K-query batches
        global ROWS_PER_GPU, NLIST_PER_GPU, NQ_PER_GPU, NPROBE
        # nprobe: SURVEY §8d suggests 64 and lets the builder retune for recall >= 0.95.  With 20 k-means iterations
        # 80 of 16384 lists give recall@10 = 0.961 on this data (112: 0.970; with the 8 iterations of round 1: 64 ->
        # 0.934, 96 -> 0.948, 112 -> 0.952).  FVDB_BENCH_CFG5_NPROBE overrides.
        np5 = int(os.environ.get("FVDB_BENCH_CFG5_NPROBE", 80))
        ROWS_PER_GPU, NLIST_PER_GPU, NQ_PER_GPU, NPROBE = 12_500_000, 2048, 1250, np5
        os.environ["FVDB_BENCH_NPROBE"] = str(np5)
        os.environ.setdefault("FVDB_BENCH_PARITY", "0")   # the unsharded host index would be 154 GB: recall vs exact instead
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.config == "cfg3":
        return run_cfg3(args) if rank == 0 else None
    if args.config == "cfg4":
        return run_cfg4(args) if rank == 0 else None

    import torch
    import torch.distributed as dist
    from fabstir_vectordb_b200 import Engine, _lib as L
    from fabstir_vectordb_b200.shard import ShardedIndex

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = L.load()
    log = (lambda m: print(f"[bench r{rank}] {m}", file=sys.stderr, flush=True))

    eng = Engine(DIM, k_max=16, device=local_rank)
    if args.mode == "exact":
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    elif args.mode == "tc":
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
        eng.set_option(L.OPT_KMEANS_TC, 1)
    sh = ShardedIndex(eng, rank, world)
    n_total, nlist, n_comp = build_index(torch, eng, rank, world, log, sh=sh)
    nq = NQ_PER_GPU * world
    NPROBE = nprobe_for(world)
    qsets = [make_queries(torch, lib, nq, n_total, n_comp, s) for s in range(N_QUERY_SETS)]

    def step(i):
        return sh.search(qsets[i % N_QUERY_SETS], K, NPROBE, tiers=L.TIER_HISTORICAL)

    # first call seals the index (regroup by list) — outside the timed region
    step(0)
    torch.cuda.synchronize()

    # ---- recall@10 against exact ground truth --------------------------------------------
    rq = qsets[0][:RECALL_QUERIES].contiguous()
    f_ids, f_dist, f_cnt = sh.search(rq, K, NPROBE, tiers=L.TIER_HISTORICAL)
    torch.cuda.synchronize()
    found = (f_ids.cpu().numpy().view(np.uint32).copy(), f_dist.cpu().numpy().copy(),
             f_cnt.cpu().numpy().view(np.uint32).copy())
    fallback_q = eng.stats().last_fallback_queries
    truth = ground_truth(torch, lib, rq, n_total, n_comp, rank, world, K)
    recall = recall_of(found[0], found[2], truth[0], truth[2], K)
    log(f"recall@{K} = {recall:.4f} over {RECALL_QUERIES} queries (fallback queries {fallback_q})")
    if os.environ.get("FVDB_BENCH_DEBUG"):
        log(f"found[0]={found[0][0].tolist()} cnt={found[2][:4].tolist()} truth[0]={truth[0][0].tolist()} cnt={truth[2][:4].tolist()}")

    # ---- timed region: HBM-resident inputs ---------------------------------------------------
    sampler = ClockSampler(local_rank)  # samples clocks through warm-up + timed region
    sampler.start()
    # at least W warm-up steps, and at least ~0.6 s of them so that the clock sampler (one
    # nvidia-smi call per ~0.1 s) sees the GPU under this very load before and during the timed steps
    # (N > 1: a FIXED count — every step is a collective, so all ranks must run the same number)
    t_w = time.perf_counter()
    w = 0
    pipe = max(1, int(os.environ.get("FVDB_BENCH_PIPE", 8)))
    n_fixed = (max(args.warmup, 300) + pipe - 1) // pipe * pipe if world > 1 else 0
    while (w < n_fixed) if world > 1 else (w < args.warmup or (time.perf_counter() - t_w < 0.6 and w < 5000)):
        if pipe > 1:   # warm up the path that is timed: stream-ordered submits (both pipeline slots), one finish per group
            sh.submit(qsets[w % N_QUERY_SETS], K, NPROBE, tiers=L.TIER_HISTORICAL, slot=w % pipe)
            if (w + 1) % pipe == 0:
                sh.finish()
        else:
            step(w)
        w += 1
    if pipe > 1:
        sh.finish()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scan_ms, launches, alg_bytes, scan_rows = [], 0, 0, 0
    torch.cuda.synchronize()
    if os.environ.get("FVDB_BENCH_PROFILE"):
        torch.cuda.profiler.start()  # ncu --profile-from-start off: profile the timed region only
    # single GPU: the batches are submitted stream-ordered (fvdb_search_device_submit) and checked every
    # PIPE batches by one fvdb_search_device_finish — the GPU does not idle while the host turns a call
    # around.  Every batch is complete (NaN flag read, proof failures repaired) before ev1.  The scan
    # kernel's duration is sampled on the last batch of every group (the engine keeps one event pair).
    ev0.record()
    for s in range(args.steps):
        if pipe > 1:
            last = sh.submit(qsets[s % N_QUERY_SETS], K, NPROBE, tiers=L.TIER_HISTORICAL, slot=s % pipe)
            if (s + 1) % pipe and s + 1 != args.steps:
                continue
            sh.finish()
        else:
            last = step(s)
        st = eng.stats()
        scan_ms.append(st.last_scan_ms)
        n_in_group = ((s % pipe) + 1) if pipe > 1 else 1
        launches += (st.last_launches + (4 if world > 1 else 0)) * n_in_group   # N > 1: + coarse slice (3) + merge
        alg_bytes = st.last_algorithmic_bytes
        scan_rows = st.last_scanned_rows
    ev1.record()
    torch.cuda.synchronize()
    if os.environ.get("FVDB_BENCH_PROFILE"):
        torch.cuda.profiler.stop()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    # before the end-to-end leg, which reuses the pipeline slots' result buffers (N > 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
        log(f"wrote the last timed step's results to {args.dump_outputs}")
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    qps = nq * args.steps / (elapsed_ms * 1e-3)

    # ---- end to end: host buffers through the C-ABI call (H2D + search + D2H per step) -------
    h_q = [q.cpu().numpy() for q in qsets]
    if world == 1:
        # the call a user makes: fvdb_search with HOST buffers.  Queries and results live in
        # page-locked buffers from fvdb_host_alloc (the copy engines read / write them directly);
        # H2D of the step's queries and D2H of its results are inside the timed region.
        from fabstir_vectordb_b200 import PinnedArray
        p_q = []
        for a in h_q:
            pa = PinnedArray(a.shape, np.float32)
            pa.array[...] = a
            p_q.append(pa)
        p_out = (PinnedArray((nq, K), np.uint32), PinnedArray((nq, K), np.float32), PinnedArray((nq,), np.uint32))
        out = tuple(x.array for x in p_out)
        for w in range(3):
            eng.search(p_q[w % N_QUERY_SETS].array, K, NPROBE, tiers=L.TIER_HISTORICAL, out=out)
        # stream-ordered: fvdb_search_submit per batch (its upload overlaps the previous batch's scan),
        # one fvdb_search_finish per E2E_PIPE batches; every batch has its own result buffers
        e2e_pipe = max(1, min(8, int(os.environ.get("FVDB_BENCH_E2E_PIPE", 8))))
        p_more = [(PinnedArray((nq, K), np.uint32), PinnedArray((nq, K), np.float32), PinnedArray((nq,), np.uint32))
                  for _ in range(e2e_pipe - 1)]   # (kept alive: the arrays are views of these buffers)
        outs = [out] + [tuple(x.array for x in t_) for t_ in p_more]
        if e2e_pipe > 1:   # warm-up of the stream-ordered path (its slots allocate on first use)
            for w in range(2 * e2e_pipe):
                eng.search_submit(p_q[w % N_QUERY_SETS].array, K, NPROBE, L.TIER_HISTORICAL, outs[w % e2e_pipe])
                if (w + 1) % e2e_pipe == 0:
                    eng.search_finish()
            eng.search_finish()
        t0 = time.perf_counter()
        for s in range(args.steps):
            if e2e_pipe > 1:
                eng.search_submit(p_q[s % N_QUERY_SETS].array, K, NPROBE, L.TIER_HISTORICAL, outs[s % e2e_pipe])
                if (s + 1) % e2e_pipe == 0 or s + 1 == args.steps:
                    eng.search_finish()
            else:
                eng.search(p_q[s % N_QUERY_SETS].array, K, NPROBE, tiers=L.TIER_HISTORICAL, out=out)
        e2e_dt = time.perf_counter() - t0
        # the synchronous call, one batch at a time
        t0 = time.perf_counter()
        for s in range(args.steps):
            eng.search(p_q[s % N_QUERY_SETS].array, K, NPROBE, tiers=L.TIER_HISTORICAL, out=out)
        e2e_sync_qps = nq * args.steps / (time.perf_counter() - t0)
        # the same call with pageable numpy buffers (staged through the handle's pinned buffer)
        t0 = time.perf_counter()
        for s in range(args.steps):
            eng.search(h_q[s % N_QUERY_SETS], K, NPROBE, tiers=L.TIER_HISTORICAL)
        e2e_pageable_qps = nq * args.steps / (time.perf_counter() - t0)
    else:
        # every rank uploads ONLY its slice of the batch (nq / world queries over its own PCIe link), the
        # slices are all-gathered over NVLink; results go to page-locked host memory with asynchronous
        # copies (every step's results are read back; one synchronisation at the end)
        per = nq // world
        pinned = [torch.from_numpy(np.ascontiguousarray(a[rank * per:(rank + 1) * per])).pin_memory() for a in h_q]
        dq_slice = torch.empty((per, DIM), dtype=torch.float32, device="cuda")
        dq = torch.empty_like(qsets[0])
        out_h = (torch.empty((nq, K), dtype=torch.int32).pin_memory(), torch.empty((nq, K), dtype=torch.float32).pin_memory(),
                 torch.empty((nq,), dtype=torch.int32).pin_memory())
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        dqs = [torch.empty_like(qsets[0]) for _ in range(pipe)]
        prev = None
        for s in range(args.steps):
            dq_slice.copy_(pinned[s % N_QUERY_SETS], non_blocking=True)
            dist.all_gather_into_tensor(dqs[s % pipe].view(-1), dq_slice.view(-1))
            cur = sh.submit(dqs[s % pipe], K, NPROBE, tiers=L.TIER_HISTORICAL, slot=s % pipe)
            if prev is not None:   # the batch before this one has been exchanged and merged (stream order)
                for dst, src in zip(out_h, prev):
                    dst.copy_(src, non_blocking=True)
            prev = cur
            if (s + 1) % pipe == 0 or s + 1 == args.steps:
                sh.finish()
                for dst, src in zip(out_h, prev):
                    dst.copy_(src, non_blocking=True)
                prev = None
        torch.cuda.synchronize()
        e2e_dt = time.perf_counter() - t0
        t = torch.tensor([e2e_dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_dt = float(t.item())
    e2e_qps = nq * args.steps / e2e_dt
    if world > 1:
        e2e_pageable_qps = None
        e2e_sync_qps = None
        e2e_submission = ("per rank: H2D of its nq/world query slice + NVLink all-gather + pipelined sharded search "
                          f"(submit per batch, finish every {pipe}) + async D2H of the results")
    else:
        e2e_submission = (f"fvdb_search_submit per batch, fvdb_search_finish every {e2e_pipe}" if e2e_pipe > 1
                          else "fvdb_search per batch")
    h2d = nq * DIM * 4            # whole job: every query crosses PCIe once (N > 1: nq / world per rank)
    d2h = (nq * K * 8 + nq * 4) * world   # every rank reads the merged results back

    # ---- roofline of the dominant kernel (posting-list scan) -----------------------------------
    peak, peak_src = measured_peak_hbm()
    scan_bytes = scan_rows * DIM * 4 + scan_rows * 4  # rows + row norms/ids touched once
    mean_scan_ms = float(np.mean(scan_ms)) if scan_ms else 0.0
    achieved = scan_bytes / (mean_scan_ms * 1e-3) / 1e9 if mean_scan_ms > 0 else 0.0
    # dram__bytes_read.sum + dram__bytes_write.sum of the scan kernels (R + W) from one ncu --set full capture of
    # this very command (profiles/scan_traffic.json, written by scripts/summarize_ncu.py --traffic).  The file is
    # stamped with a digest of the kernel sources: a capture of other code is not reported.
    traffic, traffic_note = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "scan_traffic.json")) as fh:
            tj = json.load(fh)
        if world != 1:
            traffic_note = "captured on the single-GPU workload only"
        elif tj.get("source_digest") != scan_source_digest():
            traffic_note = "profiles/scan_traffic.json was captured from different kernel sources: not reported"
        else:
            traffic = float(tj["dram_bytes_per_launch"])
    except Exception:
        traffic_note = "no capture on file"
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak if peak else None, "traffic": traffic,
                "kernel": "ivf posting-list scan", "kernel_ms": mean_scan_ms,
                "traffic_note": traffic_note, "algorithmic_bytes_per_launch": scan_bytes, "peak_source": peak_src,
                "share_of_step": mean_scan_ms / (elapsed_ms / args.steps) if elapsed_ms else None}

    # ---- CPU baseline beside it (rank 0, N == 1) -------------------------------------------------
    cpu = None
    parity = None
    if world > 1 and not args.no_cpu_baseline and os.environ.get("FVDB_BENCH_PARITY", "1") != "0":
        # oracle parity of the SHARDED search: rank 0 builds the unsharded host index (the other ranks only
        # take part in the collective search of the sample) and compares 64 queries bit for bit
        sample = min(64, nq)
        cq_dev = qsets[0][:sample].contiguous()
        g = sh.search(cq_dev, K, NPROBE, tiers=L.TIER_HISTORICAL)
        torch.cuda.synchronize()
        if rank == 0:
            import oracle as O
            ivf, _ = host_index_from_device(torch, lib, eng, n_total, n_comp)
            _, _, cres = cpu_search_qps(ivf, h_q[0][:sample], K, NPROBE)
            g_ids = g[0].cpu().numpy().view(np.uint32)
            g_dist = g[1].cpu().numpy()
            same_ids = int((g_ids == cres[0]).all(axis=1).sum())
            same_bits = int((g_dist.view(np.uint32) == cres[1].view(np.uint32)).all(axis=1).sum())
            parity = {"queries": sample, "identical_id_lists": same_ids, "identical_distance_bits": same_bits}
            log(f"sharded search vs unsharded oracle: {parity}")
    if world == 1 and not args.no_cpu_baseline:
        import oracle as O
        ivf, _ = host_index_from_device(torch, lib, eng, n_total, n_comp)
        sample = min(nq, 4 * CPU_SAMPLE_QUERIES)
        cq = h_q[0][:sample]
        cpu_qps, cpu_dt, cres = cpu_search_qps(ivf, cq, K, NPROBE)
        f1 = 16
        _, dt1, _ = cpu_search_qps(ivf, cq[:f1], K, NPROBE, threads=1)
        # parity of the GPU results with the oracle on the same queries
        g_ids, g_dist, g_cnt = eng.search(cq, K, NPROBE, tiers=L.TIER_HISTORICAL)
        same_ids = int((g_ids == cres[0]).all(axis=1).sum())
        same_bits = int((g_dist.view(np.uint32) == cres[1].view(np.uint32)).all(axis=1).sum())
        parity = {"queries": sample, "identical_id_lists": same_ids, "identical_distance_bits": same_bits}
        cpu = {"value": cpu_qps, "unit": "queries/s", "cores": O.num_threads(), "kind": "port",
               "sample": f"{sample} of {nq} queries of one batch, full index; 1-thread: "
                         f"{f1 / dt1:.1f} q/s on {f1} queries",
               "host_cpus": os.cpu_count()}
        log(f"cpu baseline {cpu_qps:.1f} q/s on {O.num_threads()} threads; parity {parity}")

    line = {
        "metric": "QPS @ recall@10>=0.95, 1M x 384 IVF", "value": qps, "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(world), "submission": (f"stream-ordered (fvdb_search_device_submit), "
                   f"checked every {pipe} batches (fvdb_search_device_finish)" if pipe > 1 else "synchronous per batch"),
                   "rows_per_gpu": ROWS_PER_GPU, "dim": DIM,
                   "nlist": nlist, "nprobe": NPROBE, "nq_per_batch": nq, "k": K, "sigma": SIGMA,
                   "mixture_components": n_comp, "scan_mode": args.mode,
                   "cache": "index (1.5 GB/GPU) >> 126 MB L2; 4 rotating query sets",
                   "sharding": (f"lists placed on {world} ranks by greedy size-balanced bin packing; coarse step sharded by "
                                f"query + all-gather of the keys; all-gather of the per-rank top-k + merge") if world > 1 else "single GPU"},
        "recall_at_10": recall, "recall_queries": RECALL_QUERIES, "fallback_queries": int(fallback_q),
        "clocks": clocks,
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "host_buffers": "page-locked (fvdb_host_alloc)" if world == 1 else "page-locked (torch)",
                "pageable_value": e2e_pageable_qps, "synchronous_value": e2e_sync_qps,
                "submission": e2e_submission},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity_vs_oracle": parity,
    }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
