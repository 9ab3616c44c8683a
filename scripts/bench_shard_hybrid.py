"""Sharded hybrid search (FVDB_TIER_BOTH) throughput, weak-scaled: cfg4's shape per GPU (300 K recent-tier rows +
700 K IVF rows, nlist 1024, nprobe 32, 1024-query batches, k 10, a filter bitmap and tombstones).  Run under torchrun,
one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29513 \\
        scripts/bench_shard_hybrid.py [--steps 20] [--warmup 5] [--out profiles/shard_hybrid.jsonl]

Rank 0 appends one JSON line: the card name and power limit read in the same run, the median per-batch time over the
timed batches and QPS; parity of a query subset against ONE unsharded handle holding every row (built on rank 0);
and, on rank 0's own handle, fvdb_search_device_tiers + the ranks-1 tiered merge against fvdb_search_device
(TIER_BOTH), alternated batch by batch (the cost of keeping the tiers apart)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fabstir_vectordb_b200 import Engine, _lib as L, synth  # noqa: E402
from fabstir_vectordb_b200.shard import ShardedIndex, tiers_pack_layout  # noqa: E402

D, NLIST, NPROBE, NQ, K = 384, 1024, 32, 1024, 10
N_IVF, N_REC = 700_000, 300_000                      # per GPU
SIGMA, SEED, CH = 1.0, 1234, 1 << 17


def gen_rows(lib, buf, r0, n, n_comp):
    assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, D, n_comp, SIGMA, SEED,
                                      torch.cuda.current_stream().cuda_stream) == 0


def load(lib, n_ivf, n_rec, n_comp, dev, recent_cb, ivf_cb):
    """Every row in chunks: IVF rows [0, n_ivf), recent rows [n_ivf, n_ivf + n_rec)."""
    buf = torch.empty((CH, D), dtype=torch.float32, device=dev)
    for lo, hi, cb in ((0, n_ivf, ivf_cb), (n_ivf, n_ivf + n_rec, recent_cb)):
        for r0 in range(lo, hi, CH):
            n = min(CH, hi - r0)
            gen_rows(lib, buf, r0, n, n_comp)
            cb(buf[:n], torch.arange(r0, r0 + n, dtype=torch.int32, device=dev))
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--parity-queries", type=int, default=64)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shard_hybrid.jsonl"))
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    lib = L.load()
    n_ivf, n_rec = N_IVF * world, N_REC * world
    n_all, n_comp = n_ivf + n_rec, 4 * NLIST
    cbuf = torch.empty((NLIST * 64, D), dtype=torch.float32, device=dev)
    gen_rows(lib, cbuf, 0, cbuf.shape[0], n_comp)
    cents = cbuf[::64].cpu().numpy().copy()          # centroids: every 64th of the first rows (no training: a timing run)
    del cbuf

    eng = Engine(D, k_max=16, device=local)
    eng.set_centroids(cents)
    sh = ShardedIndex(eng, rank, world)
    load(lib, n_ivf, n_rec, n_comp, dev, sh.add_recent_rows_device, sh.add_rows_device)
    dele = np.arange(0, n_all, 97, dtype=np.uint32)
    sh.delete(dele)
    keep_ids = np.flatnonzero(np.arange(n_all) % 10 != 3)
    words = np.zeros((n_all + 63) // 64, dtype=np.uint64)
    np.bitwise_or.at(words, keep_ids >> 6, np.uint64(1) << (keep_ids & 63).astype(np.uint64))
    filt = torch.from_numpy(words.view(np.int64)).to(dev)
    q = torch.from_numpy(synth.queries(0, NQ, D, n_all, n_comp, SIGMA, SEED, synth.default_qnoise(D, SIGMA), 5678)).to(dev)

    def batch():
        return sh.search(q, K, NPROBE, tiers=L.TIER_BOTH, filter_bits=filt, filter_nbits=filt.numel() * 64)

    for _ in range(args.warmup):
        batch()
    torch.cuda.synchronize()
    times = []
    for _ in range(args.steps):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    g = tuple(t.cpu().numpy().copy() for t in batch())
    torch.cuda.synchronize()
    ms = float(np.median(times)) * 1e3

    # one-handle overhead: split entry + ranks-1 merge vs the merged entry, alternated (rank 0's handle)
    over = None
    if rank == 0:
        o_ids = torch.empty((NQ, K), dtype=torch.int32, device=dev)
        o_dst = torch.empty((NQ, K), dtype=torch.float32, device=dev)
        o_cnt = torch.empty((NQ,), dtype=torch.int32, device=dev)
        pack = torch.empty((tiers_pack_layout(NQ, K)[4],), dtype=torch.int32, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        fb = (filt.data_ptr(), filt.numel() * 64)

        def merged():
            eng.search_device(q.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, *fb, o_ids.data_ptr(), o_dst.data_ptr(),
                              o_cnt.data_ptr(), st)

        def split():
            eng.search_device_tiers(q.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, *fb, 0, pack.data_ptr(), st)
            eng.merge_topk_tiers_packed_device(pack.data_ptr(), 1, NQ, K, o_ids.data_ptr(), o_dst.data_ptr(),
                                               o_cnt.data_ptr(), st)
        t = {"merged": [], "split": []}
        for i in range(args.warmup + args.steps):
            for name, f in (("merged", merged), ("split", split)) if i % 2 == 0 else (("split", split), ("merged", merged)):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                if i >= args.warmup:
                    t[name].append(time.perf_counter() - t0)
        over = {k_: round(float(np.median(v)) * 1e3, 4) for k_, v in t.items()}
    dist.barrier()
    eng.close()

    # parity: one unsharded handle over every row (rank 0), exact mode, on a query subset
    parity = None
    if rank == 0:
        ref = Engine(D, k_max=16, device=local)
        ref.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
        ref.set_centroids(cents)
        load(lib, n_ivf, n_rec, n_comp, dev,
             lambda x, i: ref.flat_add_device(x.data_ptr(), i.data_ptr(), x.shape[0]),
             lambda x, i: ref.ivf_add_device(x.data_ptr(), i.data_ptr(), x.shape[0]))
        ref.set_deleted(dele, True)
        m = args.parity_queries
        r_ids = torch.empty((m, K), dtype=torch.int32, device=dev)
        r_dst = torch.empty((m, K), dtype=torch.float32, device=dev)
        r_cnt = torch.empty((m,), dtype=torch.int32, device=dev)
        ref.search_device(q[:m].data_ptr(), m, K, NPROBE, L.TIER_BOTH, filt.data_ptr(), filt.numel() * 64,
                          r_ids.data_ptr(), r_dst.data_ptr(), r_cnt.data_ptr())
        torch.cuda.synchronize()
        same = 0
        for i in range(m):
            c = int(r_cnt[i])
            same += int(c == int(g[2][i]) and np.array_equal(g[0][i, :c], r_ids[i, :c].cpu().numpy())
                        and np.array_equal(g[1][i, :c].view(np.uint32), r_dst[i, :c].cpu().numpy().view(np.uint32)))
        parity = f"{same}/{m}"
        ref.close()
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True).stdout.strip()
        line = dict(workload="shard_hybrid_cfg4_weak", gpus=world, gpu=gpu, rows_per_gpu=N_IVF + N_REC,
                    recent_rows_per_gpu=N_REC, nlist=NLIST, nprobe=NPROBE, nq=NQ, k=K, steps=args.steps,
                    ms_per_batch_median=round(ms, 4), qps=round(NQ / (ms / 1e3)), parity_vs_unsharded=parity,
                    one_handle_ms_merged_vs_split=over)
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(args.out), exist_ok=True)
            with open(args.out, "a") as fh:
                fh.write(json.dumps(line) + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
