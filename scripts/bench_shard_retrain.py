"""The sharded retrain (ShardedIndex.optimize_clusters) on an IVF tier that grew by migration.  Run under torchrun,
one rank per GPU (one GPU exercises everything but the cross-GPU exchange):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29517 \\
        scripts/bench_shard_retrain.py [--steps 20] [--warmup 5] [--iters 10] [--out profiles/shard_retrain.jsonl]

Per GPU: 500 K rows loaded size-balanced (place_lists over centroids taken from them), then 500 K recent-tier rows
from a second mixture, migrated into the IVF tier (each stays on the rank that held it, in whatever list is
nearest), so the lists are fragmented over the ranks and grouped by centroids that never saw half the rows.
D 384, nlist 1024, nprobe 32, 1024-query batches (half near each mixture), k 10, IVF tier only.

Rank 0 appends one JSON line with the card name and power limit read in the same run and, before and after
optimize_clusters: the rows each rank scans per batch (max / mean over ranks), the median batch time and QPS, and
recall@10 against an exact scan of every row; and the retrain's own figures: time per Lloyd iteration, reassign
time, placement time, exchange bytes and time (max over ranks)."""
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
from fabstir_vectordb_b200.shard import ShardedIndex, place_lists  # noqa: E402

D, NLIST, NPROBE, NQ, K = 384, 1024, 32, 1024, 10
N_BASE, N_MIG = 500_000, 500_000                     # per GPU
SIGMA, SEED_BASE, SEED_MIG, CH = 1.0, 1234, 4321, 1 << 17


def gen(lib, buf, r0, n, seed):
    assert lib.fvdb_synth_rows_device(buf.data_ptr(), r0, n, D, 4 * NLIST, SIGMA, seed,
                                      torch.cuda.current_stream().cuda_stream) == 0


def chunks(lib, dev, n_base, n_mig):
    """Every row in chunks: (rows, ids); base rows [0, n_base), migrated rows [n_base, n_base + n_mig) from the
    second mixture."""
    buf = torch.empty((CH, D), dtype=torch.float32, device=dev)
    for lo, hi, seed in ((0, n_base, SEED_BASE), (n_base, n_base + n_mig, SEED_MIG)):
        for r0 in range(lo, hi, CH):
            n = min(CH, hi - r0)
            gen(lib, buf, r0 - lo, n, seed)
            torch.cuda.synchronize()          # the engine reads the rows on its own stream
            yield buf[:n], torch.arange(r0, r0 + n, dtype=torch.int32, device=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shard_retrain.jsonl"))
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    lib = L.load()
    n_base, n_mig = N_BASE * world, N_MIG * world

    cbuf = torch.empty((NLIST * 64, D), dtype=torch.float32, device=dev)
    gen(lib, cbuf, 0, cbuf.shape[0], SEED_BASE)
    cents = cbuf[::64].cpu().numpy().copy()
    del cbuf
    eng = Engine(D, k_max=16, device=local)
    eng.set_centroids(cents)
    sh = ShardedIndex(eng, rank, world)
    hist = torch.zeros((NLIST,), dtype=torch.int64, device=dev)
    for x, _ in chunks(lib, dev, n_base, 0):
        sh.list_histogram_device(x, hist)
    sh.set_placement(place_lists(hist.cpu().numpy(), world))
    for x, ids in chunks(lib, dev, n_base, n_mig):
        if int(ids[0]) < n_base:
            sh.add_rows_device(x, ids)
        else:
            sh.add_recent_rows_device(x, ids)
    torch.cuda.synchronize()
    assert sh.migrate(np.arange(n_base, n_base + n_mig, dtype=np.uint32)) == n_mig

    half = NQ // 2
    q = torch.from_numpy(np.concatenate([
        synth.queries(0, half, D, n_base, 4 * NLIST, SIGMA, SEED_BASE, synth.default_qnoise(D, SIGMA), 5678),
        synth.queries(0, NQ - half, D, n_mig, 4 * NLIST, SIGMA, SEED_MIG, synth.default_qnoise(D, SIGMA), 8765)])).to(dev)

    # ground truth on rank 0: an exact scan of every row
    truth = None
    if rank == 0:
        ref = Engine(D, k_max=16, device=local)
        ref.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
        for x, ids in chunks(lib, dev, n_base, n_mig):
            ref.flat_add_device(x.data_ptr(), ids.data_ptr(), x.shape[0])
        t_ids = torch.empty((NQ, K), dtype=torch.int32, device=dev)
        t_dst = torch.empty((NQ, K), dtype=torch.float32, device=dev)
        t_cnt = torch.empty((NQ,), dtype=torch.int32, device=dev)
        ref.search_device(q.data_ptr(), NQ, K, 0, L.TIER_RECENT, 0, 0, t_ids.data_ptr(), t_dst.data_ptr(),
                          t_cnt.data_ptr())
        torch.cuda.synchronize()
        truth = t_ids.cpu().numpy()
        ref.close()

    def measure():
        for _ in range(args.warmup):
            sh.search(q, K, NPROBE)
        torch.cuda.synchronize()
        times = []
        for _ in range(args.steps):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sh.search(q, K, NPROBE)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        ids, _, cnt = (t.cpu().numpy() for t in sh.search(q, K, NPROBE))
        torch.cuda.synchronize()
        scanned = torch.tensor([float(eng.stats().last_scanned_rows)], device=dev)
        per_rank = [torch.zeros_like(scanned) for _ in range(world)]
        dist.all_gather(per_rank, scanned)
        per_rank = [int(s.item()) for s in per_rank]
        ms = float(np.median(times)) * 1e3
        held = torch.tensor([float(eng.stats().ivf_rows)], device=dev)
        held_all = [torch.zeros_like(held) for _ in range(world)]
        dist.all_gather(held_all, held)
        out = dict(scanned_rows_per_rank=per_rank, scanned_max_over_mean=round(max(per_rank) / max(1e-9, np.mean(per_rank)), 4),
                   ivf_rows_per_rank=[int(h.item()) for h in held_all], ms_per_batch_median=round(ms, 4),
                   qps=round(NQ / (ms / 1e3)))
        if truth is not None:
            hits = sum(len(set(ids[i, :cnt[i]].tolist()) & set(truth[i].tolist())) for i in range(NQ))
            out["recall_at_10"] = round(hits / (NQ * K), 4)
        return out

    before = measure()
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sh.optimize_clusters(max_iterations=args.iters)
    torch.cuda.synchronize()
    total_s = time.perf_counter() - t0
    secs = torch.tensor([res["seconds"].get(k_, 0.0) for k_ in ("lloyd", "reassign", "placement", "exchange")],
                        dtype=torch.float64, device=dev)
    dist.all_reduce(secs, op=dist.ReduceOp.MAX)
    after = measure()

    if rank == 0:
        s = secs.cpu().numpy()
        gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True).stdout.strip()
        line = dict(workload="shard_retrain_after_migration", gpus=world, gpu=gpu, base_rows_per_gpu=N_BASE,
                    migrated_rows_per_gpu=N_MIG, dim=D, nlist=NLIST, nprobe=NPROBE, nq=NQ, k=K, steps=args.steps,
                    before=before, after=after,
                    retrain=dict(iterations=res["iterations"], converged=res["converged"],
                                 rows_reassigned=res["rows_reassigned"], rows_moved=res["rows_moved"],
                                 lloyd_ms_per_iteration=round(float(s[0]) * 1e3 / max(1, res["iterations"]), 3),
                                 reassign_ms=round(float(s[1]) * 1e3, 3), placement_ms=round(float(s[2]) * 1e3, 3),
                                 exchange_ms=round(float(s[3]) * 1e3, 3),
                                 exchange_bytes=res["rows_moved"] * (4 * D + 4),
                                 total_ms=round(total_s * 1e3, 3)))
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as fh:
                fh.write(json.dumps(line) + "\n")
    dist.barrier()
    eng.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
