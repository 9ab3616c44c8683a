"""Multi-GPU parity check (run under torchrun, one rank per GPU): list-sharded search + NCCL
all-gather + merge must equal the unsharded CPU oracle on EVERY rank, bit for bit.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29512 scripts/check_shard.py
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import oracle as O  # noqa: E402
from fabstir_vectordb_b200 import Engine, _lib as L, synth  # noqa: E402
from fabstir_vectordb_b200.shard import ShardedIndex  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dev = torch.device("cuda", local)
N, D, NLIST, NQ, K, NPROBE = 40_000, 384, 64, 96, 10, 8
x = synth.rows(0, N, D, 4 * NLIST, 1.0, 1234)
q = synth.queries(0, NQ, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678)
cents = x[:: N // NLIST][:NLIST].copy()
ok = True
for mode in (L.SCAN_EXACT, L.SCAN_TC):
    eng = Engine(D, k_max=16, device=local)
    eng.set_option(L.OPT_SCAN_MODE, mode)
    eng.set_centroids(cents)
    sh = ShardedIndex(eng, rank, world)
    dx = torch.from_numpy(x).to(dev)
    ids = torch.arange(N, dtype=torch.int32, device=dev)
    kept = sh.add_rows_device(dx, ids)
    dq = torch.from_numpy(q).to(dev)
    g_ids, g_dst, g_cnt = sh.search(dq, K, NPROBE, tiers=L.TIER_HISTORICAL)
    torch.cuda.synchronize()
    ivf = O.IVF(cents, x, np.arange(N, dtype=np.uint32))
    w_ids, w_dst, w_cnt = O.hybrid_batch_search(ivf, None, None, q, K, NPROBE, tiers=2)
    a = g_ids.cpu().numpy().view(np.uint32)
    same = (a == w_ids).all() and (g_dst.cpu().numpy().view(np.uint32) == w_dst.view(np.uint32)).all() \
        and (g_cnt.cpu().numpy().view(np.uint32) == w_cnt).all()
    print(f"rank {rank}/{world} mode {mode}: kept {kept} rows, global result identical to the oracle: {bool(same)}", flush=True)
    ok = ok and bool(same)
    # the pipelined entry (submit / finish): six batches in flight, each against the oracle
    qs = [synth.queries(100 * i, NQ, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678) for i in range(6)]
    dqs = [torch.from_numpy(a_).to(dev) for a_ in qs]
    outs = [sh.submit(dqs[i], K, NPROBE, tiers=L.TIER_HISTORICAL, slot=i) for i in range(6)]
    sh.finish()
    torch.cuda.synchronize()
    same_p = True
    for i in range(6):
        w = O.hybrid_batch_search(ivf, None, None, qs[i], K, NPROBE, tiers=2)
        same_p = same_p and (outs[i][0].cpu().numpy().view(np.uint32) == w[0]).all() \
            and (outs[i][1].cpu().numpy().view(np.uint32) == w[1].view(np.uint32)).all() \
            and (outs[i][2].cpu().numpy().view(np.uint32) == w[2]).all()
    print(f"rank {rank}/{world} mode {mode}: pipelined submit/finish identical to the oracle: {bool(same_p)}", flush=True)
    ok = ok and bool(same_p)
    eng.close()

# ---- size-balanced placement + shards with unequal row norms (the proof bound must use the largest
# norm of ALL shards: rows of the odd lists are 3x longer) ---------------------------------------------
from fabstir_vectordb_b200.shard import place_lists  # noqa: E402
x2 = x.copy()
a_full = O.assign(x2, cents)
x2[a_full % 2 == 1] *= np.float32(3.0)
a2 = O.assign(x2, cents)
eng = Engine(D, k_max=16, device=local)
eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
eng.set_centroids(cents)
sh = ShardedIndex(eng, rank, world)
hist = torch.zeros((NLIST,), dtype=torch.int64, device=dev)
dx2 = torch.from_numpy(x2).to(dev)
sh.list_histogram_device(dx2, hist)
assert hist.cpu().numpy().tolist() == np.bincount(a2, minlength=NLIST).tolist()
sh.set_placement(place_lists(hist.cpu().numpy(), world))
kept = sh.add_rows_device(dx2, torch.arange(N, dtype=torch.int32, device=dev))
loads = [None] * world
dist.all_gather_object(loads, int(kept))
ivf2 = O.IVF(cents, x2, np.arange(N, dtype=np.uint32))
g = sh.search(torch.from_numpy(q).to(dev), K, NPROBE, tiers=L.TIER_HISTORICAL)
torch.cuda.synchronize()
w = O.hybrid_batch_search(ivf2, None, None, q, K, NPROBE, tiers=2)
same2 = (g[0].cpu().numpy().view(np.uint32) == w[0]).all() and (g[1].cpu().numpy().view(np.uint32) == w[1].view(np.uint32)).all()
print(f"rank {rank}/{world}: balanced placement loads {loads} (sum {sum(loads)} of {N}), unequal-norm shards identical "
      f"to the oracle: {bool(same2)}", flush=True)
ok = ok and bool(same2) and sum(loads) == N and max(loads) - min(loads) <= int(hist.max())
eng.close()

# ---- a tensor-core proof that fails on ONE rank: rows dropped on the OTHER ranks by that rank's bounds lose
# their proof as well, so every rank must answer on the exact path (ShardedIndex._redo_exact) ----------------
x3 = x.copy()
rng3 = np.random.default_rng(11)
for j in range(60):
    x3[300 + j] = x3[100] if j % 3 == 0 else x3[100] + (1e-4 * rng3.standard_normal(D)).astype(np.float32)
q3 = np.concatenate([np.stack([x3[100] + (0.05 * rng3.standard_normal(D)).astype(np.float32) for _ in range(16)]), q[:48]])
eng = Engine(D, k_max=16, device=local)
eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
eng.set_centroids(cents)
sh = ShardedIndex(eng, rank, world)
sh.add_rows_device(torch.from_numpy(x3).to(dev), torch.arange(N, dtype=torch.int32, device=dev))
ivf3 = O.IVF(cents, x3, np.arange(N, dtype=np.uint32))
w3 = O.hybrid_batch_search(ivf3, None, None, q3, K, NPROBE, tiers=2)
dq3 = torch.from_numpy(q3).to(dev)
g3 = sh.search(dq3, K, NPROBE, tiers=L.TIER_HISTORICAL)
torch.cuda.synchronize()
same3 = (g3[0].cpu().numpy().view(np.uint32) == w3[0]).all() and (g3[1].cpu().numpy().view(np.uint32) == w3[1].view(np.uint32)).all()
o3 = sh.submit(dq3, K, NPROBE, tiers=L.TIER_HISTORICAL, slot=1)
o3b = sh.submit(dqs[0], K, NPROBE, tiers=L.TIER_HISTORICAL, slot=2)
sh.finish()
torch.cuda.synchronize()
same3p = (o3[0].cpu().numpy().view(np.uint32) == w3[0]).all() and (o3[1].cpu().numpy().view(np.uint32) == w3[1].view(np.uint32)).all()
print(f"rank {rank}/{world}: near-duplicate shell (proof fails somewhere): sync path identical to the oracle: {bool(same3)}, "
      f"pipelined path: {bool(same3p)}", flush=True)
ok = ok and bool(same3) and bool(same3p)
eng.close()

# ---- exact distance ties across ranks: binary rows (d 64) make every distance exact and give each query tie
# groups of dozens of rows spread over the lists of all ranks; the merge must order them by row id, as the
# unsharded search does, not by rank -------------------------------------------------------------------------------
rng4 = np.random.default_rng(77)
x4 = rng4.integers(0, 2, size=(20_000, 64)).astype(np.float32)
q4 = rng4.integers(0, 2, size=(70, 64)).astype(np.float32)
c4 = (0.5 + 0.3 * rng4.standard_normal((16, 64))).astype(np.float32)
ivf4 = O.IVF(c4, x4, np.arange(x4.shape[0], dtype=np.uint32))
w4 = O.hybrid_batch_search(ivf4, None, None, q4, K, 6, tiers=2)
rank_of_row = (ivf4.assign % world).astype(np.int64)
ties4 = sum(int(np.unique(rank_of_row[w4[0][i][w4[1][i] == v]]).size > 1)
            for i in range(q4.shape[0]) for v in np.unique(w4[1][i]))
same4 = ties4 > 0
for mode in (L.SCAN_EXACT, L.SCAN_TC):
    eng = Engine(64, k_max=16, device=local)
    eng.set_option(L.OPT_SCAN_MODE, mode)
    eng.set_centroids(c4)
    sh = ShardedIndex(eng, rank, world)
    sh.add_rows_device(torch.from_numpy(x4).to(dev), torch.arange(x4.shape[0], dtype=torch.int32, device=dev))
    g4 = sh.search(torch.from_numpy(q4).to(dev), K, 6, tiers=L.TIER_HISTORICAL)
    torch.cuda.synchronize()
    same4 = same4 and (g4[0].cpu().numpy().view(np.uint32) == w4[0]).all() \
        and (g4[1].cpu().numpy().view(np.uint32) == w4[1].view(np.uint32)).all() \
        and (g4[2].cpu().numpy().view(np.uint32) == w4[2]).all()
    eng.close()
print(f"rank {rank}/{world}: lattice rows with {ties4} cross-rank tie groups in the top-{K}: exact and tc paths identical "
      f"to the oracle: {bool(same4)}", flush=True)
ok = ok and bool(same4)

# ---- hybrid search (FVDB_TIER_BOTH): the lattice rows above as the IVF tier; a recent tier in slabs (id % world)
# holding copies of IVF rows under HIGHER ids (cross-tier ties across ranks), fresh rows, and 200 rows three times
# longer than any IVF row.  Delete, vacuum, then a migration that moves the long rows into the IVF arenas: the
# tensor-core proof's norm floor (FVDB_OPT_PROOF_XMAX, shared bounds) must follow them --------------------------------
n4 = x4.shape[0]
rng5 = np.random.default_rng(5)
big5 = 3 * rng5.integers(0, 2, size=(200, 64)).astype(np.float32)
fx5 = np.concatenate([x4[rng5.choice(n4, 2000, replace=False)], rng5.integers(0, 2, size=(2000, 64)).astype(np.float32), big5])
fid5 = np.arange(n4, n4 + fx5.shape[0], dtype=np.uint32)
q5 = np.concatenate([q4, big5[:8]])
dq5s = [torch.from_numpy(np.ascontiguousarray(np.roll(q5, s, axis=0))).to(dev) for s in range(3)]


def _same(g, w):
    return bool((g[0].cpu().numpy().view(np.uint32) == w[0]).all() and (g[1].cpu().numpy().view(np.uint32) == w[1].view(np.uint32)).all()
                and (g[2].cpu().numpy().view(np.uint32) == w[2]).all())


for mode in (L.SCAN_EXACT, L.SCAN_TC):
    eng = Engine(64, k_max=16, device=local)
    eng.set_option(L.OPT_SCAN_MODE, mode)
    eng.set_centroids(c4)
    sh = ShardedIndex(eng, rank, world)
    sh.add_rows_device(torch.from_numpy(x4).to(dev), torch.arange(n4, dtype=torch.int32, device=dev))
    kept5 = sh.add_recent_rows_device(torch.from_numpy(fx5).to(dev), torch.from_numpy(fid5.view(np.int32)).to(dev))
    s_x, s_ids, s_fx, s_fid = x4, np.arange(n4, dtype=np.uint32), fx5, fid5
    bm5 = None
    line = []
    for step in ("load", "delete", "vacuum", "migrate"):
        if step == "delete":
            dele5 = np.concatenate([np.arange(1, n4, 7), fid5[2::5]]).astype(np.uint32)
            sh.delete(dele5)
            bm5 = O.make_bitmap(n4 + fx5.shape[0], dele5)
        elif step == "vacuum":
            removed = sh.vacuum()
            ok = ok and removed == dele5.size
            kx, kf = ~np.isin(s_ids, dele5), ~np.isin(s_fid, dele5)
            s_x, s_ids, s_fx, s_fid, bm5 = s_x[kx], s_ids[kx], s_fx[kf], s_fid[kf], None
        elif step == "migrate":
            mig = np.concatenate([s_fid[s_fid < n4 + 4000][::2], s_fid[s_fid >= n4 + 4000]])
            moved = sh.migrate(mig)
            ok = ok and moved == mig.size
            m = np.isin(s_fid, mig)
            s_x, s_ids = np.concatenate([s_x, s_fx[m]]), np.concatenate([s_ids, s_fid[m]])
            s_fx, s_fid = s_fx[~m], s_fid[~m]
        ivf5 = O.IVF(c4, s_x, s_ids)
        ws = [O.hybrid_batch_search(ivf5, s_fx, s_fid, np.roll(q5, s, axis=0), K, 6, tiers=3, deleted=bm5) for s in range(3)]
        same_s = _same(sh.search(dq5s[0], K, 6, tiers=L.TIER_BOTH), ws[0])
        torch.cuda.synchronize()
        outs5 = [sh.submit(dq5s[s], K, 6, tiers=L.TIER_BOTH, slot=s) for s in range(3)]
        sh.finish()
        torch.cuda.synchronize()
        same_p = all(_same(outs5[s], ws[s]) for s in range(3))
        if step == "load":
            # tie groups of the oracle's top-k holding a recent row and an IVF row that sit on different ranks
            w_ids, w_dst, w_cnt = ws[0]
            r_ivf = (ivf5.assign % world).astype(np.int64)
            pos = np.full(n4 + fx5.shape[0], -1, dtype=np.int64)
            pos[s_ids] = np.arange(s_ids.size)
            ties5 = 0
            for i in range(q5.shape[0]):
                for v in np.unique(w_dst[i, :w_cnt[i]]):
                    grp = w_ids[i, :w_cnt[i]][w_dst[i, :w_cnt[i]] == v]
                    rec, iv = grp[grp >= n4], grp[grp < n4]
                    rk = set((rec % world).tolist()) | set(r_ivf[pos[iv]].tolist())
                    ties5 += int(rec.size > 0 and iv.size > 0 and len(rk) > 1)
            line.append(f"{ties5} cross-tier cross-rank tie groups")
            ok = ok and (ties5 > 0 or world == 1)
        line.append(f"{step}: sync {same_s} pipelined {same_p}")
        ok = ok and same_s and same_p
    print(f"rank {rank}/{world} mode {mode}: hybrid (TIER_BOTH), {kept5} recent rows on this rank, "
          + ", ".join(line) + f" — identical to the oracle: {all('False' not in s for s in line)}", flush=True)
    eng.close()

# ---- sharded k-means (points split over the ranks, one all-reduce per iteration) against the single-GPU
# order-faithful training from the same initial centroids ------------------------------------------------
eng = Engine(D, k_max=16, device=local)
sh = ShardedIndex(eng, rank, world)
per = (N + world - 1) // world
mine = torch.from_numpy(x[rank * per:(rank + 1) * per]).to(dev)
res = sh.train(mine, NLIST, 6, cents)
c_sh = eng.get_centroids()
ref = Engine(D, k_max=16, device=local)
r1 = ref.train(x, NLIST, 6, init_centroids=cents)
c_1 = ref.get_centroids()
err = float(np.abs(c_sh - c_1).max())
sample = x[::37]
same_assign = float((O.assign(sample, c_sh) == O.assign(sample, c_1)).mean())
print(f"rank {rank}/{world}: sharded k-means {res} vs single GPU {r1}: max |dc| {err:.2e}, identical assignments on "
      f"{sample.shape[0]} sample rows: {same_assign:.4f}", flush=True)
ok = ok and err < 1e-4 and same_assign >= 0.999 and res["iterations"] == r1["iterations"]
eng.close(); ref.close()
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
