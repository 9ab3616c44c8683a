"""World-size-2 gloo test of the multi-GPU exchange step (SURVEY §8e) on CPU: list l lives on rank
l % world, every rank searches only the lists it owns (here with the CPU oracle standing in for
the per-GPU engine), one all-gather of the per-rank [nq x k] results, then the k-way merge of
src/hybrid/core.rs:482-483.  The merged result must equal the unsharded search bit for bit."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

import oracle as O  # noqa: E402
from fabstir_vectordb_b200 import synth  # noqa: E402
from fabstir_vectordb_b200.shard import gather_layout, merge_parts_reference, owner_of_list, pack_layout  # noqa: E402

N, D, NLIST, NQ, K, NPROBE = 4000, 32, 16, 24, 10, 6


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _case():
    x = synth.rows(0, N, D, 64, 0.7, 1234)
    q = synth.queries(0, NQ, D, N, 64, 0.7, 1234, synth.default_qnoise(D, 0.7), 5678)
    cents = x[:: N // NLIST][:NLIST].copy()
    return x, q, cents


def _lattice_case():
    """Exact distance ties across ranks: integer rows, d 8, four lists on two ranks (l % 2).  Row 0 sits in
    list 1 (rank 1), row 1 in list 0 (rank 0), both at distance 1.0 from q = 0: the unsharded search returns
    row 0 first, a merge that breaks ties by rank returns row 1."""
    d, nlist = 8, 4
    cents = np.zeros((nlist, d), dtype=np.float32)
    cents[np.arange(nlist), np.arange(nlist)] = 10
    x = np.zeros((6, d), dtype=np.float32)
    x[0, 1] = 1; x[1, 0] = 1; x[2, 2] = 3; x[3, 3] = 3; x[4, 0] = 5; x[5, 1] = 5
    q = np.zeros((2, d), dtype=np.float32)
    q[1, :2] = 0.5                    # rows 0 and 1 tie again, at sqrt(0.5)
    return x, q, cents


CASES = {"synth": (_case, K, NPROBE), "lattice": (_lattice_case, 4, 4)}


def _worker(rank, world, port, out_dir, case="synth"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        make, K, NPROBE = CASES[case]
        x, q, cents = make()
        N, NQ = x.shape[0], q.shape[0]
        full = O.IVF(cents, x, np.arange(N, dtype=np.uint32))
        # this rank's shard: rows of the lists it owns, same centroids (replicated)
        mine = np.array([owner_of_list(int(l), world) == rank for l in full.assign])
        shard = O.IVF(cents, x[mine], np.arange(N, dtype=np.uint32)[mine], assign_=full.assign[mine])
        ids, dst, cnt = O.hybrid_batch_search(shard, None, None, q, K, NPROBE, tiers=2)
        # the product's exchange step: ONE all-gather of the packed chunk [ids | dist | count]
        o_i, o_d, o_c, chunk = pack_layout(NQ, K)
        pack = np.empty(chunk, dtype=np.int32)
        pack[o_i:o_i + NQ * K] = ids.astype(np.uint32).view(np.int32).ravel()
        pack[o_d:o_d + NQ * K] = dst.astype(np.float32).view(np.int32).ravel()
        pack[o_c:o_c + NQ] = cnt.astype(np.uint32).view(np.int32)
        g_pack = torch.empty((world, chunk), dtype=torch.int32)
        dist.all_gather_into_tensor(g_pack.view(-1), torch.from_numpy(pack))
        g = g_pack.numpy()
        (gs, cs) = gather_layout(NQ, K, world)
        g_ids = g[:, o_i:o_i + NQ * K].copy().view(np.uint32).reshape(gs)
        g_dst = g[:, o_d:o_d + NQ * K].copy().view(np.float32).reshape(gs)
        g_cnt = g[:, o_c:o_c + NQ].copy().view(np.uint32).reshape(cs)
        m_ids, m_dst, m_cnt = merge_parts_reference(g_ids, g_dst, g_cnt, K)
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), ids=m_ids, dst=m_dst, cnt=m_cnt)
    finally:
        dist.destroy_process_group()


def _check_sharded_search(tmp_path, case):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), case), nprocs=world, join=True)
    make, K, NPROBE = CASES[case]
    x, q, cents = make()
    full = O.IVF(cents, x, np.arange(x.shape[0], dtype=np.uint32))
    w_ids, w_dst, w_cnt = O.hybrid_batch_search(full, None, None, q, K, NPROBE, tiers=2)
    for r in range(world):
        got = np.load(tmp_path / f"rank{r}.npz")
        assert got["cnt"].tolist() == w_cnt.tolist()
        for i in range(q.shape[0]):
            c = int(w_cnt[i])
            assert got["ids"][i, :c].tolist() == w_ids[i, :c].tolist()
            assert got["dst"][i, :c].view(np.uint32).tolist() == w_dst[i, :c].view(np.uint32).tolist()
    return full, w_ids


def test_list_sharded_search_world2(tmp_path):
    _check_sharded_search(tmp_path, "synth")


def test_list_sharded_search_cross_rank_ties_world2(tmp_path):
    """Two rows at exactly the same distance in lists of different ranks, the higher id on the lower rank:
    the merge must order them by row id, as the unsharded search does, not by rank."""
    full, w_ids = _check_sharded_search(tmp_path, "lattice")
    assert full.assign[:2].tolist() == [1, 0]             # row 0 on rank 1, row 1 on rank 0
    assert w_ids[0].tolist() == [0, 1, 2, 3] and w_ids[1, :2].tolist() == [0, 1]


def test_owner_rule_partitions_lists():
    for world in (1, 2, 4, 8):
        owners = [owner_of_list(l, world) for l in range(64)]
        assert set(owners) == set(range(world))
        assert all(o == l % world for l, o in enumerate(owners))


def test_place_lists_balances_rows():
    """Greedy size-balanced placement (SURVEY §8e): every list gets exactly one owner, the heaviest and the
    lightest rank differ by at most the largest list, and the table is a pure function of the histogram."""
    from fabstir_vectordb_b200.shard import place_lists
    rng = np.random.default_rng(5)
    sizes = (rng.pareto(1.5, 4096) * 300).astype(np.int64) + 1          # a few hub lists, many small ones
    for world in (1, 2, 4, 8):
        owner = place_lists(sizes, world)
        assert owner.shape == sizes.shape and owner.max() == world - 1
        load = np.bincount(owner, weights=sizes, minlength=world)
        assert load.sum() == sizes.sum()
        assert load.max() - load.min() <= sizes.max()
        if world > 1:
            mod_load = np.bincount(np.arange(sizes.size) % world, weights=sizes, minlength=world)
            assert load.max() <= mod_load.max()                               # never worse than l % world
        assert np.array_equal(owner, place_lists(sizes.copy(), world))
    # ties go to the lower rank, equal sizes are placed in list order
    assert place_lists([5, 5, 5, 5], 2).tolist() == [0, 1, 0, 1]


def _kmeans_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fabstir_vectordb_b200.shard import kmeans_allreduce_step
        x, _, cents = _case()
        per = (N + world - 1) // world
        mine = x[rank * per:(rank + 1) * per]
        # this rank's share of one Lloyd iteration: assignment (oracle standing in for the per-GPU engine),
        # per-cluster sums / counts / squared error of ITS points
        a = O.assign(mine, cents)
        sums = np.zeros((NLIST, D), dtype=np.float32)
        np.add.at(sums, a, mine)
        counts = np.bincount(a, minlength=NLIST).astype(np.int32)
        d = O.l2_many(mine[0], cents[a[:1]])  # (shape check of the helper)
        assert d.shape == (1,)
        sq = float(sum(O.l2(mine[i], cents[a[i]]) ** 2 for i in range(mine.shape[0])))
        t_sums, t_counts = torch.from_numpy(sums), torch.from_numpy(counts)
        t_sq, t_ch = torch.tensor([sq], dtype=torch.float64), torch.tensor([1 if rank == 0 else 0], dtype=torch.int32)
        tot, changed, total = kmeans_allreduce_step(t_sums, t_counts, t_sq, t_ch)
        means = cents.copy()
        nz = t_counts.numpy() > 0
        means[nz] = t_sums.numpy()[nz] / t_counts.numpy()[nz, None].astype(np.float32)
        np.savez(os.path.join(out_dir, f"km{rank}.npz"), means=means, counts=t_counts.numpy(), tot=tot,
                 changed=changed, total=total)
    finally:
        dist.destroy_process_group()


def test_sharded_kmeans_exchange_step_world2(tmp_path):
    """Points sharded over two ranks, one all-reduce of sums / counts / error (kmeans_allreduce_step): both
    ranks end up with the same means, equal to the unsharded update_centroids (src/ivf/core.rs:388-417) up
    to the f32 summation order, with exact counts and the unsharded error."""
    world = 2
    mp.spawn(_kmeans_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    x, _, cents = _case()
    a = O.assign(x, cents)
    want = O.update_centroids(x, a, cents)
    r0, r1 = np.load(tmp_path / "km0.npz"), np.load(tmp_path / "km1.npz")
    assert np.array_equal(r0["means"].view(np.uint32), r1["means"].view(np.uint32))
    assert r0["counts"].tolist() == np.bincount(a, minlength=NLIST).tolist()
    assert int(r0["total"]) == N and int(r0["changed"]) == 1
    np.testing.assert_allclose(r0["means"], want, rtol=2e-5, atol=2e-6)
    assert abs(float(r0["tot"]) / N - O.compute_error(x, cents, a)) < 1e-4


# ---- the pipelined driver (ShardedIndex.submit / finish) over CPU tensors with a stand-in engine -----------------
class _Stats:
    nlist = NLIST
    last_fallback_queries = 0


class _StandInEngine:
    """Implements the C-ABI calls ShardedIndex.submit / finish make, over host memory, with the oracle doing the
    numeric work of this rank's shard.  Records the call order; can report a tensor-core proof failure once."""

    def __init__(self, shard_ivf, report_fallback_in_finish=0):
        import ctypes
        self.C = ctypes
        self.ivf = shard_ivf
        self.log = []
        self.mode = 1
        self._stats = _Stats()
        self._inject = report_fallback_in_finish
        self.finishes = 0

    def _f32(self, ptr, n):
        return np.ctypeslib.as_array((self.C.c_float * n).from_address(ptr))

    def _i32(self, ptr, n):
        return np.ctypeslib.as_array((self.C.c_int32 * n).from_address(ptr))

    def _i64(self, ptr, n):
        return np.ctypeslib.as_array((self.C.c_int64 * n).from_address(ptr))

    def stats(self):
        return self._stats

    def set_option(self, option, value):
        self.log.append(("set_option", option, value))
        self.mode = value

    def coarse_device_submit(self, d_q, nq, np_, d_out, stream=0):
        self.log.append(("coarse", nq))
        q = self._f32(d_q, nq * D).reshape(nq, D)
        out = self._i64(d_out, nq * np_).reshape(nq, np_)
        for i in range(nq):
            lists, dists = self.ivf.coarse(q[i], np_)
            out[i] = ((dists.view(np.uint32).astype(np.uint64) << np.uint64(32)) | lists.astype(np.uint64)).view(np.int64)

    coarse_device = coarse_device_submit

    def search_device_coarse_submit(self, d_q, nq, k, np_, tiers, d_f, fn, d_coarse, d_ids, d_dist, d_cnt, stream=0):
        self.log.append(("scan", nq, "exact" if self.mode == 0 else "tc"))
        q = self._f32(d_q, nq * D).reshape(nq, D).copy()
        ids, dst, cnt = O.hybrid_batch_search(self.ivf, None, None, q, k, np_, tiers=2)
        self._i32(d_ids, nq * k)[:] = ids.view(np.int32).ravel()
        self._f32(d_dist, nq * k)[:] = dst.ravel()
        self._i32(d_cnt, nq)[:] = cnt.view(np.int32)

    search_device_coarse = search_device_coarse_submit

    def search_device_wait(self, age, stream=0):
        self.log.append(("wait", age))

    def merge_topk_packed_device(self, d_pack, parts, nq, k, o_ids, o_dist, o_cnt, stream=0):
        self.log.append(("merge", parts))
        o_i, o_d, o_c, chunk = pack_layout(nq, k)
        g = self._i32(d_pack, parts * chunk).reshape(parts, chunk)
        ids = g[:, o_i:o_i + nq * k].copy().view(np.uint32).reshape(parts, nq, k)
        dst = g[:, o_d:o_d + nq * k].copy().view(np.float32).reshape(parts, nq, k)
        cnt = g[:, o_c:o_c + nq].copy().view(np.uint32).reshape(parts, nq)
        m_ids, m_dst, m_cnt = merge_parts_reference(ids, dst, cnt, k)
        self._i32(o_ids, nq * k)[:] = m_ids.view(np.int32).ravel()
        self._f32(o_dist, nq * k)[:] = m_dst.ravel()
        self._i32(o_cnt, nq)[:] = m_cnt.view(np.int32)

    def search_device_finish(self, stream=0):
        self.log.append(("finish",))
        self.finishes += 1
        self._stats.last_fallback_queries = self._inject if self.finishes == 1 else 0


def _pipeline_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["FVDB_SHARE_BOUNDS"] = "1"
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fabstir_vectordb_b200.shard import ShardedIndex
        x, q, cents = _case()
        full = O.IVF(cents, x, np.arange(N, dtype=np.uint32))
        mine = np.array([owner_of_list(int(l), world) == rank for l in full.assign])
        shard = O.IVF(cents, x[mine], np.arange(N, dtype=np.uint32)[mine], assign_=full.assign[mine])
        # rank 1 reports a tensor-core proof failure in the FIRST group: both ranks must redo it on the exact path
        eng = _StandInEngine(shard, report_fallback_in_finish=3 if rank == 1 else 0)
        sh = ShardedIndex(eng, rank, world)
        qs = [torch.from_numpy(np.ascontiguousarray(np.roll(q, s, axis=0))) for s in range(5)]
        res = []
        for group in (qs[:3], qs[3:]):
            outs = [sh.submit(qq, K, NPROBE, slot=i) for i, qq in enumerate(group)]
            sh.finish()
            res += [tuple(t.numpy().copy() for t in o) for o in outs]
        np.savez(os.path.join(out_dir, f"pipe{rank}.npz"), **{f"ids{i}": r[0] for i, r in enumerate(res)},
                 **{f"dst{i}": r[1] for i, r in enumerate(res)}, **{f"cnt{i}": r[2] for i, r in enumerate(res)})
        with open(os.path.join(out_dir, f"pipe{rank}.log"), "w") as fh:
            fh.write(repr(eng.log))
    finally:
        dist.destroy_process_group()


def test_pipelined_sharded_search_world2(tmp_path):
    """ShardedIndex.submit / finish on two gloo ranks with a stand-in engine: (i) every batch equals the unsharded
    oracle on both ranks; (ii) the result exchange of batch i is issued after batch i + 1's scan was handed to the
    engine (the two-deep pipeline), joined with fvdb_search_device_wait; (iii) a proof failure reported by ONE
    rank sends the whole group to the exact path on BOTH ranks, and later groups stay on the fast path."""
    world = 2
    mp.spawn(_pipeline_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    x, q, cents = _case()
    full = O.IVF(cents, x, np.arange(N, dtype=np.uint32))
    for r in range(world):
        got = np.load(tmp_path / f"pipe{r}.npz")
        for s in range(5):
            w_ids, w_dst, w_cnt = O.hybrid_batch_search(full, None, None, np.roll(q, s, axis=0), K, NPROBE, tiers=2)
            assert got[f"cnt{s}"].view(np.uint32).tolist() == w_cnt.tolist()
            assert np.array_equal(got[f"ids{s}"].view(np.uint32), w_ids)
            assert np.array_equal(got[f"dst{s}"].view(np.uint32), w_dst.view(np.uint32))
        log = eval(open(tmp_path / f"pipe{r}.log").read())
        kinds = [e[0] for e in log]
        first_finish = kinds.index("finish")
        head = log[:first_finish]
        # group 1, fast path: scan(0), scan(1), [wait age 1 = batch 0, merge], scan(2), [wait 1 = batch 1, merge]; then batch 2 at finish (age 0)
        scans = [i for i, e in enumerate(head) if e[0] == "scan"]
        waits = [i for i, e in enumerate(head) if e[0] == "wait"]
        assert len(scans) == 3 and [head[i][1] for i in waits] == [1, 1, 0]
        assert waits[0] > scans[1] and waits[1] > scans[2]          # the exchange of batch i follows the scan of batch i + 1
        # the redo: exact mode switched on, three scans on the exact path, mode restored — on BOTH ranks
        after = log[first_finish + 1:]
        assert ("set_option", 1, 0) in after and ("set_option", 1, 1) in after
        a0, a1 = after.index(("set_option", 1, 0)), after.index(("set_option", 1, 1))
        assert [e[2] for e in after[a0:a1] if e[0] == "scan"] == ["exact"] * 3
        # group 2: no failure reported -> no redo
        assert [e[2] for e in after[a1:] if e[0] == "scan"] == ["tc", "tc"]
