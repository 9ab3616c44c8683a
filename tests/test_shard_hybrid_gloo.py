"""The hybrid (FVDB_TIER_BOTH) routing of the sharded index on CPU: the chunk layout, the recent-row placement
rule, the host statement of the tiered merge, and ShardedIndex's synchronous search, pipelined search,
mutations and 3x post-filter at world 2 over gloo, with a numpy stand-in for the per-GPU engine (the oracle does
the numeric work of each rank's shard).  Every merged result must equal the unsharded oracle bit for bit."""
import ctypes
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

import oracle as O  # noqa: E402
from fabstir_vectordb_b200 import _lib as L  # noqa: E402
from fabstir_vectordb_b200.shard import (merge_parts_reference, merge_tiers_reference, owner_of_list,  # noqa: E402
                                         owner_of_recent_row, pack_layout, tiers_pack_layout)

D, NLIST, N_IVF, N_REC, NQ, K, NPROBE = 8, 4, 600, 200, 12, 6, 2


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_tiers_pack_layout_and_recent_owner():
    for nq, k in ((1, 1), (7, 10), (129, 32)):
        o_i, o_d, o_c, part, chunk = tiers_pack_layout(nq, k)
        assert (o_i, o_d, o_c, part) == pack_layout(nq, k)
        assert chunk == 2 * part == 2 * (2 * nq * k + nq)
    for world in (1, 2, 3, 8):
        assert [owner_of_recent_row(i, world) for i in range(40)] == [i % world for i in range(40)]


def test_merge_tiers_reference_cross_tier_ties():
    """Two ranks, one query, k 5.  At distance 1.0: recent rows 9 (rank 0) and 5 (rank 1), IVF rows 2 (rank 1)
    and 7 (rank 0).  Recent rows first, each tier by id: 1 | 5 9 | 2 7.  The one-tier rule gives 1 2 5 7 9."""
    inf = np.float32(np.inf)
    ids = np.array([[[9, 0, 0, 0, 0]], [[1, 7, 0, 0, 0]], [[5, 0, 0, 0, 0]], [[2, 11, 0, 0, 0]]], dtype=np.uint32)
    dst = np.array([[[1.0, inf, inf, inf, inf]], [[0.5, 1.0, inf, inf, inf]], [[1.0, inf, inf, inf, inf]],
                    [[1.0, 3.0, inf, inf, inf]]], dtype=np.float32)
    cnt = np.array([[1], [2], [1], [2]], dtype=np.uint32)
    m_ids, m_dst, m_cnt = merge_tiers_reference(ids, dst, cnt, 5)
    assert m_ids[0].tolist() == [1, 5, 9, 2, 7] and m_cnt.tolist() == [5]
    assert m_dst[0].tolist() == [0.5, 1.0, 1.0, 1.0, 1.0]
    assert merge_parts_reference(ids, dst, cnt, 5)[0][0].tolist() == [1, 2, 5, 7, 9]
    # truncation at k keeps the recent rows of a tie group; counts above k are clamped
    cnt2 = np.array([[3], [2], [1], [2]], dtype=np.uint32)
    assert merge_tiers_reference(ids, dst, cnt2, 2)[0][0].tolist() == [1, 5]


def _data():
    """Integer rows: exact distance ties everywhere.  The recent tier holds copies of 100 IVF rows under
    higher ids, and 100 fresh rows."""
    rng = np.random.default_rng(21)
    x = rng.integers(0, 3, size=(N_IVF, D)).astype(np.float32)
    fx = np.concatenate([x[rng.choice(N_IVF, 100, replace=False)], rng.integers(0, 3, size=(100, D)).astype(np.float32)])
    fids = np.arange(N_IVF, N_IVF + N_REC, dtype=np.uint32)
    q = rng.integers(0, 3, size=(NQ, D)).astype(np.float32)
    cents = np.eye(NLIST, D, dtype=np.float32) * 2
    return x, fx, fids, q, cents


class _Stats:
    nlist = NLIST
    last_fallback_queries = 0


class _HybridStandIn:
    """The C-ABI calls ShardedIndex makes for a hybrid index, over host memory: this rank's IVF rows and recent
    slab, tombstones, and the oracle doing each tier's search.  Records the call order."""

    def __init__(self, cents, x, ids):
        self.cents = cents
        self.x, self.ids = x.copy(), ids.copy()
        self.fx = np.zeros((0, D), dtype=np.float32)
        self.fids = np.zeros(0, dtype=np.uint32)
        self.deleted = set()
        self.k_max = 3 * K
        self.log = []
        self._stats = _Stats()

    def _arr(self, ptr, ctype, n):
        return np.ctypeslib.as_array((ctype * n).from_address(ptr)) if n else np.zeros(0)

    def stats(self):
        return self._stats

    def set_option(self, option, value):
        self.log.append(("set_option", option, value))

    def ivf_max_sqnorm(self):
        self.log.append(("max_sqnorm",))
        return float((self.x.astype(np.float32) ** 2).sum(axis=1).max()) if self.x.shape[0] else 0.0

    def coarse_device_submit(self, d_q, nq, np_, d_out, stream=0):
        q = self._arr(d_q, ctypes.c_float, nq * D).reshape(nq, D)
        out = self._arr(d_out, ctypes.c_int64, nq * np_).reshape(nq, np_)
        ivf = O.IVF(self.cents, np.zeros((0, D), dtype=np.float32))
        for i in range(nq):
            lists, dists = ivf.coarse(q[i], np_)
            out[i] = ((dists.view(np.uint32).astype(np.uint64) << np.uint64(32)) | lists.astype(np.uint64)).view(np.int64)

    coarse_device = coarse_device_submit

    def _bits(self):
        return O.make_bitmap(N_IVF + N_REC, sorted(self.deleted)) if self.deleted else None

    def search_device_tiers_submit(self, d_q, nq, k, np_, tiers, d_f, fn, d_coarse, d_pack, stream=0):
        self.log.append(("tiers", nq))
        q = self._arr(d_q, ctypes.c_float, nq * D).reshape(nq, D).copy()
        filt = self._arr(d_f, ctypes.c_uint64, fn // 64).copy() if d_f else None
        o_i, o_d, o_c, part, chunk = tiers_pack_layout(nq, k)
        pack = self._arr(d_pack, ctypes.c_int32, chunk)
        empty = (np.full((nq, k), 0xFFFFFFFF, dtype=np.uint32), np.full((nq, k), np.inf, dtype=np.float32),
                 np.zeros(nq, dtype=np.uint32))
        recent = O.hybrid_batch_search(None, self.fx, self.fids, q, k, 0, tiers=1, deleted=self._bits(),
                                       filter_bits=filt) if (tiers & 1) and self.fids.size else empty
        ivf = O.hybrid_batch_search(O.IVF(self.cents, self.x, self.ids), None, None, q, k, np_, tiers=2,
                                    deleted=self._bits(), filter_bits=filt) if tiers & 2 else empty
        for t, (ids, dst, cnt) in enumerate((recent, ivf)):
            base = t * part
            pack[base + o_i:base + o_d] = ids.astype(np.uint32).view(np.int32).ravel()
            pack[base + o_d:base + o_c] = dst.astype(np.float32).view(np.int32).ravel()
            pack[base + o_c:base + part] = cnt.astype(np.uint32).view(np.int32)

    search_device_tiers = search_device_tiers_submit

    def search_device_wait(self, age, stream=0):
        self.log.append(("wait", age))

    def merge_topk_tiers_packed_device(self, d_pack, ranks, nq, k, o_ids, o_dist, o_cnt, stream=0):
        self.log.append(("merge_tiers", ranks))
        o_i, o_d, o_c, part, chunk = tiers_pack_layout(nq, k)
        g = self._arr(d_pack, ctypes.c_int32, ranks * chunk).reshape(2 * ranks, part)
        m = merge_tiers_reference(g[:, o_i:o_d].copy().view(np.uint32).reshape(-1, nq, k),
                                  g[:, o_d:o_c].copy().view(np.float32).reshape(-1, nq, k),
                                  g[:, o_c:].copy().view(np.uint32), k)
        self._arr(o_ids, ctypes.c_int32, nq * k)[:] = m[0].view(np.int32).ravel()
        self._arr(o_dist, ctypes.c_float, nq * k)[:] = m[1].ravel()
        self._arr(o_cnt, ctypes.c_int32, nq)[:] = m[2].view(np.int32)

    def search_device_finish(self, stream=0):
        self.log.append(("finish",))

    def flat_add_device(self, d_x, d_ids, n):
        self.fx = np.concatenate([self.fx, self._arr(d_x, ctypes.c_float, n * D).reshape(n, D).copy()])
        self.fids = np.concatenate([self.fids, self._arr(d_ids, ctypes.c_uint32, n).copy()])

    def set_deleted(self, ids, deleted=True):
        self.log.append(("set_deleted", len(ids)))
        self.deleted = self.deleted | set(ids.tolist()) if deleted else self.deleted - set(ids.tolist())

    def vacuum(self):
        gone_x = np.isin(self.ids, list(self.deleted))
        gone_f = np.isin(self.fids, list(self.deleted))
        self.x, self.ids = self.x[~gone_x], self.ids[~gone_x]
        self.fx, self.fids = self.fx[~gone_f], self.fids[~gone_f]
        self.deleted = set()
        return int(gone_x.sum() + gone_f.sum())

    def move_flat_to_ivf(self, ids):
        mv = np.isin(self.fids, ids)
        self.x = np.concatenate([self.x, self.fx[mv]])
        self.ids = np.concatenate([self.ids, self.fids[mv]])
        self.fx, self.fids = self.fx[~mv], self.fids[~mv]
        return int(mv.sum())


def _check(got, want, what):
    g_ids, g_dst, g_cnt = (t.numpy() for t in got)
    w_ids, w_dst, w_cnt = want
    assert g_cnt.view(np.uint32).tolist() == w_cnt.tolist(), what
    for i in range(len(w_cnt)):
        c = int(w_cnt[i])
        assert g_ids[i, :c].view(np.uint32).tolist() == w_ids[i, :c].tolist(), f"{what}: ids of query {i}"
        assert g_dst[i, :c].view(np.uint32).tolist() == w_dst[i, :c].view(np.uint32).tolist(), f"{what}: dist of query {i}"


def _hybrid_worker(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["FVDB_SHARE_BOUNDS"] = "1"
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fabstir_vectordb_b200.shard import ShardedIndex
        x, fx, fids, q, cents = _data()
        ids = np.arange(N_IVF, dtype=np.uint32)
        a = O.assign(x, cents)
        mine = np.array([owner_of_list(int(l), world) == rank for l in a])
        eng = _HybridStandIn(cents, x[mine], ids[mine])
        sh = ShardedIndex(eng, rank, world)
        kept = sh.add_recent_rows_device(torch.from_numpy(fx), torch.from_numpy(fids.view(np.int32)))
        assert kept == int((fids % world == rank).sum()) and set(eng.fids.tolist()) == set(fids[fids % world == rank].tolist())
        tq = torch.from_numpy(q)

        def oracle(x_, ids_, fx_, fids_, qq=q, deleted=None):
            return O.hybrid_batch_search(O.IVF(cents, x_, ids_), fx_, fids_, qq, K, NPROBE, tiers=3, deleted=deleted)

        want = oracle(x, ids, fx, fids)
        # the case holds cross-tier ties that the one-tier rule would order differently
        w_ids, w_dst, w_cnt = want
        # (recent ids are all above the IVF ids: a recent row right before an IVF row at the same distance)
        assert sum(int(((w_ids[i, :-1] >= N_IVF) & (w_ids[i, 1:] < N_IVF) & (w_dst[i, :-1] == w_dst[i, 1:])).any())
                   for i in range(NQ)) > 0
        _check(sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH), want, "synchronous")

        # pipelined: three batches, the exchange of batch i issued after batch i + 1's scan was handed over
        qs = [torch.from_numpy(np.ascontiguousarray(np.roll(q, s, axis=0))) for s in range(3)]
        eng.log.clear()
        outs = [sh.submit(qq, K, NPROBE, tiers=L.TIER_BOTH, slot=i) for i, qq in enumerate(qs)]
        sh.finish()
        for s, o in enumerate(outs):
            _check(o, oracle(x, ids, fx, fids, qq=np.roll(q, s, axis=0)), f"pipelined batch {s}")
        kinds = [e[0] for e in eng.log]
        assert kinds.count("tiers") == 3 and kinds.count("merge_tiers") == 3
        assert kinds.index("merge_tiers") > [i for i, k_ in enumerate(kinds) if k_ == "tiers"][1]

        # delete (not an IVF-tier mutation: no re-reduction of the proof floor), vacuum, migrate
        dele = np.concatenate([np.arange(0, N_IVF, 9), np.arange(N_IVF + 1, N_IVF + N_REC, 4)]).astype(np.uint32)
        eng.log.clear()
        sh.delete(dele)
        bm = O.make_bitmap(N_IVF + N_REC, dele)
        _check(sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH), oracle(x, ids, fx, fids, deleted=bm), "after delete")
        assert not any(e[0] == "max_sqnorm" for e in eng.log)
        assert sh.vacuum() == dele.size
        keep_x, keep_f = ~np.isin(ids, dele), ~np.isin(fids, dele)
        x, ids, fx, fids = x[keep_x], ids[keep_x], fx[keep_f], fids[keep_f]
        _check(sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH), oracle(x, ids, fx, fids), "after vacuum")
        # migrate every other recent row, scaled beyond every IVF row's norm first: the proof floor must follow
        # (two fresh recent rows of norm^2 648, one per rank, join the migration)
        big_ids = np.array([N_IVF + N_REC + 1, N_IVF + N_REC + 2], dtype=np.uint32)
        sh.add_recent_rows_device(torch.full((2, D), 9.0), torch.from_numpy(big_ids.view(np.int32)))
        fx = np.concatenate([fx, np.full((2, D), 9.0, dtype=np.float32)])
        fids = np.concatenate([fids, big_ids])
        mig = np.concatenate([fids[:-2:2], big_ids])
        eng.log.clear()
        _check(sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH), oracle(x, ids, fx, fids), "recent insert")
        assert not any(e[0] == "max_sqnorm" for e in eng.log), "a recent-tier insert re-reduced the proof floor"
        assert sh.migrate(mig) == mig.size
        is_mig = np.isin(fids, mig)
        x, ids = np.concatenate([x, fx[is_mig]]), np.concatenate([ids, fids[is_mig]])
        fx, fids = fx[~is_mig], fids[~is_mig]
        eng.log.clear()
        _check(sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH), oracle(x, ids, fx, fids), "after migrate")
        xmax = [e for e in eng.log if e[0] == "set_option" and e[1] == L.OPT_PROOF_XMAX]
        assert len(xmax) == 1 and np.uint32(xmax[0][2]).view(np.float32) == np.float32(9.0 * 9.0 * D)
        eng.log.clear()
        sh.search(tq, K, NPROBE, tiers=L.TIER_BOTH)
        assert not any(e[0] == "max_sqnorm" for e in eng.log), "the proof floor was re-reduced without a mutation"

        # the 3x post-filter over the sharded hybrid result
        n_all = N_IVF + N_REC + 3
        match = O.make_bitmap(n_all, np.flatnonzero(np.arange(n_all) % 3 != 0))
        got = sh.search_postfilter(tq, K, NPROBE, torch.from_numpy(match.view(np.int64)))
        ivf = O.IVF(cents, x, ids)
        for i in range(NQ):
            w_i, w_d = O.hybrid_search_postfilter(ivf, fx, fids, q[i], K, NPROBE, match, tiers=3)
            c = len(w_i)
            assert int(got[2][i]) == c
            assert got[0][i, :c].numpy().view(np.uint32).tolist() == w_i.tolist()
            assert got[1][i, :c].numpy().view(np.uint32).tolist() == w_d.view(np.uint32).tolist()
            assert (got[0][i, c:].numpy().view(np.uint32) == 0xFFFFFFFF).all()
    finally:
        dist.destroy_process_group()


def test_sharded_hybrid_routing_world2():
    """ShardedIndex with tiers = FVDB_TIER_BOTH on two gloo ranks, a stand-in engine per rank: recent rows placed by
    id % world; the synchronous and the pipelined search equal the unsharded oracle; delete / vacuum / migrate are
    broadcast and their counts all-reduced; the proof floor (FVDB_OPT_PROOF_XMAX) is max-reduced again after an
    IVF-tier mutation, and only then; the 3x post-filter equals the reference's."""
    mp.spawn(_hybrid_worker, args=(2, _free_port()), nprocs=2, join=True)
