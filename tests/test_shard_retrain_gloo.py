"""ShardedIndex.retrain / optimize_clusters / add_clusters on CPU: two gloo ranks drive the driver over a numpy
stand-in for the per-GPU engine (the oracle assigns rows to centroids).  The index is built so that lists are
fragmented over both ranks, as migration leaves them.  Checked: both ranks train the same centroids and compute
the same placement, the all-to-all layout delivers every row exactly once to the rank that owns its new list, a
failed exchange puts the taken rows back, and the cached nlist follows the new table."""
import ctypes
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

import oracle as O  # noqa: E402
from fabstir_vectordb_b200.shard import owner_of_list, place_lists  # noqa: E402

D, NLIST, N, ITERS = 8, 6, 900, 4


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _arr(ptr, ctype, n):
    return np.ctypeslib.as_array((ctype * n).from_address(ptr)) if n else np.zeros(0)


class _Stats:
    def __init__(self, nlist):
        self.nlist = nlist


class _ArenaStandIn:
    """The C-ABI calls of a retrain over host memory: an arena of rows grouped by list (stable), a centroid
    table, the sharded k-means blocks and the take / add entries, with the oracle's assignment."""

    def __init__(self, cents):
        self.dim, self.device = D, 0
        self.cents = np.ascontiguousarray(cents, dtype=np.float32)
        self.x = np.zeros((0, D), dtype=np.float32)
        self.ids = np.zeros(0, dtype=np.uint32)
        self.lists = np.zeros(0, dtype=np.uint32)
        self.closed = False

    def stats(self):
        return _Stats(self.cents.shape[0])

    def close(self):
        self.closed = True

    def _append(self, x, ids):
        lists = O.assign(x, self.cents) if len(x) else np.zeros(0, dtype=np.uint32)
        self.x = np.concatenate([self.x, x])
        self.ids = np.concatenate([self.ids, ids])
        self.lists = np.concatenate([self.lists, lists])
        order = np.argsort(self.lists, kind="stable")
        self.x, self.ids, self.lists = (np.ascontiguousarray(a[order]) for a in (self.x, self.ids, self.lists))

    # centroids and the k-means blocks (the scratch handle)
    def set_centroids(self, c):
        self.cents = np.ascontiguousarray(c, dtype=np.float32).reshape(-1, D)
        self.x, self.ids, self.lists = self.x[:0], self.ids[:0], self.lists[:0]

    def get_centroids(self):
        return self.cents.copy()

    def kmeans_accumulate_device(self, d_data, n, d_sums, d_counts, d_sqerr, d_assign, d_changed, stream=0):
        nl = self.cents.shape[0]
        x = _arr(d_data, ctypes.c_float, n * D).reshape(n, D)
        a = O.assign(x, self.cents)
        prev = _arr(d_assign, ctypes.c_uint32, n)
        if (prev != a).any():
            _arr(d_changed, ctypes.c_uint32, 1)[0] = 1
        prev[:] = a
        sums = np.zeros((nl, D), dtype=np.float64)
        np.add.at(sums, a, x.astype(np.float64))
        _arr(d_sums, ctypes.c_float, nl * D)[:] += sums.astype(np.float32).ravel()
        _arr(d_counts, ctypes.c_uint32, nl)[:] += np.bincount(a, minlength=nl).astype(np.uint32)
        d = ((x.astype(np.float64) - self.cents[a]) ** 2).sum()
        _arr(d_sqerr, ctypes.c_double, 1)[0] += d

    def kmeans_apply_device(self, d_sums, d_counts, stream=0):
        nl = self.cents.shape[0]
        s = _arr(d_sums, ctypes.c_float, nl * D).reshape(nl, D)
        c = _arr(d_counts, ctypes.c_uint32, nl)
        self.cents = np.where(c[:, None] > 0, s / np.maximum(c, 1).astype(np.float32)[:, None], self.cents).astype(np.float32)

    # the retrain entries
    def ivf_arena_device(self):
        return self.x.ctypes.data, self.ids.ctypes.data, self.ids.shape[0]

    def ivf_reassign(self, c):
        x, ids = self.x, self.ids
        self.set_centroids(c)
        self._append(x, ids)

    def dump_lists(self):
        return self.ids.copy(), self.lists.copy()

    def ivf_take_unowned_device(self, d_owner, my_rank, world, d_rows_out=0, d_ids_out=0, cap=0, stream=0):
        owner = _arr(d_owner, ctypes.c_uint32, self.cents.shape[0])
        dest = owner[self.lists]
        counts = np.bincount(dest[dest != my_rank], minlength=world).astype(np.uint64)
        if d_rows_out:
            assert cap >= counts.sum()
            take = np.flatnonzero(dest != my_rank)
            take = take[np.argsort(dest[take], kind="stable")]
            _arr(d_rows_out, ctypes.c_float, take.size * D)[:] = self.x[take].ravel()
            _arr(d_ids_out, ctypes.c_uint32, take.size)[:] = self.ids[take]
            keep = dest == my_rank
            self.x, self.ids, self.lists = (np.ascontiguousarray(a[keep]) for a in (self.x, self.ids, self.lists))
        return counts

    def ivf_add_device(self, d_x, d_ids, n, mod=1, rem=0):
        x = _arr(d_x, ctypes.c_float, n * D).reshape(n, D).copy()
        ids = _arr(d_ids, ctypes.c_uint32, n).copy()
        if mod > 1:
            keep = O.assign(x, self.cents) % mod == rem
            x, ids = x[keep], ids[keep]
        self._append(x, ids)
        return int(ids.size)

    def ivf_add_device_owned(self, d_x, d_ids, n, d_owner, my_rank):
        x = _arr(d_x, ctypes.c_float, n * D).reshape(n, D).copy()
        ids = _arr(d_ids, ctypes.c_uint32, n).copy()
        owner = _arr(d_owner, ctypes.c_uint32, self.cents.shape[0])
        keep = owner[O.assign(x, self.cents)] == my_rank
        self._append(x[keep], ids[keep])
        return int(keep.sum())


def _data():
    rng = np.random.default_rng(5)
    centers = rng.standard_normal((12, D)).astype(np.float32) * 4
    x = (centers[rng.integers(0, 12, N)] + rng.standard_normal((N, D)).astype(np.float32)).astype(np.float32)
    return x, x[:: N // NLIST][:NLIST].copy()


def _gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t)
    return [o.numpy() for o in out]


def _gather_var(a):
    n = _gather(torch.tensor([a.size], dtype=torch.int64))
    m = int(max(v[0] for v in n))
    buf = torch.zeros(m, dtype=torch.int64)
    buf[:a.size] = torch.from_numpy(a.astype(np.int64))
    return [g[:int(c[0])] for g, c in zip(_gather(buf), n)]


def _check_placement(sh, eng, x, what):
    world = dist.get_world_size()
    owner = sh.owner_host
    owners = _gather(torch.from_numpy(owner.astype(np.int64)))
    assert all(np.array_equal(o, owners[0]) for o in owners), f"{what}: the ranks disagree on the placement"
    cents = _gather(torch.from_numpy(eng.cents.copy()))
    assert all(np.array_equal(c.view(np.uint32), cents[0].view(np.uint32)) for c in cents), f"{what}: centroids differ"
    ids, lists = eng.dump_lists()
    assert (owner[lists] == sh.rank).all(), f"{what}: rank {sh.rank} holds a row of a list it does not own"
    assert np.array_equal(lists, O.assign(x[ids], eng.cents)), f"{what}: a row is not in its nearest list"
    all_ids = np.concatenate(_gather_var(ids))
    assert np.array_equal(np.sort(all_ids), np.arange(N)), f"{what}: rows lost or duplicated"
    hist = np.bincount(O.assign(x, eng.cents), minlength=eng.cents.shape[0])
    assert np.array_equal(owner, place_lists(hist, world)), f"{what}: not the placement of the global histogram"
    loads = np.bincount(owner, weights=hist, minlength=world)
    assert ids.size == int(loads[sh.rank]), f"{what}: row count differs from the placement's load"


def _worker(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from fabstir_vectordb_b200.shard import ShardedIndex
        x, cents = _data()
        eng = _ArenaStandIn(cents)
        sh = ShardedIndex(eng, rank, world)
        scratches = []

        def new_scratch():
            scratches.append(_ArenaStandIn(np.zeros((1, D), dtype=np.float32)))
            return scratches[-1]
        sh._new_scratch = new_scratch
        # two thirds loaded by the l % world rule, the rest "migrated": each row on rank id % world, whatever
        # rank owns its list, so every list is in fragments on both ranks
        ids = np.arange(N, dtype=np.uint32)
        base = ids < 2 * N // 3
        a = O.assign(x, cents)
        mine = base & (np.array([owner_of_list(int(l), world) for l in a]) == rank)
        mine |= ~base & (ids % world == rank)
        eng._append(x[mine], ids[mine])
        before = eng.ids.size
        frag = _gather(torch.tensor([int((a[eng.ids] % world != rank).sum())]))
        assert sum(int(f[0]) for f in frag) > 0, "no row off its owner: the case tests nothing"

        sh._nlist = NLIST
        res = sh.retrain(NLIST, ITERS, cents)
        assert res["old_nlist"] == res["new_nlist"] == NLIST and res["rows_reassigned"] == N
        assert res["iterations"] <= ITERS and sh._nlist == NLIST
        assert res["rows_moved"] > 0 and eng.ids.size != before
        assert all(s.closed for s in scratches), "the scratch handle was not closed"
        o_c, _, _ = O.train_lloyd(x, cents, ITERS)
        assert float(np.abs(eng.cents - o_c).max()) < 1e-3, "centroids differ from a single-process Lloyd"
        _check_placement(sh, eng, x, "retrain")

        # optimize_clusters: same nlist, from the current centroids
        res = sh.optimize_clusters(max_iterations=2)
        assert res["new_nlist"] == NLIST
        _check_placement(sh, eng, x, "optimize_clusters")

        # add_clusters: nlist grows, the cached nlist follows
        init = np.concatenate([eng.cents, x[[1, 2, 3]]])
        res = sh.add_clusters(3, init, max_iterations=2)
        assert (res["old_nlist"], res["new_nlist"]) == (NLIST, NLIST + 3) and sh._nlist == NLIST + 3
        _check_placement(sh, eng, x, "add_clusters")

        # failure rule: the exchange of the rows fails on every rank after take_unowned -> each rank's taken rows
        # are back in its own arena, and the error propagates
        real = dist.all_to_all_single
        calls = []

        def failing(out, inp, *args, **kw):
            calls.append(inp.dtype)
            if inp.dtype == torch.float32:
                raise RuntimeError("exchange failed")
            return real(out, inp, *args, **kw)
        init = x[:: N // 4][:4].copy()
        held = set(eng.ids.tolist())
        dist.all_to_all_single = failing
        try:
            with pytest.raises(RuntimeError, match="exchange failed"):
                sh.retrain(4, 2, init)
        finally:
            dist.all_to_all_single = real
        assert torch.float32 in calls
        assert set(eng.ids.tolist()) == held and eng.ids.size == len(held), "taken rows were not put back"
        assert np.array_equal(eng.lists, O.assign(x[eng.ids], eng.cents))
        assert eng.cents.shape[0] == 4 and sh._nlist is None
        all_ids = np.concatenate(_gather_var(eng.ids))
        assert np.array_equal(np.sort(all_ids), np.arange(N))
    finally:
        dist.destroy_process_group()


def test_sharded_retrain_world2():
    mp.spawn(_worker, args=(2, _free_port()), nprocs=2, join=True)


def test_retrain_refuses_batches_in_flight():
    from fabstir_vectordb_b200.shard import ShardedIndex
    sh = ShardedIndex(_ArenaStandIn(np.zeros((2, D), dtype=np.float32)), 0, 1)
    sh._group = [object()]
    with pytest.raises(RuntimeError, match="finish"):
        sh.retrain(2, 1, np.zeros((2, D), dtype=np.float32))
