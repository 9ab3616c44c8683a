"""The sharded retrain (ShardedIndex.retrain) on ONE GPU: W Engine handles on device 0 act as the W ranks and the
test performs the driver's collective steps itself (sums of the k-means buffers, the list histogram, the
all-to-all of the rows).  The index is built size-balanced (place_lists), then recent-tier rows are migrated so
that lists lie in fragments on every handle, and some rows are tombstoned.  After the retrain every row must sit
on the handle that owns its nearest new centroid, and the sharded search must equal the CPU oracle bit for bit.

Also covered: fvdb_ivf_reassign against fvdb_ivf_retrain on one handle, fvdb_ivf_arena_device, and the edge and
error cases of fvdb_ivf_take_unowned_device."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, FvdbError, InvalidConfig, NanInput, NotTrained, _lib as L, synth
from fabstir_vectordb_b200.shard import _tensor_at, pack_layout, place_lists, tiers_pack_layout

pytestmark = pytest.mark.gpu

D, NLIST, N0, NREC, NMIG, ITERS, K, NPROBE, NQ = 128, 32, 20_000, 6_000, 4_000, 4, 10, 6, 64


def _torch():
    import torch
    return torch


def _dev(a):
    torch = _torch()
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a.copy()).cuda()


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _assert_bits(got, want, what):
    g_ids, g_dst, g_cnt = got
    w_ids, w_dst, w_cnt = want
    assert np.array_equal(g_cnt, w_cnt.astype(np.uint32)), f"{what}: counts"
    for i in range(len(w_cnt)):
        c = int(w_cnt[i])
        assert g_ids[i, :c].tolist() == w_ids[i, :c].tolist(), f"{what}: ids of query {i}"
        assert g_dst[i, :c].view(np.uint32).tolist() == w_dst[i, :c].view(np.uint32).tolist(), f"{what}: dist of query {i}"


@pytest.fixture(scope="module")
def data():
    x = synth.rows(0, N0 + NREC, D, 4 * NLIST, 1.0, 4321)
    q = synth.queries(0, NQ, D, N0 + NREC, 4 * NLIST, 1.0, 4321, synth.default_qnoise(D, 1.0), 99)
    init = x[:N0:N0 // NLIST][:NLIST].copy()
    rng = np.random.default_rng(3)
    mig = np.sort(rng.choice(np.arange(N0, N0 + NREC), NMIG, replace=False)).astype(np.uint32)
    dele = np.concatenate([np.arange(5, N0, 13), mig[::7], np.arange(N0 + 1, N0 + NREC, 17)]).astype(np.uint32)
    return dict(x=x, q=q, init=init, mig=mig, dele=np.unique(dele))


def _build(data, world):
    """A size-balanced sharded index over rows [0, N0), the recent rows on handle id % world, NMIG of them
    migrated (each into the arena of the handle that held it), tombstones on every handle."""
    torch = _torch()
    x, init = data["x"], data["init"]
    hist = np.bincount(O.assign(x[:N0], init), minlength=NLIST)
    owner = place_lists(hist, world)
    d_owner = _dev(owner)
    dx = torch.from_numpy(x[:N0]).cuda()
    dids = torch.arange(N0, dtype=torch.int32, device="cuda")
    rec_ids = np.arange(N0, N0 + NREC, dtype=np.uint32)
    recent = [(torch.from_numpy(x[m]).cuda(), _dev(m)) for m in (rec_ids[rec_ids % world == r] for r in range(world))]
    torch.cuda.synchronize()     # the engine reads the rows on its own stream
    engs = []
    for r in range(world):
        e = Engine(D, k_max=64)
        e.set_centroids(init)
        assert e.ivf_add_device_owned(dx.data_ptr(), dids.data_ptr(), N0, d_owner.data_ptr(), r) > 0
        fx, fids = recent[r]
        e.flat_add_device(fx.data_ptr(), fids.data_ptr(), fx.shape[0])
        e.move_flat_to_ivf(data["mig"])
        e.set_deleted(data["dele"], True)
        engs.append(e)
    return engs, owner


def _arena(e):
    p_rows, p_ids, n = e.ivf_arena_device()
    dev = _torch().device("cuda", 0)
    return _tensor_at(p_rows, (n, D), "<f4", dev), _tensor_at(p_ids, (n,), "<i4", dev)


def _sharded_lloyd(engs, init, iters):
    """train()'s loop with the all-reduce done by hand: scratch handles hold the working centroids."""
    torch = _torch()
    scratch = [Engine(D, k_max=1) for _ in engs]
    views = [_arena(e)[0] for e in engs]
    for s in scratch:
        s.set_centroids(init)
    assigns = [torch.zeros((max(v.shape[0], 1),), dtype=torch.int32, device="cuda") for v in views]
    for _ in range(iters):
        parts = []
        for s, v, a in zip(scratch, views, assigns):
            b = [torch.zeros((NLIST, D), dtype=torch.float32, device="cuda"),
                 torch.zeros((NLIST,), dtype=torch.int32, device="cuda"),
                 torch.zeros((1,), dtype=torch.float64, device="cuda"),
                 torch.zeros((1,), dtype=torch.int32, device="cuda")]
            s.kmeans_accumulate_device(v.data_ptr(), v.shape[0], b[0].data_ptr(), b[1].data_ptr(), b[2].data_ptr(),
                                       a.data_ptr(), b[3].data_ptr())
            parts.append(b)
        torch.cuda.synchronize()
        sums = sum(p[0] for p in parts)
        counts = sum(p[1] for p in parts)
        for s in scratch:
            s.kmeans_apply_device(sums.data_ptr(), counts.data_ptr())
        torch.cuda.synchronize()
    cents = [s.get_centroids() for s in scratch]
    for s in scratch:
        s.close()
    return cents


def _lloyd64(x, init, iters):
    c = init.astype(np.float32)
    for _ in range(iters):
        a = O.assign(x, c)
        s = np.zeros((NLIST, D))
        np.add.at(s, a, x.astype(np.float64))
        n = np.bincount(a, minlength=NLIST)
        c = np.where(n[:, None] > 0, s / np.maximum(n, 1)[:, None], c).astype(np.float32)
    return c


def _retrain(engs, data):
    """ShardedIndex.retrain's steps over the handles.  Returns (centroids, owner, rows sent per handle)."""
    torch = _torch()
    world = len(engs)
    cents = _sharded_lloyd(engs, data["init"], ITERS)
    for c in cents[1:]:
        assert np.array_equal(c.view(np.uint32), cents[0].view(np.uint32)), "ranks trained different centroids"
    cents = cents[0]
    for e in engs:
        e.ivf_reassign(cents)
    hist = sum(np.bincount(e.dump_lists()[1], minlength=NLIST) for e in engs)
    owner = place_lists(hist, world)
    d_owner = _dev(owner)
    sends = []
    for r, e in enumerate(engs):
        counts = e.ivf_take_unowned_device(d_owner.data_ptr(), r, world)
        assert counts[r] == 0
        n = int(counts.sum())
        sx = torch.empty((n, D), dtype=torch.float32, device="cuda")
        si = torch.empty((n,), dtype=torch.int32, device="cuda")
        got = e.ivf_take_unowned_device(d_owner.data_ptr(), r, world, sx.data_ptr(), si.data_ptr(), n)
        assert np.array_equal(got, counts)
        # grouped by destination rank: the owner of each row's list, ascending
        dst = owner[O.assign(sx.cpu().numpy(), cents)] if n else np.zeros(0, dtype=np.uint32)
        assert (np.diff(dst.astype(np.int64)) >= 0).all() and np.array_equal(np.bincount(dst, minlength=world), counts)
        sends.append((sx, si, counts.astype(np.int64)))
    recv = []
    for r in range(world):     # the all_to_all_single layout: from every source rank in rank order
        segs_x, segs_i = [], []
        for sx, si, c in sends:
            lo = int(c[:r].sum())
            segs_x.append(sx[lo:lo + int(c[r])])
            segs_i.append(si[lo:lo + int(c[r])])
        recv.append((torch.cat(segs_x).contiguous(), torch.cat(segs_i).contiguous()))
    torch.cuda.synchronize()
    for r, (e, (rx, ri)) in enumerate(zip(engs, recv)):
        if rx.shape[0]:
            assert e.ivf_add_device_owned(rx.data_ptr(), ri.data_ptr(), rx.shape[0], d_owner.data_ptr(), r) == rx.shape[0]
    return cents, owner, [int(s[2].sum()) for s in sends]


def _coarse(engs, dq, nprobe):
    torch = _torch()
    world, nq = len(engs), dq.shape[0]
    per = (nq + world - 1) // world
    mine = []
    for r, e in enumerate(engs):
        m = torch.full((per, nprobe), -1, dtype=torch.int64, device="cuda")
        lo = min(nq, r * per)
        n = max(0, min(nq, lo + per) - lo)
        if n:
            e.coarse_device(dq[lo:lo + n].data_ptr(), n, nprobe, m.data_ptr())
        mine.append(m)
    return torch.cat(mine)


def _search(engs, q, tiers):
    torch = _torch()
    nq, world = q.shape[0], len(engs)
    dq = torch.from_numpy(q).cuda()
    keys = _coarse(engs, dq, NPROBE)
    out = [torch.empty((nq, K), dtype=torch.int32, device="cuda"), torch.empty((nq, K), dtype=torch.float32, device="cuda"),
           torch.empty((nq,), dtype=torch.int32, device="cuda")]
    if tiers == L.TIER_BOTH:
        packs = torch.empty((world, tiers_pack_layout(nq, K)[4]), dtype=torch.int32, device="cuda")
        for e, p in zip(engs, packs):
            e.search_device_tiers(dq.data_ptr(), nq, K, NPROBE, tiers, 0, 0, keys.data_ptr(), p.data_ptr())
        engs[0].merge_topk_tiers_packed_device(packs.data_ptr(), world, nq, K, *(t.data_ptr() for t in out))
    else:
        o_i, o_d, o_c, chunk = pack_layout(nq, K)
        packs = torch.empty((world, chunk), dtype=torch.int32, device="cuda")
        for e, p in zip(engs, packs):
            e.search_device_coarse(dq.data_ptr(), nq, K, NPROBE, tiers, 0, 0, keys.data_ptr(), p[o_i:o_d].data_ptr(),
                                   p[o_d:o_c].data_ptr(), p[o_c:].data_ptr())
        engs[0].merge_topk_packed_device(packs.data_ptr(), world, nq, K, *(t.data_ptr() for t in out))
    torch.cuda.synchronize()
    return _u32(out[0]), out[1].cpu().numpy(), _u32(out[2])


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_retrain_replaces_rows(data, world):
    x, dele, mig = data["x"], data["dele"], data["mig"]
    engs, _ = _build(data, world)
    ivf_ids = np.concatenate([np.arange(N0, dtype=np.uint32), mig])
    # migration left lists in fragments: some list has rows on more than one handle
    held = [e.dump_lists() for e in engs]
    frag = sum(len(set(np.unique(l).tolist()) & set(np.unique(m).tolist()))
               for i, (_, l) in enumerate(held) for (_, m) in held[i + 1:])
    assert frag > 0, "no list in fragments: the case tests nothing"
    # the arena view is the arena
    for e, (ids, _) in zip(engs, held):
        rows, vids = _arena(e)
        assert vids.shape[0] == ids.size == e.stats().ivf_rows
        assert np.array_equal(_u32(vids), ids) and np.array_equal(rows.cpu().numpy(), x[ids])

    cents, owner, sent = _retrain(engs, data)
    assert sum(sent) > 0
    # the sums are unordered f32 atomics: agreement to rounding (a row on a cell boundary may still flip)
    ref = _lloyd64(x[ivf_ids], data["init"], ITERS)
    assert float(np.abs(cents - ref).max()) < 1e-3, "centroids differ from a float64 Lloyd"
    assert float((O.assign(x[ivf_ids], cents) == O.assign(x[ivf_ids], ref)).mean()) >= 0.999

    want_list = O.assign(x, cents)
    hist = np.bincount(want_list[ivf_ids], minlength=NLIST)
    assert np.array_equal(owner, place_lists(hist, world))
    loads = np.bincount(owner, weights=hist, minlength=world)
    seen = []
    for r, e in enumerate(engs):
        assert np.array_equal(e.get_centroids().view(np.uint32), cents.view(np.uint32))
        ids, lists = e.dump_lists()
        assert np.array_equal(lists, want_list[ids]), f"handle {r}: a row is not in its nearest new list"
        assert (owner[lists] == r).all(), f"handle {r} holds a row of a list it does not own"
        assert (np.diff(lists.astype(np.int64)) >= 0).all(), f"handle {r}: arena not grouped by list"
        assert ids.size == int(loads[r])
        seen.append(ids)
    allids = np.concatenate(seen)
    assert np.array_equal(np.sort(allids), np.sort(ivf_ids)), "rows lost or duplicated"

    # search: the proof floor re-reduced over the handles, then exact and tensor-core mode, both tier sets
    floor = int(np.float32(max(e.ivf_max_sqnorm() for e in engs)).view(np.uint32))
    live_ivf = ivf_ids[~np.isin(ivf_ids, dele)]
    rec = np.setdiff1d(np.arange(N0, N0 + NREC, dtype=np.uint32), mig)
    live_rec = rec[~np.isin(rec, dele)]
    ivf = O.IVF(cents, x[live_ivf], live_ivf)
    q = data["q"]
    for mode in (L.SCAN_EXACT, L.SCAN_TC):
        for e in engs:
            e.set_option(L.OPT_SCAN_MODE, mode)
            e.set_option(L.OPT_PROOF_XMAX, floor)
        for tiers in (L.TIER_HISTORICAL, L.TIER_BOTH):
            want = O.hybrid_batch_search(ivf, x[live_rec], live_rec, q, K, NPROBE, tiers=tiers)
            got = _search(engs, q, tiers)
            _assert_bits(got, want, f"mode {mode} tiers {tiers}")
            for i in range(NQ):
                assert not np.isin(got[0][i, :got[2][i]], dele).any(), "a tombstoned row was returned"

    # vacuum removes exactly the tombstoned rows
    gone = sum(e.vacuum() for e in engs)
    assert gone == int(np.isin(ivf_ids, dele).sum() + np.isin(rec, dele).sum())
    left = np.concatenate([e.dump_lists()[0] for e in engs])
    assert np.array_equal(np.sort(left), np.sort(live_ivf))
    for e in engs:
        e.close()


def test_reassign_equals_retrain(data):
    x = data["x"][:N0]
    ids = np.arange(N0, dtype=np.uint32)
    a, b = Engine(D), Engine(D)
    for e in (a, b):
        e.set_centroids(data["init"])
        e.ivf_add(x, ids)
    a.set_deleted(ids[::9], True)
    b.set_deleted(ids[::9], True)
    a.retrain(NLIST, ITERS, init_centroids=data["init"])
    cents = a.get_centroids()
    b.ivf_reassign(cents)
    ra, la = a.dump_lists()
    rb, lb = b.dump_lists()
    assert np.array_equal(ra, rb) and np.array_equal(la, lb)
    assert np.array_equal(lb, O.assign(x[rb], cents))
    assert b.stats().deleted_rows == a.stats().deleted_rows
    # a different nlist; then the errors
    c2 = x[::N0 // 8][:8].copy()
    b.ivf_reassign(c2)
    rb, lb = b.dump_lists()
    assert b.stats().nlist == 8 and np.array_equal(np.sort(rb), ids) and np.array_equal(lb, O.assign(x[rb], c2))
    bad = c2.copy()
    bad[3, 5] = np.nan
    with pytest.raises(NanInput):
        b.ivf_reassign(bad)
    assert np.array_equal(b.dump_lists()[1], lb), "a rejected table changed the lists"
    fresh = Engine(D)
    with pytest.raises(NotTrained):
        fresh.ivf_reassign(c2)
    cos = Engine(D, metric=L.METRIC_COS)
    for call in (lambda: cos.ivf_reassign(c2), cos.ivf_arena_device):
        with pytest.raises(InvalidConfig):
            call()
    for e in (a, b, fresh, cos):
        e.close()


def test_take_unowned_edge_cases(data):
    torch = _torch()
    x = data["x"][:5_000]
    ids = np.arange(5_000, dtype=np.uint32)
    e = Engine(D)
    e.set_centroids(data["init"])
    e.ivf_add(x, ids)
    before = e.dump_lists()
    n = before[0].size
    out_x = torch.empty((n, D), dtype=torch.float32, device="cuda")
    out_i = torch.empty((n,), dtype=torch.int32, device="cuda")
    mine, elsewhere = _dev(np.zeros(NLIST, dtype=np.uint32)), _dev(np.ones(NLIST, dtype=np.uint32))

    def same():
        now = e.dump_lists()
        return np.array_equal(now[0], before[0]) and np.array_equal(now[1], before[1])

    assert e.ivf_take_unowned_device(mine.data_ptr(), 0, 2, out_x.data_ptr(), out_i.data_ptr(), n).tolist() == [0, 0]
    assert same(), "an all-mine table changed the arena"
    assert e.ivf_take_unowned_device(elsewhere.data_ptr(), 0, 2).tolist() == [0, n]
    assert same(), "a counts-only call changed the arena"

    def code(f):
        with pytest.raises(FvdbError) as ei:
            f()
        return ei.value.code
    p = (out_x.data_ptr(), out_i.data_ptr())
    assert code(lambda: e.ivf_take_unowned_device(0, 0, 2, *p, n)) == L.ERR_INVALID_ARG
    assert code(lambda: e.ivf_take_unowned_device(elsewhere.data_ptr(), 2, 2, *p, n)) == L.ERR_INVALID_ARG
    assert code(lambda: e.ivf_take_unowned_device(elsewhere.data_ptr(), 0, 2, *p, n - 1)) == L.ERR_INVALID_ARG
    assert code(lambda: e.ivf_take_unowned_device(elsewhere.data_ptr(), 0, 2, p[0], 0, n)) == L.ERR_INVALID_ARG
    beyond = _dev(np.full(NLIST, 5, dtype=np.uint32))
    assert code(lambda: e.ivf_take_unowned_device(beyond.data_ptr(), 0, 2, *p, n)) == L.ERR_INVALID_ARG
    assert same(), "a refused call changed the arena"
    assert code(lambda: Engine(D).ivf_take_unowned_device(mine.data_ptr(), 0, 2)) == L.ERR_NOT_TRAINED
    assert code(lambda: Engine(D, metric=L.METRIC_COS).ivf_take_unowned_device(mine.data_ptr(), 0, 2)) == L.ERR_INVALID_CONFIG

    # all elsewhere: the arena empties, the rows come out in arena order
    assert e.ivf_take_unowned_device(elsewhere.data_ptr(), 0, 2, *p, n).tolist() == [0, n]
    torch.cuda.synchronize()
    assert e.stats().ivf_rows == 0 and e.dump_lists()[0].size == 0
    assert np.array_equal(_u32(out_i), before[0])
    assert np.array_equal(out_x.cpu().numpy(), x[before[0]])
    # they go back in through the owned add and land where they were
    assert e.ivf_add_device_owned(out_x.data_ptr(), out_i.data_ptr(), n, mine.data_ptr(), 0) == n
    assert same()
    e.close()


def test_sharded_index_retrain_one_rank(data):
    """ShardedIndex.retrain itself on one GPU (world 1: no exchange): the arena view, the scratch handle, the
    reassignment and the refreshed nlist."""
    from fabstir_vectordb_b200.shard import ShardedIndex
    engs, _ = _build(data, 1)
    e = engs[0]
    ids0 = np.sort(e.dump_lists()[0])
    sh = ShardedIndex(e, 0, 1)
    init = data["x"][:N0:N0 // 16][:16].copy()
    res = sh.retrain(16, ITERS, init)
    assert (res["old_nlist"], res["new_nlist"], res["rows_reassigned"], res["rows_moved"]) == (NLIST, 16, ids0.size, 0)
    assert sh._nlist == 16 and set(res["seconds"]) == {"lloyd", "reassign", "placement", "exchange"}
    cents = e.get_centroids()
    ids, lists = e.dump_lists()
    assert np.array_equal(np.sort(ids), ids0) and np.array_equal(lists, O.assign(data["x"][ids], cents))
    assert (sh.owner_host == 0).all() and sh.owner_host.size == 16
    res = sh.optimize_clusters(max_iterations=2)
    assert res["new_nlist"] == 16 and np.array_equal(np.sort(e.dump_lists()[0]), ids0)
    e.close()
