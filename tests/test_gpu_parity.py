"""GPU parity: libfvdb_b200 (through the C ABI) against the CPU oracle on the same seeded inputs.
Exact mode must be BIT-exact (ids and distance bits); the tensor-core mode must return the same
ids/distances wherever the oracle's neighbouring distances differ by more than 1e-4 relative
(BASELINE.json north_star) — in practice it is bit-exact too because the final ranking is
re-computed in fp32 in the reference's operation order."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, _lib as L, synth

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4  # north_star: ids must agree wherever distances are separated by > 1e-4 relative


def _data(n, d, seed, n_comp=16, sigma=0.6):
    return synth.rows(0, n, d, n_comp, sigma, seed)


def _queries(nq, d, n, seed, n_comp=16, sigma=0.6):
    return synth.queries(0, nq, d, n, n_comp, sigma, seed, synth.default_qnoise(d, sigma), seed + 1)


def _assert_same(ids, dist, cnt, o_ids, o_dist, o_cnt, exact=True):
    assert cnt.tolist() == o_cnt.tolist()
    for i in range(len(cnt)):
        c = int(cnt[i])
        if exact:
            assert ids[i, :c].tolist() == o_ids[i, :c].tolist(), f"query {i}"
            assert dist[i, :c].view(np.uint32).tolist() == o_dist[i, :c].view(np.uint32).tolist(), f"query {i}"
        else:
            # tolerance form: positions whose oracle distance is separated from both neighbours
            # by > REL_TOL must carry the same id; distances within REL_TOL everywhere
            od = o_dist[i, :c].astype(np.float64)
            assert np.allclose(dist[i, :c], od, rtol=REL_TOL, atol=0)
            for j in range(c):
                lo = j == 0 or (od[j] - od[j - 1]) > REL_TOL * od[j]
                hi = j == c - 1 or (od[j + 1] - od[j]) > REL_TOL * od[j]
                if lo and hi:
                    assert ids[i, j] == o_ids[i, j], f"query {i} pos {j}"


def _build(n, d, nlist, seed, mode, k_max=64, flat_n=0):
    x = _data(n + flat_n, d, seed)
    cents = x[np.random.default_rng(seed).choice(n, nlist, replace=False)].copy()
    eng = Engine(d, k_max=k_max)
    _set_mode(eng, mode)
    eng.set_centroids(cents)
    ids = np.arange(n, dtype=np.uint32)
    lists = eng.ivf_add(x[:n], ids, want_lists=True)
    ivf = O.IVF(cents, x[:n], ids)
    assert lists.tolist() == ivf.assign.tolist(), "coarse assignment differs from the oracle"
    fx, fid = None, None
    if flat_n:
        fx = x[n:]
        fid = np.arange(n, n + flat_n, dtype=np.uint32)
        eng.flat_add(fx, fid)
    return eng, ivf, x, cents, fx, fid


MODES = ["exact", "tc"]


def _set_mode(eng, mode):
    from fabstir_vectordb_b200 import InvalidConfig
    if mode == "tc":
        try:
            eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
            eng.set_option(L.OPT_KMEANS_TC, 1)
        except InvalidConfig:
            pytest.skip("tensor-core path unavailable for this dim")
    else:
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n,d,nlist,nprobe,k,nq", [
    (4000, 384, 32, 8, 10, 64),
    (3000, 128, 16, 16, 5, 33),
    (5000, 384, 64, 1, 10, 1),
    (2000, 64, 8, 3, 16, 130),
])
def test_ivf_search_parity(mode, n, d, nlist, nprobe, k, nq):
    if mode == "tc" and d % 32:
        pytest.skip("tc needs dim % 32 == 0")
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 11, mode)
    q = _queries(nq, d, n, 11)
    ids, dist, cnt = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL)
    o = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    _assert_same(ids, dist, cnt, *o)
    if mode == "tc":
        # the tensor-core path must carry these well-separated shapes itself: a proof that failed for more
        # than a stray query would mean "tc" parity is really the exact fallback's
        assert eng.stats().last_fallback_queries <= nq // 16


@pytest.mark.parametrize("d", [2, 3, 7, 30, 100])
def test_odd_dimensions_exact(d):
    n, nlist = 1500, 8
    rng = np.random.default_rng(d)
    x = rng.standard_normal((n, d)).astype(np.float32)
    cents = x[:nlist].copy()
    eng = Engine(d, k_max=32)
    eng.set_centroids(cents)
    eng.ivf_add(x, np.arange(n, dtype=np.uint32))
    ivf = O.IVF(cents, x)
    q = x[:40] + np.float32(0.01)
    ids, dist, cnt = eng.search(q, 10, 4, tiers=L.TIER_HISTORICAL)
    _assert_same(ids, dist, cnt, *O.hybrid_batch_search(ivf, None, None, q, 10, 4, tiers=2))


@pytest.mark.parametrize("mode", MODES)
def test_assign_matches_find_nearest_centroid(mode):
    d, nlist = 384, 96
    x = _data(6000, d, 5)
    cents = x[:nlist].copy()
    cents[7] = cents[3]  # duplicate centroid: strict '<' must pick the lower id
    eng = Engine(d)
    _set_mode(eng, mode)
    eng.set_centroids(cents)
    got = eng.assign(x)
    want = O.assign(x, cents)
    assert got.tolist() == want.tolist()
    assert 7 not in set(got.tolist())


@pytest.mark.parametrize("mode", MODES)
def test_flat_tier_is_exact_scan(mode):
    d, n = 384, 7000
    x = _data(n, d, 21)
    ids = (np.arange(n, dtype=np.uint32) * 3 + 5).astype(np.uint32)
    eng = Engine(d, k_max=64)
    _set_mode(eng, mode)
    eng.flat_add(x, ids)
    q = _queries(50, d, n, 21)
    got = eng.search(q, 10, 0, tiers=L.TIER_RECENT)
    want = O.hybrid_batch_search(None, x, ids, q, 10, 0, tiers=1)
    _assert_same(*got, *want)


@pytest.mark.parametrize("d", [384, 64])
def test_bulk_assignment_tensor_core_path(d):
    # rows x lists >= 64M: find_nearest_centroid (src/ivf/core.rs:373-386) runs as a tensor-core scan
    # of the centroid table with exact re-rank + proof; every assignment must equal the oracle's
    n, nlist = 65_536, 1024
    x = _data(n, d, 29, n_comp=512)
    cents = x[:: n // nlist][:nlist].copy()
    cents[7] = cents[3]                     # duplicate centroid: the lower id must win
    eng = Engine(d, k_max=16)
    _set_mode(eng, "tc")
    eng.set_centroids(cents)
    got = eng.assign(x)
    sample = np.arange(0, n, 16 if d == 384 else 2)
    want = O.assign(x[sample], cents)
    assert got[sample].tolist() == want.tolist()
    assert 7 not in set(got.tolist())
    eng.close()


@pytest.mark.parametrize("d", [384, 64])
def test_flat_tier_tensor_core_path(d):
    # large enough (rows x queries >= 4M) for the tensor-core flat scan: several row chunks and
    # query groups, a ragged last tile, tombstones and a filter bitmap; must stay bit-exact
    n, nq, k = 21_003, 210, 10
    x = _data(n, d, 23)
    ids = (np.arange(n, dtype=np.uint32) * 2 + 1).astype(np.uint32)
    eng = Engine(d, k_max=16)
    _set_mode(eng, "tc")
    eng.flat_add(x, ids)
    q = _queries(nq, d, n, 23)
    got = eng.search(q, k, 0, tiers=L.TIER_RECENT)
    want = O.hybrid_batch_search(None, x, ids, q, k, 0, tiers=1)
    _assert_same(*got, *want)
    dele = ids[::17].copy()
    eng.set_deleted(dele, True)
    nbits = int(ids.max()) + 1
    keep = ids[(ids % 3) != 0]
    fbits = O.make_bitmap((nbits + 63) // 64 * 64, keep)
    got = eng.search(q, k, 0, tiers=L.TIER_RECENT, filter_bits=fbits)
    want = O.hybrid_batch_search(None, x, ids, q, k, 0, tiers=1,
                                 deleted=O.make_bitmap((nbits + 63) // 64 * 64, dele), filter_bits=fbits)
    _assert_same(*got, *want)
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_hybrid_merge_ties_and_no_dedup(mode):
    # the same vectors live in both tiers under different ids: distance ties, recent first
    d, n = 128, 3000
    eng, ivf, x, cents, _, _ = _build(n, d, 16, 31, mode)
    fx = x[:200].copy()
    fid = np.arange(200, dtype=np.uint32) + 100_000
    eng.flat_add(fx, fid)
    q = x[:20].copy()
    got = eng.search(q, 6, 16, tiers=L.TIER_BOTH)
    want = O.hybrid_batch_search(ivf, fx, fid, q, 6, 16, tiers=3)
    _assert_same(*got, *want)
    assert got[0][0, 0] == 100_000 and got[0][0, 1] == 0


@pytest.mark.parametrize("mode", MODES)
def test_tombstones_and_filter_bitmap(mode):
    d, n, flat_n = 384, 6000, 1500
    eng, ivf, x, cents, fx, fid = _build(n, d, 32, 41, mode, flat_n=flat_n)
    total = n + flat_n
    rng = np.random.default_rng(41)
    dele = rng.choice(total, total // 50, replace=False).astype(np.uint32)
    eng.set_deleted(dele, True)
    dbits = O.make_bitmap(total, dele)
    fbits = synth.filter_bitmap((total + 63) // 64 * 64, 10, 99)
    q = _queries(64, d, total, 41)
    # tombstones only
    got = eng.search(q, 10, 8, tiers=L.TIER_BOTH)
    want = O.hybrid_batch_search(ivf, fx, fid, q, 10, 8, tiers=3, deleted=dbits)
    _assert_same(*got, *want)
    assert not set(got[0].ravel().tolist()) & set(dele.tolist())
    # tombstones AND 10% pre-filter
    got = eng.search(q, 10, 8, tiers=L.TIER_BOTH, filter_bits=fbits)
    want = O.hybrid_batch_search(ivf, fx, fid, q, 10, 8, tiers=3, deleted=dbits, filter_bits=fbits)
    _assert_same(*got, *want)
    # revive, vacuum
    eng.set_deleted(dele[:10], False)
    removed = eng.vacuum()
    assert removed == len(dele) - 10
    keep = np.setdiff1d(np.arange(total), dele[10:])
    got = eng.search(q, 10, 8, tiers=L.TIER_BOTH)
    want = O.hybrid_batch_search(ivf, fx, fid, q, 10, 8, tiers=3, deleted=O.make_bitmap(total, dele[10:]))
    _assert_same(*got, *want)
    assert eng.stats().ivf_rows + eng.stats().flat_rows == len(keep)


def test_fewer_than_k_and_empty():
    d = 16
    eng = Engine(d, k_max=16)
    q = np.zeros((3, d), np.float32)
    ids, dist, cnt = eng.search(q, 5, 4)
    assert cnt.tolist() == [0, 0, 0]  # uninitialised index -> Ok(vec![])
    cents = np.eye(4, d, dtype=np.float32)
    eng.set_centroids(cents)
    ids, dist, cnt = eng.search(q, 5, 4)
    assert cnt.tolist() == [0, 0, 0]
    eng.ivf_add(cents[:3] * 0.5, np.array([7, 8, 9], np.uint32))
    ids, dist, cnt = eng.search(q, 10, 4)
    assert cnt.tolist() == [3, 3, 3]
    assert sorted(ids[0, :3].tolist()) == [7, 8, 9]
    assert ids[0, 3] == 0xFFFFFFFF and np.isinf(dist[0, 3])
    # nprobe larger than nlist is clamped (truncate(n_probe), src/ivf/core.rs:656)
    ids, dist, cnt = eng.search(q, 10, 100)
    assert cnt.tolist() == [3, 3, 3]


def test_error_codes():
    from fabstir_vectordb_b200 import (DuplicateVector, FvdbError, InsufficientTrainingData,
                                       NanInput, NotTrained, VectorNotFound)
    d = 8
    eng = Engine(d, k_max=8)
    x = np.random.default_rng(0).standard_normal((20, d)).astype(np.float32)
    with pytest.raises(NotTrained):
        eng.ivf_add(x, np.arange(20, dtype=np.uint32))
    with pytest.raises(NotTrained):
        eng.assign(x)
    with pytest.raises(InsufficientTrainingData):
        eng.train(x[:3], 4, 5)
    eng.set_centroids(x[:4])
    eng.ivf_add(x, np.arange(20, dtype=np.uint32))
    with pytest.raises(DuplicateVector):
        eng.ivf_add(x[:1], np.array([3], np.uint32))
    with pytest.raises(DuplicateVector):
        eng.flat_add(x[:1], np.array([3], np.uint32))
    with pytest.raises(VectorNotFound):
        eng.set_deleted([999], True)
    bad = x[:2].copy()
    bad[1, 3] = np.nan
    with pytest.raises(NanInput):
        eng.search(bad, 3, 2)
    with pytest.raises(NanInput):
        eng.flat_add(bad, np.array([100, 101], np.uint32))
    with pytest.raises(FvdbError):
        eng.search(x[:2], 9, 2)  # k > k_max
    ids, dist, cnt = eng.search(x[:2], 3, 2)  # handle still usable after errors
    assert cnt.tolist() == [3, 3]


def test_move_flat_to_ivf():
    d, n = 64, 2000
    x = _data(n, d, 51)
    cents = x[:8].copy()
    eng = Engine(d, k_max=16)
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    eng.set_centroids(cents)
    ids = np.arange(n, dtype=np.uint32)
    eng.flat_add(x, ids)
    moved = eng.move_flat_to_ivf(ids[::2])
    assert moved == n // 2
    s = eng.stats()
    assert s.flat_rows == n // 2 and s.ivf_rows == n // 2
    q = x[:30] + np.float32(0.001)
    got = eng.search(q, 8, 8, tiers=L.TIER_BOTH)
    ivf = O.IVF(cents, x[::2], ids[::2])
    want = O.hybrid_batch_search(ivf, x[1::2], ids[1::2], q, 8, 8, tiers=3)
    _assert_same(*got, *want)


@pytest.mark.parametrize("n,d,nlist,iters", [(3000, 16, 12, 8), (20000, 384, 64, 5), (9, 2, 3, 10)])
def test_kmeans_lloyd_parity_shared_init(n, d, nlist, iters):
    """Lloyd loop of IVFIndex::train from shared initial centroids: assignments are exact, the
    update sums members in data order, the error is a sequential f32 fold — so centroids,
    iteration count, converged flag and both errors must match the oracle bit for bit."""
    if n == 9:
        from test_oracle_kat import TRAIN_2D
        x = TRAIN_2D
        init = x[[0, 6, 4]].copy()
    else:
        x = _data(n, d, 61, n_comp=nlist)
        init = x[np.random.default_rng(1).choice(n, nlist, replace=False)].copy()
    eng = Engine(d)
    res = eng.train(x, nlist, iters, init_centroids=init)
    cent, assign, want = O.train_lloyd(x, init, iters)
    got_c = eng.get_centroids()
    assert res["iterations"] == want["iterations"]
    assert res["converged"] == want["converged"]
    assert np.float32(res["initial_error"]).view(np.uint32) == np.float32(want["initial_error"]).view(np.uint32)
    assert np.float32(res["final_error"]).view(np.uint32) == np.float32(want["final_error"]).view(np.uint32)
    assert got_c.view(np.uint32).tolist() == cent.view(np.uint32).tolist()
    assert eng.stats().ivf_rows == 0  # training leaves the lists empty


@pytest.mark.parametrize("n,d,nlist,seed", [(6000, 32, 12, 42), (20000, 384, 64, 7), (500, 8, 40, 123456789012345)])
def test_kmeanspp_seeded_training_equals_the_oracle(n, d, nlist, seed):
    """IVFIndex::train with a seed (src/ivf/core.rs:176-179, 240-371): the device draws from the
    reference's own generator (rand 0.8 StdRng = ChaCha12, restated in engine.cu) and makes the
    sequential f32 prefix pick of :357-367, so on the same seed the k-means++ centroids — and with them
    the whole training run — equal the oracle's fo_kmeanspp_init + Lloyd loop bit for bit.  (Both are
    restatements of rand's published algorithm: parity with the crate itself stays unpinned, SURVEY §8c.)"""
    x = _data(n, d, 71, n_comp=nlist, sigma=0.2)
    init, picked = O.kmeanspp_init(x, nlist, seed)
    assert len(picked) == nlist
    # max_iterations = 1: centroids after one Lloyd step from the k-means++ start
    eng = Engine(d)
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    res = eng.train(x, nlist, 1, seed=seed)
    o_c, _, o_r = O.train_lloyd(x, init, 1)
    assert np.array_equal(eng.get_centroids().view(np.uint32), o_c.view(np.uint32))
    assert np.float32(res["initial_error"]).view(np.uint32) == np.float32(o_r["initial_error"]).view(np.uint32)
    # the full run
    iters = 10
    res = eng.train(x, nlist, iters, seed=seed)
    o_c, _, o_r = O.train_lloyd(x, init, iters)
    assert res["iterations"] == o_r["iterations"] and res["converged"] == o_r["converged"]
    assert np.array_equal(eng.get_centroids().view(np.uint32), o_c.view(np.uint32))
    assert np.float32(res["final_error"]).view(np.uint32) == np.float32(o_r["final_error"]).view(np.uint32)
    # another seed, another start
    eng.train(x, nlist, 1, seed=seed + 1)
    assert not np.array_equal(eng.get_centroids().view(np.uint32), O.train_lloyd(x, init, 1)[0].view(np.uint32))


@pytest.mark.parametrize("mode", MODES)
def test_coarse_entry_and_search_with_given_coarse(mode):
    # fvdb_coarse_device == the oracle's coarse ranking (src/ivf/core.rs:646-656) bit for bit, and
    # fvdb_search_device_coarse fed with it == fvdb_search (the multi-GPU driver's two-step path)
    import torch
    d, n, nlist, nq, k, nprobe = 384, 12000, 96, 70, 10, 12
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 53, mode)
    q = _queries(nq, d, n, 53)
    dq = torch.from_numpy(q).cuda()
    keys = torch.empty((nq, nprobe), dtype=torch.int64, device="cuda")
    eng.coarse_device(dq.data_ptr(), nq, nprobe, keys.data_ptr())
    torch.cuda.synchronize()
    hk = keys.cpu().numpy().view(np.uint64)
    for i in range(nq):
        ol, od = ivf.coarse(q[i], nprobe)
        assert (hk[i] & np.uint64(0xFFFFFFFF)).astype(np.uint32).tolist() == ol.tolist()
        assert (hk[i] >> np.uint64(32)).astype(np.uint32).tolist() == od.view(np.uint32).tolist()
    o_ids = torch.empty((nq, k), dtype=torch.int32, device="cuda")
    o_dst = torch.empty((nq, k), dtype=torch.float32, device="cuda")
    o_cnt = torch.empty((nq,), dtype=torch.int32, device="cuda")
    eng.search_device_coarse(dq.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0, keys.data_ptr(),
                             o_ids.data_ptr(), o_dst.data_ptr(), o_cnt.data_ptr())
    torch.cuda.synchronize()
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    _assert_same(o_ids.cpu().numpy().view(np.uint32), o_dst.cpu().numpy(), o_cnt.cpu().numpy().view(np.uint32), *want)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_page_locked_buffers_same_results(mode):
    """fvdb_search with page-locked caller buffers (fvdb_host_alloc: no staging copy, result copies
    in front of the batch's single synchronisation point) returns the bits of the pageable path
    and of the oracle; mixing one pinned and one pageable side is legal too."""
    from fabstir_vectordb_b200 import PinnedArray
    n, d, nlist, nprobe, k, nq = 4000, 384, 32, 8, 10, 70
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 23, mode)
    q = _queries(nq, d, n, 23)
    ref = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL)
    pq = PinnedArray(q.shape, np.float32)
    pq.array[...] = q
    po = (PinnedArray((nq, k), np.uint32), PinnedArray((nq, k), np.float32), PinnedArray((nq,), np.uint32))
    out = tuple(a.array for a in po)
    ids, dist, cnt = eng.search(pq.array, k, nprobe, tiers=L.TIER_HISTORICAL, out=out)
    assert ids is out[0] and dist is out[1] and cnt is out[2]
    for a, b in zip((ids, dist.view(np.uint32), cnt), (ref[0], ref[1].view(np.uint32), ref[2])):
        assert np.array_equal(a, b)
    o = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    _assert_same(ids, dist, cnt, *o)
    mixed = eng.search(pq.array, k, nprobe, tiers=L.TIER_HISTORICAL)          # pinned in, pageable out
    assert np.array_equal(mixed[0], ref[0]) and np.array_equal(mixed[2], ref[2])
    out2 = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL, out=out)          # pageable in, pinned out
    assert np.array_equal(out2[0], ref[0]) and np.array_equal(out2[1].view(np.uint32), ref[1].view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_retrain_on_device_parity(mode):
    """fvdb_ivf_retrain (IVFIndex::retrain, src/ivf/operations.rs:148-193) from shared initial
    centroids: the resident rows are the training set in arena order; centroids, the new list of
    every row and the searches afterwards (tombstones kept) equal the oracle's bit for bit."""
    n, d, nlist, new_nlist, iters = 6000, 64, 12, 20, 6
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 31, mode)
    dead = np.arange(0, n, 97, dtype=np.uint32)
    eng.set_deleted(dead, True)
    init = x[np.random.default_rng(5).choice(n, new_nlist, replace=False)].copy()
    res = eng.retrain(new_nlist, iters, init_centroids=init)
    new_ivf, order, want = O.retrain_lloyd(ivf, init, iters)
    assert res["iterations"] == want["iterations"] and res["converged"] == want["converged"]
    assert np.float32(res["final_error"]).view(np.uint32) == np.float32(want["final_error"]).view(np.uint32)
    assert eng.get_centroids().view(np.uint32).tolist() == new_ivf.centroids.view(np.uint32).tolist()
    rows, lists = eng.dump_lists()
    assert rows.size == n and eng.stats().ivf_rows == n and eng.stats().nlist == new_nlist
    got = dict(zip(rows.tolist(), lists.tolist()))
    assert got == dict(zip(new_ivf.ids.tolist(), new_ivf.assign.tolist()))
    assert (np.diff(lists.astype(np.int64)) >= 0).all()          # arena grouped by list
    q = _queries(40, d, n, 31)
    ids, dist, cnt = eng.search(q, 10, 5, tiers=L.TIER_HISTORICAL)
    o = O.hybrid_batch_search(new_ivf, None, None, q, 10, 5, tiers=2, deleted=O.make_bitmap(n, dead))
    _assert_same(ids, dist, cnt, *o)
    # errors of the reference: fewer rows than clusters (the inner train fails, core.rs:250-255)
    from fabstir_vectordb_b200 import InsufficientTrainingData
    with pytest.raises(InsufficientTrainingData):
        eng.retrain(n + 1, 3)
    assert eng.stats().ivf_rows == n and eng.stats().trained == 1   # nothing was touched


@pytest.mark.gpu
def test_mirror_maintenance_operations():
    """IVFIndex.retrain / add_clusters / optimize_clusters / get_cluster_stats / balance_clusters of
    the host mirror (src/ivf/operations.rs:147-288, 422-492) on top of the device retrain."""
    from fabstir_vectordb_b200 import IVFConfig, IVFIndex, InvalidParameter, NotTrained
    n, d = 3000, 32
    x = _data(n, d, 7, n_comp=8)
    idx = IVFIndex(IVFConfig(n_clusters=8, n_probe=4, max_iterations=5, seed=3))
    with pytest.raises(NotTrained):
        idx.add_clusters(2)
    idx.train(x[:500])
    idx.batch_insert([f"v{i}" for i in range(n)], x)
    idx.mark_deleted("v5")
    st0 = idx.get_cluster_stats()
    assert st0.n_clusters == 8 and st0.total_vectors == n and abs(st0.avg_cluster_size - n / 8) < 1e-3
    rr = idx.retrain(IVFConfig(n_clusters=16, n_probe=4, max_iterations=5, seed=9))
    assert (rr.old_clusters, rr.new_clusters, rr.vectors_reassigned) == (8, 16, n)
    assert idx.total_vectors() == n and idx.is_deleted("v5") and sum(idx.get_cluster_sizes().values()) == n
    # every vector sits in the list of its nearest centroid (insert, src/ivf/core.rs:431-455)
    cents = idx.get_centroids()
    want = O.assign(x, cents)
    assert [idx._lists[f"v{i}"] for i in range(n)] == want.tolist()
    ar = idx.add_clusters(4)
    assert ar.clusters_added == 4 and ar.vectors_reassigned == n and idx.config.n_clusters == 20
    with pytest.raises(InvalidParameter):
        idx.add_clusters(0)
    opt = idx.optimize_clusters()
    assert opt.iterations >= 1 and opt.improvement >= 0.0 and idx.get_cluster_stats().total_vectors == n
    with pytest.raises(InvalidParameter):
        idx.balance_clusters(1.5)
    assert idx.balance_clusters(0.2).vectors_moved == 0
    res = idx.search(x[17], 3)
    assert res[0].vector_id == "v17" and res[0].distance < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_concurrent_single_query_calls_are_coalesced(mode):
    """Many OS threads calling fvdb_search with one query each (the reference's usage: `&self`
    searches behind an RwLock, one query per call): the submission queue runs queued calls as one
    device batch; every caller gets exactly the result of its own separate call (= the oracle's)."""
    import threading
    n, d, nlist, nprobe, k = 4000, 384, 32, 8, 10
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 41, mode)
    n_threads, per = 12, 25
    q = _queries(n_threads * per, d, n, 41)
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    got = [None] * (n_threads * per)
    seen_batch = []
    errors = []

    def worker(t):
        try:
            for j in range(per):
                i = t * per + j
                got[i] = eng.search(q[i], k, nprobe, tiers=L.TIER_HISTORICAL)
                if j % 8 == 0:
                    seen_batch.append(eng.stats().last_batch_calls)
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(n_threads)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    ids = np.concatenate([g[0] for g in got])
    dist = np.concatenate([g[1] for g in got])
    cnt = np.concatenate([g[2] for g in got])
    _assert_same(ids, dist, cnt, *want)
    assert max(seen_batch) >= 1
    # a bad call must not fail the calls it is batched with, and sees its own error
    from fabstir_vectordb_b200 import NanInput
    bad = q[0].copy()
    bad[3] = np.nan
    res = {}

    def good_call():
        res["good"] = eng.search(q[1], k, nprobe, tiers=L.TIER_HISTORICAL)

    def bad_call():
        try:
            eng.search(bad, k, nprobe, tiers=L.TIER_HISTORICAL)
            res["bad"] = "no error"
        except NanInput:
            res["bad"] = "nan"

    ts = [threading.Thread(target=f) for f in (good_call, bad_call, good_call)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert res["bad"] == "nan"
    assert np.array_equal(res["good"][0], got[1][0]) and np.array_equal(res["good"][1].view(np.uint32), got[1][1].view(np.uint32))
    # serialised mode gives the same bits
    eng.set_option(L.OPT_COALESCE, 0)
    one = eng.search(q[2], k, nprobe, tiers=L.TIER_HISTORICAL)
    assert np.array_equal(one[0], got[2][0]) and eng.stats().last_batch_calls == 1


def test_load_chunk_bulk_path():
    """SURVEY §8f rows 1-2: a stored VectorChunk (CBOR) goes through ONE decode and ONE assignment launch;
    list membership and searches equal the oracle's per-vector `find_cluster` + insert
    (src/hybrid/persistence.rs:626-653)."""
    from fabstir_vectordb_b200 import IVFConfig, IVFIndex, encode_vector_chunk
    rng = np.random.default_rng(21)
    n, d, nlist = 3000, 64, 16
    x = rng.standard_normal((n, d)).astype(np.float32)
    x[rng.random((n, d)) < 0.05] = 0.5           # some half-float-exact values in the chunk
    cents = x[rng.choice(n, nlist, replace=False)].copy()
    ids = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    idx = IVFIndex(IVFConfig(n_clusters=nlist, n_probe=4))
    idx.set_trained(cents, d)
    added = 0
    for c0 in range(0, n, 1000):                 # three chunks
        added += idx.load_chunk(encode_vector_chunk(f"chunk-{c0 // 1000}", c0, c0 + 999, ids[c0:c0 + 1000], x[c0:c0 + 1000]))
    assert added == n and idx.total_vectors() == n
    want_lists = O.assign(x, cents)
    got = np.array([idx._lists[bytes(b)] for b in ids])
    assert np.array_equal(got, want_lists)
    o = O.IVF(cents, x)                         # oracle ids = row numbers
    q = x[:16] + np.float32(0.01)
    for i in range(16):
        want_ids, want_dist = o.search(q[i], 5, 4)
        res = idx.search_with_config(q[i], 5, 4)
        assert [r.vector_id for r in res] == [bytes(ids[j]) for j in want_ids]
        assert np.array_equal(np.array([r.distance for r in res], np.float32).view(np.uint32),
                              np.asarray(want_dist, np.float32).view(np.uint32))


@pytest.mark.parametrize("nlist", [2048, 4096])
def test_coarse_selection_with_clumped_centroid_ids(nlist):
    """Centroids whose ids share a residue mod 128 are near-duplicates of one another (what a k-means
    initialised from clumped seeds leaves behind): all of a query's nearest centroids then sit in ONE
    thread's share of the coarse selection.  The kernel must notice and re-select exactly: same
    results as the oracle, and the queries are NOT handed to the exact fallback path wholesale (before
    the in-kernel re-selection every one of them was)."""
    rng = np.random.default_rng(nlist)
    d, n, nprobe, k, nq = 64, 20000, 16, 10, 96

    def unit(a):
        return (a / np.linalg.norm(a, axis=1, keepdims=True)).astype(np.float32)

    seeds = unit(rng.standard_normal((128, d)))
    cents = unit(seeds[np.arange(nlist) % 128] + 0.01 * rng.standard_normal((nlist, d)))
    x = unit(cents[rng.integers(0, nlist, n)] + 0.05 * rng.standard_normal((n, d)))
    q = unit(seeds[rng.integers(0, 128, nq)] + 0.02 * rng.standard_normal((nq, d)))
    eng = Engine(d, k_max=32)
    _set_mode(eng, "tc")
    eng.set_centroids(cents)
    eng.ivf_add(x, np.arange(n, dtype=np.uint32))
    ivf = O.IVF(cents, x)
    ids, dist, cnt = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL)
    o = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    _assert_same(ids, dist, cnt, *o)
    assert eng.stats().last_fallback_queries < nq // 2


@pytest.mark.parametrize("kernel", ["R", "W", "hybrid"])
def test_hub_list_is_split_into_row_ranges(kernel, monkeypatch):
    """A hub posting list (thousands of rows, probed by every query) is cut into row ranges with one work
    item and one shortlist slot each (DESIGN §3.1).  Results — with tombstones and a filter bitmap on —
    must equal the oracle's bit for bit: with kernel R alone, with kernel W alone (every list goes to the
    wide-tile kernel) and with the product's split (the hub list to kernel W, the others to kernel R)."""
    if kernel != "hybrid":
        monkeypatch.setenv("FVDB_TC_KERNEL", kernel)
    rng = np.random.default_rng(77)
    d, nlist, nq, k, nprobe = 128, 12, 150, 10, 6
    cents = rng.standard_normal((nlist, d)).astype(np.float32)
    # list 0 is the hub: 7000 of the 10000 rows sit around its centroid; all queries come from there
    owner = np.concatenate([np.zeros(7000, np.int64), rng.integers(1, nlist, 3000)])
    rng.shuffle(owner)
    x = (cents[owner] + np.float32(0.4) * rng.standard_normal((len(owner), d))).astype(np.float32)
    q = (cents[0] + np.float32(0.5) * rng.standard_normal((nq, d))).astype(np.float32)
    n = len(x)
    eng = Engine(d, k_max=32)
    _set_mode(eng, "tc")
    eng.set_centroids(cents)
    ids = np.arange(n, dtype=np.uint32)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    assert max(ivf.list_len(l) for l in range(nlist)) > 4096       # long enough to be split
    dele = np.arange(3, n, 41, dtype=np.uint32)
    eng.set_deleted(dele, True)
    fbits = O.make_bitmap(n, np.arange(0, n, 2, dtype=np.uint32))   # every other row passes the filter
    got = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL, filter_bits=fbits)
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2, deleted=O.make_bitmap(n, dele),
                                 filter_bits=fbits)
    _assert_same(*got, *want)
    got = eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL)
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2, deleted=O.make_bitmap(n, dele))
    _assert_same(*got, *want)


@pytest.mark.parametrize("mode", MODES)
def test_stream_ordered_submit_finish(mode):
    """fvdb_search_device_submit x N + one fvdb_search_device_finish == N synchronous calls: same bits as the
    oracle, including queries whose tensor-core proof fails (near-duplicate neighbourhoods: repaired on the
    exact path at finish time) and a NaN batch (reported by finish)."""
    import torch
    from fabstir_vectordb_b200 import NanInput
    d, n, nlist, nq, k, nprobe = 128, 9000, 24, 80, 10, 6
    rng = np.random.default_rng(5)
    x = _data(n, d, 91)
    # 120 near-copies of row 0 (1e-4 apart): the 32 best approximate distances of a query there are
    # indistinguishable in TF32, so the proof must fail and the exact path must answer
    x[1:121] = x[0] + np.float32(1e-4) * rng.standard_normal((120, d)).astype(np.float32)
    cents = x[rng.choice(n, nlist, replace=False)].copy()
    eng = Engine(d, k_max=32)
    _set_mode(eng, mode)
    eng.set_centroids(cents)
    ids = np.arange(n, dtype=np.uint32)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    qs = [_queries(nq, d, n, 100 + i) for i in range(3)]
    qs[1][:7] = x[0] + np.float32(1e-4) * rng.standard_normal((7, d)).astype(np.float32)
    dq = [torch.from_numpy(q).cuda() for q in qs]
    outs = [(torch.empty((nq, k), dtype=torch.int32, device="cuda"), torch.empty((nq, k), dtype=torch.float32, device="cuda"),
             torch.empty((nq,), dtype=torch.int32, device="cuda")) for _ in qs]
    for q_, o_ in zip(dq, outs):
        eng.search_device_submit(q_.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0,
                                 o_[0].data_ptr(), o_[1].data_ptr(), o_[2].data_ptr())
    eng.search_device_finish()
    if mode == "tc":
        assert eng.stats().last_fallback_queries >= 7
    for q_, o_ in zip(qs, outs):
        want = O.hybrid_batch_search(ivf, None, None, q_, k, nprobe, tiers=2)
        _assert_same(o_[0].cpu().numpy().view(np.uint32), o_[1].cpu().numpy(), o_[2].cpu().numpy().view(np.uint32), *want)
    # a NaN batch between two good ones: finish reports it, later calls work again
    bad = dq[0].clone()
    bad[3, 5] = float("nan")
    eng.search_device_submit(dq[2].data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0,
                             outs[2][0].data_ptr(), outs[2][1].data_ptr(), outs[2][2].data_ptr())
    eng.search_device_submit(bad.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0,
                             outs[0][0].data_ptr(), outs[0][1].data_ptr(), outs[0][2].data_ptr())
    with pytest.raises(NanInput):
        eng.search_device_finish()
    eng.search_device_submit(dq[0].data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0,
                             outs[0][0].data_ptr(), outs[0][1].data_ptr(), outs[0][2].data_ptr())
    eng.search_device_finish()
    want = O.hybrid_batch_search(ivf, None, None, qs[0], k, nprobe, tiers=2)
    _assert_same(outs[0][0].cpu().numpy().view(np.uint32), outs[0][1].cpu().numpy(), outs[0][2].cpu().numpy().view(np.uint32), *want)
    eng.close()


@pytest.mark.parametrize("mode", MODES)
def test_host_buffer_submit_finish(mode):
    """fvdb_search_submit x N + fvdb_search_finish with page-locked buffers == N fvdb_search calls (the upload of
    a batch overlaps the scan of the one before); pageable buffers are refused."""
    from fabstir_vectordb_b200 import FvdbError, PinnedArray
    d, n, nlist, nq, k, nprobe = 128, 8000, 20, 64, 10, 5
    eng, ivf, x, cents, _, _ = _build(n, d, nlist, 61, mode)
    qs = [_queries(nq, d, n, 200 + i) for i in range(6)]
    pq = [PinnedArray((nq, d), np.float32) for _ in qs]
    po = [(PinnedArray((nq, k), np.uint32), PinnedArray((nq, k), np.float32), PinnedArray((nq,), np.uint32)) for _ in qs]
    for a, q_ in zip(pq, qs):
        a.array[...] = q_
    for rnd in range(2):          # two rounds: the slots and their device buffers are reused
        for i in range(3 * rnd, 3 * rnd + 3):
            eng.search_submit(pq[i].array, k, nprobe, L.TIER_HISTORICAL, tuple(b.array for b in po[i]))
        eng.search_finish()
    for i, q_ in enumerate(qs):
        want = O.hybrid_batch_search(ivf, None, None, q_, k, nprobe, tiers=2)
        _assert_same(po[i][0].array, po[i][1].array, po[i][2].array, *want)
    with pytest.raises(FvdbError):
        eng.search_submit(qs[0], k, nprobe, L.TIER_HISTORICAL, tuple(b.array for b in po[0]))   # pageable queries
    eng.search_finish()           # nothing pending: a no-op
    eng.close()


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("metric", ["cos", "dot"])
@pytest.mark.parametrize("d,n,nq", [(384, 12000, 300), (64, 9000, 70), (30, 2000, 9)])
def test_cosine_and_dot_metrics(mode, metric, d, n, nq):
    """FVDB_METRIC_COS / FVDB_METRIC_DOT (src/core/vector_ops.rs:35-49, ranked as top_k_indices does :12-23):
    a similarity handle scores the flat tier exhaustively; ids and similarity BITS equal the oracle's
    batch scoring + stable descending sort, in the exact mode and through kernel W + exact re-rank."""
    if mode == "tc" and d % 32:
        pytest.skip("tc needs dim % 32 == 0")
    m = L.METRIC_COS if metric == "cos" else L.METRIC_DOT
    om = O.COSINE if metric == "cos" else O.DOT
    rng = np.random.default_rng(d + n)
    x = _data(n, d, 41, n_comp=24, sigma=0.7) * rng.uniform(0.2, 3.0, size=(n, 1)).astype(np.float32)   # unequal norms
    x[17] = 0.0                                                                                          # a zero row scores 0
    x[n - 5] = x[11]                                                                                     # an exact tie: lower id first
    q = _queries(nq, d, n, 41, n_comp=24, sigma=0.7) * rng.uniform(0.5, 2.0, size=(nq, 1)).astype(np.float32)
    q[3] = 0.0                                                                                           # a zero query: every cosine is 0
    ids = np.arange(n, dtype=np.uint32)
    eng = Engine(d, k_max=16, metric=m)
    _set_mode(eng, mode)
    eng.flat_add(x, ids)
    dele = np.arange(5, n, 61, dtype=np.uint32)
    eng.set_deleted(dele, True)
    got = eng.search(q, 10, 0, tiers=L.TIER_RECENT)
    want = O.flat_search_metric(x, ids, q, 10, om, deleted=O.make_bitmap(n, dele))
    assert got[2].tolist() == want[2].tolist()
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    if mode == "tc" and d == 384:
        assert eng.stats().last_fallback_queries <= max(2, nq // 16)   # kernel W carries it (the zero query falls back)
    # with a filter bitmap; fewer than k live rows
    fb = O.make_bitmap(n, np.arange(0, n, 7))
    got = eng.search(q[:20], 10, 0, tiers=L.TIER_RECENT, filter_bits=fb)
    want = O.flat_search_metric(x, ids, q[:20], 10, om, deleted=O.make_bitmap(n, dele), filter_bits=fb)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    few = O.make_bitmap(n, [1, 2, 3])
    got = eng.search(q[:4], 10, 0, tiers=L.TIER_RECENT, filter_bits=few)
    assert got[2].tolist() == [3] * 4
    # the IVF tier is L2 only, as in the reference
    from fabstir_vectordb_b200 import InvalidConfig
    with pytest.raises(InvalidConfig):
        eng.set_centroids(x[:8])


def test_near_duplicate_neighbourhood_falls_back_and_still_matches():
    """The adversarial case for the tensor-core proof: 60 rows within 1e-4 of one another sit exactly where the
    k-th neighbour is, so the 32-entry approximate shortlist cannot be proven to contain the exact top-k (the TF32
    bound is wider than their gaps).  Such queries MUST take the exact fallback — and the result must still be
    the oracle's, bit for bit, with ties in id order."""
    d, n, nlist = 384, 6000, 8
    rng = np.random.default_rng(7)
    x = _data(n, d, 91, n_comp=8, sigma=0.6)
    base = x[100].copy()
    for j in range(60):                       # a shell of near-duplicates around one row (some exact copies)
        x[200 + j] = base if j % 3 == 0 else base + (1e-4 * rng.standard_normal(d)).astype(np.float32)
    cents = x[rng.choice(n, nlist, replace=False)].copy()
    ids = np.arange(n, dtype=np.uint32)
    eng = Engine(d, k_max=64)
    _set_mode(eng, "tc")
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    q = np.stack([base + (0.05 * rng.standard_normal(d)).astype(np.float32) for _ in range(24)] +
                 [x[i] + np.float32(0.01) for i in range(1000, 1040)])
    got = eng.search(q, 10, nlist, tiers=L.TIER_HISTORICAL)
    fb = eng.stats().last_fallback_queries
    _assert_same(*got, *O.hybrid_batch_search(ivf, None, None, q, 10, nlist, tiers=2))
    assert fb >= 12, f"the queries inside the duplicate shell must fail the proof (fell back: {fb})"
    assert fb < len(q), "the ordinary queries must not"
    # the same batch through the stream-ordered entry: repaired at finish time
    import torch
    dq = torch.from_numpy(q).cuda()
    o = (torch.empty((len(q), 10), dtype=torch.int32, device="cuda"), torch.empty((len(q), 10), dtype=torch.float32, device="cuda"),
         torch.empty((len(q),), dtype=torch.int32, device="cuda"))
    s = torch.cuda.current_stream().cuda_stream
    eng.search_device_submit(dq.data_ptr(), len(q), 10, nlist, L.TIER_HISTORICAL, 0, 0, o[0].data_ptr(), o[1].data_ptr(),
                             o[2].data_ptr(), s)
    eng.search_device_finish(s)
    want = O.hybrid_batch_search(ivf, None, None, q, 10, nlist, tiers=2)
    assert np.array_equal(o[0].cpu().numpy().view(np.uint32), want[0])
    assert np.array_equal(o[1].cpu().numpy().view(np.uint32), want[1].view(np.uint32))


def test_two_slot_pipeline_many_batches_and_mutation_between_groups():
    """The stream-ordered entries run consecutive batches in two pipeline slots (own stream, own scratch).  Twelve
    batches in flight, each against the oracle; rows added and tombstoned BETWEEN groups must be seen by the next
    group (every other entry point drains the slots first); FVDB_OPT_PIPELINE = 0 gives the same bits."""
    import torch
    d, n, nlist, nq, k, nprobe = 384, 30000, 48, 200, 10, 8
    x = _data(n + 4000, d, 77, n_comp=64, sigma=0.8)
    cents = x[np.random.default_rng(3).choice(n, nlist, replace=False)].copy()
    ids = np.arange(n + 4000, dtype=np.uint32)
    eng = Engine(d, k_max=16)
    _set_mode(eng, "tc")
    eng.set_centroids(cents)
    eng.ivf_add(x[:n], ids[:n])
    qs = [_queries(nq, d, n, 300 + i, n_comp=64, sigma=0.8) for i in range(12)]
    dq = [torch.from_numpy(q).cuda() for q in qs]
    outs = [(torch.empty((nq, k), dtype=torch.int32, device="cuda"), torch.empty((nq, k), dtype=torch.float32, device="cuda"),
             torch.empty((nq,), dtype=torch.int32, device="cuda")) for _ in qs]
    s = torch.cuda.current_stream().cuda_stream

    def run_group():
        for q_, o_ in zip(dq, outs):
            eng.search_device_submit(q_.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0,
                                     o_[0].data_ptr(), o_[1].data_ptr(), o_[2].data_ptr(), s)
        eng.search_device_finish(s)
        return [tuple(t.cpu().numpy() for t in o_) for o_ in outs]

    def check(res, ivf, deleted=None):
        for q_, (i_, d_, c_) in zip(qs, res):
            want = O.hybrid_batch_search(ivf, None, None, q_, k, nprobe, tiers=2, deleted=deleted)
            _assert_same(i_.view(np.uint32), d_, c_.view(np.uint32), *want)

    piped = run_group()
    check(piped, O.IVF(cents, x[:n], ids[:n]))
    assert eng.stats().last_fallback_queries <= 3
    # mutate between groups: more rows, some tombstones
    eng.ivf_add(x[n:], ids[n:])
    dele = np.arange(3, n + 4000, 53, dtype=np.uint32)
    eng.set_deleted(dele, True)
    check(run_group(), O.IVF(cents, x, ids), deleted=O.make_bitmap(n + 4000, dele))
    # pipeline off: the same bits
    on = run_group()
    eng.set_option(6, 0)     # FVDB_OPT_PIPELINE
    off = run_group()
    for a, b in zip(on, off):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32)) and np.array_equal(a[2], b[2])
    eng.close()
