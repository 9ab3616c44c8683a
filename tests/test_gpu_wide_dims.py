"""The tensor-core search at widths above 512 (544 .. 2048), against the CPU oracle.

Above D = 512 kernel R alone scans, with items of 32 queries up to D = 1024 and of 16 queries above (the query
tile of an item stays resident in shared memory), and the re-rank's proof bound grows with D.  Kernel W and the
tensor-core coarse step stay at D <= 384.  Every case compares with the oracle bit for bit (ids and distance
bits), runs again in exact mode on the same handle with identical bits, reads the launched kernels with
`torch.profiler` to check that kernel R ran and kernels W / Q did not, and bounds the queries whose proof failed
(nq / 16 unless the case is built to make them fail)."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, FvdbError, _lib as L, synth
from fabstir_vectordb_b200.shard import owner_of_list, pack_layout

pytestmark = pytest.mark.gpu

# the first and last width of each item class (32 queries: 544..1024, 16 queries: 1056..2048) and two model widths
DIMS = [544, 768, 1024, 1056, 1536, 2048]
K_R = "tc_scan_kernel"          # kernel R (rows on lanes)
K_W = "tc_scan_wide_kernel"     # kernel W: D <= 384 only
K_Q = "tc_scan_q_kernel"        # the tensor-core coarse step: D <= 384 only
TC_KERNELS = (K_R, K_W, K_Q, "rerank_kernel")


def _assert_same(got, want, k=None, what=""):
    """got == want bit for bit; `want` may come from a larger k (the oracle's (distance, id) order is total, so
    its first k entries are the top-k)."""
    ids, dist, cnt = got
    w_ids, w_dist, w_cnt = want
    k = ids.shape[1] if k is None else k
    w_cnt = np.minimum(w_cnt[:len(cnt)], k)
    assert cnt.tolist() == w_cnt.tolist(), f"{what}: counts"
    for i in range(len(cnt)):
        c = int(cnt[i])
        assert ids[i, :c].tolist() == w_ids[i, :c].tolist(), f"{what}: ids of query {i}"
        assert dist[i, :c].view(np.uint32).tolist() == w_dist[i, :c].view(np.uint32).tolist(), f"{what}: query {i}"


def _profiled(run):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run()
        torch.cuda.synchronize()
    names = {e.key for e in prof.key_averages()}
    assert any("_kernel" in n for n in names), f"the profiler recorded no kernel of the library: {sorted(names)}"
    return out, names


def _ran(names, kernel):
    return any(kernel in n for n in names)


def _run_tc(eng, run, nq, fb_bound=None):
    """A search on a tensor-core handle: kernel R ran, kernels W and Q did not, at most `fb_bound` (default
    max(1, nq // 16)) queries failed their proof; then the same search in exact mode launches no tensor-core
    kernel and returns the same bits.  Returns (result, fallback queries)."""
    got, names = _profiled(run)
    fb = eng.stats().last_fallback_queries
    assert _ran(names, K_R), f"kernel R did not run; kernels: {sorted(names)}"
    assert not _ran(names, K_W) and not _ran(names, K_Q), sorted(names)
    bound = max(1, nq // 16) if fb_bound is None else fb_bound
    assert fb <= bound, f"{fb} of {nq} queries fell back to the exact path (bound {bound})"
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    try:
        ex, ex_names = _profiled(run)
    finally:
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    assert not any(_ran(ex_names, kn) for kn in TC_KERNELS), sorted(ex_names)
    assert np.array_equal(got[2], ex[2]) and np.array_equal(got[0], ex[0])
    assert np.array_equal(got[1].view(np.uint32), ex[1].view(np.uint32))
    return got, fb


def _lists(d, sizes, nq, seed, hub, n_hub_q):
    """Unit-norm centroids; the rows of list l are its centroid plus noise of norm ~0.5 in a 16-dimensional
    subspace of its own, regenerated until each row lies closest to its own centroid (list l holds exactly
    sizes[l] rows).  Lists 0-3 sit next to list `hub`; `n_hub_q` of the queries sit around the hub centroid, so
    the hub and its neighbours are probed by several items' worth of queries.  Returns centroids, rows
    (shuffled) and queries (shuffled)."""
    rng = np.random.default_rng(seed)
    nlist, r = len(sizes), 16
    cents = rng.standard_normal((nlist, d)) / np.sqrt(d)
    for s in range(4):
        cents[s] = cents[hub] + 0.6 * rng.standard_normal(d) / np.sqrt(d)
    cents = cents.astype(np.float32)
    basis = rng.standard_normal((nlist, r, d)).astype(np.float32) / np.float32(np.sqrt(d))
    sigma = 0.5 / np.sqrt(r)
    c64 = cents.astype(np.float64)
    cn = (c64 * c64).sum(1)
    rows = []
    for l, n in enumerate(sizes):
        got = np.empty((0, d), np.float32)
        while len(got) < n:
            x = (cents[l] + sigma * rng.standard_normal((2 * n + 8, r)).astype(np.float32) @ basis[l]).astype(np.float32)
            d2 = cn[None, :] - 2.0 * x.astype(np.float64) @ c64.T
            own = np.argsort(d2, axis=1)[:, :2]
            keep = (own[:, 0] == l) & (d2[np.arange(len(x)), own[:, 1]] - d2[:, l] > 1e-3)
            got = np.concatenate([got, x[keep]])
        rows.append(got[:n])
    x = np.concatenate(rows)
    x = x[rng.permutation(len(x))]
    ql = np.concatenate([np.full(n_hub_q, hub), rng.integers(0, nlist, nq - n_hub_q)])
    z = rng.standard_normal((nq, r))
    q = cents[ql] + sigma * np.einsum("qr,qrd->qd", z, basis[ql]) + 0.05 * rng.standard_normal((nq, d)) / np.sqrt(d)
    q = q[rng.permutation(nq)].astype(np.float32)
    return cents, x, q


def _tc_engine(d, k_max=16):
    eng = Engine(d, k_max=k_max)
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    eng.set_option(L.OPT_KMEANS_TC, 1)
    return eng


# 260 lists, so that nprobe 256 is not clamped: lists of 1 / 127 / 128 / 129 rows next to a hub of 2600 rows (cut
# into row ranges), 255 more of 20-40 rows.  257 queries, 130 of them around the hub.
SIZES = [1, 127, 128, 129, 2600] + [20 + (7 * i) % 21 for i in range(255)]
NQ = 257


@pytest.mark.parametrize("d", DIMS)
def test_ivf_wide_dimension_sweep(d):
    cents, x, q = _lists(d, SIZES, NQ, 6000 + d, hub=4, n_hub_q=130)
    ids = (np.arange(len(x), dtype=np.uint32) * 3 + 1).astype(np.uint32)
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    assert [ivf.list_len(l) for l in range(len(SIZES))] == SIZES
    for nprobe in (1, 32, 112, 256):
        want = O.hybrid_batch_search(ivf, None, None, q, 16, nprobe, tiers=2)
        for k in (1, 10, 16):
            got, _ = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL), NQ)
            _assert_same(got, want, k, f"nprobe {nprobe} k {k}")
        if nprobe == 32:
            # ragged batches around the 16- and 32-query item edges
            for nq in (1, 15, 16, 17, 31, 33):
                qq = q[:nq]
                got, _ = _run_tc(eng, lambda: eng.search(qq, 10, nprobe, tiers=L.TIER_HISTORICAL), nq)
                _assert_same(got, want, 10, f"nq {nq}")
    # tombstones and a filter bitmap
    k, nprobe = 10, 32
    dele = ids[5::37].copy()
    fbits = O.make_bitmap(int(ids.max()) + 1, ids[(np.arange(len(ids)) % 3) != 1])
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2,
                                 deleted=O.make_bitmap(int(ids.max()) + 1, dele), filter_bits=fbits)
    eng.set_deleted(dele, True)
    got, _ = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL, filter_bits=fbits), NQ)
    _assert_same(got, want, k, "tombstones + filter")
    eng.close()


@pytest.mark.parametrize("d", [768, 2048])
def test_hybrid_and_flat_tier(d):
    # flat rows x queries >= 4M: the tensor-core flat scan (kernel R) in both tiers of a hybrid search
    k, nprobe, nq, n = 10, 8, 300, 14_011
    cents, x, q = _lists(d, SIZES[:64], nq, 7000 + d, hub=4, n_hub_q=100)
    ids = np.arange(len(x), dtype=np.uint32)
    _, xf, _ = _lists(d, [n // 8] * 7 + [n - 7 * (n // 8)], 8, 7100 + d, hub=0, n_hub_q=0)
    xf = xf + np.float32(0.2) * cents[np.arange(n) % 64]      # recent rows near the IVF lists
    idf = (np.arange(n, dtype=np.uint32) * 2 + 1_000_001).astype(np.uint32)
    assert n * nq >= 4 << 20
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    eng.flat_add(xf, idf)
    ivf = O.IVF(cents, x, ids)
    got, _ = _run_tc(eng, lambda: eng.search(q, k, 0, tiers=L.TIER_RECENT), nq)
    _assert_same(got, O.hybrid_batch_search(None, xf, idf, q, k, 0, tiers=1), what="flat tier")
    got, _ = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_BOTH), nq)
    _assert_same(got, O.hybrid_batch_search(ivf, xf, idf, q, k, nprobe, tiers=3), what="hybrid")
    eng.close()


@pytest.mark.parametrize("d", [768, 2048])
def test_bulk_assignment(d):
    # rows x lists >= 64M and nlist >= 256: the tensor-core nearest-centroid scan (kernel R, k = 1, re-rank of 4)
    n, nlist = 65_536, 1024
    x = synth.rows(0, n, d, 512, 0.6, 31 + d)
    cents = x[:: n // nlist][:nlist].copy()
    cents[9] = cents[5]                     # duplicate centroid: the lower id must win
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    got, names = _profiled(lambda: eng.assign(x))
    assert _ran(names, K_R) and not _ran(names, K_W), sorted(names)
    sample = np.arange(0, n, 8)
    assert got[sample].tolist() == O.assign(x[sample], cents).tolist()
    assert 9 not in set(got.tolist())
    assert got[5 * (n // nlist)] == 5
    eng.close()


def test_seeded_training_at_768():
    # IVFIndex::train with a seed on a tensor-core handle: k-means++ and Lloyd whose assignment passes run on
    # kernel R (rows x lists >= 64M) equal the oracle's run bit for bit
    d, n, nlist, seed, iters = 768, 65_536, 1024, 7, 2
    x = synth.rows(0, n, d, nlist, 0.3, 71)
    init, _ = O.kmeanspp_init(x, nlist, seed)
    o_c, _, o_r = O.train_lloyd(x, init, iters)
    eng = _tc_engine(d)
    res, names = _profiled(lambda: eng.train(x, nlist, iters, seed=seed))
    assert _ran(names, K_R), sorted(names)
    assert res["iterations"] == o_r["iterations"]
    assert np.array_equal(eng.get_centroids().view(np.uint32), o_c.view(np.uint32))
    assert np.float32(res["final_error"]).view(np.uint32) == np.float32(o_r["final_error"]).view(np.uint32)
    eng.close()


def test_proof_under_load_at_2048():
    """Rows whose squared norms are 1 + j * 2e-6 and queries of norm ~1e-3: the exact distances of a query's 32
    nearest rows lie within ~6e-5 of one another, inside the relative error term of a 2048-term sum
    (2052 * 2^-24 = 1.2e-4) but outside the 3.1e-5 that bounds a 512-term one.  Every proof must fail and the
    exact path must answer; a bound sized for D = 512 would let proofs pass here."""
    d, n, nq, k = 2048, 6000, 64, 10
    rng = np.random.default_rng(23)
    u = rng.standard_normal((n, d))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    x = (u * np.sqrt(1.0 + 2e-6 * rng.permutation(n))[:, None]).astype(np.float32)
    q = (1e-3 * rng.standard_normal((nq, d)) / np.sqrt(d)).astype(np.float32)
    ids = rng.permutation(n).astype(np.uint32)
    cents = x[rng.choice(n, 8, replace=False)].copy()
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    want = O.hybrid_batch_search(ivf, None, None, q, k, 8, tiers=2)
    got, fb = _run_tc(eng, lambda: eng.search(q, k, 8, tiers=L.TIER_HISTORICAL), nq, fb_bound=nq)
    assert fb == nq, f"only {fb} of {nq} proofs failed"
    _assert_same(got, want, what="flood")
    eng.close()


def test_list_sharded_search_at_1024():
    """The list-sharded driver's steps on one GPU (as tests/test_gpu_shard_parts.py): three handles with the same
    centroids each hold the lists they own, the query-sharded coarse slices are concatenated, every shard scans
    into its packed chunk with the proof floor FVDB_OPT_PROOF_XMAX set to the largest row norm of all shards,
    and the packed merge equals the unsharded oracle."""
    import torch
    d, n, nlist, nq, k, nprobe, world = 1024, 40_000, 64, 70, 10, 8, 3
    x = synth.rows(0, n, d, 4 * nlist, 1.0, 1234)
    q = synth.queries(0, nq, d, n, 4 * nlist, 1.0, 1234, synth.default_qnoise(d, 1.0), 5678)
    a = O.assign(x, x[:: n // nlist][:nlist].copy())
    x[a % 2 == 1] *= np.float32(3.0)                       # unequal row norms across the shards
    cents = x[:: n // nlist][:nlist].copy()
    ivf = O.IVF(cents, x, np.arange(n, dtype=np.uint32))
    dx = torch.from_numpy(x).cuda()
    dids = torch.arange(n, dtype=torch.int32, device="cuda")
    engs = []
    for r in range(world):
        e = _tc_engine(d)
        e.set_centroids(cents)
        e.ivf_add_device(dx.data_ptr(), dids.data_ptr(), n, world, r)
        engs.append(e)
    floor = max(e.ivf_max_sqnorm() for e in engs)
    for e in engs:
        e.set_option(L.OPT_PROOF_XMAX, int(np.float32(floor).view(np.uint32)))
    assert all(owner_of_list(l, world) == l % world for l in range(nlist))

    def sharded():
        dq = torch.from_numpy(q).cuda()
        per = (nq + world - 1) // world
        keys = []
        for r, e in enumerate(engs):
            m = torch.full((per, nprobe), -1, dtype=torch.int64, device="cuda")
            lo = min(nq, r * per)
            if min(nq, lo + per) > lo:
                e.coarse_device(dq[lo:].data_ptr(), min(nq, lo + per) - lo, nprobe, m.data_ptr())
            keys.append(m)
        keys = torch.cat(keys)
        o_i, o_d, o_c, chunk = pack_layout(nq, k)
        packs = torch.empty((world, chunk), dtype=torch.int32, device="cuda")
        for e, p in zip(engs, packs):
            e.search_device_coarse(dq.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0, keys.data_ptr(),
                                   p[o_i:o_d].data_ptr(), p[o_d:o_c].data_ptr(), p[o_c:].data_ptr())
        out = [torch.empty((nq, k), dtype=torch.int32, device="cuda"),
               torch.empty((nq, k), dtype=torch.float32, device="cuda"),
               torch.empty((nq,), dtype=torch.int32, device="cuda")]
        engs[0].merge_topk_packed_device(packs.data_ptr(), world, nq, k, *(t.data_ptr() for t in out))
        torch.cuda.synchronize()
        return (out[0].cpu().numpy().view(np.uint32), out[1].cpu().numpy(), out[2].cpu().numpy().view(np.uint32))

    got, names = _profiled(sharded)
    assert _ran(names, K_R) and not _ran(names, K_W) and not _ran(names, K_Q), sorted(names)
    assert sum(e.stats().last_fallback_queries for e in engs) <= nq // 16
    _assert_same(got, O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2), what="sharded")
    for e in engs:
        e.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    ex = sharded()
    assert np.array_equal(got[0], ex[0]) and np.array_equal(got[1].view(np.uint32), ex[1].view(np.uint32))
    for e in engs:
        e.close()


@pytest.mark.parametrize("d,tc", [(2048, True), (2080, False), (560, False)])
def test_width_limits(d, tc):
    # a new handle defaults to the tensor-core scan exactly where it can serve the width
    n, nq, k, nprobe = 3000, 40, 10, 4
    rng = np.random.default_rng(d)
    x = rng.standard_normal((n, d)).astype(np.float32)
    q = (x[:nq] + 0.1 * rng.standard_normal((nq, d))).astype(np.float32)
    cents = x[:: n // 16][:16].copy()
    eng = Engine(d, k_max=16)
    eng.set_centroids(cents)
    eng.ivf_add(x, np.arange(n, dtype=np.uint32))
    got, names = _profiled(lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL))
    assert _ran(names, K_R) == tc, sorted(names)
    ivf = O.IVF(cents, x, np.arange(n, dtype=np.uint32))
    _assert_same(got, O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2), what=f"d {d}")
    if not tc:
        with pytest.raises(FvdbError) as e:
            eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
        assert e.value.code == L.ERR_INVALID_CONFIG
    eng.close()
