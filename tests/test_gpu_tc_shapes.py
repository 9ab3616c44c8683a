"""The tensor-core search at every shape class it dispatches on, against the CPU oracle.

Every dimension class of the scan kernels (k-blocks per stage of kernel W, the shared-memory ring of
kernel R, kernel R alone above D = 384), the k and nprobe limits of the tensor-core path, ragged query
groups, posting lists of 1 / 127 / 128 / 129 / > 2048 rows, the flat tier, bulk assignment and
candidate floods.  Results must equal the oracle's bit for bit (ids and distance bits).

The exact re-rank and the proof hide part of a broken scan: a query whose proof fails is re-run on the
exact path, so its result is right whatever the scan did.  `_run_tc` therefore bounds the number of
such queries and checks, from the kernels the search launched, that the tensor-core kernels ran.
(`fvdb_stats.last_launches` cannot tell the two paths apart: above D = 384, and with the tensor-core
coarse step below it, the tensor-core search and the exact one launch the same number of kernels.)"""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, FvdbError, _lib as L, synth

pytestmark = pytest.mark.gpu

# tc_supported: D % 32 == 0, 32 <= D <= 512.  KB = D / 32 k-blocks: 1 (one block per kernel W stage),
# 3, 5, 7, 11 (primes: one block per stage), 8, 9, 12 and the kernel-R-only class 13..16
DIMS = [32, 96, 160, 224, 256, 288, 352, 384, 416, 448, 480, 512]
W_MAX_D = 384            # kernel W and the tensor-core coarse step need the query tile in tensor memory
TC_MAX_K = 16
TC_MAX_NPROBE = 256
TC_MAX_NPROBE_COARSE = 112

K_R = "tc_scan_kernel"          # kernel R (rows on lanes)
K_W = "tc_scan_wide_kernel"     # kernel W (wide query tiles on CTA pairs)
K_Q = "tc_scan_q_kernel"        # kernel Q: the tensor-core coarse step
TC_KERNELS = (K_R, K_W, K_Q, "rerank_kernel")


def _assert_same(ids, dist, cnt, o_ids, o_dist, o_cnt):
    assert cnt.tolist() == o_cnt.tolist()
    for i in range(len(cnt)):
        c = int(cnt[i])
        assert ids[i, :c].tolist() == o_ids[i, :c].tolist(), f"query {i}"
        assert dist[i, :c].view(np.uint32).tolist() == o_dist[i, :c].view(np.uint32).tolist(), f"query {i}"


def _assert_identical(a, b):
    assert np.array_equal(a[2], b[2])
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


def _profiled(run):
    """run() and the names of the CUDA kernels it launched (in this process, whoever launched them)."""
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
    return any(kernel in n for n in names)     # no kernel name is a part of another one


def _run_tc(eng, run, nq, expect, absent=(), fb_bound=None):
    """Run a search on a tensor-core handle, then once more on the same handle in exact mode.  Asserts
    that the kernels in `expect` ran and those in `absent` did not, that at most `fb_bound` (default
    nq // 16) queries were handed to the exact path by a failed proof, and that the exact run returns
    the same bits without launching any tensor-core kernel.  Returns the tensor-core result."""
    got, names = _profiled(run)
    fb = eng.stats().last_fallback_queries
    for kname in expect:
        assert _ran(names, kname), f"{kname} did not run; kernels: {sorted(names)}"
    for kname in absent:
        assert not _ran(names, kname), f"{kname} ran; kernels: {sorted(names)}"
    bound = nq // 16 if fb_bound is None else fb_bound
    assert fb <= bound, f"{fb} of {nq} queries fell back to the exact path (bound {bound})"
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    try:
        ex, ex_names = _profiled(run)
    finally:
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    assert not any(_ran(ex_names, kn) for kn in TC_KERNELS), sorted(ex_names)
    _assert_identical(got, ex)
    return got


def _run_exact_path(eng, run):
    """A tensor-core handle whose search must take the exact path (shape outside the tensor-core limits)."""
    got, names = _profiled(run)
    assert not any(_ran(names, kn) for kn in TC_KERNELS), sorted(names)
    assert eng.stats().last_fallback_queries == 0
    return got


def _tc_engine(d, k_max=16, metric=L.METRIC_L2):
    eng = Engine(d, k_max=k_max, metric=metric)
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    eng.set_option(L.OPT_KMEANS_TC, 1)
    return eng


# ---- data: lists of chosen lengths around chosen centroids ---------------------------------------
def _lists(d, sizes, nq, seed, near=(), hub=None, n_hub_q=0):
    """Unit-norm centroids; the rows of list l are its centroid plus noise of norm ~0.5 in a 16-dimensional
    subspace of its own, so that the k nearest rows are well separated from the 32nd (the tensor-core proof
    holds for almost every query).  Lists `near` get centroids close to that of list `hub`, and `n_hub_q` of
    the `nq` queries sit around the hub centroid: those queries all probe the hub and the `near` lists, so
    these lists are probed by more than 128 queries of the batch.  Rows are regenerated until each lies
    closest to its own centroid, so list l holds exactly sizes[l] rows.  Returns centroids, rows in a
    shuffled insertion order, and the queries (also shuffled)."""
    rng = np.random.default_rng(seed)
    nlist, r = len(sizes), 16
    cents = rng.standard_normal((nlist, d)) / np.sqrt(d)
    for s in near:
        cents[s] = cents[hub] + 0.6 * rng.standard_normal(d) / np.sqrt(d)
    cents = cents.astype(np.float32)
    basis = rng.standard_normal((nlist, r, d)) / np.sqrt(d)
    sigma = 0.5 / np.sqrt(r)
    c64 = cents.astype(np.float64)
    cn = (c64 * c64).sum(1)
    rows = []
    for l, n in enumerate(sizes):
        got = np.empty((0, d), np.float32)
        while len(got) < n:
            x = (cents[l] + sigma * rng.standard_normal((2 * n + 8, r)) @ basis[l]).astype(np.float32)
            d2 = cn[None, :] - 2.0 * x.astype(np.float64) @ c64.T
            own = np.argsort(d2, axis=1)[:, :2]
            keep = (own[:, 0] == l) & (d2[np.arange(len(x)), own[:, 1]] - d2[:, l] > 1e-3)
            got = np.concatenate([got, x[keep]])
        rows.append(got[:n])
    x = np.concatenate(rows)
    x = x[rng.permutation(len(x))]
    ql = np.concatenate([np.full(n_hub_q, hub if hub is not None else 0), rng.integers(0, nlist, nq - n_hub_q)])
    z = rng.standard_normal((nq, r))
    q = cents[ql] + sigma * np.einsum("qr,qrd->qd", z, basis[ql]) + 0.05 * rng.standard_normal((nq, d)) / np.sqrt(d)
    q = q[rng.permutation(nq)].astype(np.float32)
    return cents, x, q


# list 4 is a hub of 2600 rows (cut into three row ranges), lists 0-3 hold 1, 127, 128 and 129 rows and sit
# next to it; 59 more lists of 40-89 rows
SIZES = [1, 127, 128, 129, 2600] + [40 + (7 * i) % 50 for i in range(59)]
NQ = 300


def _ivf_case(d, seed):
    cents, x, q = _lists(d, SIZES, NQ, seed, near=(0, 1, 2, 3), hub=4, n_hub_q=150)
    ids = (np.arange(len(x), dtype=np.uint32) * 3 + 1).astype(np.uint32)
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    assert [ivf.list_len(l) for l in range(len(SIZES))] == SIZES
    return eng, ivf, ids, q


def _variants(d):
    """(name, environment, kernels that must run, kernels that must not) of the scan-kernel choice."""
    if d > W_MAX_D:
        return [("default", {}, (K_R,), (K_W, K_Q)), ("R", {"FVDB_TC_KERNEL": "R"}, (K_R,), (K_W, K_Q))]
    return [("default", {}, (K_R, K_W, K_Q), ()),       # hub + its neighbours to W, the rest to R
            ("R", {"FVDB_TC_KERNEL": "R"}, (K_R, K_Q), (K_W,)),
            ("W", {"FVDB_TC_WIDE_MIN": "1"}, (K_W, K_Q), ())]


@pytest.mark.parametrize("d", DIMS)
def test_ivf_dimension_sweep(d, monkeypatch):
    k, nprobe = 10, 8
    eng, ivf, ids, q = _ivf_case(d, 1000 + d)
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    filtered = d in (256, 448)      # one dimension of each kernel-selection class
    if filtered:
        dele = ids[5::37].copy()
        fbits = O.make_bitmap(int(ids.max()) + 1, ids[(np.arange(len(ids)) % 3) != 1])
        want_f = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2,
                                       deleted=O.make_bitmap(int(ids.max()) + 1, dele), filter_bits=fbits)
    for name, env, expect, absent in _variants(d):
        for key in ("FVDB_TC_KERNEL", "FVDB_TC_WIDE_MIN"):
            monkeypatch.delenv(key, raising=False)
        for key, val in env.items():
            monkeypatch.setenv(key, val)
        got = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL), NQ, expect, absent)
        _assert_same(*got, *want)
        if filtered:
            eng.set_deleted(dele, True)
            got = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL, filter_bits=fbits), NQ,
                          expect, absent)
            _assert_same(*got, *want_f)
            eng.set_deleted(dele, False)
    eng.close()


@pytest.mark.parametrize("d", [384, 512])
def test_ragged_query_counts(d):
    # query groups of kernel R (64) and work items of kernel W (256) that end ragged; at D = 384 the lists
    # reach 129 probing queries only from nq = 129 on
    k, nprobe = 10, 8
    eng, ivf, ids, q = _ivf_case(d, 2000 + d)
    expect = (K_R,) if d > W_MAX_D else (K_R, K_Q)
    for nq in (63, 64, 65, 128, 129, 255, 256, 257):
        qq = q[:nq]
        got = _run_tc(eng, lambda: eng.search(qq, k, nprobe, tiers=L.TIER_HISTORICAL), nq, expect,
                      fb_bound=max(1, nq // 16))
        _assert_same(*got, *O.hybrid_batch_search(ivf, None, None, qq, k, nprobe, tiers=2))
    eng.close()


@pytest.mark.parametrize("d", [384, 512])
def test_k_and_nprobe_limits(d):
    # nlist > 512, so that nprobe = 513 is not clamped to nlist and is refused
    nlist, nq = 600, 256
    sizes = [6 + (5 * i) % 11 for i in range(nlist)]
    cents, x, q = _lists(d, sizes, nq, 3000 + d)
    ids = np.arange(len(x), dtype=np.uint32)
    eng = _tc_engine(d, k_max=32)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    for nprobe in (112, 113, 256, 257, 512):
        for k in (1, 15, 16, 17):
            run = lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL)   # noqa: E731
            if k <= TC_MAX_K and nprobe <= TC_MAX_NPROBE:
                coarse = d <= W_MAX_D and nprobe <= TC_MAX_NPROBE_COARSE
                # k = 16: the 32-entry shortlist is tightest, the same bound holds
                got = _run_tc(eng, run, nq, (K_R, K_Q) if coarse else (K_R,), () if coarse else (K_Q,))
            else:
                got = _run_exact_path(eng, run)
            _assert_same(*got, *O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2))
    with pytest.raises(FvdbError) as e:
        eng.search(q[:4], 10, 513, tiers=L.TIER_HISTORICAL)
    assert e.value.code == L.ERR_INVALID_ARG
    eng.close()


@pytest.mark.parametrize("d", DIMS)
def test_flat_tier_dimension_sweep(d):
    # flat rows x queries >= 4M: the tensor-core flat scan (kernel W up to D = 384, kernel R alone above);
    # a ragged last tile and a ragged last query group
    n, k = 14_011, 10
    cents, x, q = _lists(d, [n // 8] * 7 + [n - 7 * (n // 8)], NQ, 4000 + d)
    assert len(x) * NQ >= 4 << 20
    ids = (np.arange(n, dtype=np.uint32) * 2 + 3).astype(np.uint32)
    eng = _tc_engine(d)
    eng.flat_add(x, ids)
    run = lambda: eng.search(q, k, 0, tiers=L.TIER_RECENT)   # noqa: E731
    got = _run_tc(eng, run, NQ, (K_W,) if d <= W_MAX_D else (K_R,), (K_R,) if d <= W_MAX_D else (K_W,))
    _assert_same(*got, *O.hybrid_batch_search(None, x, ids, q, k, 0, tiers=1))
    eng.close()


@pytest.mark.parametrize("metric", ["cos", "dot"])
def test_similarity_flat_tier_above_kernel_w_limit_is_exact(metric):
    # cosine / dot scans need kernel W (D <= 384): at D = 416 a tensor-core handle answers on the exact path
    d, n = 416, 14_000
    m, om = (L.METRIC_COS, O.COSINE) if metric == "cos" else (L.METRIC_DOT, O.DOT)
    _, x, q = _lists(d, [n // 4] * 4, NQ, 5000)
    ids = np.arange(n, dtype=np.uint32)
    eng = _tc_engine(d, metric=m)
    eng.flat_add(x, ids)
    got = _run_exact_path(eng, lambda: eng.search(q, 10, 0, tiers=L.TIER_RECENT))
    want = O.flat_search_metric(x, ids, q, 10, om)
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    eng.close()


@pytest.mark.parametrize("d", [32, 160, 512])
def test_bulk_assignment_dimension_classes(d):
    # rows x lists >= 64M and nlist >= 256: the tensor-core nearest-centroid scan (kernel W with one block
    # per stage at D = 32 and 160, kernel R alone at D = 512).  Its fallback rows are counted only inside
    # the handle (not in fvdb_stats), so only the assignments are compared here.
    n, nlist = 65_536, 1024
    x = synth.rows(0, n, d, 512, 0.6, 29 + d)
    cents = x[:: n // nlist][:nlist].copy()
    cents[9] = cents[5]                     # duplicate centroid: the lower id must win
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    got, names = _profiled(lambda: eng.assign(x))
    assert _ran(names, K_W if d <= W_MAX_D else K_R), sorted(names)
    sample = np.arange(0, n, 8)
    assert got[sample].tolist() == O.assign(x[sample], cents).tolist()
    assert 9 not in set(got.tolist())
    assert got[5 * (n // nlist)] == 5
    eng.close()


def _flood_case():
    """{0, 1} rows in D = 128.  20 disjoint query patterns of three ones in dims 64..123; per pattern
    3 exact copies (d2 = 0), 6 rows at d2 = 1 and 6 at d2 = 2, so the 10 nearest rows of a query hold tie
    groups that cross the k-th position.  5000 background rows with two ones in dims 0..5 (15 patterns)
    sit at d2 = 5 from every query: a tile passes up to 128 candidates per query at one distance until the
    bound settles, and the 33rd nearest is still 3 above the 10th, so the proof holds."""
    rng = np.random.default_rng(17)
    d = 128
    near = []
    pats = [np.arange(64 + 3 * j, 67 + 3 * j) for j in range(20)]
    for p in pats:
        base = np.zeros(d, np.float32)
        base[p] = 1
        near += [base] * 3
        for e in (124, 125, 126):                      # one extra one: d2 = 1
            v = base.copy(); v[e] = 1; near.append(v)
        for b in p:                                    # one missing one: d2 = 1
            v = base.copy(); v[b] = 0; near.append(v)
        for b in p:                                    # one moved one: d2 = 2
            for e in (126, 127):
                v = base.copy(); v[b] = 0; v[e] = 1; near.append(v)
    bg = np.zeros((5000, d), np.float32)
    pairs = [(a, b) for a in range(6) for b in range(a + 1, 6)]
    for i in range(len(bg)):
        bg[i, list(pairs[rng.integers(len(pairs))])] = 1
    x = np.concatenate([np.stack(near), bg])
    order = rng.permutation(len(x))
    x = x[order]
    ids = rng.permutation(len(x)).astype(np.uint32)       # tie order by id is not insertion order
    q = np.zeros((NQ, d), np.float32)
    for i in range(NQ):
        q[i, pats[i % 20]] = 1
    cents = x[rng.choice(len(x), 6, replace=False)].copy()
    cents += np.float32(0.01) * rng.standard_normal(cents.shape).astype(np.float32)
    return d, x, ids, q, cents


@pytest.mark.parametrize("kernel", ["R", "W"])
def test_candidate_floods(kernel, monkeypatch):
    monkeypatch.setenv(*(("FVDB_TC_KERNEL", "R") if kernel == "R" else ("FVDB_TC_WIDE_MIN", "1")))
    d, x, ids, q, cents = _flood_case()
    k = 10
    eng = _tc_engine(d)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    ivf = O.IVF(cents, x, ids)
    nprobe = len(cents)                                   # every list: the near rows may sit in any of them
    want = O.hybrid_batch_search(ivf, None, None, q, k, nprobe, tiers=2)
    assert (want[1][:, 0] == 0.0).all() and (want[1][:, 9] == np.float32(np.sqrt(2.0))).all()
    # binary operands are exact in TF32, so no tie group is split by rounding and every proof holds
    got = _run_tc(eng, lambda: eng.search(q, k, nprobe, tiers=L.TIER_HISTORICAL), NQ,
                  (K_R,) if kernel == "R" else (K_W,), (K_W,) if kernel == "R" else ())
    _assert_same(*got, *want)
    # the same rows in the flat tier
    eng2 = _tc_engine(d)
    xf = np.concatenate([x] * 3)
    idf = np.arange(len(xf), dtype=np.uint32)[::-1].copy()
    eng2.flat_add(xf, idf)
    wantf = O.hybrid_batch_search(None, xf, idf, q, k, 0, tiers=1)
    got = _run_tc(eng2, lambda: eng2.search(q, k, 0, tiers=L.TIER_RECENT), NQ, (K_R,) if kernel == "R" else (K_W,))
    _assert_same(*got, *wantf)
    eng.close()
    eng2.close()
