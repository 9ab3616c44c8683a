"""Sharded HYBRID search (FVDB_TIER_BOTH over a list-sharded IVF tier and recent-tier slabs) tested on ONE GPU:
W Engine handles on device 0 act as the W shards and the test performs the driver's collective steps itself
(concatenate the coarse-key slices, stack the per-rank fvdb_search_device_tiers chunks), as
test_gpu_shard_parts.py does for the IVF tier.  Every sharded result is compared bit for bit (ids, distance
bits, counts) with the CPU oracle's unsharded HybridIndex::search.

Covered: fvdb_merge_topk_tiers_packed_device against merge_tiers_reference; fvdb_search_device_tiers against
the one-tier and both-tier results of the existing entry on one handle (exact and tensor-core, tombstones, a
filter, a recent tier below and above the tensor-core threshold); the sharded hybrid search with cross-tier,
cross-rank distance ties; delete / vacuum / migrate; the pipelined _tiers_submit entry including the deferred
exact repair; the sharded 3x post-filter."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, FvdbError, _lib as L, synth
from fabstir_vectordb_b200.shard import (ShardedIndex, merge_tiers_reference, owner_of_list, owner_of_recent_row,
                                         place_lists, tiers_pack_layout)
from test_gpu_shard_parts import ID_NONE, INF_BITS, _assert_bits, _coarse_keys, _dev, _f32, _random_parts, _set_mode, _u32

pytestmark = pytest.mark.gpu

K = 10


def _torch():
    import torch
    return torch


def _out(nq, k):
    torch = _torch()
    return [torch.empty((nq, k), dtype=torch.int32, device="cuda"),
            torch.empty((nq, k), dtype=torch.float32, device="cuda"),
            torch.empty((nq,), dtype=torch.int32, device="cuda")]


def _host(out):
    _torch().cuda.synchronize()
    return _u32(out[0]), _f32(out[1]), _u32(out[2])


def _unpack_tiers(chunks, nq, k):
    """[ranks][chunk] -> ids / dist [2 ranks][nq][k], counts [2 ranks][nq] (part 2r recent, 2r + 1 IVF)."""
    o_i, o_d, o_c, part, _ = tiers_pack_layout(nq, k)
    g = chunks.cpu().numpy().reshape(-1, part)
    return (g[:, o_i:o_d].copy().view(np.uint32).reshape(-1, nq, k),
            g[:, o_d:o_c].copy().view(np.float32).reshape(-1, nq, k),
            g[:, o_c:].copy().view(np.uint32))


def _merge_host_tiered(ids, dist, cnt, k, tiered=True):
    """Vectorised (distance, tier, row id) merge — or (distance, row id) with tiered=False."""
    parts, nq, kk = ids.shape
    valid = np.arange(kk)[None, None, :] < np.minimum(cnt.astype(np.int64), k)[:, :, None]
    flat = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2)).reshape(nq, parts * kk)  # noqa: E731
    d = flat(np.where(valid, dist, np.inf).astype(np.float32))
    i = flat(ids).astype(np.int64)
    tier = flat(np.broadcast_to((np.arange(parts) & 1)[:, None, None], ids.shape)) if tiered else np.zeros_like(i)
    order = np.lexsort((i, tier, d, flat(~valid)), axis=-1)[:, :k]
    n_ok = np.minimum(valid.sum(axis=(0, 2)), k)
    pos = np.arange(k)[None, :] < n_ok[:, None]
    o_ids = np.where(pos, np.take_along_axis(i, order, axis=1), ID_NONE).astype(np.uint32)
    o_dst = np.where(pos, np.take_along_axis(d, order, axis=1), np.inf).astype(np.float32)
    return o_ids, o_dst, n_ok.astype(np.uint32)


@pytest.fixture(scope="module")
def merge_eng():
    eng = Engine(8, k_max=64)
    yield eng
    eng.close()


# ---- a. the tiered merge ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("ranks", [1, 2, 4, 8, 32])
@pytest.mark.parametrize("k", [1, 7, 10, 32])
def test_tiered_merge_matches_reference(merge_eng, ranks, k):
    torch = _torch()
    rng = np.random.default_rng(1000 * ranks + k)
    reorders = 0
    for nq in (1, 127, 128, 129, 4097):
        ids, dist, cnt = _random_parts(rng, 2 * ranks, nq, k)
        want = _merge_host_tiered(ids, dist, cnt, k)
        if nq <= 129:
            ref = merge_tiers_reference(ids, dist, cnt, k)
            for a, b in zip(ref, want):
                assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"nq {nq}: host statements disagree"
        reorders += int((want[0] != _merge_host_tiered(ids, dist, cnt, k, tiered=False)[0]).any(axis=1).sum())
        o_i, o_d, o_c, part, chunk = tiers_pack_layout(nq, k)
        pack = np.empty((2 * ranks, part), dtype=np.uint32)
        pack[:, o_i:o_d] = ids.reshape(2 * ranks, -1)
        pack[:, o_d:o_c] = dist.reshape(2 * ranks, -1).view(np.uint32)
        pack[:, o_c:] = cnt
        d_pack = _dev(pack.reshape(ranks, chunk))
        out = _out(nq, k)
        merge_eng.merge_topk_tiers_packed_device(d_pack.data_ptr(), ranks, nq, k, *(t.data_ptr() for t in out))
        got = _host(out)
        assert np.array_equal(got[2], want[2]), f"nq {nq}: counts"
        assert np.array_equal(got[0], want[0]), f"nq {nq}: ids (tails included)"
        assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), f"nq {nq}: distance bits"
        del d_pack
    torch.cuda.synchronize()
    assert reorders > 0, "no cross-tier tie where (distance, id) and (distance, tier, id) disagree"


def test_tiered_merge_rejects_bad_arguments(merge_eng):
    torch = _torch()
    buf = torch.zeros((66 * 8,), dtype=torch.int32, device="cuda")
    out = torch.zeros((8,), dtype=torch.int32, device="cuda")
    for ranks in (0, 33):
        with pytest.raises(FvdbError):
            merge_eng.merge_topk_tiers_packed_device(buf.data_ptr(), ranks, 1, 1, out.data_ptr(), out.data_ptr(),
                                                     out.data_ptr())
    cos = Engine(8, k_max=16, metric=L.METRIC_COS)
    with pytest.raises(FvdbError):
        cos.merge_topk_tiers_packed_device(buf.data_ptr(), 1, 1, 1, out.data_ptr(), out.data_ptr(), out.data_ptr())
    dq = torch.zeros((1, 8), dtype=torch.float32, device="cuda")
    with pytest.raises(FvdbError):
        cos.search_device_tiers(dq.data_ptr(), 1, 1, 1, L.TIER_BOTH, 0, 0, 0, buf.data_ptr())
    cos.close()


# ---- data sets ------------------------------------------------------------------------------------------------------
N, D, NLIST, NPROBE = 40_000, 384, 64, 8


@pytest.fixture(scope="module")
def synth_case():
    r = 6000
    x = synth.rows(0, N + r, D, 4 * NLIST, 1.0, 1234)
    q = synth.queries(0, 70, D, N + r, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678)
    cents = x[:N:N // NLIST][:NLIST].copy()
    return dict(x=x[:N], fx=x[N:], fids=np.arange(N, N + r, dtype=np.uint32), q=q, cents=cents, nprobe=NPROBE)


LAT_N, LAT_D, LAT_NLIST, LAT_NPROBE = 20_000, 64, 16, 6


@pytest.fixture(scope="module")
def lattice_case():
    """Binary rows (d 64), every squared distance an integer.  The recent tier holds copies of 2000 IVF rows
    under HIGHER ids (same distance to every query as the IVF copy with the lower id) and 2000 fresh rows: the
    recent-first rule and a (distance, id) rule order every such pair differently."""
    rng = np.random.default_rng(77)
    x = rng.integers(0, 2, size=(LAT_N, LAT_D)).astype(np.float32)
    q = rng.integers(0, 2, size=(70, LAT_D)).astype(np.float32)
    cents = (0.5 + 0.3 * rng.standard_normal((LAT_NLIST, LAT_D))).astype(np.float32)
    fx = np.concatenate([x[rng.choice(LAT_N, 2000, replace=False)],
                         rng.integers(0, 2, size=(2000, LAT_D)).astype(np.float32)])
    return dict(x=x, fx=fx, fids=np.arange(LAT_N, LAT_N + 4000, dtype=np.uint32), q=q, cents=cents,
                nprobe=LAT_NPROBE)


def _without_slab(case, world, rank):
    """The case with the recent rows of `rank` removed: that rank holds an empty recent slab."""
    keep = np.array([owner_of_recent_row(int(i), world) != rank for i in case["fids"]])
    return dict(case, fx=case["fx"][keep], fids=case["fids"][keep])


def _oracle(case, q, k, tiers=3, deleted=None, filt=None):
    ivf = O.IVF(case["cents"], case["x"], case.get("ids", np.arange(case["x"].shape[0], dtype=np.uint32)))
    return O.hybrid_batch_search(ivf, case["fx"], case["fids"], q, k, case["nprobe"], tiers=tiers, deleted=deleted,
                                 filter_bits=filt)


def _hybrid_shards(case, world, mode, placement="mod"):
    """`world` handles: IVF rows by list placement (l % world or place_lists), recent rows by id % world."""
    torch = _torch()
    x, cents, fx, fids = case["x"], case["cents"], case["fx"], case["fids"]
    dx = torch.from_numpy(x).cuda()
    dids = torch.arange(x.shape[0], dtype=torch.int32, device="cuda")
    owner = place_lists(np.bincount(O.assign(x, cents), minlength=cents.shape[0]), world) if placement == "place" else None
    d_owner = _dev(owner) if owner is not None else None
    engs = []
    for r in range(world):
        e = Engine(x.shape[1], k_max=64)
        _set_mode(e, mode)
        e.set_centroids(cents)
        if owner is None:
            e.ivf_add_device(dx.data_ptr(), dids.data_ptr(), x.shape[0], world, r)
        else:
            e.ivf_add_device_owned(dx.data_ptr(), dids.data_ptr(), x.shape[0], d_owner.data_ptr(), r)
        mine = np.array([owner_of_recent_row(int(i), world) == r for i in fids], dtype=bool)
        if mine.any():
            fdx = torch.from_numpy(np.ascontiguousarray(fx[mine])).cuda()
            fdi = _dev(fids[mine])
            e.flat_add_device(fdx.data_ptr(), fdi.data_ptr(), int(mine.sum()))
        engs.append(e)
    torch.cuda.synchronize()
    return engs, owner


def _close(engs):
    for e in engs:
        e.close()


def _tiered_search(engs, q, k, nprobe, tiers=L.TIER_BOTH, filt=None, submit=False):
    """ShardedIndex.search's TIER_BOTH steps over `engs`: coarse slices, every shard's fvdb_search_device_tiers
    into its chunk, the tiered merge.  Returns (merged result, the gathered chunks)."""
    torch = _torch()
    nq = q.shape[0]
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    keys = _coarse_keys(engs, dq, nprobe)
    chunks = torch.empty((len(engs), tiers_pack_layout(nq, k)[4]), dtype=torch.int32, device="cuda")
    f_ptr, f_bits = (filt.data_ptr(), filt.numel() * 64) if filt is not None else (0, 0)
    for e, c in zip(engs, chunks):
        e.search_device_tiers(dq.data_ptr(), nq, k, nprobe, tiers, f_ptr, f_bits, keys.data_ptr(), c.data_ptr())
    out = _out(nq, k)
    engs[0].merge_topk_tiers_packed_device(chunks.data_ptr(), len(engs), nq, k, *(t.data_ptr() for t in out))
    return _host(out), chunks


# ---- b. the split entry on one handle ---------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["exact", "tc"])
@pytest.mark.parametrize("flat_n", [3000, 64_000])
def test_split_entry_equals_existing_entry(mode, flat_n):
    """flat_n 64 000 x 70 queries is above the 4M-pair tensor-core threshold of the recent tier, 3000 below."""
    torch = _torch()
    nq, n = 70, 20_000
    x = synth.rows(0, n + flat_n, D, 4 * NLIST, 1.0, 4321)
    q = synth.queries(0, nq, D, n + flat_n, 4 * NLIST, 1.0, 4321, synth.default_qnoise(D, 1.0), 8765)
    cents = x[:n:n // NLIST][:NLIST].copy()
    e = Engine(D, k_max=64)
    _set_mode(e, mode)
    e.set_centroids(cents)
    e.ivf_add(x[:n], np.arange(n, dtype=np.uint32))
    e.flat_add(x[n:], np.arange(n, n + flat_n, dtype=np.uint32))
    dq = torch.from_numpy(q).cuda()
    dele = np.arange(5, n + flat_n, 13, dtype=np.uint32)
    keep = O.make_bitmap(n + flat_n, np.flatnonzero(np.arange(n + flat_n) % 4 != 2))
    case = dict(x=x[:n], fx=x[n:], fids=np.arange(n, n + flat_n, dtype=np.uint32), cents=cents, nprobe=NPROBE)
    for step in ("plain", "tombstones", "filter"):
        if step == "tombstones":
            e.set_deleted(dele, True)
        filt = _dev(keep) if step == "filter" else None
        f_ptr, f_bits = (filt.data_ptr(), filt.numel() * 64) if filt is not None else (0, 0)

        def existing(tiers):
            out = _out(nq, K)
            e.search_device_coarse(dq.data_ptr(), nq, K, NPROBE, tiers, f_ptr, f_bits, 0, *(t.data_ptr() for t in out))
            return _host(out)

        def split(tiers):
            chunk = torch.empty((tiers_pack_layout(nq, K)[4],), dtype=torch.int32, device="cuda")
            e.search_device_tiers(dq.data_ptr(), nq, K, NPROBE, tiers, f_ptr, f_bits, 0, chunk.data_ptr())
            out = _out(nq, K)
            e.merge_topk_tiers_packed_device(chunk.data_ptr(), 1, nq, K, *(t.data_ptr() for t in out))
            return _host(out), _unpack_tiers(chunk[None], nq, K)

        what = f"{mode}, flat {flat_n}, {step}"
        both, parts = split(L.TIER_BOTH)
        _assert_bits(both, existing(L.TIER_BOTH), f"{what}: ranks-1 merge of the split chunk")
        recent, hist = existing(L.TIER_RECENT), existing(L.TIER_HISTORICAL)
        p_ids, p_dst, p_cnt = parts
        _assert_bits((p_ids[0], p_dst[0], p_cnt[0]), recent, f"{what}: recent part")
        _assert_bits((p_ids[1], p_dst[1], p_cnt[1]), hist, f"{what}: IVF part")
        # tails of both parts as a lone tier writes them
        for t in (0, 1):
            tail = np.arange(K)[None, :] >= p_cnt[t][:, None]
            assert (p_ids[t][tail] == ID_NONE).all() and (p_dst[t][tail].view(np.uint32) == INF_BITS).all()
        for tiers, empty in ((L.TIER_RECENT, 1), (L.TIER_HISTORICAL, 0)):
            _, (s_ids, s_dst, s_cnt) = split(tiers)
            assert (s_cnt[empty] == 0).all(), f"{what}: tiers {tiers} filled the other part"
            _assert_bits((s_ids[1 - empty], s_dst[1 - empty], s_cnt[1 - empty]), recent if tiers == L.TIER_RECENT else hist,
                         f"{what}: tiers {tiers}")
        bm_del = O.make_bitmap(n + flat_n, dele) if step != "plain" else None
        _assert_bits(both, _oracle(case, q, K, deleted=bm_del, filt=keep if step == "filter" else None), f"{what}: oracle")
    e.close()


# ---- c. sharded hybrid search ------------------------------------------------------------------------------------------
def _cross_tier_rank_ties(want, n_ivf, rank_of_ivf_row, world):
    """Tie groups in the oracle's top-k holding a recent row and an IVF row that sit on different ranks."""
    ids, dst, cnt = want
    n = 0
    for i in range(len(cnt)):
        c = int(cnt[i])
        for v in np.unique(dst[i, :c]):
            grp = ids[i, :c][dst[i, :c] == v]
            rec, ivf = grp[grp >= n_ivf], grp[grp < n_ivf]
            ranks = set((rec % world).tolist()) | set(rank_of_ivf_row[ivf].tolist())
            n += int(bool(rec.size and ivf.size) and len(ranks) > 1)
    return n


@pytest.mark.parametrize("mode", ["exact", "tc"])
@pytest.mark.parametrize("placement", ["mod", "place"])
@pytest.mark.parametrize("data", ["synth", "lattice"])
@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_hybrid_equals_oracle(request, mode, placement, data, world):
    case = _without_slab(request.getfixturevalue(f"{data}_case"), world, world - 1)
    q, nprobe = case["q"], case["nprobe"]
    n_all = case["x"].shape[0] + case["fx"].shape[0]
    engs, owner = _hybrid_shards(case, world, mode, placement)
    assert engs[world - 1].stats().flat_rows == 0 and all(e.stats().flat_rows > 0 for e in engs[:-1])

    want = _oracle(case, q, K)
    got, chunks = _tiered_search(engs, q, K, nprobe)
    _assert_bits(got, want, "sharded hybrid")
    if data == "lattice":
        a = O.assign(case["x"], case["cents"])
        rank_of_ivf = (owner[a] if owner is not None else a % world).astype(np.int64)
        assert _cross_tier_rank_ties(want, case["x"].shape[0], rank_of_ivf, world) >= 20, \
            "too few cross-tier, cross-rank ties in the top-k"
        old = _merge_host_tiered(*_unpack_tiers(chunks, q.shape[0], K), K, tiered=False)
        assert not np.array_equal(old[0], want[0]), "a (distance, id) merge would pass: the case tests nothing"

    dele = np.arange(3, n_all, 11, dtype=np.uint32)
    for e in engs:
        e.set_deleted(dele, True)
    bm_del = O.make_bitmap(n_all, dele)
    _assert_bits(_tiered_search(engs, q, K, nprobe)[0], _oracle(case, q, K, deleted=bm_del), "sharded hybrid + tombstones")
    keep = O.make_bitmap(n_all, np.flatnonzero(np.arange(n_all) % 3 != 1))
    got = _tiered_search(engs, q, K, nprobe, filt=_dev(keep))[0]
    _assert_bits(got, _oracle(case, q, K, deleted=bm_del, filt=keep), "sharded hybrid + tombstones + filter")
    _close(engs)


# ---- d. mutations -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("placement", ["mod", "place"])
@pytest.mark.parametrize("mode", ["exact", "tc"])
def test_sharded_mutations(lattice_case, mode, placement):
    """With a place_lists table a migrated row often joins a list another rank owns: it stays on its rank."""
    world = 3
    case = dict(lattice_case)
    q, nprobe = case["q"], case["nprobe"]
    n_ivf = case["x"].shape[0]
    n_all = n_ivf + case["fx"].shape[0]
    engs, owner = _hybrid_shards(case, world, mode, placement)
    dele = np.concatenate([np.arange(1, n_ivf, 7), np.arange(n_ivf + 2, n_all, 5)]).astype(np.uint32)
    for e in engs:
        e.set_deleted(dele, True)
    _assert_bits(_tiered_search(engs, q, K, nprobe)[0], _oracle(case, q, K, deleted=O.make_bitmap(n_all, dele)), "after delete")
    removed = sum(e.vacuum() for e in engs)
    assert removed == dele.size
    gone = np.zeros(n_all, dtype=bool)
    gone[dele] = True
    case = dict(case, x=case["x"][~gone[:n_ivf]], ids=np.flatnonzero(~gone[:n_ivf]).astype(np.uint32),
                fx=case["fx"][~gone[n_ivf:]], fids=case["fids"][~gone[n_ivf:]])
    _assert_bits(_tiered_search(engs, q, K, nprobe)[0], _oracle(case, q, K), "after vacuum")
    # migrate every other recent row: each rank moves those it holds into its own arena
    mig = case["fids"][::2]
    moved = sum(e.move_flat_to_ivf(mig) for e in engs)
    assert moved == mig.size
    if owner is not None:
        lists = O.assign(case["fx"][np.isin(case["fids"], mig)], case["cents"])
        held = mig % world
        assert (owner[lists] != held).any(), "no migrated row joins a list another rank owns: the case tests nothing"
    is_mig = np.isin(case["fids"], mig)
    case = dict(case, x=np.concatenate([case["x"], case["fx"][is_mig]]),
                ids=np.concatenate([case["ids"], case["fids"][is_mig]]), fx=case["fx"][~is_mig], fids=case["fids"][~is_mig])
    _assert_bits(_tiered_search(engs, q, K, nprobe)[0], _oracle(case, q, K), "after migrate")
    _close(engs)


# ---- e. the pipelined entry ---------------------------------------------------------------------------------------------
def _pipelined_tiers(engs, qs, k, nprobe):
    """ShardedIndex.submit's TIER_BOTH steps: per batch every shard's stream-ordered coarse slice and
    fvdb_search_device_tiers_submit, the merge of batch i - 1 after wait(age=1), the last after wait(0), finish."""
    torch = _torch()
    nq = qs[0].shape[0]
    dqs = [torch.from_numpy(np.ascontiguousarray(q)).cuda() for q in qs]
    chunk = tiers_pack_layout(nq, k)[4]
    bufs, outs = [], []

    def merge(chunks):
        out = _out(nq, k)
        engs[0].merge_topk_tiers_packed_device(chunks.data_ptr(), len(engs), nq, k, *(t.data_ptr() for t in out))
        return out

    for i, dq in enumerate(dqs):
        keys = _coarse_keys(engs, dq, nprobe, submit=True)
        chunks = torch.empty((len(engs), chunk), dtype=torch.int32, device="cuda")
        for e, c in zip(engs, chunks):
            e.search_device_tiers_submit(dq.data_ptr(), nq, k, nprobe, L.TIER_BOTH, 0, 0, keys.data_ptr(), c.data_ptr())
        bufs.append((keys, chunks))
        if i:
            for e in engs:
                e.search_device_wait(1)
            outs.append(merge(bufs[i - 1][1]))
    for e in engs:
        e.search_device_wait(0)
    outs.append(merge(bufs[-1][1]))
    for e in engs:
        e.search_device_finish()
    # the chunks after finish (a deferred repair rewrites them) merged again
    final = [_host(merge(b[1])) for b in bufs]
    res = [_host(o) for o in outs]
    return res, final, [e.stats().last_fallback_queries for e in engs]


def test_pipelined_tiers_entry(synth_case):
    world = 3
    case = synth_case
    engs, _ = _hybrid_shards(case, world, "tc")
    qs = [synth.queries(100 * i, 64, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678) for i in range(4)]
    sync = [_tiered_search(engs, q, K, NPROBE)[0] for q in qs]
    res, final, fb = _pipelined_tiers(engs, qs, K, NPROBE)
    for i, q in enumerate(qs):
        want = _oracle(case, q, K)
        _assert_bits(sync[i], want, f"sync batch {i}")
        _assert_bits(final[i], want, f"pipelined batch {i} after finish")
        if not max(fb):
            _assert_bits(res[i], want, f"pipelined batch {i}")
    _close(engs)

    # a near-duplicate shell in the IVF tier (check_shard.py §3) makes the tensor-core proof fail on the shard
    # holding it: fvdb_search_device_finish re-runs those queries exactly and rewrites BOTH parts of the chunk
    x3 = case["x"].copy()
    rng = np.random.default_rng(11)
    for j in range(60):
        x3[300 + j] = x3[100] if j % 3 == 0 else x3[100] + (1e-4 * rng.standard_normal(D)).astype(np.float32)
    q3 = np.concatenate([np.stack([x3[100] + (0.05 * rng.standard_normal(D)).astype(np.float32) for _ in range(16)]),
                         case["q"][:48]])
    case3 = dict(case, x=x3)
    engs, _ = _hybrid_shards(case3, world, "tc")
    group = [q3, qs[0], q3[::-1].copy(), qs[1]]
    _, final, fb = _pipelined_tiers(engs, group, K, NPROBE)
    holder = owner_of_list(int(O.assign(x3[100:101], case["cents"])[0]), world)
    assert fb[holder] > 0, f"no proof failure on the shard holding the shell (fallback counts {fb})"
    for i, q in enumerate(group):
        _assert_bits(final[i], _oracle(case3, q, K), f"repaired batch {i}")
    _close(engs)


POISON = 0x7A7A7A7A


def test_deferred_repair_rewrites_both_parts(synth_case):
    """The deferred exact repair of fvdb_search_device_finish on a split batch.  Two shards, each holding 70 000
    recent rows (70 000 x 64 queries is above the 4M-pair tensor-core threshold of the recent tier) and a share of
    an IVF tier with a near-duplicate shell; a second shell sits in the recent tier.  After the scans the chunks are
    overwritten with a marker, then finish() runs: exactly the repaired queries get both parts back, and both
    equal the exact-mode split search of the same handle."""
    torch = _torch()
    world, nq, r = 2, 64, 140_000
    case = synth_case
    x3 = case["x"].copy()
    rng = np.random.default_rng(11)
    for j in range(60):
        x3[300 + j] = x3[100] if j % 3 == 0 else x3[100] + (1e-4 * rng.standard_normal(D)).astype(np.float32)
    fx = synth.rows(N, r, D, 4 * NLIST, 1.0, 99)
    for j in range(1, 60):
        fx[j] = fx[0] if j % 3 == 0 else fx[0] + (1e-4 * rng.standard_normal(D)).astype(np.float32)
    near = lambda row, n: np.stack([row + (0.05 * rng.standard_normal(D)).astype(np.float32) for _ in range(n)])  # noqa: E731
    q = np.concatenate([near(x3[100], 8), near(fx[0], 8), case["q"][:48]]).astype(np.float32)
    case3 = dict(case, x=x3, fx=fx, fids=np.arange(N, N + r, dtype=np.uint32))
    engs, _ = _hybrid_shards(case3, world, "tc")
    assert all(e.stats().flat_rows * nq >= (4 << 20) for e in engs)
    dq = torch.from_numpy(q).cuda()
    keys = _coarse_keys(engs, dq, NPROBE)
    o_i, o_d, o_c, part, chunk = tiers_pack_layout(nq, K)
    group = [dq, dq.flip(0).contiguous()]
    chunks = [torch.empty((world, chunk), dtype=torch.int32, device="cuda") for _ in group]
    gkeys = [keys, _coarse_keys(engs, group[1], NPROBE)]
    for b, (qq, kk) in enumerate(zip(group, gkeys)):
        for e, c in zip(engs, chunks[b]):
            e.search_device_tiers_submit(qq.data_ptr(), nq, K, NPROBE, L.TIER_BOTH, 0, 0, kk.data_ptr(), c.data_ptr())
    torch.cuda.synchronize()
    for c in chunks:
        c.fill_(POISON)
    torch.cuda.synchronize()
    for e in engs:
        e.search_device_finish()
    fb = [e.stats().last_fallback_queries for e in engs]
    torch.cuda.synchronize()
    for e in engs:
        e.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    repaired = [0] * world
    for b, (qq, kk) in enumerate(zip(group, gkeys)):
        for r_, e in enumerate(engs):
            ref = torch.empty((chunk,), dtype=torch.int32, device="cuda")
            e.search_device_tiers(qq.data_ptr(), nq, K, NPROBE, L.TIER_BOTH, 0, 0, kk.data_ptr(), ref.data_ptr())
            got = chunks[b][r_].cpu().numpy().reshape(2, part)
            want = ref.cpu().numpy().reshape(2, part)
            fixed = [got[t, o_c:] != POISON for t in (0, 1)]
            assert np.array_equal(fixed[0], fixed[1]), f"batch {b} rank {r_}: a repair rewrote one part only"
            for t in (0, 1):
                rows = np.flatnonzero(fixed[t])
                g3 = got[t, :o_c].reshape(2, nq, K)
                w3 = want[t, :o_c].reshape(2, nq, K)
                assert np.array_equal(g3[:, rows], w3[:, rows]), f"batch {b} rank {r_} part {t}: repaired rows differ"
                assert np.array_equal(got[t, o_c:][rows], want[t, o_c:][rows])
            repaired[r_] += int(fixed[0].sum())
    assert repaired == fb, f"repaired rows {repaired} vs reported fallbacks {fb}"
    holder = owner_of_list(int(O.assign(x3[100:101], case["cents"])[0]), world)
    assert fb[holder] > 0, f"no proof failure on the shard holding the IVF shell (fallback counts {fb})"
    _close(engs)


# ---- f. the sharded post-filter ---------------------------------------------------------------------------------------------
def test_sharded_postfilter(lattice_case):
    torch = _torch()
    world = 3
    case = lattice_case
    q, nprobe = case["q"], case["nprobe"]
    n_all = case["x"].shape[0] + case["fx"].shape[0]
    engs, _ = _hybrid_shards(case, world, "tc")
    match = O.make_bitmap(n_all, np.flatnonzero(np.arange(n_all) % 4 != 0))
    # the driver's post-filter over the emulated sharded search (its collective steps are done here)
    sh = ShardedIndex(engs[0], 0, 1)
    sh.search = lambda qq, k, nprobe_, tiers=L.TIER_BOTH: tuple(
        torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).cuda()
        for a in _tiered_search(engs, qq.cpu().numpy(), k, nprobe_, tiers)[0])
    got = sh.search_postfilter(torch.from_numpy(q).cuda(), K, nprobe, _dev(match))
    g_ids, g_dst, g_cnt = _u32(got[0]), _f32(got[1]), _u32(got[2])
    ivf = O.IVF(case["cents"], case["x"], np.arange(case["x"].shape[0], dtype=np.uint32))
    for i in range(q.shape[0]):
        w_ids, w_dst = O.hybrid_search_postfilter(ivf, case["fx"], case["fids"], q[i], K, nprobe, match, tiers=3)
        c = len(w_ids)
        assert int(g_cnt[i]) == c, f"query {i}: count"
        assert g_ids[i, :c].tolist() == w_ids.tolist(), f"query {i}: ids"
        assert g_dst[i, :c].view(np.uint32).tolist() == w_dst.view(np.uint32).tolist(), f"query {i}: dist"
        assert (g_ids[i, c:] == ID_NONE).all()
    with pytest.raises(ValueError):
        sh.search_postfilter(torch.from_numpy(q).cuda(), 22, nprobe, _dev(match))
    _close(engs)
