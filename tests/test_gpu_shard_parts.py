"""The device entry points the list-sharded multi-GPU driver (fabstir_vectordb_b200/shard.py) is built from, tested
on ONE GPU: W Engine handles on device 0 with the same centroids act as the W shards, and the test performs the
driver's collective steps itself (concatenate the coarse-key slices, stack the packed result chunks).  Every
sharded result is compared with the unsharded CPU oracle bit for bit (ids, distance bits, counts).

Covered: fvdb_merge_topk_device / _packed_device against a host (distance, row id) merge; list-sharded loading
(fvdb_ivf_add_device mod / rem, fvdb_ivf_add_device_owned, fvdb_assign_device); the synchronous sharded search
(fvdb_coarse_device + fvdb_search_device_coarse + packed merge) in exact and tensor-core mode, on synthetic rows
and on integer-lattice rows whose exact distance ties straddle ranks; "probe nothing" key rows; the pipelined
entries (fvdb_coarse_device_submit / fvdb_search_device_coarse_submit / fvdb_search_device_wait / _finish);
fvdb_ivf_max_sqnorm with FVDB_OPT_PROOF_XMAX; the sharded k-means blocks (fvdb_kmeans_accumulate_device /
fvdb_kmeans_apply_device)."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, FvdbError, _lib as L, synth
from fabstir_vectordb_b200.shard import ShardedIndex, owner_of_list, pack_layout, place_lists

pytestmark = pytest.mark.gpu

ID_NONE = 0xFFFFFFFF
INF_BITS = 0x7F800000

# the data set of scripts/check_shard.py
N, D, NLIST, K, NPROBE = 40_000, 384, 64, 10, 8


def _torch():
    import torch
    return torch


def _dev(a):
    """Host array -> CUDA tensor with the same bytes (u32 as i32, u64 as i64)."""
    torch = _torch()
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    elif a.dtype == np.uint64:
        a = a.view(np.int64)
    return torch.from_numpy(a.copy()).cuda()


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _f32(t):
    return t.cpu().numpy().view(np.float32)


def _assert_bits(got, want, what=""):
    g_ids, g_dst, g_cnt = got
    w_ids, w_dst, w_cnt = want
    assert np.array_equal(np.asarray(g_cnt, dtype=np.uint32), np.asarray(w_cnt, dtype=np.uint32)), f"{what}: counts"
    for i in range(len(w_cnt)):
        c = int(w_cnt[i])
        assert g_ids[i, :c].tolist() == w_ids[i, :c].tolist(), f"{what}: ids of query {i}"
        assert g_dst[i, :c].view(np.uint32).tolist() == w_dst[i, :c].view(np.uint32).tolist(), f"{what}: dist of query {i}"


def _merge_host(ids, dist, cnt, k, by_part=False):
    """The merge in float64-free host terms: candidates are the first min(count, k) entries of every part,
    ordered by (distance, row id) — or, with by_part, by (distance, part, position), the order the merge
    kernel used before ties were broken by row id.  Tails are ID_NONE / +inf."""
    parts, nq, kk = ids.shape
    valid = np.arange(kk)[None, None, :] < np.minimum(cnt.astype(np.int64), k)[:, :, None]
    flat = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2)).reshape(nq, parts * kk)  # noqa: E731
    d = flat(np.where(valid, dist, np.inf).astype(np.float32))
    i = flat(ids).astype(np.int64)
    second = np.broadcast_to(np.arange(parts * kk), (nq, parts * kk)) if by_part else i
    order = np.lexsort((second, d, flat(~valid)), axis=-1)[:, :k]
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


# ---- a. the merge kernels -------------------------------------------------------------------------------------
def _random_parts(rng, parts, nq, k):
    """Per-part partial results sorted by (distance, id), ids distinct across the parts of a query, distances
    from five values (cross-part ties everywhere), counts 0, below k and above k; tails ID_NONE / +inf."""
    levels = np.array([0.25, 1.0, 1.5, 2.0, 7.0], dtype=np.float32)
    li = rng.integers(0, levels.size, size=(parts, nq, k))
    perm = np.argsort(rng.random((nq, parts * k)), axis=1).astype(np.int64)          # distinct per query
    ids = perm.reshape(nq, parts, k).transpose(1, 0, 2) * 3 + 5
    order = np.argsort((li << 32) | ids, axis=-1)
    li = np.take_along_axis(li, order, axis=-1)
    ids = np.take_along_axis(ids, order, axis=-1).astype(np.uint32)
    dist = levels[li]
    cnt = rng.choice(np.array([0, 1, max(k - 1, 0), k, k + 3], dtype=np.uint32), size=(parts, nq))
    tail = np.arange(k)[None, None, :] >= cnt[:, :, None]
    ids[tail] = ID_NONE
    dist[tail] = np.inf
    return ids, dist, cnt


@pytest.mark.parametrize("parts", [1, 2, 3, 8, 64])
@pytest.mark.parametrize("k", [1, 7, 10, 32])
def test_merge_kernels_match_host_merge(merge_eng, parts, k):
    torch = _torch()
    rng = np.random.default_rng(1000 * parts + k)
    reorders = 0
    for nq in (1, 127, 128, 129, 4097):
        ids, dist, cnt = _random_parts(rng, parts, nq, k)
        want = _merge_host(ids, dist, cnt, k)
        reorders += int((want[0] != _merge_host(ids, dist, cnt, k, by_part=True)[0]).any(axis=1).sum())
        out = [torch.empty((nq, k), dtype=torch.int32, device="cuda"),
               torch.empty((nq, k), dtype=torch.float32, device="cuda"),
               torch.empty((nq,), dtype=torch.int32, device="cuda")]
        d_ids, d_dst, d_cnt = _dev(ids), _dev(dist), _dev(cnt)
        merge_eng.merge_topk_device(d_ids.data_ptr(), d_dst.data_ptr(), d_cnt.data_ptr(), parts, nq, k,
                                    *(t.data_ptr() for t in out))
        # the packed twin: parts x [ids nq*k | dist nq*k | count nq] (the chunk length is odd when nq is)
        o_i, o_d, o_c, chunk = pack_layout(nq, k)
        pack = np.empty((parts, chunk), dtype=np.uint32)
        pack[:, o_i:o_d] = ids.reshape(parts, -1)
        pack[:, o_d:o_c] = dist.reshape(parts, -1).view(np.uint32)
        pack[:, o_c:] = cnt
        d_pack = _dev(pack)
        out_p = [torch.empty_like(t) for t in out]
        merge_eng.merge_topk_packed_device(d_pack.data_ptr(), parts, nq, k, *(t.data_ptr() for t in out_p))
        torch.cuda.synchronize()
        got = (_u32(out[0]), _f32(out[1]), _u32(out[2]))
        assert np.array_equal(got[2], want[2]), f"nq {nq}: counts"
        assert np.array_equal(got[0], want[0]), f"nq {nq}: ids (tails included)"
        assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32)), f"nq {nq}: distance bits"
        assert (got[1][np.arange(k)[None, :] >= got[2][:, None]].view(np.uint32) == INF_BITS).all()
        for a, b in zip(out, out_p):
            assert torch.equal(a, b), f"nq {nq}: packed and unpacked merges differ"
    if parts > 1:
        assert reorders > 0, "no cross-part tie where the two tie rules disagree: the case tests nothing"


def test_merge_part_count_is_checked(merge_eng):
    torch = _torch()
    buf = torch.zeros((65 * 8,), dtype=torch.int32, device="cuda")
    out = torch.zeros((8,), dtype=torch.int32, device="cuda")
    for parts in (0, 65):
        with pytest.raises(FvdbError):
            merge_eng.merge_topk_device(buf.data_ptr(), buf.data_ptr(), buf.data_ptr(), parts, 1, 1,
                                        out.data_ptr(), out.data_ptr(), out.data_ptr())
        with pytest.raises(FvdbError):
            merge_eng.merge_topk_packed_device(buf.data_ptr(), parts, 1, 1, out.data_ptr(), out.data_ptr(),
                                               out.data_ptr())


# ---- data sets ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def synth_case():
    x = synth.rows(0, N, D, 4 * NLIST, 1.0, 1234)
    q = synth.queries(0, 70, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678)
    cents = x[:: N // NLIST][:NLIST].copy()
    return dict(x=x, q=q, cents=cents, ivf=O.IVF(cents, x, np.arange(N, dtype=np.uint32)), nprobe=NPROBE)


LAT_N, LAT_D, LAT_NLIST, LAT_NPROBE = 20_000, 64, 16, 6


@pytest.fixture(scope="module")
def lattice_case():
    """Binary rows (d 64): every squared distance is an integer, so exact in f32 on every path, and a query's
    nearest rows share a handful of distances — tie groups of dozens of rows, spread over the lists of all
    ranks by Gaussian centroids."""
    rng = np.random.default_rng(77)
    x = rng.integers(0, 2, size=(LAT_N, LAT_D)).astype(np.float32)
    q = rng.integers(0, 2, size=(70, LAT_D)).astype(np.float32)
    cents = (0.5 + 0.3 * rng.standard_normal((LAT_NLIST, LAT_D))).astype(np.float32)
    return dict(x=x, q=q, cents=cents, ivf=O.IVF(cents, x, np.arange(LAT_N, dtype=np.uint32)), nprobe=LAT_NPROBE)


def _set_mode(eng, mode):
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC if mode == "tc" else L.SCAN_EXACT)


def _shards(case, world, mode, owner=None):
    """`world` handles with the case's centroids, each loaded with the rows of the lists it owns."""
    torch = _torch()
    x, cents = case["x"], case["cents"]
    dx = torch.from_numpy(x).cuda()
    dids = torch.arange(x.shape[0], dtype=torch.int32, device="cuda")
    engs, kept = [], []
    d_owner = _dev(owner) if owner is not None else None
    for r in range(world):
        e = Engine(x.shape[1], k_max=64)
        _set_mode(e, mode)
        e.set_centroids(cents)
        if owner is None:
            kept.append(e.ivf_add_device(dx.data_ptr(), dids.data_ptr(), x.shape[0], world, r))
        else:
            kept.append(e.ivf_add_device_owned(dx.data_ptr(), dids.data_ptr(), x.shape[0], d_owner.data_ptr(), r))
        engs.append(e)
    return engs, kept


def _close(engs):
    for e in engs:
        e.close()


def _coarse_keys(engs, dq, nprobe, submit=False):
    """The driver's query-sharded coarse step: rank r ranks rows [r*per, r*per + per) of the batch, the slices
    are concatenated, rows of a short or empty slice stay 0xFF..FF ("probe nothing")."""
    torch = _torch()
    world, nq = len(engs), dq.shape[0]
    per = (nq + world - 1) // world
    mine = []
    for r, e in enumerate(engs):
        m = torch.full((per, nprobe), -1, dtype=torch.int64, device="cuda")
        lo = min(nq, r * per)
        n_mine = max(0, min(nq, lo + per) - lo)
        if n_mine:
            f = e.coarse_device_submit if submit else e.coarse_device
            f(dq[lo:lo + n_mine].data_ptr(), n_mine, nprobe, m.data_ptr())
        mine.append(m)
    return torch.cat(mine)


def _pack_bufs(nq, k, world):
    torch = _torch()
    o_i, o_d, o_c, chunk = pack_layout(nq, k)
    packs = torch.empty((world, chunk), dtype=torch.int32, device="cuda")
    views = [(p[o_i:o_d].data_ptr(), p[o_d:o_c].data_ptr(), p[o_c:].data_ptr()) for p in packs]
    return packs, views


def _unpack(packs, nq, k):
    o_i, o_d, o_c, _ = pack_layout(nq, k)
    g = packs.cpu().numpy()
    world = g.shape[0]
    return (g[:, o_i:o_d].copy().view(np.uint32).reshape(world, nq, k),
            g[:, o_d:o_c].copy().view(np.float32).reshape(world, nq, k),
            g[:, o_c:].copy().view(np.uint32))


def _merge_dev(eng, packs, nq, k):
    torch = _torch()
    out = [torch.empty((nq, k), dtype=torch.int32, device="cuda"),
           torch.empty((nq, k), dtype=torch.float32, device="cuda"),
           torch.empty((nq,), dtype=torch.int32, device="cuda")]
    eng.merge_topk_packed_device(packs.data_ptr(), packs.shape[0], nq, k, *(t.data_ptr() for t in out))
    return out


def _host(out):
    _torch().cuda.synchronize()
    return _u32(out[0]), _f32(out[1]), _u32(out[2])


def _sharded_search(engs, q, k, nprobe, filt=None):
    """ShardedIndex.search's steps over `engs`: coarse slices, concatenation, every shard's scan into its packed
    chunk, the packed merge.  Returns (merged result, the gathered per-shard parts)."""
    torch = _torch()
    nq = q.shape[0]
    dq = torch.from_numpy(np.ascontiguousarray(q)).cuda()
    keys = _coarse_keys(engs, dq, nprobe)
    packs, views = _pack_bufs(nq, k, len(engs))
    f_ptr, f_bits = (filt.data_ptr(), filt.numel() * 64) if filt is not None else (0, 0)
    for e, (pi, pd, pc) in zip(engs, views):
        e.search_device_coarse(dq.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, f_ptr, f_bits, keys.data_ptr(), pi, pd, pc)
    out = _merge_dev(engs[0], packs, nq, k)
    got = _host(out)
    return got, _unpack(packs, nq, k)


# ---- b. list-sharded loading --------------------------------------------------------------------------------------
def _check_shards(engs, kept, x_ids_pos, want_list, owner_of):
    n = want_list.shape[0]
    assert sum(kept) == n
    seen = np.zeros(n, dtype=np.int64)
    for r, (e, kr) in enumerate(zip(engs, kept)):
        ids, lists = e.dump_lists()
        assert ids.shape[0] == kr
        pos = x_ids_pos[ids]                                    # input position of every arena row
        seen[pos] += 1
        assert np.array_equal(lists, want_list[pos]), f"rank {r}: a row is in the wrong list"
        assert all(owner_of(int(l)) == r for l in np.unique(lists)), f"rank {r} holds a list it does not own"
        # grouped by list, insertion order inside a list
        assert (np.diff(lists.astype(np.int64)) >= 0).all(), f"rank {r}: arena not grouped by list"
        same = lists[1:] == lists[:-1]
        assert (np.diff(pos)[same] > 0).all(), f"rank {r}: insertion order lost inside a list"
    assert (seen == 1).all(), "the shards do not partition the rows"


@pytest.mark.parametrize("world", [2, 3, 8])
def test_sharded_loading(synth_case, world):
    torch = _torch()
    x, cents = synth_case["x"][:12_000], synth_case["cents"]
    n = x.shape[0]
    rng = np.random.default_rng(world)
    row_ids = (rng.permutation(n) * 2 + 1).astype(np.uint32)      # insertion order != id order
    pos_of = np.full(2 * n + 2, -1, dtype=np.int64)
    pos_of[row_ids] = np.arange(n)
    want = O.assign(x, cents)
    dx, dids = torch.from_numpy(x).cuda(), _dev(row_ids)

    engs = []
    for r in range(world):
        e = Engine(D)
        e.set_centroids(cents)
        engs.append(e)
    kept = [e.ivf_add_device(dx.data_ptr(), dids.data_ptr(), n, world, r) for r, e in enumerate(engs)]
    _check_shards(engs, kept, pos_of, want, lambda l: owner_of_list(l, world))

    # size-balanced placement from a histogram made without moving rows
    a = torch.empty((n,), dtype=torch.int32, device="cuda")
    engs[0].assign_device(dx.data_ptr(), n, a.data_ptr())
    hist = np.bincount(_u32(a), minlength=NLIST)
    assert hist.tolist() == np.bincount(want, minlength=NLIST).tolist()
    owner = place_lists(hist, world)
    d_owner = _dev(owner)
    owned = []
    for r in range(world):
        e = Engine(D)
        e.set_centroids(cents)
        owned.append(e)
    kept = [e.ivf_add_device_owned(dx.data_ptr(), dids.data_ptr(), n, d_owner.data_ptr(), r) for r, e in enumerate(owned)]
    _check_shards(owned, kept, pos_of, want, lambda l: int(owner[l]))
    _close(engs + owned)


# ---- c. synchronous sharded search ------------------------------------------------------------------------------------
def _row_rank(case, world):
    return np.array([owner_of_list(int(l), world) for l in range(case["cents"].shape[0])])[case["ivf"].assign]


def _cross_rank_ties(w, world_of_row):
    """Tie groups in the oracle's top-k whose rows lie on more than one rank."""
    ids, dst, cnt = w
    n = 0
    for i in range(len(cnt)):
        c = int(cnt[i])
        for v in np.unique(dst[i, :c]):
            grp = ids[i, :c][dst[i, :c] == v]
            n += int(grp.size > 1 and np.unique(world_of_row[grp]).size > 1)
    return n


@pytest.mark.parametrize("mode", ["exact", "tc"])
@pytest.mark.parametrize("data", ["synth", "lattice"])
@pytest.mark.parametrize("world,nq", [(3, 70), (8, 5)])
def test_sharded_search_equals_oracle(request, mode, data, world, nq):
    case = request.getfixturevalue(f"{data}_case")
    x, ivf, nprobe = case["x"], case["ivf"], case["nprobe"]
    q = case["q"][:nq]
    n = x.shape[0]
    engs, kept = _shards(case, world, mode)
    assert sum(kept) == n

    want = O.hybrid_batch_search(ivf, None, None, q, K, nprobe, tiers=2)
    got, parts = _sharded_search(engs, q, K, nprobe)
    _assert_bits(got, want, "sharded")
    # every part is in (distance, id) order: the order the merge relies on
    p_ids, p_dst, p_cnt = parts
    for r in range(world):
        for i in range(nq):
            c = int(p_cnt[r, i])
            key = list(zip(p_dst[r, i, :c].tolist(), p_ids[r, i, :c].tolist()))
            assert key == sorted(key) and len(set(p_ids[r, i, :c].tolist())) == c
    if data == "lattice":
        assert _cross_rank_ties(want, _row_rank(case, world)) >= (20 if nq > 5 else 2), \
            "the lattice case has too few cross-rank ties in the top-k"
        if nq > 5:
            old = _merge_host(p_ids, p_dst, p_cnt, K, by_part=True)
            assert not np.array_equal(old[0], want[0]), "a rank-order merge would pass: the case tests nothing"

    # tombstones (the same id set on every shard: a shard accepts ids it does not hold), then also a filter
    dele = np.arange(3, n, 11, dtype=np.uint32)
    for e in engs:
        e.set_deleted(dele, True)
    bm_del = O.make_bitmap(n, dele)
    want = O.hybrid_batch_search(ivf, None, None, q, K, nprobe, tiers=2, deleted=bm_del)
    _assert_bits(_sharded_search(engs, q, K, nprobe)[0], want, "sharded + tombstones")
    keep = O.make_bitmap(n, np.flatnonzero(np.arange(n) % 3 != 1))
    want = O.hybrid_batch_search(ivf, None, None, q, K, nprobe, tiers=2, deleted=bm_del, filter_bits=keep)
    got = _sharded_search(engs, q, K, nprobe, filt=_dev(keep))[0]
    _assert_bits(got, want, "sharded + tombstones + filter")
    _close(engs)


@pytest.mark.parametrize("mode", ["exact", "tc"])
def test_unsharded_handle_on_lattice(lattice_case, mode):
    """Control: one handle over all lattice rows already returns the oracle's (distance, id) order."""
    e = Engine(LAT_D, k_max=64)
    _set_mode(e, mode)
    e.set_centroids(lattice_case["cents"])
    e.ivf_add(lattice_case["x"], np.arange(LAT_N, dtype=np.uint32))
    q = lattice_case["q"]
    got = e.search(q, K, LAT_NPROBE, tiers=L.TIER_HISTORICAL)
    _assert_bits(got, O.hybrid_batch_search(lattice_case["ivf"], None, None, q, K, LAT_NPROBE, tiers=2), "unsharded")
    e.close()


# ---- d. "probe nothing" key rows -------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["exact", "tc"])
def test_probe_nothing_rows(synth_case, mode):
    torch = _torch()
    engs, _ = _shards(synth_case, 1, mode)
    e = engs[0]
    q = synth_case["q"]
    nq = q.shape[0]
    dq = torch.from_numpy(q).cuda()
    keys = torch.empty((nq, NPROBE), dtype=torch.int64, device="cuda")
    e.coarse_device(dq.data_ptr(), nq, NPROBE, keys.data_ptr())

    def run(k_):
        out = [torch.empty((nq, K), dtype=torch.int32, device="cuda"),
               torch.empty((nq, K), dtype=torch.float32, device="cuda"),
               torch.empty((nq,), dtype=torch.int32, device="cuda")]
        e.search_device_coarse(dq.data_ptr(), nq, K, NPROBE, L.TIER_HISTORICAL, 0, 0, k_.data_ptr(),
                               *(t.data_ptr() for t in out))
        return _host(out)

    base = run(keys)
    _assert_bits(base, O.hybrid_batch_search(synth_case["ivf"], None, None, q, K, NPROBE, tiers=2), "given keys")
    wiped = [0, 5, 31, 32, nq - 1]
    k2 = keys.clone()
    k2[wiped] = -1
    got = run(k2)
    rest = np.setdiff1d(np.arange(nq), wiped)
    assert (got[2][wiped] == 0).all()
    assert (got[0][wiped] == ID_NONE).all() and (got[1][wiped].view(np.uint32) == INF_BITS).all()
    assert np.array_equal(got[2][rest], base[2][rest])
    assert np.array_equal(got[0][rest], base[0][rest])
    assert np.array_equal(got[1][rest].view(np.uint32), base[1][rest].view(np.uint32))
    _close(engs)


# ---- e. the pipelined entries on real engines ---------------------------------------------------------------------------
def _pipelined_group(engs, qs, k, nprobe):
    """ShardedIndex.submit / finish's steps: per batch, every shard's coarse slice (stream-ordered) and scan
    submit; the merge of batch i - 1 after every shard's wait(age=1); the last merge after wait(0); finish."""
    torch = _torch()
    nq = qs[0].shape[0]
    dqs = [torch.from_numpy(np.ascontiguousarray(q)).cuda() for q in qs]
    bufs, outs = [], []
    for i, dq in enumerate(dqs):
        keys = _coarse_keys(engs, dq, nprobe, submit=True)
        packs, views = _pack_bufs(nq, k, len(engs))
        for e, (pi, pd, pc) in zip(engs, views):
            e.search_device_coarse_submit(dq.data_ptr(), nq, k, nprobe, L.TIER_HISTORICAL, 0, 0, keys.data_ptr(), pi, pd, pc)
        bufs.append((keys, packs))
        if i:
            for e in engs:
                e.search_device_wait(1)
            outs.append(_merge_dev(engs[0], bufs[i - 1][1], nq, k))
    for e in engs:
        e.search_device_wait(0)
    outs.append(_merge_dev(engs[0], bufs[-1][1], nq, k))
    for e in engs:
        e.search_device_finish()
    res = [_host(o) for o in outs]
    del dqs, bufs
    return res, [e.stats().last_fallback_queries for e in engs]


def test_pipelined_sharded_search(synth_case):
    world = 3
    x, ivf = synth_case["x"], synth_case["ivf"]
    engs, _ = _shards(synth_case, world, "tc")
    qs = [synth.queries(100 * i, 64, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678) for i in range(5)]
    res, fb = _pipelined_group(engs, qs, K, NPROBE)
    if max(fb):
        # a proof failed on some shard: results exchanged before the repair are void, the driver answers the
        # group on the exact path (ShardedIndex._redo_exact); the shell group below checks that redo
        for e in engs:
            e.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
        res = [_sharded_search(engs, q, K, NPROBE)[0] for q in qs]
    for i, q in enumerate(qs):
        _assert_bits(res[i], O.hybrid_batch_search(ivf, None, None, q, K, NPROBE, tiers=2), f"batch {i} (fallback counts {fb})")
    _close(engs)

    # a near-duplicate shell (check_shard.py §3): 60 copies / near-copies of row 100 make the proof fail on
    # the shard that holds them; results exchanged from the unrepaired scan are not trusted, the group is
    # re-run on the exact path on every shard and equals the oracle
    x3 = x.copy()
    rng = np.random.default_rng(11)
    for j in range(60):
        x3[300 + j] = x3[100] if j % 3 == 0 else x3[100] + (1e-4 * rng.standard_normal(D)).astype(np.float32)
    q3 = np.concatenate([np.stack([x3[100] + (0.05 * rng.standard_normal(D)).astype(np.float32) for _ in range(16)]),
                         synth_case["q"][:48]])
    case3 = dict(x=x3, cents=synth_case["cents"])
    ivf3 = O.IVF(synth_case["cents"], x3, np.arange(N, dtype=np.uint32))
    engs, _ = _shards(case3, world, "tc")
    group = [q3, qs[0], q3[::-1].copy(), qs[1]]
    _, fb = _pipelined_group(engs, group, K, NPROBE)
    holder = owner_of_list(int(ivf3.assign[100]), world)
    assert fb[holder] > 0, f"no proof failure on the shard holding the shell (fallback counts {fb})"
    for e in engs:
        e.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    for i, q in enumerate(group):
        got, _ = _sharded_search(engs, q, K, NPROBE)
        _assert_bits(got, O.hybrid_batch_search(ivf3, None, None, q, K, NPROBE, tiers=2), f"redo of batch {i}")
    _close(engs)


# ---- f. unequal row norms and the proof floor ---------------------------------------------------------------------------
def test_unequal_norms_and_proof_floor(synth_case):
    x, cents = synth_case["x"], synth_case["cents"]
    world = 3
    x2 = x.copy()
    a = synth_case["ivf"].assign
    x2[a % 2 == 1] *= np.float32(3.0)
    case2 = dict(x=x2, cents=cents)
    ivf2 = O.IVF(cents, x2, np.arange(N, dtype=np.uint32))
    engs, _ = _shards(case2, world, "tc")
    sq = (x2.astype(np.float64) ** 2).sum(axis=1)
    rank_of_row = np.array([owner_of_list(int(l), world) for l in range(NLIST)])[ivf2.assign]
    xmax = []
    for r, e in enumerate(engs):
        got = e.ivf_max_sqnorm()
        ref = sq[rank_of_row == r].max()
        assert abs(got - ref) <= 1e-6 * ref, f"rank {r}: {got} vs {ref}"
        xmax.append(got)
    empty = Engine(D)
    empty.set_centroids(cents)
    assert empty.ivf_max_sqnorm() == 0.0
    for bad in (-1.0, float("nan")):
        with pytest.raises(FvdbError):
            empty.set_option(L.OPT_PROOF_XMAX, int(np.float32(bad).view(np.uint32)))
    empty.close()
    floor = int(np.float32(max(xmax)).view(np.uint32))
    for e in engs:
        e.set_option(L.OPT_PROOF_XMAX, floor)
    q = synth_case["q"]
    got, _ = _sharded_search(engs, q, K, NPROBE)
    _assert_bits(got, O.hybrid_batch_search(ivf2, None, None, q, K, NPROBE, tiers=2), "proof floor")
    _close(engs)


# ---- g. the sharded k-means blocks ---------------------------------------------------------------------------------------
def _accumulate(eng, dx, nlist, assign=None):
    torch = _torch()
    n, d = dx.shape
    sums = torch.zeros((nlist, d), dtype=torch.float32, device="cuda")
    counts = torch.zeros((nlist,), dtype=torch.int32, device="cuda")
    sqerr = torch.zeros((1,), dtype=torch.float64, device="cuda")
    changed = torch.zeros((1,), dtype=torch.int32, device="cuda")
    if assign is None:
        assign = torch.zeros((n,), dtype=torch.int32, device="cuda")
    eng.kmeans_accumulate_device(dx.data_ptr(), n, sums.data_ptr(), counts.data_ptr(), sqerr.data_ptr(),
                                 assign.data_ptr(), changed.data_ptr())
    torch.cuda.synchronize()
    return sums.cpu().numpy(), _u32(counts), float(sqerr.item()), int(changed.item()), assign


def test_sharded_kmeans_blocks():
    torch = _torch()
    d, nlist, world, n = 384, 64, 3, 30_000
    x = synth.rows(0, n, d, 4 * nlist, 1.0, 99)
    cents = x[:: n // nlist][:nlist].copy()
    per = (n + world - 1) // world
    sums = np.zeros((nlist, d), dtype=np.float64)
    counts = np.zeros(nlist, dtype=np.int64)
    sqerr = 0.0
    assigns = []
    for r in range(world):
        e = Engine(d)
        e.set_centroids(cents)
        xs = x[r * per:(r + 1) * per]
        dx = torch.from_numpy(xs).cuda()
        s, c, se, ch, a = _accumulate(e, dx, nlist)
        ha = _u32(a).copy()
        assert np.array_equal(ha, O.assign(xs, cents)), f"slice {r}: assignment differs from the oracle"
        assert ch == 1
        assert np.array_equal(c, np.bincount(ha, minlength=nlist)), f"slice {r}: counts"
        # a repeat with the same centroids: the assignment held in the buffer does not change
        _, c2, _, ch2, _ = _accumulate(e, dx, nlist, assign=a)
        assert ch2 == 0 and np.array_equal(c2, c)
        sums += s
        counts += c
        sqerr += se
        assigns.append(ha)
        e.close()
    a = np.concatenate(assigns)
    assert np.array_equal(counts, np.bincount(a, minlength=nlist))
    x64 = x.astype(np.float64)
    exact = np.zeros((nlist, d))
    absum = np.zeros((nlist, d))
    np.add.at(exact, a, x64)
    np.add.at(absum, a, np.abs(x64))
    bound = counts[:, None] * 2.0 ** -23 * absum
    assert (np.abs(sums - exact) <= bound).all(), "per-cluster sums outside the f32 summation bound"
    dist = np.empty(n, dtype=np.float32)
    for c in range(nlist):
        m = a == c
        if m.any():
            dist[m] = O.l2_many(cents[c], x[m])
    ref = float((dist.astype(np.float64) ** 2).sum())
    assert abs(sqerr - ref) <= 1e-9 * ref

    # apply: host sums and counts, count 0 keeps the previous centroid bits
    e = Engine(d)
    e.set_centroids(cents)
    rng = np.random.default_rng(3)
    h_sums = rng.standard_normal((nlist, d)).astype(np.float32) * np.float32(50)
    h_cnt = rng.integers(1, 5000, size=nlist).astype(np.uint32)
    h_cnt[[0, 7, nlist - 1]] = 0
    d_s, d_c = _dev(h_sums), _dev(h_cnt)
    e.kmeans_apply_device(d_s.data_ptr(), d_c.data_ptr())
    torch.cuda.synchronize()
    want = np.where(h_cnt[:, None] > 0, h_sums / np.maximum(h_cnt, 1).astype(np.float32)[:, None], cents).astype(np.float32)
    assert np.array_equal(e.get_centroids().view(np.uint32), want.view(np.uint32))
    e.close()


def test_kmeans_apply_invalidates_tensor_core_centroid_cache():
    """n x nlist >= 64M and nlist >= 256: the assignment runs on the tensor cores over a cached centroid tile
    set.  accumulate -> apply -> accumulate: the second assignment must see the applied centroids."""
    torch = _torch()
    d, nlist, n = 384, 1024, 65_536
    rng = np.random.default_rng(8)
    centers = rng.standard_normal((256, d)).astype(np.float32)
    x = (centers[rng.integers(0, 256, n)] + np.float32(0.5) * rng.standard_normal((n, d)).astype(np.float32))
    cents = x[rng.choice(n, nlist, replace=False)].copy()
    e = Engine(d)
    e.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    e.set_centroids(cents)
    dx = torch.from_numpy(x).cuda()
    sample = np.arange(0, n, 16)
    s, c, _, _, a = _accumulate(e, dx, nlist)
    assert np.array_equal(_u32(a)[sample], O.assign(x[sample], cents))
    d_s, d_c = _dev(s), _dev(c)
    e.kmeans_apply_device(d_s.data_ptr(), d_c.data_ptr())
    applied = e.get_centroids()
    assert not np.array_equal(applied, cents)
    _, _, _, ch, a2 = _accumulate(e, dx, nlist, assign=a)
    assert np.array_equal(_u32(a2)[sample], O.assign(x[sample], applied)), "assignment used stale centroids"
    assert ch == 1
    e.close()


def test_sharded_train_world1_matches_oracle_lloyd():
    torch = _torch()
    d, nlist, n, iters = 384, 64, 30_000, 6
    x = synth.rows(0, n, d, 4 * nlist, 1.0, 4321)
    init = x[:: n // nlist][:nlist].copy()
    e = Engine(d)
    res = ShardedIndex(e, 0, 1).train(torch.from_numpy(x).cuda(), nlist, iters, init)
    got = e.get_centroids()
    o_c, _, o_res = O.train_lloyd(x, init, iters)
    assert res["iterations"] == o_res["iterations"], (res, o_res)
    assert float(np.abs(got - o_c).max()) < 1e-4
    sample = x[::37]
    assert float((O.assign(sample, got) == O.assign(sample, o_c)).mean()) >= 0.999
    e.close()
