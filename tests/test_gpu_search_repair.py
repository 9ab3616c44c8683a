"""The exact repair of tensor-core proof failures in a hybrid search (FVDB_TIER_BOTH) on one handle.

Near-duplicate shells make the proof fail: one shell sits in both tiers at the same place, one in the IVF tier
alone and one in the recent tier alone, so a batch holds queries that fail in both tiers and queries that fail in
one tier only.  The recent tier (40 000 rows x 128 queries) is above the tensor-core threshold of 4M pairs.  The
synchronous entries, the stream-ordered ones and the split ("tiers") entry must all give the oracle's bits, and
the synchronous and stream-ordered entries must report the same number of re-run queries: each query once,
whichever tiers it failed in."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, _lib as L, synth
from fabstir_vectordb_b200.shard import tiers_pack_layout

pytestmark = pytest.mark.gpu

N, R, D, NLIST, NPROBE, K, NQ = 40_000, 40_000, 128, 64, 8, 10, 128


def _shell(rows, at, lo, n, rng):
    """rows[lo:lo + n] become near-copies of `at`: every third one exact, the others 1e-4 away."""
    for j in range(n):
        rows[lo + j] = at if j % 3 == 0 else at + (1e-4 * rng.standard_normal(D)).astype(np.float32)


@pytest.fixture(scope="module")
def case():
    import torch
    rng = np.random.default_rng(21)
    x = synth.rows(0, N, D, 4 * NLIST, 1.0, 1234)
    fx = synth.rows(N, R, D, 4 * NLIST, 1.0, 99)
    both, ivf_only, recent_only = x[100].copy(), x[20_000].copy(), fx[30_000].copy()
    _shell(x, both, 300, 80, rng)
    _shell(fx, both, 0, 80, rng)
    _shell(x, ivf_only, 20_300, 80, rng)
    _shell(fx, recent_only, 30_100, 80, rng)
    near = lambda at, n: [at + (0.05 * rng.standard_normal(D)).astype(np.float32) for _ in range(n)]  # noqa: E731
    q0 = synth.queries(0, NQ - 48, D, N, 4 * NLIST, 1.0, 1234, synth.default_qnoise(D, 1.0), 5678)
    q = np.stack(near(both, 16) + near(ivf_only, 16) + near(recent_only, 16) + list(q0)).astype(np.float32)
    q = q[rng.permutation(NQ)].copy()
    cents = x[:: N // NLIST][:NLIST].copy()
    ids = np.arange(N, dtype=np.uint32)
    fids = np.arange(N, N + R, dtype=np.uint32)
    eng = Engine(D, k_max=16)
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
    eng.set_centroids(cents)
    eng.ivf_add(x, ids)
    eng.flat_add(fx, fids)
    want = O.hybrid_batch_search(O.IVF(cents, x, ids), fx, fids, q, K, NPROBE, tiers=3)
    yield dict(eng=eng, q=q, dq=torch.from_numpy(q).cuda(), want=want)
    eng.close()


def _out():
    import torch
    return (torch.empty((NQ, K), dtype=torch.int32, device="cuda"), torch.empty((NQ, K), dtype=torch.float32, device="cuda"),
            torch.empty((NQ,), dtype=torch.int32, device="cuda"))


def _bits(out):
    import torch
    torch.cuda.synchronize()
    return tuple(t.cpu().numpy().view(np.uint32) for t in out)


def _assert_oracle(got, want, what):
    g_ids, g_dist, g_cnt = (np.asarray(a).view(np.uint32) for a in got)
    w_ids, w_dist, w_cnt = want
    assert np.array_equal(g_cnt, w_cnt), f"{what}: counts"
    for i in range(NQ):
        c = int(w_cnt[i])
        assert g_ids[i, :c].tolist() == w_ids[i, :c].tolist(), f"{what}: ids of query {i}"
        assert g_dist[i, :c].tolist() == w_dist[i, :c].view(np.uint32).tolist(), f"{what}: distance bits of query {i}"


def _fallbacks(eng, dq, tiers):
    out = _out()
    eng.search_device(dq.data_ptr(), NQ, K, NPROBE, tiers, 0, 0, *(t.data_ptr() for t in out))
    return eng.stats().last_fallback_queries


def test_case_fails_in_both_tiers_and_in_one(case):
    """The batch is what the other tests need: queries whose proof fails in both tiers, and in each tier alone."""
    eng, dq = case["eng"], case["dq"]
    assert eng.stats().flat_rows * NQ >= (4 << 20), "the recent tier must be scanned on the tensor cores"
    f_ivf = _fallbacks(eng, dq, L.TIER_HISTORICAL)
    f_recent = _fallbacks(eng, dq, L.TIER_RECENT)
    f_both = _fallbacks(eng, dq, L.TIER_BOTH)
    assert f_both < f_ivf + f_recent, f"no query fails in both tiers ({f_ivf} IVF, {f_recent} recent, {f_both} in all)"
    assert f_both > f_recent, f"no query fails in the IVF tier alone ({f_ivf} IVF, {f_recent} recent, {f_both} in all)"
    assert f_both > f_ivf, f"no query fails in the recent tier alone ({f_ivf} IVF, {f_recent} recent, {f_both} in all)"
    assert f_both <= 48 + NQ // 16, f"ordinary queries fell back too ({f_both})"


def test_synchronous_and_stream_ordered_repair_agree(case):
    import torch
    eng, dq, want = case["eng"], case["dq"], case["want"]
    sync = _out()
    eng.search_device(dq.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, 0, 0, *(t.data_ptr() for t in sync))
    st = eng.stats()
    fb_sync = st.last_fallback_queries
    assert fb_sync > 0, "no proof failed: the case tests nothing"
    assert st.last_nq == NQ, "the figures of a repaired call describe the caller's batch"
    got_sync = _bits(sync)
    _assert_oracle(got_sync, want, "synchronous device entry")

    s = torch.cuda.current_stream().cuda_stream
    deferred = _out()
    eng.search_device_submit(dq.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, 0, 0, *(t.data_ptr() for t in deferred), s)
    eng.search_device_finish(s)
    assert eng.stats().last_fallback_queries == fb_sync, "both entries count each re-run query once"
    got_deferred = _bits(deferred)
    for a, b in zip(got_deferred, got_sync):
        assert np.array_equal(a, b), "stream-ordered and synchronous results differ"

    host = eng.search(case["q"], K, NPROBE, tiers=L.TIER_BOTH)   # host buffers: the repair rewrites them too
    assert eng.stats().last_fallback_queries == fb_sync
    _assert_oracle(host, want, "host-buffer entry")


def test_split_entry_repair(case):
    """fvdb_search_device_tiers and its stream-ordered form give the same packed chunk, both parts repaired."""
    import torch
    eng, dq = case["eng"], case["dq"]
    chunk = tiers_pack_layout(NQ, K)[4]
    sync = torch.empty((chunk,), dtype=torch.int32, device="cuda")
    eng.search_device_tiers(dq.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, 0, 0, 0, sync.data_ptr())
    fb_sync = eng.stats().last_fallback_queries
    assert fb_sync > 0
    deferred = torch.full((chunk,), 0x7A7A7A7A, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()   # the marker is written before the engine's stream writes the chunk
    eng.search_device_tiers_submit(dq.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, 0, 0, 0, deferred.data_ptr())
    eng.search_device_finish()
    assert eng.stats().last_fallback_queries == fb_sync
    torch.cuda.synchronize()
    assert np.array_equal(sync.cpu().numpy(), deferred.cpu().numpy()), "synchronous and stream-ordered chunks differ"
    eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
    try:
        exact = torch.empty((chunk,), dtype=torch.int32, device="cuda")
        eng.search_device_tiers(dq.data_ptr(), NQ, K, NPROBE, L.TIER_BOTH, 0, 0, 0, exact.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(sync.cpu().numpy(), exact.cpu().numpy()), "the repaired chunk differs from exact mode"
    finally:
        eng.set_option(L.OPT_SCAN_MODE, L.SCAN_TC)
