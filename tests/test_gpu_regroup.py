"""The order of the IVF arena after every step that regroups a row tier: seal, the list-sharded adds (mod / rem and
owner table), vacuum, move_flat_to_ivf and take_unowned.  DESIGN §2 promises insertion order inside a list, and
fvdb_ivf_dump_lists exposes it, so the expected arena is built on the host as a stable sort by list, the lists coming
from the oracle's assignment, and compared exactly: ids and lists with dump_lists(), rows bit for bit with
fvdb_ivf_arena_device.  Insertion orders are shuffled, so a grouping that is not stable shows.

Also: device_bytes comes back to the same value after two identical add / move / delete / vacuum cycles."""
import numpy as np
import pytest

import oracle as O
from fabstir_vectordb_b200 import Engine, synth
from fabstir_vectordb_b200.shard import _tensor_at

pytestmark = pytest.mark.gpu

D, NLIST, N = 128, 32, 12_000


def _torch():
    import torch
    return torch


def _dev(a):
    torch = _torch()
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a.copy()).cuda()


@pytest.fixture(scope="module")
def data():
    x = synth.rows(0, N, D, 4 * NLIST, 1.0, 2468)
    cents = x[:: N // NLIST][:NLIST].copy()
    lists = O.assign(x, cents)   # row id i is row x[i]
    return dict(x=x, cents=cents, lists=lists, order=np.random.default_rng(11).permutation(N).astype(np.uint32))


def _engine(data):
    e = Engine(D, k_max=16)
    e.set_centroids(data["cents"])
    return e


def _expect(data, inserted):
    """(ids, lists) of an arena whose rows were inserted in the order `inserted`."""
    inserted = np.asarray(inserted, dtype=np.uint32)
    lists = data["lists"][inserted]
    o = np.argsort(lists, kind="stable")
    return inserted[o], lists[o]


def _check(e, data, want, what):
    ids, lists = e.dump_lists()
    assert np.array_equal(ids, want[0]), f"{what}: arena ids / order"
    assert np.array_equal(lists, want[1]), f"{what}: arena lists"
    p_rows, p_ids, n = e.ivf_arena_device()
    assert n == ids.size
    dev = _torch().device("cuda", 0)
    rows = _tensor_at(p_rows, (n, D), "<f4", dev).cpu().numpy()
    assert np.array_equal(rows.view(np.uint32), data["x"][ids].view(np.uint32)), f"{what}: arena rows"
    assert np.array_equal(_tensor_at(p_ids, (n,), "<i4", dev).cpu().numpy().view(np.uint32), ids)


def test_seal_onto_sealed_arena(data):
    x, order = data["x"], data["order"]
    a, b = order[:5_000], order[5_000:9_000]
    e = _engine(data)
    e.ivf_add(x[a], a)
    e.search(x[:8], 10, 4)   # seals the first batch
    _check(e, data, _expect(data, a), "first seal")
    e.ivf_add(x[b], b)       # pending rows behind a non-empty arena
    _check(e, data, _expect(data, np.concatenate([a, b])), "second seal")
    e.close()


def test_list_sharded_adds(data):
    torch = _torch()
    x, lists, order = data["x"], data["lists"], data["order"]
    sel = order[:8_000]
    dx, dids = torch.from_numpy(x[sel]).cuda(), _dev(sel)
    torch.cuda.synchronize()

    e = _engine(data)
    kept = e.ivf_add_device(dx.data_ptr(), dids.data_ptr(), sel.size, mod=3, rem=1)
    mine = sel[lists[sel] % 3 == 1]
    assert kept == mine.size
    _check(e, data, _expect(data, mine), "mod 3 rem 1")
    e.close()

    owner = np.random.default_rng(5).integers(0, 3, NLIST).astype(np.uint32)
    assert len(set(owner.tolist())) == 3
    d_owner = _dev(owner)
    e = _engine(data)
    kept = e.ivf_add_device_owned(dx.data_ptr(), dids.data_ptr(), sel.size, d_owner.data_ptr(), 1)
    mine = sel[owner[lists[sel]] == 1]
    assert kept == mine.size
    _check(e, data, _expect(data, mine), "owner table, rank 1")
    # a second owned add lands behind the first in every list
    more = order[8_000:10_000]
    mx, mids = torch.from_numpy(x[more]).cuda(), _dev(more)
    torch.cuda.synchronize()
    kept2 = e.ivf_add_device_owned(mx.data_ptr(), mids.data_ptr(), more.size, d_owner.data_ptr(), 1)
    more_mine = more[owner[lists[more]] == 1]
    assert kept2 == more_mine.size
    _check(e, data, _expect(data, np.concatenate([mine, more_mine])), "owner table, second add")
    e.close()


def test_vacuum_both_tiers(data):
    x, order = data["x"], data["order"]
    ivf, flat = order[:7_000], order[7_000:10_000]
    e = _engine(data)
    e.ivf_add(x[ivf], ivf)
    e.flat_add(x[flat], flat)
    rng = np.random.default_rng(7)
    dele = rng.choice(order[:10_000], 2_500, replace=False).astype(np.uint32)
    revive = dele[::5]
    e.set_deleted(dele, True)
    e.set_deleted(revive, False)
    gone = np.setdiff1d(dele, revive)
    assert e.vacuum() == gone.size
    _check(e, data, _expect(data, ivf[~np.isin(ivf, gone)]), "vacuum")
    st = e.stats()
    assert st.flat_rows == np.count_nonzero(~np.isin(flat, gone))
    assert st.deleted_rows == 0
    e.close()


def test_move_flat_to_ivf_follows_existing_rows(data):
    x, order = data["x"], data["order"]
    ivf, flat = order[:6_000], order[6_000:10_000]
    e = _engine(data)
    e.ivf_add(x[ivf], ivf)
    _check(e, data, _expect(data, ivf), "before the move")
    e.flat_add(x[flat], flat)
    move = np.random.default_rng(9).choice(flat, 1_500, replace=False).astype(np.uint32)   # not in flat order
    assert e.move_flat_to_ivf(move) == move.size
    moved_in_flat_order = flat[np.isin(flat, move)]
    _check(e, data, _expect(data, np.concatenate([ivf, moved_in_flat_order])), "move")
    assert e.stats().flat_rows == flat.size - move.size
    e.close()


def test_take_unowned_order(data):
    torch = _torch()
    x, lists, order = data["x"], data["lists"], data["order"]
    ins = order[:9_000]
    e = _engine(data)
    e.ivf_add(x[ins], ins)
    before = _expect(data, ins)
    _check(e, data, before, "before take")
    world, rank = 3, 0
    owner = np.random.default_rng(13).integers(0, world, NLIST).astype(np.uint32)
    d_owner = _dev(owner)
    dst = owner[before[1]]
    n_out = int(np.count_nonzero(dst != rank))
    out_x = torch.empty((n_out, D), dtype=torch.float32, device="cuda")
    out_i = torch.empty((n_out,), dtype=torch.int32, device="cuda")
    counts = e.ivf_take_unowned_device(d_owner.data_ptr(), rank, world, out_x.data_ptr(), out_i.data_ptr(), n_out)
    torch.cuda.synchronize()
    assert counts.tolist() == [int(np.count_nonzero(dst == r)) if r != rank else 0 for r in range(world)]
    # grouped by destination rank, in arena order within a rank
    want_taken = np.concatenate([before[0][dst == r] for r in range(world) if r != rank])
    taken = out_i.cpu().numpy().view(np.uint32)
    assert np.array_equal(taken, want_taken)
    assert np.array_equal(out_x.cpu().numpy().view(np.uint32), x[taken].view(np.uint32))
    kept = dst == rank
    _check(e, data, (before[0][kept], before[1][kept]), "kept after take")
    # the list offsets follow the compacted arena: an exact search equals the oracle over the kept rows
    q = x[order[9_000:9_064]]
    got = e.search(q, 10, 6)
    ivf = O.IVF(data["cents"], x[before[0][kept]], before[0][kept])
    want = O.hybrid_batch_search(ivf, None, None, q, 10, 6, tiers=3)
    assert np.array_equal(got[2], want[2].astype(np.uint32))
    for i, c in enumerate(want[2]):
        assert got[0][i, :c].tolist() == want[0][i, :c].tolist()
        assert got[1][i, :c].view(np.uint32).tolist() == want[1][i, :c].view(np.uint32).tolist()
    e.close()


def test_device_bytes_steady_state(data):
    x, order = data["x"], data["order"]
    ivf, flat = order[:6_000], order[6_000:9_000]
    e = _engine(data)
    after = []
    for _ in range(2):
        e.ivf_add(x[ivf], ivf)
        e.flat_add(x[flat], flat)
        assert e.move_flat_to_ivf(flat) == flat.size
        e.set_deleted(np.concatenate([ivf, flat]), True)
        assert e.vacuum() == ivf.size + flat.size
        st = e.stats()
        assert st.ivf_rows == 0 and st.flat_rows == 0
        after.append(st.device_bytes)
    assert after[0] == after[1], f"device_bytes drifts: {after}"
    e.close()
