"""Multi-GPU sharded hybrid index (SURVEY §8e): one process per GPU, torch.distributed for the
plumbing.  IVF list l lives on rank (l % world, or a place_lists table); centroids are replicated, so
every rank runs the same coarse step, scans only the probed lists it owns (the others are empty in its
arena) and emits a local top-k.  Recent-tier ("HNSW") rows live in slabs: row id r on rank r % world
(owner_of_recent_row), scanned exhaustively by the rank that holds them.

One exchange step: all-gather of the packed per-rank results, then the k-way merge of
src/hybrid/core.rs:482-483.  A one-tier search (FVDB_TIER_HISTORICAL, or FVDB_TIER_RECENT) gathers one part
per rank (ids | dist | count) and merges in (distance, row id) order (`fvdb_merge_topk_packed_device`).  A
FVDB_TIER_BOTH search keeps the tiers apart on every rank (`fvdb_search_device_tiers`: a recent part and an
IVF part per chunk) and merges the 2 * world parts in (distance, tier with recent first, row id) order
(`fvdb_merge_topk_tiers_packed_device`): exactly one unsharded FVDB_TIER_BOTH search, however the rows of
both tiers are split over the ranks.

Mutations (delete, vacuum, migrate) are broadcast: every rank applies them to the rows it holds.  The
tombstone and filter bitmaps are indexed by global row id, so a rank accepts ids it does not hold.  A
migrated row joins its nearest list in the arena of the rank that held it, whichever rank owns that list.
retrain / optimize_clusters re-cluster the IVF rows where they are and then move every row to the rank that
owns its new list, which restores a size-balanced placement.

The collective is torch.distributed (NCCL on GPUs; gloo in the CPU tests of the layout logic).
"""
from __future__ import annotations

import os
import time
from typing import Optional, Tuple

import numpy as np

from . import _lib as L
from .engine import Engine, NanInput


def owner_of_list(list_id: int, world: int) -> int:
    """List -> rank placement rule; must match fvdb_ivf_add_device(list_filter_mod=world)."""
    return list_id % world


def owner_of_recent_row(row_id: int, world: int) -> int:
    """Recent-tier row -> rank placement rule (slabs by id): a pure function of the id, so every rank agrees
    which rank holds a row without any table."""
    return row_id % world


def place_lists(sizes, world: int) -> np.ndarray:
    """Size-balanced list -> rank placement (SURVEY §8e): greedy bin packing, longest list first, each to
    the rank that holds the fewest rows so far (ties: the lower rank; equal sizes: the lower list id first),
    so that every GPU streams the same number of rows per batch.  Deterministic: every rank computes the
    same table from the same histogram.  Returns owner[nlist] (u32).  `l % world` (owner_of_list) is the
    fallback when no histogram is known."""
    sizes = np.asarray(sizes, dtype=np.int64)
    owner = np.zeros(sizes.shape[0], dtype=np.uint32)
    load = [0] * world
    for l in np.lexsort((np.arange(sizes.shape[0]), -sizes)):
        r = min(range(world), key=lambda i: (load[i], i))
        owner[l] = r
        load[r] += int(sizes[l])
    return owner


def kmeans_allreduce_step(sums, counts, sqerr, changed, group=None):
    """The exchange step of sharded k-means (SURVEY §8e, C2): every rank holds the per-cluster f32 sums
    [nlist x dim], counts [nlist], the squared-error sum and the "some assignment changed" flag of ITS
    points; one all-reduce (sum) of each makes them global, in place.  torch tensors on any device (NCCL on
    GPUs, gloo in the CPU tests).  Returns (total squared error, changed points, total points)."""
    import torch.distributed as dist
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(sqerr, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(changed, op=dist.ReduceOp.SUM, group=group)
    return float(sqerr.item()), int(changed.item()), int(counts.sum().item())


def gather_layout(nq: int, k: int, world: int) -> Tuple[Tuple[int, ...], Tuple[int, ...]]:
    """Shapes of the all-gathered buffers consumed by fvdb_merge_topk_device:
    ids/dist [world][nq][k], count [world][nq]."""
    return (world, nq, k), (world, nq)


def pack_layout(nq: int, k: int) -> Tuple[int, int, int, int]:
    """One rank's chunk of the single-collective exchange, in 32-bit words:
    (offset of ids [nq x k], offset of dist [nq x k], offset of count [nq], chunk length).
    Must match fvdb_merge_topk_packed_device."""
    nk = nq * k
    return 0, nk, 2 * nk, 2 * nk + nq


def tiers_pack_layout(nq: int, k: int) -> Tuple[int, int, int, int, int]:
    """One rank's chunk of a FVDB_TIER_BOTH exchange (fvdb_search_device_tiers), in 32-bit words: two
    pack_layout parts back to back, the recent tier then the IVF tier.  Returns (offset of ids, of dist, of
    count inside a part, part length, chunk length); part t starts at t * part length.  Must match
    fvdb_merge_topk_tiers_packed_device."""
    o_ids, o_dist, o_cnt, part = pack_layout(nq, k)
    return o_ids, o_dist, o_cnt, part, 2 * part


def merge_parts_reference(ids: np.ndarray, dist: np.ndarray, cnt: np.ndarray, k: int):
    """Host statement of the merge rule of fvdb_merge_topk_device, used by the CPU gloo tests to validate
    the gather layout; the product path merges on the GPU.  Order: (distance, row id), the ABI's tie rule,
    so that the merged result equals the unsharded search whichever rank holds which of two rows at the
    same distance.  The parts hold disjoint rows of one tier (an IVF-only sharded search, or recent-tier
    slabs); the first min(count, k) entries of each part count."""
    return _merge_reference(ids, dist, cnt, k, tiered=False)


def merge_tiers_reference(ids: np.ndarray, dist: np.ndarray, cnt: np.ndarray, k: int):
    """Host statement of fvdb_merge_topk_tiers_packed_device: ids / dist [2 * ranks][nq][k], cnt
    [2 * ranks][nq], part 2r = recent tier of rank r, part 2r + 1 = IVF tier of rank r.  Order: (distance,
    tier with recent first, row id), the order of one unsharded FVDB_TIER_BOTH search (the stable sort of
    src/hybrid/core.rs:482-483 over recent-then-IVF results, each tier in (distance, row id) order)."""
    return _merge_reference(ids, dist, cnt, k, tiered=True)


def _merge_reference(ids, dist, cnt, k, tiered):
    parts, nq, _ = ids.shape
    out_ids = np.full((nq, k), 0xFFFFFFFF, dtype=np.uint32)
    out_dist = np.full((nq, k), np.inf, dtype=np.float32)
    out_cnt = np.zeros(nq, dtype=np.uint32)
    for q in range(nq):
        cand = []
        for p in range(parts):
            for j in range(min(int(cnt[p, q]), k)):
                cand.append((float(dist[p, q, j]), p & 1 if tiered else 0, int(ids[p, q, j])))
        cand.sort()
        cand = cand[:k]
        out_cnt[q] = len(cand)
        for o, c in enumerate(cand):
            out_ids[q, o] = c[2]
            out_dist[q, o] = c[0]
    return out_ids, out_dist, out_cnt


def _cur_stream(t=None) -> int:
    """The caller's CUDA stream (0 when the tensors live on the host: the gloo tests drive this class with a
    stand-in engine over CPU tensors)."""
    import torch
    if t is not None and not t.is_cuda:
        return 0
    return torch.cuda.current_stream().cuda_stream


def _tensor_at(ptr: int, shape, typestr: str, device):
    """A torch tensor over memory the engine owns (no copy): __cuda_array_interface__ on a GPU, the raw bytes on
    the host (the gloo tests' stand-in engines)."""
    import ctypes
    import torch
    n = int(np.prod(shape))
    dtype = {"<f4": torch.float32, "<i4": torch.int32}[typestr]
    if n == 0:
        return torch.empty(shape, dtype=dtype, device=device)
    if device.type == "cuda":
        # torch refuses the read-only flag; the callers only read through the tensor
        view = type("_DeviceView", (), {"__cuda_array_interface__": dict(shape=tuple(shape), typestr=typestr,
                                                                          data=(ptr, False), version=3)})()
        return torch.as_tensor(view, device=device)
    return torch.frombuffer((ctypes.c_char * (4 * n)).from_address(ptr), dtype=dtype).view(shape)


class ShardedIndex:
    """One rank's shard + the exchange step.  All tensors are torch CUDA tensors."""

    def __init__(self, engine: Engine, rank: int, world: int, group=None):
        self.eng = engine
        self.rank = rank
        self.world = world
        self.group = group
        self.shard_coarse = os.environ.get("FVDB_SHARD_COARSE", "1") != "0"
        self.share_bounds = os.environ.get("FVDB_SHARE_BOUNDS", "1") != "0"
        self._bounds_cap = 0
        self._bufs = {}
        self.owner = None
        self.owner_host = None
        self._inflight = None      # pipelined sharded search: the batch whose results are not exchanged yet
        self._group = []           # ... and every batch submitted since the last finish()
        self._nlist = None
        self._deferred_error = None
        # an IVF-tier mutation can raise a rank's largest row norm: FVDB_OPT_PROOF_XMAX is max-reduced again
        # before the next search (every rank mutates in the same order, so every rank sees the same flag)
        self._xmax_dirty = False
        # the coarse step of a pipelined batch: stream-ordered until a proof failure shows up there (dense
        # centroid tables, e.g. nlist 16384), then the synchronous, self-repairing entry (see submit / finish)
        self.coarse_async = os.environ.get("FVDB_SHARD_COARSE_ASYNC", "1") == "1"

    def _setup_bound_sharing(self, nq: int, device):
        """Exchange the inter-process handles of the per-query bound arrays (once per capacity)."""
        import torch
        import torch.distributed as dist
        # no rank may free its exported array while a peer still has it mapped
        self.eng.bounds_close_peers()
        dist.barrier(group=self.group)
        self._reduce_xmax(device)
        mine = torch.frombuffer(bytearray(self.eng.bounds_export(nq)), dtype=torch.uint8).to(device)
        allh = torch.empty((self.world * 64,), dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(allh, mine, group=self.group)
        self.eng.bounds_import(bytes(allh.cpu().numpy().tobytes()), self.world, self.rank)
        self._bounds_cap = nq

    def _reduce_xmax(self, device):
        """Rows of this shard can be dropped by a bound a peer published: the tensor-core proof of every shard
        uses the largest row norm of ALL shards (FVDB_OPT_PROOF_XMAX).  One all-reduce (max)."""
        import torch
        import torch.distributed as dist
        xm = torch.tensor([self.eng.ivf_max_sqnorm()], dtype=torch.float32, device=device)
        dist.all_reduce(xm, op=dist.ReduceOp.MAX, group=self.group)
        self.eng.set_option(L.OPT_PROOF_XMAX, int(np.float32(xm.item()).view(np.uint32)))
        self._xmax_dirty = False

    def _begin_batch(self, q, nq: int, stream: int):
        """NVLink bound sharing: reset this rank's bound array BEFORE the coarse all-gather (which orders the
        reset before any peer's scan of this batch); the proof floor is re-reduced first after an IVF-tier
        mutation."""
        if not (self.share_bounds and self.world <= 8):
            return
        if q.is_cuda and nq > self._bounds_cap:
            self._setup_bound_sharing(nq, q.device)
        elif self._xmax_dirty:
            self._reduce_xmax(q.device)
        if q.is_cuda:
            self.eng.bounds_begin_batch(nq, stream)

    def _device(self):
        """Where this rank's collectives run: the host under gloo (the CPU tests), else the current GPU."""
        import torch
        import torch.distributed as dist
        if self.world > 1 and dist.is_initialized() and dist.get_backend(self.group) == "gloo":
            return torch.device("cpu")
        return torch.device("cuda", torch.cuda.current_device())

    def set_placement(self, owner):
        """Install a list -> rank table (place_lists) in place of the l % world rule; `owner` is a host
        array [nlist].  Rows loaded afterwards are kept when owner[list] == rank."""
        import torch
        self.owner_host = np.ascontiguousarray(owner, dtype=np.uint32)
        self.owner = torch.from_numpy(self.owner_host.view(np.int32)).to(self._device())

    def list_histogram_device(self, x, hist):
        """hist[l] += number of rows of x (CUDA tensor [n x dim]) whose nearest centroid is l: the input of
        place_lists, computed without moving rows (fvdb_assign_device)."""
        import torch
        a = torch.empty((x.shape[0],), dtype=torch.int32, device=x.device)
        self.eng.assign_device(x.data_ptr(), x.shape[0], a.data_ptr(), torch.cuda.current_stream().cuda_stream)
        hist += torch.bincount(a.long(), minlength=hist.shape[0])

    def add_rows_device(self, x, row_ids) -> int:
        """Assign rows to lists and keep those this rank owns (every rank calls this with the same rows)."""
        self._xmax_dirty = True
        if getattr(self, "owner", None) is not None:
            return self.eng.ivf_add_device_owned(x.data_ptr(), row_ids.data_ptr(), x.shape[0], self.owner.data_ptr(),
                                                 self.rank)
        return self.eng.ivf_add_device(x.data_ptr(), row_ids.data_ptr(), x.shape[0], self.world, self.rank)

    def add_recent_rows_device(self, x, row_ids) -> int:
        """Recent-tier insert (HNSWIndex::insert, src/hnsw/core.rs:226): every rank is handed the same rows
        (CUDA tensors x [n x dim], row_ids [n] int32) and keeps those it holds by owner_of_recent_row.
        Returns the number of rows kept on this rank."""
        if self.world > 1:
            mine = (row_ids.long() & 0xFFFFFFFF) % self.world == self.rank
            x, row_ids = x[mine].contiguous(), row_ids[mine].contiguous()
        n = int(x.shape[0])
        if n:
            self.eng.flat_add_device(x.data_ptr(), row_ids.data_ptr(), n)
        return n

    def _sum_over_ranks(self, v: int) -> int:
        if self.world == 1:
            return int(v)
        import torch
        import torch.distributed as dist
        t = torch.tensor([int(v)], dtype=torch.int64, device=self._device())
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return int(t.item())

    def delete(self, row_ids, deleted: bool = True):
        """IVFIndex::mark_deleted / HNSWIndex::mark_deleted on every rank (fvdb_set_deleted): `row_ids` is a
        host array, the same on every rank.  The tombstone bitmap is indexed by global row id, so every rank
        takes the whole list; sharded handles (loaded through the device entries) do not track which ids they
        hold, so ids held by other ranks, or by none, are accepted."""
        self.eng.set_deleted(np.ascontiguousarray(row_ids, dtype=np.uint32), deleted)

    def vacuum(self) -> int:
        """fvdb_vacuum on every rank: drop the tombstoned rows each rank holds.  Returns the rows removed on
        all ranks."""
        self._xmax_dirty = True
        return self._sum_over_ranks(self.eng.vacuum())

    def migrate(self, row_ids) -> int:
        """HybridIndex::migrate_with_threshold (fvdb_move_flat_to_ivf) on every rank: each rank moves those of
        `row_ids` (host array, the same on every rank) that sit in its recent slab into its IVF arena.  A moved
        row joins its nearest list on the rank that held it, even when another rank owns that list: results
        do not change (every rank scans its own rows of every probed list), but the per-rank scan load drifts
        from the placement's balance as rows migrate.  Returns the rows moved on all ranks."""
        self._xmax_dirty = True
        return self._sum_over_ranks(self.eng.move_flat_to_ivf(np.ascontiguousarray(row_ids, dtype=np.uint32)))

    def train(self, points, nlist: int, max_iterations: int, init_centroids, eng: Optional[Engine] = None):
        """IVFIndex::train (src/ivf/core.rs:240-334) with the points sharded over the ranks (SURVEY §8e):
        `points` is THIS rank's slice (CUDA tensor [n_r x dim]), `init_centroids` [nlist x dim] (host array,
        the same on every rank).  The centroids are trained on `eng` (default: this rank's engine; retrain
        passes a scratch handle).  Per iteration every rank assigns its points against the replicated
        centroid table and accumulates per-cluster sums and counts (fvdb_kmeans_accumulate_device), one
        all-reduce makes them global (kmeans_allreduce_step), every rank installs the same means
        (fvdb_kmeans_apply_device; an empty cluster keeps its centroid, :410-415).  Stop rule of :303-321 on
        the mean squared distance measured at assignment time.  The sums are unordered f32 atomics, so the
        centroids agree with the single-GPU (order-faithful) ones to rounding, not bit for bit.
        Returns dict(iterations, converged, initial_error, final_error); like the reference, training
        leaves every posting list empty."""
        import torch
        eng = self.eng if eng is None else eng
        dev = points.device
        dim = points.shape[1]
        n_r = points.shape[0]
        stream = _cur_stream(points)
        eng.set_centroids(np.ascontiguousarray(init_centroids, dtype=np.float32))
        sums = torch.zeros((nlist, dim), dtype=torch.float32, device=dev)
        counts = torch.zeros((nlist,), dtype=torch.int32, device=dev)
        sqerr = torch.zeros((1,), dtype=torch.float64, device=dev)
        changed = torch.zeros((1,), dtype=torch.int32, device=dev)
        assign = torch.zeros((max(n_r, 1),), dtype=torch.int32, device=dev)    # vec![ClusterId(0); n]
        prev_err, initial, err = float("inf"), None, 0.0
        converged, iterations = False, 0
        for it in range(max_iterations):
            iterations = it + 1
            sums.zero_(); counts.zero_(); sqerr.zero_(); changed.zero_()
            if n_r:
                eng.kmeans_accumulate_device(points.data_ptr(), n_r, sums.data_ptr(), counts.data_ptr(),
                                             sqerr.data_ptr(), assign.data_ptr(), changed.data_ptr(), stream)
            if self.world > 1:
                tot, n_changed, n_total = kmeans_allreduce_step(sums, counts, sqerr, changed, self.group)
            else:
                tot, n_changed, n_total = float(sqerr.item()), int(changed.item()), int(counts.sum().item())
            err = tot / max(1, n_total)
            if initial is None:
                initial = err
            eng.kmeans_apply_device(sums.data_ptr(), counts.data_ptr(), stream)
            if iterations >= max_iterations:
                break
            if n_changed == 0 or (prev_err != float("inf") and abs(prev_err - err) / prev_err < 1e-4):
                converged = True
                break
            prev_err = err
        if points.is_cuda:
            torch.cuda.synchronize()
        return dict(iterations=iterations, converged=converged, initial_error=initial, final_error=err)

    def retrain(self, nlist: int, max_iterations: int, init_centroids) -> dict:
        """IVFIndex::retrain (src/ivf/operations.rs:148-193) over the list-sharded IVF tier, without a host copy of
        any row.  Every rank calls it with the same arguments; `init_centroids` [nlist x dim] is a host array.

        1. The sharded Lloyd of train() runs on a scratch handle over this rank's arena as it is
           (fvdb_ivf_arena_device: every IVF row, tombstoned rows included); this handle's centroids keep
           grouping the arena meanwhile.  The final centroids are bit-identical on every rank (all-reduced sums).
        2. fvdb_ivf_reassign installs them and moves every row to its nearest new list, in place.
        3. The list histogram is all-reduced and place_lists makes the new placement (set_placement).
        4. fvdb_ivf_take_unowned_device takes out the rows of lists other ranks own; two all_to_all_single
           exchanges (the counts, then the rows and ids) deliver them, and each rank adds what it received
           (add_rows_device).
        Afterwards every row sits on the rank that owns its list, as after a fresh balanced build.

        Failure rule: a row on a rank that does not own its list is legal (migrate makes such rows), so when the
        exchange fails each rank puts the rows it took back into its own arena (fvdb_ivf_add_device, mod 1) and
        the error propagates: results stay exact, only the balance is lost.

        Peak device memory per rank is about three times its arena: the arena, the rows it sends and the rows it
        receives, while the received rows are added.

        Pipelined batches must be finished first (RuntimeError otherwise).  Returns dict(old_nlist, new_nlist,
        rows_reassigned and rows_moved summed over the ranks, converged, iterations, seconds): `seconds` holds this
        rank's host-clock time of each step (lloyd, reassign, placement, exchange); every step ends in a
        synchronisation."""
        import torch
        import torch.distributed as dist
        if self._inflight is not None or self._group:
            raise RuntimeError("retrain: submitted search batches are in flight; call finish() first")
        dev = self._device()
        old_nlist = int(self.eng.stats().nlist)
        init = np.ascontiguousarray(init_centroids, dtype=np.float32).reshape(nlist, self.eng.dim)

        secs, t0 = {}, time.perf_counter()

        def lap(name):
            nonlocal t0
            t1 = time.perf_counter()
            secs[name], t0 = t1 - t0, t1

        # 1. Lloyd on a scratch handle over the arena as it stands
        p_rows, _, n = self.eng.ivf_arena_device()
        rows = _tensor_at(p_rows, (n, self.eng.dim), "<f4", dev)
        scratch = self._new_scratch()
        try:
            tr = self.train(rows, nlist, max_iterations, init, eng=scratch)
            cents = scratch.get_centroids()
        finally:
            scratch.close()
        del rows
        lap("lloyd")
        try:
            # 2. every row to its nearest new list, in place
            self.eng.ivf_reassign(cents)
            lap("reassign")
            # 3. the new placement from the global list histogram
            _, lists = self.eng.dump_lists()
            hist = torch.from_numpy(np.bincount(lists, minlength=nlist).astype(np.int64)).to(dev)
            if self.world > 1:
                dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=self.group)
            self.set_placement(place_lists(hist.cpu().numpy(), self.world))
            lap("placement")
            # 4. rows to their owners
            moved = self._exchange_unowned(dev) if self.world > 1 else 0
            lap("exchange")
        finally:
            # the centroid table (and with it nlist) and the rows of the IVF tier have changed
            self._xmax_dirty = True
            self._nlist = None
            self._bufs = {k: v for k, v in self._bufs.items() if k[0] != "coarse"}
        self._nlist = nlist
        return dict(old_nlist=old_nlist, new_nlist=nlist, rows_reassigned=self._sum_over_ranks(n),
                    rows_moved=self._sum_over_ranks(moved), converged=tr["converged"], iterations=tr["iterations"],
                    seconds=secs)

    def optimize_clusters(self, max_iterations: int = 25) -> dict:
        """IVFIndex::optimize_clusters (src/ivf/operations.rs:221-260) on the sharded index: retrain with the same
        nlist, starting from the current centroids."""
        cents = self.eng.get_centroids()
        return self.retrain(cents.shape[0], max_iterations, cents)

    def add_clusters(self, n_clusters_to_add: int, init_centroids, max_iterations: int = 25) -> dict:
        """IVFIndex::add_clusters (src/ivf/operations.rs:195-219) on the sharded index: retrain with nlist +
        n_clusters_to_add from `init_centroids` [nlist + n x dim] (host, the same on every rank)."""
        return self.retrain(int(self.eng.stats().nlist) + n_clusters_to_add, max_iterations, init_centroids)

    def _new_scratch(self) -> Engine:
        """The handle the working centroids of a retrain live on (this rank's device, no rows)."""
        return Engine(self.eng.dim, k_max=1, device=self.eng.device)

    def _exchange_unowned(self, dev) -> int:
        """Step 4 of retrain: take out the rows of other ranks' lists, exchange, add.  Returns the rows sent."""
        import torch
        import torch.distributed as dist
        stream = _cur_stream(self.owner)
        counts = self.eng.ivf_take_unowned_device(self.owner.data_ptr(), self.rank, self.world, stream=stream)
        n_send = int(counts.sum())
        send_x = torch.empty((n_send, self.eng.dim), dtype=torch.float32, device=dev)
        send_ids = torch.empty((n_send,), dtype=torch.int32, device=dev)
        if n_send:
            self.eng.ivf_take_unowned_device(self.owner.data_ptr(), self.rank, self.world, send_x.data_ptr(),
                                             send_ids.data_ptr(), n_send, stream)
        try:
            send_counts = torch.from_numpy(counts.astype(np.int64)).to(dev)
            recv_counts = torch.empty_like(send_counts)
            dist.all_to_all_single(recv_counts, send_counts, group=self.group)
            recv_counts = recv_counts.cpu().numpy().tolist()
            recv_x = torch.empty((sum(recv_counts), self.eng.dim), dtype=torch.float32, device=dev)
            recv_ids = torch.empty((sum(recv_counts),), dtype=torch.int32, device=dev)
            split = counts.astype(np.int64).tolist()
            dist.all_to_all_single(recv_x, send_x, recv_counts, split, group=self.group)
            dist.all_to_all_single(recv_ids, send_ids, recv_counts, split, group=self.group)
        except Exception:
            if n_send:      # the failure rule: the taken rows go back into this rank's own arena
                self.eng.ivf_add_device(send_x.data_ptr(), send_ids.data_ptr(), n_send, 1, 0)
            raise
        del send_x, send_ids
        n_recv = int(recv_x.shape[0])
        if recv_x.is_cuda:      # the engine reads the rows on its own stream
            torch.cuda.current_stream().synchronize()
        if n_recv:
            kept = self.add_rows_device(recv_x, recv_ids)
            if kept != n_recv:
                raise RuntimeError(f"retrain: rank {self.rank} kept {kept} of the {n_recv} rows it received")
        return n_send

    def _buffers(self, nq: int, k: int, device, slot: int = 0, tiered: bool = False):
        import torch
        key = (nq, k, slot, tiered)
        if key not in self._bufs:
            o_ids, o_dist, o_cnt, chunk = pack_layout(nq, k)
            if tiered:     # two parts, recent tier then IVF tier (tiers_pack_layout); ids / dist / cnt: the first
                chunk = tiers_pack_layout(nq, k)[4]
            # this rank's results are written straight into the three sections of its packed chunk
            pack = torch.empty((chunk,), dtype=torch.int32, device=device)
            self._bufs[key] = dict(
                pack=pack,
                ids=pack[o_ids:o_ids + nq * k].view(nq, k),
                dist=pack[o_dist:o_dist + nq * k].view(torch.float32).view(nq, k),
                cnt=pack[o_cnt:o_cnt + nq],
                g_pack=torch.empty((self.world, chunk), dtype=torch.int32, device=device),
                o_ids=torch.empty((nq, k), dtype=torch.int32, device=device),
                o_dist=torch.empty((nq, k), dtype=torch.float32, device=device),
                o_cnt=torch.empty((nq,), dtype=torch.int32, device=device),
            )
        return self._bufs[key]

    def submit(self, q, k: int, nprobe: int, tiers: int = L.TIER_HISTORICAL, slot: int = 0):
        """Stream-ordered search: enqueue the batch and return its result tensors, which are valid after
        finish().  `slot` selects one of several buffer sets, so that batches in flight do not share one;
        `q` must stay alive and untouched until finish().

        One GPU: fvdb_search_device_submit.  Several GPUs: a two-deep software pipeline over the same four
        steps as search() — while the engine scans batch i in one of its pipeline slots, batch i + 1's
        coarse slice and the all-gather of its keys are already running on the caller's stream, and batch
        i's result exchange (one all-gather of the packed chunks + merge) is enqueued only after batch
        i + 1's scan has been handed to the engine (fvdb_search_device_wait joins it on the device).  No
        host synchronisation per batch.  The NVLink bound arrays stay safe: a rank's reset for batch i + 2
        is ordered behind its all-gather of batch i's results, which needs every peer's finished scan of i.

        tiers: FVDB_TIER_HISTORICAL, or FVDB_TIER_BOTH (fvdb_search_device_tiers_submit + the tiered merge).
        A rank that holds recent-tier rows runs a hybrid batch on the handle's own stream, not in a pipeline
        slot: it is stream-ordered and correct but does not overlap its neighbours."""
        import torch
        import torch.distributed as dist
        nq = q.shape[0]
        tiered = self.world > 1 and tiers == L.TIER_BOTH
        b = self._buffers(nq, k, q.device, slot, tiered)
        stream = _cur_stream(q)
        if self.world == 1:
            self.eng.search_device_submit(q.data_ptr(), nq, k, nprobe, tiers, 0, 0, b["ids"].data_ptr(),
                                          b["dist"].data_ptr(), b["cnt"].data_ptr(), stream)
            return b["ids"], b["dist"], b["cnt"]
        assert tiers in (L.TIER_HISTORICAL, L.TIER_BOTH) and nprobe > 0 and self.shard_coarse, \
            "pipelined sharded search: the IVF tier, or both tiers"
        np_ = min(nprobe, self.eng.stats().nlist) if self._nlist is None else min(nprobe, self._nlist)
        if self._nlist is None:
            self._nlist = self.eng.stats().nlist
        self._begin_batch(q, nq, stream)
        per = (nq + self.world - 1) // self.world
        key = ("coarse", nq, np_, slot)
        if key not in self._bufs:
            self._bufs[key] = (torch.empty((per, np_), dtype=torch.int64, device=q.device),
                               torch.empty((self.world * per, np_), dtype=torch.int64, device=q.device))
        mine, allk = self._bufs[key]
        lo = min(nq, self.rank * per)
        n_mine = max(0, min(nq, lo + per) - lo)
        if n_mine < per:
            mine.fill_(-1)
        if n_mine:
            # The coarse step of the slice: the stream-ordered entry (no host round trip; a proof failure makes
            # finish() re-run the group) until such a failure has been seen once — dense centroid tables (nlist
            # 16384) produce a few per batch — then the synchronous entry, which repairs them on the spot and
            # whose host synchronisation only waits for THIS stream while the previous batch keeps scanning.
            try:
                if self.coarse_async:
                    self.eng.coarse_device_submit(q[lo:lo + n_mine].data_ptr(), n_mine, np_, mine.data_ptr(), stream)
                else:
                    self.eng.coarse_device(q[lo:lo + n_mine].data_ptr(), n_mine, np_, mine.data_ptr(), stream)
            except NanInput as e:      # every rank has to reach the collectives: raise at finish()
                mine.fill_(-1)
                self._deferred_error = e
        dist.all_gather_into_tensor(allk, mine, group=self.group)
        if tiered:
            self.eng.search_device_tiers_submit(q.data_ptr(), nq, k, np_, tiers, 0, 0, allk.data_ptr(),
                                                b["pack"].data_ptr(), stream)
        else:
            self.eng.search_device_coarse_submit(q.data_ptr(), nq, k, np_, tiers, 0, 0, allk.data_ptr(),
                                                 b["ids"].data_ptr(), b["dist"].data_ptr(), b["cnt"].data_ptr(), stream)
        if self._inflight is not None:
            self._exchange(self._inflight, age=1)
        self._inflight = (b, nq, k, tiered)
        self._group.append((q, k, nprobe, tiers, slot))
        return b["o_ids"], b["o_dist"], b["o_cnt"]

    def _exchange(self, rec, age: int):
        """Result exchange of a submitted batch: join its scan on the device, ONE all-gather, merge."""
        import torch
        import torch.distributed as dist
        b, nq, k, tiered = rec
        stream = _cur_stream(b["pack"])
        self.eng.search_device_wait(age, stream)
        dist.all_gather_into_tensor(b["g_pack"].view(-1), b["pack"], group=self.group)
        self._merge(b, nq, k, tiered, stream)

    def _merge(self, b, nq: int, k: int, tiered: bool, stream: int):
        merge = self.eng.merge_topk_tiers_packed_device if tiered else self.eng.merge_topk_packed_device
        merge(b["g_pack"].data_ptr(), self.world, nq, k, b["o_ids"].data_ptr(), b["o_dist"].data_ptr(),
              b["o_cnt"].data_ptr(), stream)

    def finish(self):
        """Wait for every submitted batch.  Raises NanInput if one held a NaN query.  Several GPUs: if the
        tensor-core proof failed for some query on ANY rank (rare), every rank re-runs the group through the
        synchronous path, which repairs such queries before results are exchanged."""
        import torch
        import torch.distributed as dist
        on_host = self._inflight is not None and not self._inflight[0]["pack"].is_cuda
        stream = 0 if on_host else _cur_stream()
        if self.world > 1 and self._inflight is not None:
            self._exchange(self._inflight, age=0)
            self._inflight = None
        try:
            self.eng.search_device_finish(stream)
        finally:
            err, self._deferred_error = self._deferred_error, None
        if err is not None:
            self._group = []
            raise err
        if self.world > 1:
            group, self._group = self._group, []
            fb = torch.tensor([self.eng.stats().last_fallback_queries], dtype=torch.int32,
                              device=torch.device("cpu") if on_host else torch.device("cuda", torch.cuda.current_device()))
            dist.all_reduce(fb, op=dist.ReduceOp.MAX, group=self.group)
            if int(fb.item()) > 0:
                self.coarse_async = False     # (every rank sees the same all-reduced count)
                self._redo_exact(group)

    def _redo_exact(self, group):
        """A tensor-core proof failed for some query on SOME rank.  Rows of that query may have been dropped on
        OTHER ranks by a bound the failing rank published — their exclusion rested on the proof that failed — so
        no rank's tensor-core result can be kept: every rank answers the batches on the exact path."""
        import torch
        mode = L.SCAN_TC
        self.eng.set_option(L.OPT_SCAN_MODE, L.SCAN_EXACT)
        try:
            for q, k, nprobe, tiers, slot in group:
                self.search(q, k, nprobe, tiers=tiers, slot=slot, _check=False)
            if group and group[0][0].is_cuda:
                torch.cuda.synchronize()
        finally:
            self.eng.set_option(L.OPT_SCAN_MODE, mode)

    def search(self, q, k: int, nprobe: int, tiers: int = L.TIER_HISTORICAL, filter_bits=None,
               filter_nbits: int = 0, slot: int = 0, _check: bool = True):
        """q: [nq x dim] CUDA tensor, identical on every rank.  Returns (ids, dist, cnt) CUDA
        tensors holding the GLOBAL top-k on every rank.  tiers = FVDB_TIER_BOTH is HybridIndex::search over
        both tiers (fvdb_search_device_tiers on every rank, the tiered merge); one tier alone merges by
        (distance, row id)."""
        import torch
        import torch.distributed as dist
        nq = q.shape[0]
        tiered = self.world > 1 and tiers == L.TIER_BOTH
        b = self._buffers(nq, k, q.device, slot, tiered)
        stream = _cur_stream(q)
        f_ptr = filter_bits.data_ptr() if filter_bits is not None else 0
        if self.world == 1:
            self.eng.search_device(q.data_ptr(), nq, k, nprobe, tiers, f_ptr, filter_nbits,
                                   b["ids"].data_ptr(), b["dist"].data_ptr(), b["cnt"].data_ptr(), stream)
            return b["ids"], b["dist"], b["cnt"]
        coarse = 0
        if (tiers & L.TIER_HISTORICAL) and nprobe > 0 and self.shard_coarse:
            # the coarse step is sharded by QUERY: each rank ranks its slice of the batch against the
            # (replicated) centroid table, one small all-gather hands every rank the whole ranking
            np_ = min(nprobe, self.eng.stats().nlist)
            self._begin_batch(q, nq, stream)
            per = (nq + self.world - 1) // self.world
            key = ("coarse", nq, np_)
            if key not in self._bufs:
                self._bufs[key] = (torch.empty((per, np_), dtype=torch.int64, device=q.device),
                                   torch.empty((self.world * per, np_), dtype=torch.int64, device=q.device))
            mine, allk = self._bufs[key]
            lo = min(nq, self.rank * per)
            n_mine = max(0, min(nq, lo + per) - lo)
            if n_mine < per:
                mine.fill_(-1)                                   # 0xFF..FF keys: "probe nothing"
            if n_mine:
                self.eng.coarse_device(q[lo:lo + n_mine].data_ptr(), n_mine, np_, mine.data_ptr(), stream)
            dist.all_gather_into_tensor(allk, mine, group=self.group)
            coarse, nprobe = allk.data_ptr(), np_
        if tiered:
            self.eng.search_device_tiers(q.data_ptr(), nq, k, nprobe, tiers, f_ptr, filter_nbits, coarse,
                                         b["pack"].data_ptr(), stream)
        else:
            self.eng.search_device_coarse(q.data_ptr(), nq, k, nprobe, tiers, f_ptr, filter_nbits, coarse,
                                          b["ids"].data_ptr(), b["dist"].data_ptr(), b["cnt"].data_ptr(), stream)
        # ONE exchange step: all-gather of the packed per-rank chunks (ids | dist | count), then the merge
        dist.all_gather_into_tensor(b["g_pack"].view(-1), b["pack"], group=self.group)
        self._merge(b, nq, k, tiered, stream)
        if _check and filter_bits is None and self._tc_mode():
            # one more small collective on this (synchronous) path: did the proof fail anywhere?  (see _redo_exact)
            fb = torch.tensor([self.eng.stats().last_fallback_queries], dtype=torch.int32, device=q.device)
            dist.all_reduce(fb, op=dist.ReduceOp.MAX, group=self.group)
            if int(fb.item()) > 0:
                self._redo_exact([(q, k, nprobe, tiers, slot)])
        return b["o_ids"], b["o_dist"], b["o_cnt"]

    def search_postfilter(self, q, k: int, nprobe: int, keep_bits, tiers: int = L.TIER_BOTH):
        """HybridIndex::search_with_filter (src/hybrid/core.rs:513-549), the reference's 3x post-filter, over
        the sharded index: a sharded search of 3k, then — in order — the candidates whose row id has its bit
        set in `keep_bits` (int64 tensor of u64 words over row ids, on q's device; ids beyond it fail), truncated
        to k.  Like fvdb_search_postfilter it may return fewer than k rows although more match, and needs
        3k <= k_max.  Returns (ids, dist, cnt) tensors."""
        import torch
        k3 = 3 * k
        k_max = getattr(self.eng, "k_max", None)
        if k_max is not None and k3 > k_max:
            raise ValueError(f"search_postfilter needs 3k <= k_max ({k3} > {k_max})")
        ids, dst, cnt = self.search(q, k3, nprobe, tiers=tiers)
        nq = ids.shape[0]
        rid = ids.long() & 0xFFFFFFFF
        nwords = keep_bits.numel()
        word = keep_bits[(rid >> 6).clamp(max=max(nwords - 1, 0))] if nwords else torch.zeros_like(rid)
        ok = (torch.arange(k3, device=ids.device)[None, :] < cnt.long()[:, None]) & (rid < nwords * 64) & \
             (((word >> (rid & 63)) & 1) != 0)
        pos = torch.cumsum(ok.long(), dim=1) - 1
        dest = torch.where(ok & (pos < k), pos, torch.full_like(pos, k))      # column k collects what is dropped
        o_ids = torch.full((nq, k + 1), -1, dtype=torch.int32, device=ids.device).scatter_(1, dest, ids)
        o_dst = torch.full((nq, k + 1), float("inf"), dtype=torch.float32, device=ids.device).scatter_(1, dest, dst)
        o_cnt = ok.sum(dim=1).clamp(max=k).to(torch.int32)
        return o_ids[:, :k].contiguous(), o_dst[:, :k].contiguous(), o_cnt

    def _tc_mode(self) -> bool:
        return os.environ.get("FVDB_SHARD_CHECK", "1") != "0" and self.share_bounds
