"""Thin numpy-facing wrapper over the C ABI (include/fvdb.h).  One Engine == one fvdb_index
handle == the device state of one HybridIndex.  No numeric work happens in Python."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


class PinnedArray:
    """numpy view of a page-locked host buffer from fvdb_host_alloc (freed with the object).  Passed
    to Engine.search(..., out=...) or as the query matrix, the copy engines read / write it
    directly (no staging memcpy)."""

    def __init__(self, shape, dtype):
        lib = L.load()
        self.shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.dtype = np.dtype(dtype)
        n = int(np.prod(self.shape)) * self.dtype.itemsize
        self._ptr = C.c_void_p()
        rc = lib.fvdb_host_alloc(max(n, 1), C.byref(self._ptr))
        if rc != 0:
            raise MemoryError(f"fvdb_host_alloc({n}) failed with code {rc}")
        self._lib = lib
        buf = (C.c_char * max(n, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def __del__(self):
        p, self._ptr = getattr(self, "_ptr", None), None
        if p is not None and p.value:
            self._lib.fvdb_host_free(p)


class FvdbError(Exception):
    """Base of the error enums of the reference (IVFError src/ivf/core.rs:14-39, HNSWError,
    HybridError src/hybrid/core.rs:16-35)."""
    code = None

    def __init__(self, message="", code=None):
        super().__init__(message)
        if code is not None:
            self.code = code


class NotTrained(FvdbError):
    code = L.ERR_NOT_TRAINED


class DuplicateVector(FvdbError):
    code = L.ERR_DUPLICATE


class DimensionMismatch(FvdbError):
    code = L.ERR_DIM_MISMATCH

    def __init__(self, expected=None, actual=None, message=None):
        super().__init__(message or f"Dimension mismatch: expected {expected}, got {actual}")
        self.expected, self.actual = expected, actual


class InsufficientTrainingData(FvdbError):
    code = L.ERR_INSUFFICIENT_TRAINING


class InconsistentDimensions(FvdbError):
    code = L.ERR_INCONSISTENT_DIM


class InvalidConfig(FvdbError):
    code = L.ERR_INVALID_CONFIG


class VectorNotFound(FvdbError):
    code = L.ERR_NOT_FOUND


class NanInput(FvdbError):
    code = L.ERR_NAN


class NoDevice(FvdbError):
    code = L.ERR_NO_DEVICE


_BY_CODE = {c.code: c for c in (NotTrained, DuplicateVector, InsufficientTrainingData,
                                InconsistentDimensions, InvalidConfig, VectorNotFound, NanInput,
                                NoDevice)}


def _raise(code: int, msg: str):
    if code == L.ERR_DIM_MISMATCH:
        raise DimensionMismatch(message=msg)
    cls = _BY_CODE.get(code)
    if cls is not None:
        raise cls(msg)
    raise FvdbError(msg or f"fvdb error {code}", code=code)


def _f32(a, shape_cols=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape_cols is not None:
        a = a.reshape(-1, shape_cols)
    return a


def _p(a, typ):
    return a.ctypes.data_as(typ)


_f32p = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)


def _stream(stream: int):
    """cudaStream_t argument.  0 is torch's (legacy) default stream, but NULL means "the handle's
    own stream" in the C ABI, so 0 is passed as cudaStreamLegacy (0x1): the work is then ordered
    with whatever the caller enqueued on the default stream (NCCL collectives, copies)."""
    return C.c_void_p(stream if stream else 1)


class Engine:
    def __init__(self, dim: int, k_max: int = 128, device: int = 0, metric: int = L.METRIC_L2):
        self._lib = L.load()
        self._h = C.c_void_p()
        self.dim = int(dim)
        self.k_max = int(k_max)
        self.device = int(device)
        self.metric = int(metric)
        rc = self._lib.fvdb_create(device, dim, self.metric, k_max, C.byref(self._h))
        if rc != 0:
            msg = self._lib.fvdb_last_error(None)
            self._h = None
            _raise(rc, msg.decode() if msg else "")

    # -- plumbing -------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.fvdb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def _ck(self, rc):
        if rc != 0:
            msg = self._lib.fvdb_last_error(self._h)
            _raise(rc, msg.decode() if msg else "")

    def set_option(self, option: int, value: int):
        self._ck(self._lib.fvdb_set_option(self._h, option, value))

    def stats(self) -> L.Stats:
        s = L.Stats()
        self._ck(self._lib.fvdb_get_stats(self._h, C.byref(s)))
        return s

    # -- centroids / training -------------------------------------------------------------
    def set_centroids(self, centroids):
        c = _f32(centroids, self.dim)
        self._ck(self._lib.fvdb_ivf_set_centroids(self._h, _p(c, _f32p), c.shape[0]))

    def get_centroids(self) -> np.ndarray:
        n = C.c_uint32()
        self._ck(self._lib.fvdb_ivf_get_centroids(self._h, None, C.byref(n)))
        out = np.empty((n.value, self.dim), dtype=np.float32)
        self._ck(self._lib.fvdb_ivf_get_centroids(self._h, _p(out, _f32p), C.byref(n)))
        return out

    def train(self, data, nlist: int, max_iterations: int, init_centroids=None, seed: int = 0):
        x = _f32(data, self.dim)
        res = L.TrainResult()
        ip = None
        if init_centroids is not None:
            ic = _f32(init_centroids, self.dim)
            if ic.shape[0] != nlist:
                raise InvalidConfig("init_centroids must be [nlist x dim]")
            ip = _p(ic, _f32p)
        self._ck(self._lib.fvdb_ivf_train(self._h, _p(x, _f32p), x.shape[0], nlist, max_iterations,
                                          ip, seed & 0xFFFFFFFFFFFFFFFF, C.byref(res)))
        return dict(iterations=res.iterations, converged=bool(res.converged),
                    initial_error=res.initial_error, final_error=res.final_error)

    def retrain(self, nlist: int, max_iterations: int, init_centroids=None, seed: int = 0):
        """k-means over the resident IVF rows + reassignment, all on the device (fvdb_ivf_retrain)."""
        res = L.TrainResult()
        ip = None
        if init_centroids is not None:
            ic = _f32(init_centroids, self.dim)
            if ic.shape[0] != nlist:
                raise InvalidConfig("init_centroids must be [nlist x dim]")
            ip = _p(ic, _f32p)
        self._ck(self._lib.fvdb_ivf_retrain(self._h, nlist, max_iterations, ip, seed & 0xFFFFFFFFFFFFFFFF,
                                            C.byref(res)))
        return dict(iterations=res.iterations, converged=bool(res.converged),
                    initial_error=res.initial_error, final_error=res.final_error)

    def dump_lists(self):
        """(row ids, lists) of the IVF tier in arena order."""
        n = C.c_uint64()
        self._ck(self._lib.fvdb_ivf_dump_lists(self._h, None, None, 0, C.byref(n)))
        ids = np.empty(n.value, dtype=np.uint32)
        lists = np.empty(n.value, dtype=np.uint32)
        if n.value:
            self._ck(self._lib.fvdb_ivf_dump_lists(self._h, _p(ids, _u32p), _p(lists, _u32p), n.value, C.byref(n)))
        return ids, lists

    def assign(self, x) -> np.ndarray:
        x = _f32(x, self.dim)
        out = np.empty(x.shape[0], dtype=np.uint32)
        self._ck(self._lib.fvdb_assign(self._h, _p(x, _f32p), x.shape[0], _p(out, _u32p)))
        return out

    # -- insertion / deletion -------------------------------------------------------------
    def ivf_add(self, x, row_ids, want_lists: bool = False):
        x = _f32(x, self.dim)
        ids = np.ascontiguousarray(row_ids, dtype=np.uint32)
        assert ids.shape[0] == x.shape[0]
        out = np.empty(x.shape[0], dtype=np.uint32) if want_lists else None
        self._ck(self._lib.fvdb_ivf_add(self._h, _p(x, _f32p), _p(ids, _u32p), x.shape[0],
                                        _p(out, _u32p) if want_lists else None))
        return out

    def flat_add(self, x, row_ids):
        x = _f32(x, self.dim)
        ids = np.ascontiguousarray(row_ids, dtype=np.uint32)
        assert ids.shape[0] == x.shape[0]
        self._ck(self._lib.fvdb_flat_add(self._h, _p(x, _f32p), _p(ids, _u32p), x.shape[0]))

    def move_flat_to_ivf(self, row_ids) -> int:
        ids = np.ascontiguousarray(row_ids, dtype=np.uint32)
        moved = C.c_uint64()
        self._ck(self._lib.fvdb_move_flat_to_ivf(self._h, _p(ids, _u32p), ids.shape[0],
                                                 C.byref(moved)))
        return moved.value

    def set_deleted(self, row_ids, deleted: bool = True):
        ids = np.ascontiguousarray(row_ids, dtype=np.uint32)
        self._ck(self._lib.fvdb_set_deleted(self._h, _p(ids, _u32p), ids.shape[0], int(deleted)))

    def vacuum(self) -> int:
        removed = C.c_uint64()
        self._ck(self._lib.fvdb_vacuum(self._h, C.byref(removed)))
        return removed.value

    # -- search ---------------------------------------------------------------------------
    def search(self, queries, k: int, nprobe: int, tiers: int = L.TIER_BOTH, filter_bits=None, out=None):
        """Returns (ids [nq,k] u32, dist [nq,k] f32, count [nq] u32); host buffers both ways.
        `out` = (ids, dist, count) arrays to fill (e.g. PinnedArray(...).array views)."""
        q = _f32(queries)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.shape[1] != self.dim:
            raise DimensionMismatch(self.dim, q.shape[1])
        nq = q.shape[0]
        if out is not None:
            ids, dist, cnt = out
            if ids.shape != (nq, k) or dist.shape != (nq, k) or cnt.shape != (nq,) or ids.dtype != np.uint32 \
                    or dist.dtype != np.float32 or cnt.dtype != np.uint32:
                raise ValueError("out must be (u32 [nq,k], f32 [nq,k], u32 [nq])")
            cnt[:] = 0
        else:
            ids = np.empty((nq, k), dtype=np.uint32)
            dist = np.empty((nq, k), dtype=np.float32)
            cnt = np.zeros(nq, dtype=np.uint32)
        fp, fn = None, 0
        if filter_bits is not None:
            fb = np.ascontiguousarray(filter_bits, dtype=np.uint64)
            fp, fn = _p(fb, _u64p), fb.size * 64
            if fb.size == 0:
                fb = np.zeros(1, dtype=np.uint64)
                fp, fn = _p(fb, _u64p), 0
        self._ck(self._lib.fvdb_search(self._h, _p(q, _f32p), nq, k, nprobe, tiers, fp, fn,
                                       _p(ids, _u32p), _p(dist, _f32p), _p(cnt, _u32p)))
        return ids, dist, cnt

    def search_postfilter(self, queries, k: int, nprobe: int, keep_bits, tiers: int = L.TIER_BOTH):
        """The reference's 3x post-filter (fvdb_search_postfilter): search(3k), keep rows whose bit is set in
        `keep_bits` (u64 words over row ids), truncate to k."""
        q = _f32(queries)
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.shape[1] != self.dim:
            raise DimensionMismatch(self.dim, q.shape[1])
        nq = q.shape[0]
        ids = np.empty((nq, k), dtype=np.uint32)
        dist = np.empty((nq, k), dtype=np.float32)
        cnt = np.zeros(nq, dtype=np.uint32)
        kb = np.ascontiguousarray(keep_bits, dtype=np.uint64)
        nbits = kb.size * 64
        if kb.size == 0:
            kb = np.zeros(1, dtype=np.uint64)
        self._ck(self._lib.fvdb_search_postfilter(self._h, _p(q, _f32p), nq, k, nprobe, tiers, _p(kb, _u64p), nbits,
                                                  _p(ids, _u32p), _p(dist, _f32p), _p(cnt, _u32p)))
        return ids, dist, cnt

    def search_submit(self, queries: np.ndarray, k: int, nprobe: int, tiers: int, out):
        """Stream-ordered fvdb_search: `queries` and `out` = (ids, dist, count) must be views of PinnedArray
        buffers; they belong to the engine until search_finish() returns."""
        nq = queries.shape[0]
        ids, dist, cnt = out
        if queries.dtype != np.float32 or queries.ndim != 2 or queries.shape[1] != self.dim or not queries.flags.c_contiguous:
            raise ValueError("queries must be a contiguous f32 [nq, dim] array")
        if ids.shape != (nq, k) or dist.shape != (nq, k) or cnt.shape != (nq,) or ids.dtype != np.uint32 \
                or dist.dtype != np.float32 or cnt.dtype != np.uint32:
            raise ValueError("out must be (u32 [nq,k], f32 [nq,k], u32 [nq])")
        self._ck(self._lib.fvdb_search_submit(self._h, _p(queries, _f32p), nq, k, nprobe, tiers,
                                              _p(ids, _u32p), _p(dist, _f32p), _p(cnt, _u32p)))

    def search_finish(self):
        self._ck(self._lib.fvdb_search_finish(self._h))

    def search_device(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                      filter_nbits: int, d_out_ids: int, d_out_dist: int, d_out_count: int,
                      stream: int = 0):
        """Device-pointer variant (ints are raw device addresses, e.g. tensor.data_ptr())."""
        self._ck(self._lib.fvdb_search_device(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                              filter_nbits, d_out_ids, d_out_dist, d_out_count,
                                              _stream(stream)))

    def search_device_submit(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                             filter_nbits: int, d_out_ids: int, d_out_dist: int, d_out_count: int,
                             stream: int = 0):
        """Stream-ordered search: enqueue and return; the results are valid after search_device_finish."""
        self._ck(self._lib.fvdb_search_device_submit(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                                     filter_nbits, d_out_ids, d_out_dist, d_out_count,
                                                     _stream(stream)))

    def search_device_finish(self, stream: int = 0):
        """Wait for every submitted batch; raises NanInput if one of them held a NaN query."""
        self._ck(self._lib.fvdb_search_device_finish(self._h, _stream(stream)))

    def coarse_device(self, d_q: int, nq: int, nprobe: int, d_out_keys: int, stream: int = 0):
        """Coarse ranking only: keys [nq x nprobe] u64 (device)."""
        self._ck(self._lib.fvdb_coarse_device(self._h, d_q, nq, nprobe, d_out_keys, _stream(stream)))

    def search_device_coarse(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                             filter_nbits: int, d_coarse_keys: int, d_out_ids: int, d_out_dist: int,
                             d_out_count: int, stream: int = 0):
        self._ck(self._lib.fvdb_search_device_coarse(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                                     filter_nbits, d_coarse_keys or None, d_out_ids,
                                                     d_out_dist, d_out_count, _stream(stream)))

    def coarse_device_submit(self, d_q: int, nq: int, nprobe: int, d_out_keys: int, stream: int = 0):
        self._ck(self._lib.fvdb_coarse_device_submit(self._h, d_q, nq, nprobe, d_out_keys, _stream(stream)))

    def search_device_coarse_submit(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                                    filter_nbits: int, d_coarse_keys: int, d_out_ids: int, d_out_dist: int,
                                    d_out_count: int, stream: int = 0):
        self._ck(self._lib.fvdb_search_device_coarse_submit(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                                            filter_nbits, d_coarse_keys or None, d_out_ids,
                                                            d_out_dist, d_out_count, _stream(stream)))

    def search_device_wait(self, age: int = 0, stream: int = 0):
        self._ck(self._lib.fvdb_search_device_wait(self._h, age, _stream(stream)))

    def search_device_tiers(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                            filter_nbits: int, d_coarse_keys: int, d_out_pack: int, stream: int = 0):
        """search_device_coarse with the tiers kept apart: d_out_pack receives two packed parts, recent tier
        then IVF tier (see shard.tiers_pack_layout)."""
        self._ck(self._lib.fvdb_search_device_tiers(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                                    filter_nbits, d_coarse_keys or None, d_out_pack,
                                                    _stream(stream)))

    def search_device_tiers_submit(self, d_q: int, nq: int, k: int, nprobe: int, tiers: int, d_filter: int,
                                   filter_nbits: int, d_coarse_keys: int, d_out_pack: int, stream: int = 0):
        """Stream-ordered search_device_tiers; the chunk is valid after search_device_finish."""
        self._ck(self._lib.fvdb_search_device_tiers_submit(self._h, d_q, nq, k, nprobe, tiers, d_filter or None,
                                                           filter_nbits, d_coarse_keys or None, d_out_pack,
                                                           _stream(stream)))

    def merge_topk_device(self, d_ids: int, d_dist: int, d_count: int, parts: int, nq: int, k: int,
                          d_out_ids: int, d_out_dist: int, d_out_count: int, stream: int = 0):
        self._ck(self._lib.fvdb_merge_topk_device(self._h, d_ids, d_dist, d_count, parts, nq, k,
                                                  d_out_ids, d_out_dist, d_out_count,
                                                  _stream(stream)))

    def ivf_max_sqnorm(self) -> float:
        v = C.c_float()
        self._ck(self._lib.fvdb_ivf_max_sqnorm(self._h, C.byref(v)))
        return float(v.value)

    def bounds_close_peers(self):
        self._ck(self._lib.fvdb_bounds_import(self._h, None, 0, 0))

    def bounds_export(self, nq_cap: int) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self._lib.fvdb_bounds_export(self._h, nq_cap, buf))
        return buf.raw

    def bounds_import(self, handles: bytes, n_ranks: int, my_rank: int):
        self._ck(self._lib.fvdb_bounds_import(self._h, C.c_char_p(handles), n_ranks, my_rank))

    def bounds_begin_batch(self, nq: int, stream: int = 0):
        self._ck(self._lib.fvdb_bounds_begin_batch(self._h, nq, _stream(stream)))

    def merge_topk_packed_device(self, d_pack: int, parts: int, nq: int, k: int, d_out_ids: int, d_out_dist: int,
                                 d_out_count: int, stream: int = 0):
        """parts x [ids nq*k | dist nq*k | count nq] 32-bit words (see shard.pack_layout)."""
        self._ck(self._lib.fvdb_merge_topk_packed_device(self._h, d_pack, parts, nq, k, d_out_ids, d_out_dist,
                                                         d_out_count, _stream(stream)))

    def merge_topk_tiers_packed_device(self, d_pack: int, ranks: int, nq: int, k: int, d_out_ids: int,
                                       d_out_dist: int, d_out_count: int, stream: int = 0):
        """ranks x search_device_tiers chunks -> the (distance, tier, row id) merge of both tiers."""
        self._ck(self._lib.fvdb_merge_topk_tiers_packed_device(self._h, d_pack, ranks, nq, k, d_out_ids, d_out_dist,
                                                               d_out_count, _stream(stream)))

    def ivf_add_device(self, d_x: int, d_ids: int, n: int, mod: int = 1, rem: int = 0) -> int:
        kept = C.c_uint64()
        self._ck(self._lib.fvdb_ivf_add_device(self._h, d_x, d_ids, n, mod, rem, C.byref(kept)))
        return kept.value

    def ivf_add_device_owned(self, d_x: int, d_ids: int, n: int, d_owner: int, my_rank: int) -> int:
        kept = C.c_uint64()
        self._ck(self._lib.fvdb_ivf_add_device_owned(self._h, d_x, d_ids, n, d_owner, my_rank, C.byref(kept)))
        return kept.value

    def assign_device(self, d_x: int, n: int, d_out: int, stream: int = 0):
        self._ck(self._lib.fvdb_assign_device(self._h, d_x, n, d_out, _stream(stream)))

    def flat_add_device(self, d_x: int, d_ids: int, n: int):
        self._ck(self._lib.fvdb_flat_add_device(self._h, d_x, d_ids, n))

    def train_device(self, d_data: int, n: int, nlist: int, max_iterations: int, d_init: int = 0,
                     seed: int = 0):
        res = L.TrainResult()
        self._ck(self._lib.fvdb_ivf_train_device(self._h, d_data, n, nlist, max_iterations,
                                                 d_init or None, seed, C.byref(res)))
        return dict(iterations=res.iterations, converged=bool(res.converged),
                    initial_error=res.initial_error, final_error=res.final_error)

    def kmeans_accumulate_device(self, d_data, n, d_sums, d_counts, d_sqerr, d_assign, d_changed,
                                 stream=0):
        self._ck(self._lib.fvdb_kmeans_accumulate_device(self._h, d_data, n, d_sums, d_counts,
                                                         d_sqerr, d_assign, d_changed,
                                                         _stream(stream)))

    def kmeans_apply_device(self, d_sums, d_counts, stream=0):
        self._ck(self._lib.fvdb_kmeans_apply_device(self._h, d_sums, d_counts, _stream(stream)))
