/*
 * fvdb.h — C ABI of libfvdb_b200.so, the B200 (sm_100a) engine for the one data-parallel
 * hot path of Fabstir/fabstir-vectordb: batched query x database L2 distance + top-k behind
 * HybridIndex::search (IVF coarse assignment, IVF posting-list scan, exact scan of the
 * recent tier, k-means centroid training).
 *
 * The reference has no FFI seam for this path today (SURVEY.md §8b): the seam is the Rust
 * method set of IVFIndex / HNSWIndex / HybridIndex.  Every entry point below names the
 * reference function body it replaces (paths relative to the reference repository).
 * The Rust-side `extern "C"` block that binds these symbols is shown in INTEGRATION.md.
 *
 * Conventions
 *   - every function returns int: FVDB_OK (0) or a negative fvdb_status; no exceptions and
 *     no panics cross the ABI; fvdb_last_error() returns a human-readable message.
 *   - the caller owns every host buffer; the library copies (pinned staging inside).
 *   - ids crossing the boundary are dense caller-chosen u32 row ids.  The 32-byte VectorId
 *     <-> row-id map, timestamps, JSON metadata and duplicate detection stay in the host
 *     language (reference: src/core/types.rs:10-35, src/hybrid/core.rs:206,368).
 *   - distances returned are TRUE L2 (sqrt applied), ascending, exactly as
 *     euclidean_distance_scalar (src/core/vector_ops.rs:51-57) computes them:
 *     sequential f32 accumulation in index order, no FMA contraction.
 *   - ties: (distance, row id) ascending.  The reference's own order of equal distances is
 *     HashMap iteration order (undefined); coarse ties resolve to the lower cluster id, as the
 *     reference's stable sort does (src/ivf/core.rs:655), argmin to the lowest id (:379).
 *   - NaN in any input returns FVDB_ERR_NAN (the reference panics: src/ivf/core.rs:655,677).
 *   - there is NO CPU fallback: without a CUDA device fvdb_create returns FVDB_ERR_NO_DEVICE.
 *   - a handle may be searched from several OS threads at once (searches serialise on an
 *     internal mutex per handle for now); mutation is exclusive, like the reference's
 *     tokio RwLock (src/hybrid/core.rs:202-213).
 */
#ifndef FVDB_H_
#define FVDB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define FVDB_ABI_VERSION 1

typedef struct fvdb_index fvdb_index; /* opaque engine handle: one per HybridIndex */

/* Status codes.  -1..-8 map 1:1 onto IVFError (src/ivf/core.rs:14-39) / HNSWError /
 * HybridError (src/hybrid/core.rs:16-35); the rest are ABI-level. */
typedef enum fvdb_status {
    FVDB_OK = 0,
    FVDB_ERR_NOT_TRAINED = -1,           /* IVFError::NotTrained */
    FVDB_ERR_DUPLICATE = -2,             /* IVFError::DuplicateVector (row id already present) */
    FVDB_ERR_DIM_MISMATCH = -3,          /* IVFError::DimensionMismatch */
    FVDB_ERR_INSUFFICIENT_TRAINING = -4, /* IVFError::InsufficientTrainingData */
    FVDB_ERR_INCONSISTENT_DIM = -5,      /* IVFError::InconsistentDimensions (host side) */
    FVDB_ERR_INVALID_CONFIG = -6,        /* IVFError::InvalidConfig */
    FVDB_ERR_CHUNK_LOAD = -7,            /* IVFError::ChunkLoadError (host side; reserved) */
    FVDB_ERR_NOT_FOUND = -8,             /* IVFError::VectorNotFound */
    FVDB_ERR_NAN = -9,                   /* NaN in an input (reference panics) */
    FVDB_ERR_CUDA = -10,                 /* CUDA runtime / driver failure, see last_error */
    FVDB_ERR_NO_DEVICE = -11,            /* no usable sm_100 device: there is no CPU path */
    FVDB_ERR_INVALID_ARG = -12,
    FVDB_ERR_K_TOO_LARGE = -13,          /* k > k_max given at create */
    FVDB_ERR_OOM = -14
} fvdb_status;

/* How a (query, row) pair is scored.  The reference's indexes (IVFIndex, HNSWIndex, HybridIndex) are L2
 * only; cosine and dot product exist as scalar kernels ranked exhaustively (batch_cosine_similarity +
 * top_k_indices, src/core/vector_ops.rs:8-23).  A COS / DOT handle therefore serves the FLAT tier
 * (fvdb_flat_add + fvdb_search with FVDB_TIER_RECENT): every row is scored, the k LARGEST similarities
 * are returned best first, ties to the lower row id (top_k_indices is a stable descending sort), and
 * out_dist holds the similarity itself, bit-identical to the scalar kernels (sequential f32, no FMA;
 * cosine = dot / (sqrt(dot(a,a)) * sqrt(dot(b,b))), 0 when either norm is 0).  Tombstones and the filter
 * bitmap apply as for L2.  The fvdb_ivf_* entries return FVDB_ERR_INVALID_CONFIG on such a handle. */
typedef enum fvdb_metric {
    FVDB_METRIC_L2 = 0,  /* euclidean_distance_scalar, src/core/vector_ops.rs:51-57 */
    FVDB_METRIC_COS = 1, /* cosine_similarity_scalar :39-49, Embedding::cosine_similarity src/core/types.rs:79-103 */
    FVDB_METRIC_DOT = 2  /* dot_product_scalar :35-37 */
} fvdb_metric;

/* Tier selection bits for fvdb_search: HybridSearchConfig.search_recent /
 * search_historical, src/hybrid/core.rs:173-196. */
#define FVDB_TIER_RECENT 1u     /* the "HNSW" tier, served by an exact flat scan */
#define FVDB_TIER_HISTORICAL 2u /* the IVF tier */
#define FVDB_TIER_BOTH 3u

/* Search precision modes (fvdb_set_option FVDB_OPT_SCAN_MODE). */
#define FVDB_SCAN_EXACT 0u /* fp32 CUDA-core scan in the reference's own operation order */
#define FVDB_SCAN_TC 1u    /* tcgen05 TF32 shortlist + exact fp32 re-rank + proof check,   \
                              falling back to EXACT for any query whose proof fails */

typedef enum fvdb_option {
    FVDB_OPT_SCAN_MODE = 1,   /* FVDB_SCAN_EXACT | FVDB_SCAN_TC (default TC when dim%32==0) */
    FVDB_OPT_SHORTLIST = 2,   /* shortlist length k' of the TC mode (default max(32, ..)) */
    FVDB_OPT_KMEANS_TC = 3,   /* 1: k-means assignment on tensor cores with exact verify */
    FVDB_OPT_COALESCE = 4,    /* 1 (default): concurrent fvdb_search calls are coalesced into one device batch */
    FVDB_OPT_PIPELINE = 6,    /* 1 (default): batches of the stream-ordered entries alternate between two
                                 internal streams with their own scratch, so that a batch's coarse step and
                                 bucketing overlap the previous batch's scan tail, merge and re-rank */
    FVDB_OPT_SCAN_SMS = 7,    /* pipelined batches: the posting-list scan kernels run on this many SMs (0 = all),
                                 the rest stay free for the neighbouring batches' coarse step, bucketing, merge,
                                 re-rank and — multi-GPU — the NCCL kernels, which otherwise only run in the
                                 scans' gaps (the scan kernels are persistent and fill every SM) */
    FVDB_OPT_PROOF_XMAX = 5   /* list-sharded multi-GPU search with shared bounds: f32 bits of the largest
                                 |x|^2 over ALL shards (fvdb_ivf_max_sqnorm, max-reduced by the driver).  A
                                 row of this shard may be dropped by a bound a peer published, so the
                                 tensor-core proof must not use a smaller norm term than the peer's. */
} fvdb_option;

/* TrainResult, src/ivf/core.rs:103-109. */
typedef struct fvdb_train_result {
    uint32_t iterations;
    uint32_t converged; /* bool */
    float initial_error;
    float final_error;
} fvdb_train_result;

typedef struct fvdb_stats {
    uint32_t dim;
    uint32_t nlist;        /* 0 until centroids are set / trained */
    uint32_t trained;      /* IVFIndex::is_trained */
    uint64_t ivf_rows;     /* IVFIndex::total_vectors (including tombstoned) */
    uint64_t flat_rows;    /* recent-tier rows (including tombstoned) */
    uint64_t deleted_rows; /* rows tombstoned and not yet vacuumed */
    uint64_t device_bytes; /* HBM held by the handle */
    /* counters of the most recent fvdb_search call */
    uint32_t last_nq;
    uint32_t last_fallback_queries; /* TC mode: queries re-run on the exact path */
    uint64_t last_scanned_rows;     /* distinct posting-list + flat rows streamed */
    uint64_t last_algorithmic_bytes;/* SURVEY §8(d) bytes: each probed list once + flat tier +
                                       queries + centroids + bitmaps + outputs */
    float last_device_ms;           /* device time of the last search (CUDA events) */
    float last_scan_ms;             /* device time of the posting-list scan kernel alone */
    uint32_t last_launches;         /* kernels launched by the last search */
    uint32_t last_batch_calls;      /* fvdb_search calls served by the last device batch (submission queue) */
} fvdb_stats;

/* ---- lifecycle ------------------------------------------------------------------------- */

/* IVFIndex::new / HNSWIndex::new / HybridIndex::new (src/ivf/core.rs:171, src/hnsw/core.rs,
 * src/hybrid/core.rs).  device: CUDA ordinal.  k_max: largest k any search will ask for
 * (1..512; FVDB_ERR_INVALID_CONFIG otherwise).  Fails with FVDB_ERR_NO_DEVICE when no CUDA device is usable. */
int fvdb_create(int device, uint32_t dim, int metric, uint32_t k_max, fvdb_index **out);
void fvdb_destroy(fvdb_index *h);
const char *fvdb_last_error(const fvdb_index *h); /* h may be NULL: last create error */
int fvdb_abi_version(void);
int fvdb_set_option(fvdb_index *h, int option, uint64_t value);
int fvdb_get_stats(fvdb_index *h, fvdb_stats *out);

/* ---- IVF centroids / training ---------------------------------------------------------- */

/* IVFIndex::set_trained (src/ivf/core.rs:509-520): install centroids [nlist x dim], mark the
 * index trained and clear every posting list. */
int fvdb_ivf_set_centroids(fvdb_index *h, const float *centroids, uint32_t nlist);
/* IVFIndex::get_centroids (:236).  out may be NULL to query nlist only. */
int fvdb_ivf_get_centroids(fvdb_index *h, float *out, uint32_t *nlist);

/* IVFIndex::train (src/ivf/core.rs:240-334): Lloyd k-means with the reference's stop rule
 * (:303-321), empty-cluster rule (:410-415) and error definition (:419-429).
 *   init_centroids != NULL : Lloyd starts from these [nlist x dim] (shared-init parity mode).
 *   init_centroids == NULL : k-means++ (:336-371) driven by `seed`; same distribution as the
 *                            reference, not the same rand-0.8 bit stream (parity unpinned).
 * Errors: n == 0 or n < nlist -> FVDB_ERR_INSUFFICIENT_TRAINING (:242-254).
 * Like the reference, training leaves every posting list empty (:273-277). */
int fvdb_ivf_train(fvdb_index *h, const float *data, uint64_t n, uint32_t nlist,
                   uint32_t max_iterations, const float *init_centroids, uint64_t seed,
                   fvdb_train_result *out);

/* IVFIndex::find_cluster / find_nearest_centroid (src/ivf/core.rs:373-386,493-499) for a batch:
 * out_list[i] = argmin_c L2(x_i, c), strict '<' so the lowest cluster id wins ties.  Also the
 * bulk re-assignment of load_index_chunked (src/hybrid/persistence.rs:626-653). */
int fvdb_assign(fvdb_index *h, const float *x, uint64_t n, uint32_t *out_list);

/* ---- insertion -------------------------------------------------------------------------- */

/* IVFIndex::insert / batch_insert (src/ivf/core.rs:431-455, src/ivf/operations.rs:107): assign
 * each row to its nearest centroid and append it to that posting list.  out_list (nullable)
 * receives the chosen list per row.  FVDB_ERR_NOT_TRAINED before centroids exist. */
int fvdb_ivf_add(fvdb_index *h, const float *x, const uint32_t *row_ids, uint64_t n,
                 uint32_t *out_list);
/* HNSWIndex::insert (src/hnsw/core.rs:226) for the recent tier: append rows to the flat tier. */
int fvdb_flat_add(fvdb_index *h, const float *x, const uint32_t *row_ids, uint64_t n);
/* HybridIndex::migrate_with_threshold (src/hybrid/core.rs:600-649): move the given recent-tier
 * rows into the IVF tier (assign + append) and drop them from the flat tier. */
int fvdb_move_flat_to_ivf(fvdb_index *h, const uint32_t *row_ids, uint64_t n, uint64_t *moved);

/* ---- soft delete ------------------------------------------------------------------------ */

/* IVFIndex::mark_deleted / HNSWIndex::mark_deleted (src/ivf/operations.rs:569-600): tombstone
 * (deleted=1) or revive (0) rows by id; tombstoned rows are skipped by every search
 * (src/ivf/core.rs:667, src/hnsw/core.rs:452-459). */
int fvdb_set_deleted(fvdb_index *h, const uint32_t *row_ids, uint64_t n, int deleted);
/* IVFIndex::vacuum / HNSWIndex::vacuum (src/ivf/operations.rs:625): physically drop
 * tombstoned rows from both tiers. */
int fvdb_vacuum(fvdb_index *h, uint64_t *removed);

/* ---- search ----------------------------------------------------------------------------- */

/* Batched HybridIndex::search_with_config (src/hybrid/core.rs:425-486) =
 *   HNSWIndex::search of the recent tier (replaced by an exact scan, src/hnsw/core.rs:398-467)
 *   ∪ IVFIndex::search_with_config (src/ivf/core.rs:626-681), stable-sorted by distance with
 *   recent-tier rows first on ties, truncated to k, no de-duplication across tiers.
 * One call = IVFIndex::batch_search (src/ivf/operations.rs:132-145) done as one batch.
 *   q            [nq x dim] host, row-major
 *   nprobe       lists probed per query (clamped to nlist, like truncate(n_probe) :656; more than 512
 *                after clamping is FVDB_ERR_INVALID_ARG)
 *   tiers        FVDB_TIER_* bits; FVDB_TIER_HISTORICAL is ignored until trained
 *                (src/hybrid/core.rs:465)
 *   filter_bits  NULL, or a bitmap over row ids (bit id set = row passes): the in-kernel
 *                pre-filter (semantics of bindings/wasm/src/index.rs:164-186); rows with
 *                id >= filter_nbits fail.  The reference's 3x post-filter
 *                (src/hybrid/core.rs:513-549) is reproduced by the host mirror on top of this.
 *   out_ids      [nq x k], out_dist [nq x k], out_count [nq] (<= k valid entries per query;
 *                fewer than k is legal, src/ivf/core.rs:386-398 of the tests).
 * Empty index or untrained+no recent rows: counts are 0 (Ok(vec![]) :431-434).
 * Concurrency: may be called from many OS threads at once (the reference's `&self` searches behind
 * an RwLock, src/hybrid/core.rs:202-213).  Calls without a filter bitmap pass through a submission
 * queue: the first caller leads, takes every queued call with the same (k, nprobe, tiers) and runs
 * them as ONE device batch (results are those of the separate calls, bit for bit — every query of a
 * batch is independent), then hands the lead to the next waiting caller.  FVDB_OPT_COALESCE = 0
 * serialises the calls instead. */
int fvdb_search(fvdb_index *h, const float *q, uint32_t nq, uint32_t k, uint32_t nprobe,
                uint32_t tiers, const uint64_t *filter_bits, uint64_t filter_nbits,
                uint32_t *out_ids, float *out_dist, uint32_t *out_count);

/* HybridIndex::search_with_filter (src/hybrid/core.rs:513-549), the reference's 3x oversampling
 * POST-filter, for a batch: search(3k) over the selected tiers exactly as fvdb_search does, keep — in
 * order — the candidates whose row id has its bit set in keep_bits, truncate to k (:529-546).
 * keep_bits is the host's evaluation of `metadata_map.get(id)` + `filter.matches` once per row (a row
 * without metadata has bit 0, :536-541; ids >= keep_nbits fail).  Like the reference it may return
 * fewer than k results although >= k matching rows exist (the in-kernel pre-filter of fvdb_search
 * does not).  Needs 3k <= k_max (FVDB_ERR_K_TOO_LARGE otherwise).  Tombstoned rows never appear. */
int fvdb_search_postfilter(fvdb_index *h, const float *q, uint32_t nq, uint32_t k, uint32_t nprobe,
                           uint32_t tiers, const uint64_t *keep_bits, uint64_t keep_nbits,
                           uint32_t *out_ids, float *out_dist, uint32_t *out_count);

/* IVFIndex::retrain (src/ivf/operations.rs:148-193; add_clusters :195-219 and optimize_clusters
 * :221-260 are the same operation with nlist + n / the same nlist): k-means over every row the
 * IVF tier holds, then every row is reassigned to its nearest new centroid.  The rows never leave
 * the device.  Training order = arena order (by list, insertion order inside a list); the
 * reference trains on HashMap iteration order, which is unspecified.  init_centroids / seed as in
 * fvdb_ivf_train.  Row ids, tombstones and the recent tier are unchanged.
 * Errors: NOT_TRAINED (:149-151), INSUFFICIENT_TRAINING when fewer rows than nlist (the train call
 * inside the reference fails the same way, src/ivf/core.rs:250-255). */
int fvdb_ivf_retrain(fvdb_index *h, uint32_t nlist, uint32_t max_iterations,
                     const float *init_centroids, uint64_t seed, fvdb_train_result *out);

/* (row id, list) of every row of the IVF tier in arena order — the membership the host keeps
 * per VectorId (InvertedList, src/ivf/core.rs:112-157) after a retrain, and what
 * save_index_chunked (src/hybrid/persistence.rs:188) walks.  NULL buffers: only *n_out. */
int fvdb_ivf_dump_lists(fvdb_index *h, uint32_t *out_row_ids, uint32_t *out_lists, uint64_t cap,
                        uint64_t *n_out);

/* Page-locked host buffers for the host-buffer entry points (replaces the `Vec<f32>` the Rust
 * callers of HybridIndex::search hand in, src/hybrid/core.rs:425).  Query and result buffers
 * allocated here are copied by the GPU's copy engines directly; pageable buffers remain legal
 * everywhere and are staged through the handle's own pinned buffer (one extra memcpy each way).
 * No handle is needed; returns FVDB_ERR_OOM when the allocation fails. */
int fvdb_host_alloc(size_t bytes, void **out);
void fvdb_host_free(void *p);

/* Same, with every buffer already resident in device memory of the handle's GPU and the
 * work enqueued on `stream` (a cudaStream_t; NULL = the handle's own stream).  Used for
 * HBM-resident throughput measurement and by the multi-GPU shard driver, which all-gathers
 * the per-GPU [nq x k] partial results over NCCL and merges them with fvdb_merge_topk_device.
 * Returns after enqueueing unless a fallback pass is needed (which synchronises). */
int fvdb_search_device(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k,
                       uint32_t nprobe, uint32_t tiers, const uint64_t *d_filter_bits,
                       uint64_t filter_nbits, uint32_t *d_out_ids, float *d_out_dist,
                       uint32_t *d_out_count, void *stream);

/* Stream-ordered pair for back-to-back batches (a serving loop that always has the next batch
 * ready): _submit enqueues the whole batch behind whatever `stream` holds and returns WITHOUT waiting, so
 * the GPU never idles between batches while the host turns a call around.  Consecutive batches run in two
 * internal pipeline slots (FVDB_OPT_PIPELINE): their scans are serialised, the smaller steps around the
 * scans overlap.  The result arrays are valid — also for work enqueued on `stream` afterwards — once
 * _finish has returned.  _finish waits for every submitted batch of the handle, reports
 * FVDB_ERR_NAN if any of them held a NaN query, and re-runs on the exact path (replacing their result
 * rows) the queries whose tensor-core proof failed.  Up to 64 batches may be pending; the query and
 * result buffers of a batch must stay alive and untouched by the caller until _finish returns.
 * (fvdb_search_device = _submit + _finish of one batch.) */
int fvdb_search_device_submit(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k,
                              uint32_t nprobe, uint32_t tiers, const uint64_t *d_filter_bits,
                              uint64_t filter_nbits, uint32_t *d_out_ids, float *d_out_dist,
                              uint32_t *d_out_count, void *stream);
int fvdb_search_device_finish(fvdb_index *h, void *stream);

/* The same pair for HOST buffers, which must be page-locked (fvdb_host_alloc; else
 * FVDB_ERR_INVALID_ARG): the upload of a batch runs on a second stream while the previous batch is
 * still being scanned, the result copies follow the batch.  At most 8 batches may be pending; query
 * and result buffers belong to the library until fvdb_search_finish returns.  No filter bitmap. */
int fvdb_search_submit(fvdb_index *h, const float *q, uint32_t nq, uint32_t k, uint32_t nprobe,
                       uint32_t tiers, uint32_t *out_ids, float *out_dist, uint32_t *out_count);
int fvdb_search_finish(fvdb_index *h);

/* The coarse step alone (src/ivf/core.rs:646-656) for nq device-resident queries:
 * d_out_keys [nq x nprobe] = (f32 bits of the exact centroid distance << 32) | list id, ascending,
 * ties to the lower list id (the reference's stable sort).  1 <= nprobe <= nlist.  Used by the
 * multi-GPU driver: each GPU ranks a slice of the batch against the replicated centroids and the
 * slices are all-gathered, so the coarse cost per GPU does not grow with the number of GPUs. */
int fvdb_coarse_device(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t nprobe,
                       uint64_t *d_out_keys, void *stream);
/* fvdb_search_device with the coarse ranking handed in (d_coarse_keys [nq x nprobe] as written
 * by fvdb_coarse_device; rows of 0xFF..FF keys = "probe nothing"; NULL = compute it here). */
int fvdb_search_device_coarse(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k,
                              uint32_t nprobe, uint32_t tiers, const uint64_t *d_filter_bits,
                              uint64_t filter_nbits, const uint64_t *d_coarse_keys,
                              uint32_t *d_out_ids, float *d_out_dist, uint32_t *d_out_count,
                              void *stream);

/* Stream-ordered twins of the two calls above for a pipelined multi-GPU driver (no host synchronisation
 * per batch): _coarse_device_submit enqueues the coarse step of a query slice; _search_device_coarse_submit
 * enqueues a batch whose coarse ranking is handed in — in one of the handle's pipeline slots, behind
 * whatever `stream` holds (e.g. the all-gather of the coarse keys); fvdb_search_device_wait makes `stream`
 * wait, on the device, for the batch submitted `age` submits ago (0 = the latest), so that a collective
 * on `stream` can consume its results while the NEXT batch is already scanning.  fvdb_search_device_finish
 * ends a group as usual: NaN -> FVDB_ERR_NAN; queries whose tensor-core proof failed are repaired locally
 * (scan) or merely counted (coarse step) and reported in fvdb_stats.last_fallback_queries — a sharded
 * driver then re-runs the group through the synchronous entries, because results it has already
 * exchanged were built from the unrepaired ones. */
int fvdb_coarse_device_submit(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t nprobe,
                              uint64_t *d_out_keys, void *stream);
int fvdb_search_device_coarse_submit(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k,
                                     uint32_t nprobe, uint32_t tiers, const uint64_t *d_filter_bits,
                                     uint64_t filter_nbits, const uint64_t *d_coarse_keys,
                                     uint32_t *d_out_ids, float *d_out_dist, uint32_t *d_out_count,
                                     void *stream);
int fvdb_search_device_wait(fvdb_index *h, uint32_t age, void *stream);

/* fvdb_search_device_coarse, but the result of each tier is written separately into ONE packed chunk:
 *   [recent ids nq*k | recent dist nq*k | recent count nq | IVF ids nq*k | IVF dist nq*k | IVF count nq]
 * (two fvdb_merge_topk_packed_device parts back to back; 2 * (2 nq k + nq) 32-bit words).  Each part is what
 * a search of that tier alone returns.  A tier not searched, or empty on this handle, has counts 0.
 * d_coarse_keys may be NULL.  This is the per-rank step of a sharded FVDB_TIER_BOTH search: the chunks of
 * all ranks are all-gathered and merged with fvdb_merge_topk_tiers_packed_device.  L2 handles only
 * (FVDB_ERR_INVALID_CONFIG otherwise).  _submit is the stream-ordered twin (arguments and pipeline rules of
 * fvdb_search_device_coarse_submit), finished by fvdb_search_device_finish, whose exact re-run of proof
 * failures rewrites both parts. */
int fvdb_search_device_tiers(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                             uint32_t tiers, const uint64_t *d_filter_bits, uint64_t filter_nbits,
                             const uint64_t *d_coarse_keys, uint32_t *d_out_pack, void *stream);
int fvdb_search_device_tiers_submit(fvdb_index *h, const float *d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                                    uint32_t tiers, const uint64_t *d_filter_bits, uint64_t filter_nbits,
                                    const uint64_t *d_coarse_keys, uint32_t *d_out_pack, void *stream);

/* Multi-GPU bound sharing over NVLink peer memory (one process per GPU, lists sharded by
 * l % world as above).  During the posting-list scan every query carries a running upper bound of
 * its 32nd-nearest approximate distance; rows above it are dropped in the epilogue.  A shard that
 * does not hold a query's nearest lists would scan with a loose bound: these calls let the shards
 * push their bounds into each other's arrays with NVLink atomics while they scan.
 *   fvdb_bounds_export      allocates this handle's [2][nq_cap] bound array and writes its
 *                           FVDB_BOUNDS_HANDLE_BYTES-byte inter-process handle (all-gather these);
 *   fvdb_bounds_import      opens the arrays of the other ranks (handles of ALL ranks, rank-major);
 *                           n_ranks == 0 closes them again — every rank does that, then a barrier, BEFORE
 *                           any rank re-exports (fvdb_bounds_export frees the previous array);
 *   fvdb_bounds_begin_batch flips the batch parity and resets this rank's half to +inf on `stream`.
 * Protocol (every rank, every batch): begin_batch -> fvdb_coarse_device on a slice -> all-gather of
 * the coarse keys -> fvdb_search_device_coarse.  The all-gather orders every rank's reset before
 * any peer's scan of that batch, and the parity keeps a rank that is one batch ahead out of the
 * array a slower peer still reads.  Results are independent of the sharing (bounds only ever drop
 * rows that cannot be among a query's 32 nearest); without these calls each rank uses a private array. */
/* Largest squared row norm of the IVF tier (0 when empty): input of FVDB_OPT_PROOF_XMAX. */
int fvdb_ivf_max_sqnorm(fvdb_index *h, float *out);
#define FVDB_BOUNDS_HANDLE_BYTES 64
int fvdb_bounds_export(fvdb_index *h, uint32_t nq_cap, void *handle_out);
int fvdb_bounds_import(fvdb_index *h, const void *handles, uint32_t n_ranks, uint32_t my_rank);
int fvdb_bounds_begin_batch(fvdb_index *h, uint32_t nq, void *stream);

/* The same merge over ONE packed buffer per part — [ids nq*k | dist nq*k | count nq] 32-bit words,
 * parts back to back — so that the exchange step is a single all-gather: a rank lets
 * fvdb_search_device write its results into the three sections of its own chunk and gathers the
 * chunks.  Order and preconditions as for fvdb_merge_topk_device below.  Device pointers. */
int fvdb_merge_topk_packed_device(fvdb_index *h, const uint32_t *d_pack, uint32_t parts, uint32_t nq,
                                  uint32_t k, uint32_t *d_out_ids, float *d_out_dist,
                                  uint32_t *d_out_count, void *stream);

/* K-way merge of `parts` per-query partial results laid out [parts][nq][k] (ids, dist) with
 * counts [parts][nq] into [nq][k]: the `sort_by(distance); truncate(k)` of
 * src/hybrid/core.rs:482-483 applied across GPUs after the all-gather.  Order: (distance, row id),
 * the ABI's tie rule, so the merged result equals one unsharded search however the rows are split.
 * The parts must hold disjoint rows of ONE tier, each part sorted by (distance, row id) — as the
 * list-sharded IVF search (FVDB_TIER_HISTORICAL) and a recent-tier scan split into slabs produce them.
 * A FVDB_TIER_BOTH search orders recent-tier rows first on equal distances; a part here does not carry
 * the tier of its rows, so FVDB_TIER_BOTH results are merged with fvdb_merge_topk_tiers_packed_device.
 * Counts above k are clamped to k; parts must be in 1..64.  Device pointers. */
int fvdb_merge_topk_device(fvdb_index *h, const uint32_t *d_ids, const float *d_dist,
                           const uint32_t *d_count, uint32_t parts, uint32_t nq, uint32_t k,
                           uint32_t *d_out_ids, float *d_out_dist, uint32_t *d_out_count,
                           void *stream);

/* After the all-gather of the per-rank fvdb_search_device_tiers chunks: 2 * ranks parts, part 2r = recent
 * tier of rank r, part 2r + 1 = IVF tier of rank r.  Order: (distance, tier with recent first, row id), i.e.
 * the merge of src/hybrid/core.rs:482-483 applied across GPUs, equal to one unsharded FVDB_TIER_BOTH search
 * however the rows of both tiers are split over the ranks.  Counts above k are clamped to k.  ranks 1..32;
 * L2 handles only (FVDB_ERR_INVALID_CONFIG otherwise).  Device pointers. */
int fvdb_merge_topk_tiers_packed_device(fvdb_index *h, const uint32_t *d_pack, uint32_t ranks, uint32_t nq,
                                        uint32_t k, uint32_t *d_out_ids, float *d_out_dist,
                                        uint32_t *d_out_count, void *stream);

/* Device-resident variants of the bulk loaders (row data already in HBM, e.g. generated on
 * the device for the 100M-row sharded configuration).  `list_filter_mod`/`list_filter_rem`:
 * when mod > 1 only rows whose assigned list satisfies list % mod == rem are kept — the
 * list-sharding rule of the multi-GPU driver (SURVEY §8e). */
int fvdb_ivf_add_device(fvdb_index *h, const float *d_x, const uint32_t *d_row_ids, uint64_t n,
                        uint32_t list_filter_mod, uint32_t list_filter_rem, uint64_t *kept);
int fvdb_flat_add_device(fvdb_index *h, const float *d_x, const uint32_t *d_row_ids, uint64_t n);
/* fvdb_ivf_add_device with a list -> GPU placement TABLE instead of the l % mod rule: a row is kept when
 * d_owner[its list] == my_rank (d_owner: [nlist] u32, device).  The multi-GPU driver fills the table by
 * greedy size-balanced bin packing of the lists (SURVEY §8e), so that every GPU streams the same number
 * of rows per batch. */
int fvdb_ivf_add_device_owned(fvdb_index *h, const float *d_x, const uint32_t *d_row_ids, uint64_t n,
                              const uint32_t *d_owner, uint32_t my_rank, uint64_t *kept);
/* fvdb_assign (find_nearest_centroid for a batch, src/ivf/core.rs:373-386) with device buffers: the list
 * histogram the placement above is computed from, without moving rows. */
int fvdb_assign_device(fvdb_index *h, const float *d_x, uint64_t n, uint32_t *d_out_list, void *stream);
int fvdb_ivf_train_device(fvdb_index *h, const float *d_data, uint64_t n, uint32_t nlist,
                          uint32_t max_iterations, const float *d_init_centroids, uint64_t seed,
                          fvdb_train_result *out);

/* One Lloyd iteration on device data with externally reduced sums — the multi-GPU k-means
 * building blocks (SURVEY §2a C2): step 1 assigns this rank's points and accumulates
 * per-cluster f32 sums [nlist x dim] and counts [nlist] (u32) plus the squared-error sum
 * (f64 scalar, device) into caller buffers; the caller all-reduces them; step 2 installs
 * means (empty cluster keeps its centroid, src/ivf/core.rs:410-415). */
int fvdb_kmeans_accumulate_device(fvdb_index *h, const float *d_data, uint64_t n,
                                  float *d_sums, uint32_t *d_counts, double *d_sqerr,
                                  uint32_t *d_assign, uint32_t *d_changed, void *stream);
int fvdb_kmeans_apply_device(fvdb_index *h, const float *d_sums, const uint32_t *d_counts,
                             void *stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* FVDB_H_ */
