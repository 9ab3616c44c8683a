// kernels.cuh — launcher declarations shared by the engine translation units.
#pragma once

#include "common.cuh"

namespace fvdb {

// ---- exact_scan.cu --------------------------------------------------------------------------
struct ExactScanArgs {
    const float* X;            // row matrix [rows x D] (device)
    const uint32_t* ids;       // row ids per row, or nullptr => id = row index
    const float* Q;            // queries [nq x D]
    uint32_t D;
    const ScanItem* items;
    const uint32_t* item_count;  // device count, or nullptr => n_items
    uint32_t n_items;
    const uint32_t* pair_q;    // non-identity items: query index per pair
    const uint32_t* pair_slot; //                     partial slot per pair
    uint32_t P;                // partial slots per query
    uint32_t k;
    const uint64_t* tomb;      // tombstone bitmap over ids (bit set = deleted) or nullptr
    uint64_t tomb_bits;
    const uint64_t* filt;      // filter bitmap over ids (bit set = passes) or nullptr
    uint64_t filt_bits;
    uint64_t* partial;         // [nq][P][k] sorted keys
    int metric = 0;            // METRIC_L2 | METRIC_COS | METRIC_DOT (common.cuh): how a (query, row) pair is scored
};

size_t exact_scan_smem_bytes(uint32_t k);
uint32_t exact_scan_tq();
uint32_t exact_scan_tr();
cudaError_t launch_exact_scan(const ExactScanArgs& a, uint32_t grid, cudaStream_t stream);
cudaError_t launch_build_identity_items(ScanItem* items, uint32_t nq, uint32_t row_begin,
                                        uint32_t row_end, uint32_t nsplit, uint32_t* n_items_out,
                                        cudaStream_t stream);
cudaError_t launch_probe_bucketing(const uint64_t* coarse_keys, uint32_t nq, uint32_t nprobe,
                                   const uint32_t* list_off, uint32_t nlist, uint32_t tile_q,
                                   uint32_t* list_cnt, uint32_t* pair_off, uint32_t* cursor,
                                   uint32_t* pair_q, uint32_t* pair_slot, ScanItem* items,
                                   uint32_t* n_items, uint64_t* scanned_rows, cudaStream_t stream,
                                   const uint32_t* list_order = nullptr, uint32_t rows_cap = 0,
                                   // optional second table: lists probed by >= wide_min queries become items
                                   // of tile_q_w queries in items_w (the wide-tile scan kernel's share)
                                   uint32_t wide_min = 0, uint32_t tile_q_w = 0, ScanItem* items_w = nullptr,
                                   uint32_t* n_items_w = nullptr,
                                   // optional (with list_order): the non-empty lists, ascending — only those are walked
                                   const uint32_t* live_ids = nullptr, uint32_t n_live = 0);
// one warp per (query, probed list): sparse batches (few queries per list)
cudaError_t launch_exact_pair_scan(const uint64_t* coarse_keys, uint32_t nq, uint32_t nprobe, const uint32_t* list_off,
                                   const float* X, const uint32_t* ids, const float* Q, uint32_t D, uint32_t P,
                                   uint32_t k, const uint64_t* tomb, uint64_t tomb_bits, const uint64_t* filt,
                                   uint64_t filt_bits, uint64_t* partial, cudaStream_t stream);
cudaError_t launch_merge_partials(const uint64_t* in, uint32_t nq, uint32_t P, uint32_t k,
                                  uint64_t* out, cudaStream_t stream);
// same for P rows of 32 keys each that may be unsorted or empty (tensor-core scan output)
cudaError_t launch_merge_rows32(const uint64_t* in, uint32_t nq, uint32_t P, uint64_t* out,
                                cudaStream_t stream, const uint32_t* row_stamp, uint32_t stamp);
// ivf_ids / ivf_dist / ivf_count given: the tiers are not merged, the IVF tier goes to this second set
cudaError_t launch_finalize(const uint64_t* recent, const uint64_t* ivf, uint32_t nq, uint32_t k,
                            uint32_t* out_ids, float* out_dist, uint32_t* out_count,
                            cudaStream_t stream, int metric = 0, uint32_t* ivf_ids = nullptr,
                            float* ivf_dist = nullptr, uint32_t* ivf_count = nullptr);
// tiered: part p holds rows of tier p & 1, order (distance, tier, row id)
cudaError_t launch_merge_parts(const uint32_t* ids, const float* dist, const uint32_t* cnt,
                               uint32_t parts, uint32_t nq, uint32_t k, uint32_t* out_ids,
                               float* out_dist, uint32_t* out_count, cudaStream_t stream,
                               size_t stride_kv = 0, size_t stride_c = 0, bool tiered = false);
// dst[idx[i]][0..k) = src[i][0..k)
cudaError_t launch_scatter_result_rows(const uint32_t* ids, const float* dist, const uint32_t* cnt,
                                       const uint32_t* idx, uint32_t n, uint32_t k, uint32_t* out_ids,
                                       float* out_dist, uint32_t* out_cnt, cudaStream_t stream);
// 3x post-filter of src/hybrid/core.rs:529-546: keep the candidates whose id bit is set, truncate to k
cudaError_t launch_postfilter_rows(const uint32_t* ids, const float* dist, const uint32_t* cnt, uint32_t nq,
                                   uint32_t k3, uint32_t k, const uint64_t* keep, uint64_t keep_bits,
                                   uint32_t* out_ids, float* out_dist, uint32_t* out_cnt, cudaStream_t stream);
cudaError_t launch_scatter_keys(const uint64_t* src, const uint32_t* idx, uint32_t n, uint32_t k,
                                uint64_t* dst, cudaStream_t stream);
cudaError_t launch_nan_check(const float* x, size_t n, int* flag, cudaStream_t stream);

// ---- layout.cu: stable grouping, gathers, bitmaps -------------------------------------------
// Stable counting sort of n keys (< nkeys; key == nkeys means "drop") into groups.
//   offsets [nkeys+2] (device): group g occupies [offsets[g], offsets[g+1]); dropped rows after
//   perm    [n]: perm[new_pos] = old index, order inside a group = original order (stable)
// scratch: see stable_group_scratch_bytes.
size_t stable_group_scratch_bytes(uint64_t n, uint32_t nkeys);
cudaError_t launch_stable_group(const uint32_t* keys, uint64_t n, uint32_t nkeys, uint32_t* offsets,
                                uint32_t* perm, void* scratch, cudaStream_t stream);
// dst[i] = src[perm[i]] for rows of D floats (two sources: index < n0 from src0 else src1).
cudaError_t launch_gather_rows(const float* src0, uint64_t n0, const float* src1, const uint32_t* perm,
                               uint64_t n, uint32_t D, float* dst, cudaStream_t stream);
cudaError_t launch_gather_u32(const uint32_t* src0, uint64_t n0, const uint32_t* src1,
                              const uint32_t* perm, uint64_t n, uint32_t* dst, cudaStream_t stream);
// keys[i] = bit(ids[i]) ? key_if_set : keys_else[i] (keys_else nullptr => key_if_clear)
cudaError_t launch_keys_from_bitmap(const uint32_t* ids, uint64_t n, const uint64_t* bits,
                                    uint64_t nbits, uint32_t key_if_set, const uint32_t* keys_else,
                                    uint32_t key_if_clear, uint32_t* keys, cudaStream_t stream);
cudaError_t launch_set_bits(uint64_t* bits, uint64_t nbits, const uint32_t* ids, uint64_t n, int value,
                            cudaStream_t stream);
// keys_out[i] = (keys[i] % mod == rem) ? keys[i] : drop
cudaError_t launch_filter_keys_mod(const uint32_t* keys, uint64_t n, uint32_t mod, uint32_t rem,
                                   uint32_t drop, uint32_t* keys_out, cudaStream_t stream);
// keys[i] = owner[lists[i]] == rank ? lists[i] : nlist + owner[lists[i]]  (nlist + world when the owner is
// >= world): launch_stable_group over nlist + world keys then puts the kept rows first, grouped by list, and
// the rows of every other rank after them, rank by rank.  With world = 0 those rows all get nlist, the drop group
// of a grouping over nlist keys: the owned IVF add keeps the rows of its own lists that way.
cudaError_t launch_owner_keys(const uint32_t* lists, uint64_t n, const uint32_t* owner, uint32_t rank,
                              uint32_t world, uint32_t nlist, uint32_t* keys, cudaStream_t stream);
cudaError_t launch_extract_assign(const uint64_t* keys, uint64_t n, uint32_t* assign, float* dist,
                                  const uint32_t* prev_assign, uint32_t* changed, cudaStream_t stream);

// ---- kmeans.cu ------------------------------------------------------------------------------
// Order-faithful centroid update (src/ivf/core.rs:388-417): thread (cluster, dim) sums its
// cluster's members in data order (perm from launch_stable_group), mean = sum / count.
cudaError_t launch_centroid_update(const float* data, uint32_t D, const uint32_t* offsets,
                                   const uint32_t* perm, uint32_t nlist, float* centroids,
                                   cudaStream_t stream);
// dist[i] = L2(data[i], centroids[assign[i]]) in reference order (compute_error :419-429).
cudaError_t launch_rowwise_dist(const float* data, uint64_t n, uint32_t D, const float* centroids,
                                const uint32_t* assign, float* dist, cudaStream_t stream);
// unordered accumulation for the multi-GPU path: sums[assign[i]] += data[i] (f32 atomics),
// counts, squared error (f64).
cudaError_t launch_accumulate_sums(const float* data, uint64_t n, uint32_t D, const uint32_t* assign,
                                   const float* dist, float* sums, uint32_t* counts, double* sqerr,
                                   cudaStream_t stream);
cudaError_t launch_apply_means(const float* sums, const uint32_t* counts, uint32_t nlist, uint32_t D,
                               float* centroids, cudaStream_t stream);
cudaError_t launch_copy_row(const float* data, const uint32_t* idx, uint32_t D, float* dst,
                            cudaStream_t stream);

}  // namespace fvdb
