// tc_scan.cuh — interface of the tensor-core (tcgen05 / TMEM / TMA) scan path.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "common.cuh"

namespace fvdb {

struct TcScratchImpl;

// Per-handle state of the tensor-core path: row norms, TMA descriptors, work buffers.
// The *_dirty flags are raised by the engine whenever the corresponding matrix moved.
struct TcScratch {
    bool arena_dirty = true;
    bool flat_dirty = true;
    bool centroids_dirty = true;
    TcScratchImpl* impl = nullptr;
};

constexpr uint32_t TC_MAX_K = 16;        // largest k served by the 32-entry shortlist
constexpr uint32_t TC_MAX_NPROBE = 256;  // partial lists merged in one pass
constexpr uint32_t TC_MAX_NPROBE_COARSE = 112;  // tensor-core coarse step (else exact coarse)
constexpr uint32_t TC_TILE_Q = 64;       // queries per work item of kernel R up to D = 512 (32 up to 1024, 16 above)
constexpr uint32_t TC_MAX_D = 2048;      // widest row served (kernel R alone above D = 384)
constexpr uint32_t TC_WIDE_MIN_QUERIES = 129;  // lists probed by at least this many queries of a batch go to kernel W
constexpr uint32_t TC_MAX_PEERS = 7;     // peer GPUs whose bound arrays one scan can push to

struct TcSearchArgs {
    const float* rows;        // IVF arena [n_rows x D]
    const uint32_t* ids;      // [n_rows]
    uint64_t n_rows;
    const uint32_t* list_off; // [nlist + 1] device
    uint32_t nlist;
    const float* Q;           // [nq x D]
    uint32_t nq, D, k, nprobe;
    const float* centroids;       // [nlist x D]
    const uint64_t* coarse_keys;  // [nq][nprobe] exact coarse ranking (low 32 bits = list id), or
                                  // nullptr: computed here on the tensor cores (nprobe <= 128)
    uint64_t* coarse_out;         // when computed here: [nq][nprobe] exact keys (may be nullptr)
    bool coarse_only = false;     // stop after the coarse step (keys in coarse_out); the arena is not touched
    const uint64_t* tomb;
    uint64_t tomb_bits;
    const uint64_t* filt;
    uint64_t filt_bits;
    uint64_t* out_keys;       // [nq][k] exact keys (distance bits << 32 | row id), sorted
    uint64_t* d_scanned_rows; // device counter (distinct posting-list rows streamed)
    uint32_t* d_fallback_count;   // device: number of queries whose proof failed
    uint32_t* d_fallback_idx;     // device [nq]: their indices
    cudaEvent_t ev_scan0, ev_scan1;
    int sm_count;
    // multi-GPU bound sharing (optional): the per-query bound array of this batch lives in memory
    // the peer GPUs can reach (already reset to +inf by the caller); a bound tightened here is
    // also pushed into the peers' arrays with NVLink atomics, so that a shard which does not hold
    // a query's nearest lists still scans with that query's tight threshold
    uint32_t* thr_ext = nullptr;
    uint32_t* thr_peers[TC_MAX_PEERS] = {};
    uint32_t n_peers = 0;
    cudaEvent_t wait_before_scan = nullptr;    // pipeline slots: the scan kernels start behind this event ...
    cudaEvent_t record_after_scan = nullptr;   // ... and this one is recorded behind them
    uint32_t scan_sms = 0;            // CTAs of the scan kernels (0 = one per SM); see FVDB_OPT_SCAN_SMS
    float xmax_floor_sq = 0.f;        // lower bound of the max |x|^2 term of the proof (max over all shards)
    // optional fusions with the caller's steps (both save a launch per batch):
    int* d_nan = nullptr;             // set to 1 when Q holds a NaN (the query-norm pass sees every element)
    uint32_t* fin_ids = nullptr;      // when given, the re-rank also writes the caller-facing result
    float* fin_dist = nullptr;        //   arrays [nq][k] / [nq] (what finalize_kernel derives from
    uint32_t* fin_count = nullptr;    //   out_keys when no other tier takes part)
};

// Tensor-core scan of the recent ("HNSW") tier: every query against every flat row.
struct TcFlatArgs {
    const float* rows;        // flat tier [n_rows x D]
    const uint32_t* ids;      // [n_rows]
    uint64_t n_rows;
    const float* Q;           // [nq x D]
    uint32_t nq, D, k;
    const uint64_t* tomb;
    uint64_t tomb_bits;
    const uint64_t* filt;
    uint64_t filt_bits;
    uint64_t* out_keys;           // [nq][k] exact keys, sorted
    uint32_t* d_fallback_count;   // device: queries whose proof failed
    uint32_t* d_fallback_idx;     // device [nq]
    int sm_count;
    // which cached row set (norms + TMA descriptor): 0 = the recent tier (invalidated by
    // TcScratch::flat_dirty), 1 = the centroid table scanned by batched nearest-centroid
    // assignment (invalidated when `version` changes)
    uint32_t state = 0;
    uint64_t version = 0;
    uint32_t rerank_r = 0;        // shortlist entries re-ranked exactly (0 = all 32)
    int metric = 0;               // METRIC_L2 | METRIC_COS | METRIC_DOT (common.cuh)
    bool argmin_only = false;     // k = 1 and the caller wants ids only: provably separated queries skip the exact re-rank
    cudaEvent_t ev_scan0 = nullptr, ev_scan1 = nullptr;   // optional: recorded around the scan kernel
};

// dim % 32 == 0 (one 128-byte swizzle atom per k-block), 32 <= dim <= TC_MAX_D (the query tile of a kernel R
// item, at most 128 KB, stays resident in shared memory)
bool tc_supported(uint32_t D);

// Tensor-core shortlist scan of the probed posting lists + exact fp32 re-rank + proof check.
// Enqueues everything on `st`; queries whose proof fails are listed in d_fallback_idx and must
// be re-run on the exact path by the caller.
int tc_ivf_search(TcScratch& s, const TcSearchArgs& a, cudaStream_t st, size_t* dev_bytes,
                  uint32_t* launches, std::string* err);
// Same machinery for the flat tier (replaces HNSWIndex::search, src/hnsw/core.rs:398-467, by an
// exhaustive scan): work items = (64-query group) x (row chunk), shortlist + exact re-rank + proof.
int tc_flat_search(TcScratch& s, const TcFlatArgs& a, cudaStream_t st, size_t* dev_bytes, uint32_t* launches,
                   std::string* err);
void tc_release(TcScratch& s);
cudaError_t launch_fill_u32(uint32_t* p, uint64_t n, uint32_t v, cudaStream_t stream);
// norms[i] = |x_i|^2 (scratch, n floats), *max_bits = max over rows as f32 bits (caller zeroes it)
cudaError_t launch_max_sqnorm(const float* x, uint64_t n, uint32_t D, float* scratch_norms, uint32_t* max_bits,
                              cudaStream_t stream);

}  // namespace fvdb
