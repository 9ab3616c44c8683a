// engine.cu — handle state, HBM layout management and the C ABI of include/fvdb.h.
//
// Device state behind one handle (= one HybridIndex, src/hybrid/core.rs:202-213):
//   centroids  C[nlist x D] fp32                            (Vec<Centroid>, src/ivf/core.rs:156)
//   IVF arena  X[ivf_n x D] fp32, rows of list l contiguous at [list_off[l], list_off[l+1]),
//              ids[ivf_n] (caller row ids), list[ivf_n]      (inverted_lists, :157)
//   pending    rows appended since the last seal (assigned, not yet grouped)
//   flat tier  R[flat_n x D] fp32 + ids[flat_n]              (HNSW nodes, src/hnsw/core.rs:141)
//   tombstones u64 bitmap over row ids                       (deleted: HashSet, src/ivf/core.rs:167)
// There is no CPU fallback anywhere in this file: every numeric result comes from a kernel.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fvdb.h"
#include "common.cuh"
#include "kernels.cuh"
#include "tc_scan.cuh"

using namespace fvdb;

namespace {

std::mutex g_err_mu;
std::string g_create_err;

template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    // grow to >= n elements; preserve the first `keep` elements
    cudaError_t ensure(size_t n, size_t keep, cudaStream_t s, size_t* total_bytes, bool exact = false) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = exact ? n : std::max(n, cap + cap / 2);
        T* np = nullptr;
        cudaError_t e = cudaMalloc(&np, ncap * sizeof(T));
        if (e != cudaSuccess) return e;
        if (keep && p) {
            e = cudaMemcpyAsync(np, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) { cudaFree(np); return e; }
            e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) { cudaFree(np); return e; }
        }
        if (p) cudaFree(p);
        if (total_bytes) *total_bytes += (ncap - cap) * sizeof(T);
        p = np;
        cap = ncap;
        return cudaSuccess;
    }
    void swap(DevBuf& o) { std::swap(p, o.p); std::swap(cap, o.cap); }
};

// rand 0.8's StdRng as IVFIndex::new seeds it (`StdRng::seed_from_u64`, src/ivf/core.rs:176-179) and as
// initialize_centroids draws from it (`gen_range(0..n)` :341, `gen::<f32>()` :359), restated from the
// published algorithms: rand_core 0.6 seed_from_u64 = a PCG32 stream expanded into the 32-byte key;
// StdRng = ChaCha with 12 rounds, 64-bit block counter from 0, stream 0, four blocks (64 words) per
// refill, words consumed in order; next_u64 = two consecutive words, low first; u64 sample_single =
// widening multiply with a rejection zone; Standard f32 = (next_u32 >> 8) * 2^-24.
// rand is an un-vendored, un-pinned dependency of the reference (Cargo.toml:41; SURVEY App. B): parity
// with it is unpinned.  What IS tested: this generator == the oracle's independent restatement, and the
// picks made with it == the oracle's fo_kmeanspp_init on the same seed.
struct StdRng08 {
    uint32_t key[8];
    uint64_t counter = 0;
    uint32_t buf[64];
    uint32_t index = 64;   // next unread word; 64 = empty

    explicit StdRng08(uint64_t seed) {
        const uint64_t MUL = 6364136223846793005ull, INC = 11634580027462260723ull;
        for (int i = 0; i < 8; ++i) {
            seed = seed * MUL + INC;
            const uint32_t xs = (uint32_t)(((seed >> 18) ^ seed) >> 27);
            const uint32_t rot = (uint32_t)(seed >> 59);
            key[i] = (xs >> rot) | (xs << ((32u - rot) & 31u));
        }
    }
    static uint32_t rotl(uint32_t v, int c) { return (v << c) | (v >> (32 - c)); }
    static void quarter(uint32_t* x, int a, int b, int c, int d) {
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 16);
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 12);
        x[a] += x[b]; x[d] = rotl(x[d] ^ x[a], 8);
        x[c] += x[d]; x[b] = rotl(x[b] ^ x[c], 7);
    }
    void block(uint64_t ctr, uint32_t* out) const {
        uint32_t in[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3],
                           key[4], key[5], key[6], key[7], (uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u};
        uint32_t x[16];
        std::memcpy(x, in, sizeof(x));
        for (int r = 0; r < 6; ++r) {   // 12 rounds: six column + diagonal double rounds
            quarter(x, 0, 4, 8, 12); quarter(x, 1, 5, 9, 13); quarter(x, 2, 6, 10, 14); quarter(x, 3, 7, 11, 15);
            quarter(x, 0, 5, 10, 15); quarter(x, 1, 6, 11, 12); quarter(x, 2, 7, 8, 13); quarter(x, 3, 4, 9, 14);
        }
        for (int i = 0; i < 16; ++i) out[i] = x[i] + in[i];
    }
    void refill() {
        for (int b = 0; b < 4; ++b) block(counter + (uint64_t)b, buf + 16 * b);
        counter += 4;
        index = 0;
    }
    uint32_t next_u32() {
        if (index >= 64) refill();
        return buf[index++];
    }
    uint64_t next_u64() {   // BlockRng::next_u64, including the word that straddles a refill
        if (index < 63) {
            const uint64_t lo = buf[index], hi = buf[index + 1];
            index += 2;
            return (hi << 32) | lo;
        }
        if (index >= 64) {
            refill();
            index = 2;
            return ((uint64_t)buf[1] << 32) | buf[0];
        }
        const uint64_t lo = buf[63];
        refill();
        index = 1;
        return ((uint64_t)buf[0] << 32) | lo;
    }
    uint64_t gen_range(uint64_t range) {   // gen_range(0..range), range > 0
        const uint64_t zone = (range << __builtin_clzll(range)) - 1;
        for (;;) {
            const unsigned __int128 m = (unsigned __int128)next_u64() * range;
            if ((uint64_t)m <= zone) return (uint64_t)(m >> 64);
        }
    }
    float gen_f32() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
};

// Pinned host destinations of a batch's results: the device -> host copies ride in front of the
// batch's single synchronisation point (the NaN flag / fallback counter read-back).
struct HostOut {
    void* ids;
    void* dist;
    void* cnt;
    size_t ob, cb;  // bytes of ids / dist, of cnt
};

// The per-batch scratch of a search: counter words, the IVF tier's proof-failure list, coarse and IVF keys,
// tensor-core tables and the timing events.  The handle owns one for the batches on its own stream; each
// pipeline slot owns another.
struct BatchScratch {
    // misc words: [0] nan flag, [2..3] scanned rows (u64), [4] kmeans changed, [6] item count,
    // [8] kmeans++ pick, [10] IVF fallback count, [11] flat fallback count, [12] assign fallback count,
    // [13] max |x|^2 bits
    DevBuf<uint32_t> misc, fb_idx;
    DevBuf<uint64_t> coarse, ivf_keys;
    TcScratch tc;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;     // around the batch
    cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;   // around the scan kernel
    cudaError_t create_events() {
        cudaError_t e = cudaSuccess;
        for (cudaEvent_t* ev : {&ev_a, &ev_b, &ev_s0, &ev_s1})
            if (e == cudaSuccess) e = cudaEventCreate(ev);
        return e;
    }
    void release() {
        tc_release(tc);
        for (cudaEvent_t ev : {ev_a, ev_b, ev_s0, ev_s1})
            if (ev) cudaEventDestroy(ev);
    }
};

}  // namespace

// One fvdb_search call waiting in the handle's submission queue (see fvdb_search).
struct SearchReq {
    const float* q;
    uint32_t nq, k, nprobe, tiers;
    uint32_t* out_ids;
    float* out_dist;
    uint32_t* out_count;
    int rc = FVDB_OK;
    enum State { WAITING, LEAD, DONE } state = WAITING;
    std::condition_variable cv;
};

struct fvdb_index {
    int device = 0;
    uint32_t dim = 0, k_max = 0;
    int metric = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string err;
    uint32_t scan_mode = FVDB_SCAN_EXACT;
    uint32_t shortlist = 0;
    uint32_t kmeans_tc = 0;
    uint32_t scan_sms = 0;              // FVDB_OPT_SCAN_SMS
    float proof_xmax_sq = 0.f;          // FVDB_OPT_PROOF_XMAX: max |x|^2 over ALL shards of a list-sharded index
    uint64_t centroids_version = 0;     // bumped whenever the centroid table changes
    uint64_t assign_fallback_rows = 0;  // rows re-assigned exactly after a failed tensor-core proof
    size_t dev_bytes = 0;

    uint32_t nlist = 0;
    bool trained = false;
    DevBuf<float> centroids;

    DevBuf<float> ivf_rows;
    DevBuf<uint32_t> ivf_ids, ivf_list;
    uint64_t ivf_n = 0;
    DevBuf<uint32_t> list_off;  // nlist + 2

    DevBuf<float> pend_rows;
    DevBuf<uint32_t> pend_ids, pend_list;
    uint64_t pend_n = 0;

    DevBuf<float> flat_rows;
    DevBuf<uint32_t> flat_ids;
    uint64_t flat_n = 0;

    DevBuf<uint64_t> tomb;
    uint64_t tomb_bits = 0;
    uint64_t deleted_count = 0;

    // host-side presence map over row ids: 0 absent, 1 flat, 2 ivf; bit 7 = tombstoned.
    std::vector<uint8_t> id_state;
    bool track_ids = true;

    // scratch (grow-only)
    BatchScratch scratch;                // per-batch scratch of everything that runs on the handle's stream
    DevBuf<float> s_q, s_x;              // staged queries / staged rows
    DevBuf<uint32_t> s_u32a, s_u32b, s_u32c, s_perm, s_keys32;
    DevBuf<uint64_t> s_filter;
    DevBuf<uint64_t> s_partial, s_partial2, s_flat_keys;
    DevBuf<ScanItem> s_items, s_items2;
    DevBuf<uint32_t> s_list_cnt, s_pair_off, s_cursor, s_pair_q, s_pair_slot;
    DevBuf<unsigned char> s_group;
    DevBuf<uint32_t> s_out_ids, s_out_cnt;
    DevBuf<float> s_out_dist, s_f32a;
    DevBuf<double> s_f64;
    DevBuf<uint64_t> s_tmpbits;
    DevBuf<uint32_t> s_fb_idx_flat;
    // A page-locked block of u32 words and its size: the read-back record of a stream-ordered batch.
    using Record = std::pair<uint32_t*, size_t>;
    // A search batch whose kernels are enqueued: what a repair of its proof failures re-runs and where its figures
    // come from.  The stream-ordered entries keep it until fvdb_search_device_finish.
    struct Pending {
        const float* d_q; uint32_t nq, k, nprobe, tiers;
        const uint64_t* d_filter; uint64_t filter_bits;
        uint32_t* d_out_ids; float* d_out_dist; uint32_t* d_out_count;
        HostOut ho;           // the caller's pinned result buffers (ids NULL: none)
        bool split;           // fvdb_search_device_tiers: the outputs are a two-part packed chunk
        bool used_tc, flat_tc, use_ivf, use_flat;
        uint32_t n_bitmaps;   // tombstone / filter bitmaps read per row (for the algorithmic-bytes figure)
        int slot;             // pipeline slot the batch ran in (-1: the handle's own stream and scratch)
        BatchScratch* scratch;   // the scratch it ran with (its timing events)
        Record rec;           // stream-ordered: [16] counter words, [2 nq] IVF fallback ids, [2 nq] flat fallback ids
    };
    // fvdb_search_submit: device-side query / result buffers of the batches in flight and the copy stream
    // their uploads run on (so that batch i + 1 uploads while batch i is scanned)
    struct HostSlot {
        DevBuf<float> q;
        DevBuf<uint32_t> ids, cnt;
        DevBuf<float> dist;
        cudaEvent_t uploaded = nullptr, done = nullptr;
        bool used = false;
    };
    static constexpr int HOST_SLOTS = 8;
    HostSlot host_slots[HOST_SLOTS];
    uint32_t host_slot_next = 0;
    cudaStream_t copy_stream = nullptr;
    std::vector<Pending> pending;
    std::vector<Record> pending_coarse;   // records of fvdb_coarse_device_submit
    std::vector<Record> pending_pool;     // recycled page-locked blocks
    DevBuf<float> s_fb_q;
    DevBuf<uint64_t> s_fb_keys, s_fb_coarse;
    DevBuf<uint32_t> s_fb_rows;          // the queries a proof-failure repair re-runs
    // Software pipeline of the stream-ordered entries (fvdb_search_device_submit / fvdb_search_submit):
    // consecutive batches alternate between two SLOTS, each with its own stream and its own per-batch
    // scratch (tensor-core tables, coarse keys, counters).  The scans of consecutive batches are
    // serialised by an event (each one fills the machine), but batch i + 1's query norms, coarse step and
    // bucketing and batch i's shortlist merge and re-rank no longer queue behind one another: they run in
    // the scans' ramps and tails and next to kernel R's CTAs wherever registers and shared memory allow.
    struct Slot {
        BatchScratch b;
        cudaStream_t stream = nullptr;
        cudaEvent_t ev_in = nullptr, ev_scan_end = nullptr, ev_done = nullptr;
        bool busy = false;
    };
    static constexpr int N_SLOTS = 2;
    Slot slots[N_SLOTS];
    uint32_t slot_next = 0;
    cudaEvent_t prev_scan_end = nullptr;   // recorded behind the most recently enqueued slot scan
    uint32_t pipeline = 1;                 // FVDB_OPT_PIPELINE
    // submission queue of fvdb_search: concurrent host-buffer calls are coalesced into one batch
    std::mutex qmu;
    std::deque<SearchReq*> queue;
    bool leader_active = false;
    uint32_t coalesce = 1;
    uint32_t last_batch_calls = 0;
    // multi-GPU bound sharing (fvdb_bounds_*): [2][bounds_cap] u32, one half per batch parity
    uint32_t* bounds = nullptr;
    uint32_t bounds_cap = 0, bounds_parity = 0, bounds_armed_nq = 0;
    std::vector<uint32_t*> peer_bounds;   // peers' arrays (cudaIpcOpenMemHandle)

    // pinned staging
    void* pin = nullptr;
    size_t pin_bytes = 0;

    fvdb_stats stats{};

    int fail(int code, const std::string& m) {
        err = m;
        return code;
    }
    int fail_cuda(cudaError_t e, const char* what) {
        err = std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what;
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? FVDB_ERR_OOM : FVDB_ERR_CUDA;
    }
    cudaError_t ensure_pin(size_t bytes) {
        if (bytes <= pin_bytes) return cudaSuccess;
        if (pin) cudaFreeHost(pin);
        pin = nullptr;
        pin_bytes = 0;
        size_t nb = std::max(bytes, (size_t)1 << 20);
        cudaError_t e = cudaMallocHost(&pin, nb);
        if (e == cudaSuccess) pin_bytes = nb;
        return e;
    }
};

static inline void mark_arena_dirty(fvdb_index* h) {
    h->scratch.tc.arena_dirty = true;
    for (auto& sl : h->slots) sl.b.tc.arena_dirty = true;
}
static inline void mark_centroids_dirty(fvdb_index* h) {
    h->scratch.tc.centroids_dirty = true;
    for (auto& sl : h->slots) sl.b.tc.centroids_dirty = true;
}
// Every batch still running in a pipeline slot has to finish before anything it reads may move.
static inline void quiesce_slots(fvdb_index* h) {
    for (auto& sl : h->slots)
        if (sl.busy && sl.stream) { cudaStreamSynchronize(sl.stream); sl.busy = false; }
}

#define CK(call)                                                      \
    do {                                                              \
        cudaError_t e__ = (call);                                     \
        if (e__ != cudaSuccess) return h->fail_cuda(e__, #call);      \
    } while (0)
#define RET(call)                         \
    do {                                  \
        int r__ = (call);                 \
        if (r__ != FVDB_OK) return r__;   \
    } while (0)

namespace {

// ---- host <-> device staging through pinned memory ------------------------------------------
int h2d(fvdb_index* h, void* dst, const void* src, size_t bytes) {
    const size_t CH = (size_t)64 << 20;
    CK(h->ensure_pin(std::min(bytes, CH)));
    size_t off = 0;
    while (off < bytes) {
        const size_t n = std::min(CH, bytes - off);
        std::memcpy(h->pin, (const char*)src + off, n);
        CK(cudaMemcpyAsync((char*)dst + off, h->pin, n, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        off += n;
    }
    return FVDB_OK;
}
int d2h(fvdb_index* h, void* dst, const void* src, size_t bytes) {
    const size_t CH = (size_t)64 << 20;
    CK(h->ensure_pin(std::min(bytes, CH)));
    size_t off = 0;
    while (off < bytes) {
        const size_t n = std::min(CH, bytes - off);
        CK(cudaMemcpyAsync(h->pin, (const char*)src + off, n, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        std::memcpy((char*)dst + off, h->pin, n);
        off += n;
    }
    return FVDB_OK;
}

int check_nan_device(fvdb_index* h, const float* d_x, size_t n, cudaStream_t st) {
    CK(h->scratch.misc.ensure(64, 0, st, &h->dev_bytes));
    int* flag = reinterpret_cast<int*>(h->scratch.misc.p);
    CK(cudaMemsetAsync(flag, 0, sizeof(int), st));
    CK(launch_nan_check(d_x, n, flag, st));
    int hf = 0;
    CK(cudaMemcpyAsync(&hf, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (hf) return h->fail(FVDB_ERR_NAN, "NaN in input (the reference panics on partial_cmp().unwrap())");
    return FVDB_OK;
}

uint32_t pick_nsplit(fvdb_index* h, uint32_t nq, uint64_t rows) {
    const uint32_t n_qt = (nq + exact_scan_tq() - 1) / exact_scan_tq();
    const uint32_t tiles = (uint32_t)((rows + exact_scan_tr() - 1) / exact_scan_tr());
    uint32_t target = (uint32_t)h->sm_count * 4;
    uint32_t s = (target + n_qt - 1) / std::max(1u, n_qt);
    s = std::max(1u, std::min(s, std::max(1u, tiles)));
    s = std::min(s, 256u);
    return s;
}

// Scan every query against rows [0,rows) of X; result keys[nq][k] sorted (exact arithmetic).
int scan_all_exact(fvdb_index* h, const float* X, const uint32_t* ids, uint64_t rows, const float* Q,
                   uint32_t nq, uint32_t k, const uint64_t* tomb, uint64_t tomb_bits,
                   const uint64_t* filt, uint64_t filt_bits, uint64_t* out_keys, cudaStream_t st,
                   int metric = FVDB_METRIC_L2) {
    if (rows >= 0xFFFFFFFFull) return h->fail(FVDB_ERR_INVALID_ARG, "row count exceeds u32");
    const uint32_t nsplit = pick_nsplit(h, nq, rows);
    uint32_t n_items = 0;
    const uint32_t n_qt = (nq + exact_scan_tq() - 1) / exact_scan_tq();
    CK(h->s_items2.ensure((size_t)n_qt * nsplit, 0, st, &h->dev_bytes));
    CK(launch_build_identity_items(h->s_items2.p, nq, 0, (uint32_t)rows, nsplit, &n_items, st));
    uint64_t* partial = out_keys;
    if (nsplit > 1) {
        CK(h->s_partial2.ensure((size_t)nq * nsplit * k, 0, st, &h->dev_bytes));
        partial = h->s_partial2.p;
        CK(cudaMemsetAsync(partial, 0xFF, (size_t)nq * nsplit * k * sizeof(uint64_t), st));
    } else {
        CK(cudaMemsetAsync(partial, 0xFF, (size_t)nq * k * sizeof(uint64_t), st));
    }
    ExactScanArgs a{};
    a.X = X; a.ids = ids; a.Q = Q; a.D = h->dim;
    a.items = h->s_items2.p; a.item_count = nullptr; a.n_items = n_items;
    a.pair_q = nullptr; a.pair_slot = nullptr;
    a.P = nsplit; a.k = k;
    a.tomb = tomb; a.tomb_bits = tomb_bits; a.filt = filt; a.filt_bits = filt_bits;
    a.partial = partial;
    a.metric = metric;
    CK(launch_exact_scan(a, n_items, st));
    h->stats.last_launches += 3;
    if (nsplit > 1) {
        CK(launch_merge_partials(partial, nq, nsplit, k, out_keys, st));
        h->stats.last_launches += 1;
    }
    return FVDB_OK;
}

// Regroup sealed + pending IVF rows so every list is one contiguous row range.
int seal(fvdb_index* h) {
    if (h->pend_n == 0) return FVDB_OK;
    quiesce_slots(h);   // the arena is about to be replaced
    cudaStream_t st = h->stream;
    const uint64_t total = h->ivf_n + h->pend_n;
    if (total >= 0xFFFFFFF0ull) return h->fail(FVDB_ERR_INVALID_ARG, "IVF tier exceeds u32 rows");
    const uint32_t D = h->dim;
    CK(h->s_keys32.ensure(total, 0, st, &h->dev_bytes));
    if (h->ivf_n)
        CK(cudaMemcpyAsync(h->s_keys32.p, h->ivf_list.p, h->ivf_n * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->s_keys32.p + h->ivf_n, h->pend_list.p, h->pend_n * 4,
                       cudaMemcpyDeviceToDevice, st));
    CK(h->s_perm.ensure(total, 0, st, &h->dev_bytes));
    CK(h->s_group.ensure(stable_group_scratch_bytes(total, h->nlist), 0, st, &h->dev_bytes));
    CK(h->list_off.ensure(h->nlist + 2, 0, st, &h->dev_bytes));
    CK(launch_stable_group(h->s_keys32.p, total, h->nlist, h->list_off.p, h->s_perm.p, h->s_group.p, st));
    uint32_t kept = 0;
    CK(cudaMemcpyAsync(&kept, h->list_off.p + h->nlist, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    DevBuf<float> nrows;
    DevBuf<uint32_t> nids, nlist_ids;
    CK(nrows.ensure((size_t)std::max<uint64_t>(kept, 1) * D, 0, st, &h->dev_bytes, true));
    CK(nids.ensure(std::max<uint64_t>(kept, 1), 0, st, &h->dev_bytes, true));
    CK(nlist_ids.ensure(std::max<uint64_t>(kept, 1), 0, st, &h->dev_bytes, true));
    CK(launch_gather_rows(h->ivf_rows.p, h->ivf_n, h->pend_rows.p, h->s_perm.p, kept, D, nrows.p, st));
    CK(launch_gather_u32(h->ivf_ids.p, h->ivf_n, h->pend_ids.p, h->s_perm.p, kept, nids.p, st));
    CK(launch_gather_u32(h->ivf_list.p, h->ivf_n, h->pend_list.p, h->s_perm.p, kept, nlist_ids.p, st));
    CK(cudaStreamSynchronize(st));
    h->dev_bytes -= h->ivf_rows.cap * sizeof(float) + (h->ivf_ids.cap + h->ivf_list.cap) * 4;
    h->dev_bytes -= h->pend_rows.cap * sizeof(float) + (h->pend_ids.cap + h->pend_list.cap) * 4;
    h->ivf_rows.swap(nrows);
    h->ivf_ids.swap(nids);
    h->ivf_list.swap(nlist_ids);
    h->pend_rows.release();
    h->pend_ids.release();
    h->pend_list.release();
    h->ivf_n = kept;
    h->pend_n = 0;
    mark_arena_dirty(h);
    return FVDB_OK;
}

int ensure_tomb(fvdb_index* h, uint64_t nbits) {
    if (nbits <= h->tomb_bits) return FVDB_OK;
    const uint64_t words_old = (h->tomb_bits + 63) / 64;
    uint64_t nb = std::max<uint64_t>(nbits, h->tomb_bits * 2);
    nb = (nb + 4095) / 4096 * 4096;
    const uint64_t words = nb / 64;
    CK(h->tomb.ensure(words, words_old, h->stream, &h->dev_bytes));
    CK(cudaMemsetAsync(h->tomb.p + words_old, 0, (words - words_old) * 8, h->stream));
    h->tomb_bits = nb;
    return FVDB_OK;
}

int append_pending(fvdb_index* h, const float* d_x, const uint32_t* d_ids, const uint32_t* d_list,
                   uint64_t n) {
    if (n == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    CK(h->pend_rows.ensure((h->pend_n + n) * D, h->pend_n * D, st, &h->dev_bytes));
    CK(h->pend_ids.ensure(h->pend_n + n, h->pend_n, st, &h->dev_bytes));
    CK(h->pend_list.ensure(h->pend_n + n, h->pend_n, st, &h->dev_bytes));
    CK(cudaMemcpyAsync(h->pend_rows.p + h->pend_n * D, d_x, n * D * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->pend_ids.p + h->pend_n, d_ids, n * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->pend_list.p + h->pend_n, d_list, n * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    h->pend_n += n;
    return FVDB_OK;
}

// assign rows to their nearest centroid: out d_assign[n] (and optionally distances)
int assign_device(fvdb_index* h, const float* d_x, uint64_t n, uint32_t* d_assign, float* d_dist,
                  const uint32_t* prev, uint32_t* d_changed, cudaStream_t st) {
    if (n == 0) return FVDB_OK;
    if (n >= 0xFFFFFFFFull) return h->fail(FVDB_ERR_INVALID_ARG, "batch exceeds u32 rows");
    BatchScratch& b = h->scratch;
    CK(b.ivf_keys.ensure(n, 0, st, &h->dev_bytes));
    // Large batches (k-means iterations, bulk insert / load): the rows play the "queries", the
    // centroid table the scanned row set of the tensor-core flat scan; the four approximately
    // nearest centroids are re-ranked in the reference's arithmetic and the fifth bounds the rest
    // (proof as in tc_scan.cu); rows whose proof fails are re-assigned by the exact kernel.
    const bool tc = h->scan_mode == FVDB_SCAN_TC && tc_supported(h->dim) && h->nlist >= 256 &&
                    n * (uint64_t)h->nlist >= (64ull << 20);
    if (tc) {
        const uint64_t CH = 1u << 18;   // rows per pass: bounds the shortlist scratch (256 B per row)
        CK(b.misc.ensure(64, 0, st, &h->dev_bytes));
        uint32_t* d_fb = b.misc.p + 12;
        for (uint64_t r0 = 0; r0 < n; r0 += CH) {
            const uint32_t m = (uint32_t)std::min<uint64_t>(CH, n - r0);
            CK(h->s_fb_idx_flat.ensure((size_t)2 * m, 0, st, &h->dev_bytes));
            CK(cudaMemsetAsync(d_fb, 0, 4, st));
            TcFlatArgs fa{};
            fa.rows = h->centroids.p; fa.ids = nullptr; fa.n_rows = h->nlist;
            fa.Q = d_x + r0 * h->dim; fa.nq = m; fa.D = h->dim; fa.k = 1;
            fa.out_keys = b.ivf_keys.p + r0;
            fa.d_fallback_count = d_fb; fa.d_fallback_idx = h->s_fb_idx_flat.p;
            fa.sm_count = h->sm_count;
            fa.state = 1; fa.version = h->centroids_version; fa.rerank_r = 4;
            fa.argmin_only = d_dist == nullptr;
            uint32_t launches = 0;
            int r = tc_flat_search(b.tc, fa, st, &h->dev_bytes, &launches, &h->err);
            if (r != FVDB_OK) return r;
            uint32_t n_fb = 0;
            CK(cudaMemcpyAsync(&n_fb, d_fb, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            n_fb = std::min(n_fb, 2 * m);
            if (n_fb) {
                CK(h->s_fb_q.ensure((size_t)n_fb * h->dim, 0, st, &h->dev_bytes));
                CK(h->s_fb_keys.ensure((size_t)n_fb, 0, st, &h->dev_bytes));
                CK(launch_gather_rows(d_x + r0 * h->dim, m, nullptr, h->s_fb_idx_flat.p, n_fb, h->dim, h->s_fb_q.p, st));
                RET(scan_all_exact(h, h->centroids.p, nullptr, h->nlist, h->s_fb_q.p, n_fb, 1, nullptr, 0, nullptr, 0,
                                   h->s_fb_keys.p, st));
                CK(launch_scatter_keys(h->s_fb_keys.p, h->s_fb_idx_flat.p, n_fb, 1, b.ivf_keys.p + r0, st));
            }
            h->assign_fallback_rows += n_fb;
        }
    } else {
        RET(scan_all_exact(h, h->centroids.p, nullptr, h->nlist, d_x, (uint32_t)n, 1, nullptr, 0,
                           nullptr, 0, b.ivf_keys.p, st));
    }
    CK(launch_extract_assign(b.ivf_keys.p, n, d_assign, d_dist, prev, d_changed, st));
    return FVDB_OK;
}

int ivf_add_device_impl(fvdb_index* h, const float* d_x, const uint32_t* d_ids, uint64_t n,
                        uint32_t mod, uint32_t rem, uint64_t* kept_out, uint32_t* h_out_list,
                        const uint32_t* d_owner = nullptr) {
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (kept_out) *kept_out = 0;
    if (n == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    RET(check_nan_device(h, d_x, n * D, st));
    CK(h->s_u32a.ensure(n, 0, st, &h->dev_bytes));
    RET(assign_device(h, d_x, n, h->s_u32a.p, nullptr, nullptr, nullptr, st));
    if (h_out_list) RET(d2h(h, h_out_list, h->s_u32a.p, n * 4));
    if (mod <= 1) {
        RET(append_pending(h, d_x, d_ids, h->s_u32a.p, n));
        if (kept_out) *kept_out = n;
        return FVDB_OK;
    }
    // list-sharded load: keep only rows whose list % mod == rem, compacted (grouped by list)
    CK(h->s_u32b.ensure(n, 0, st, &h->dev_bytes));
    if (d_owner) CK(launch_filter_keys_owner(h->s_u32a.p, n, d_owner, rem, h->nlist, h->s_u32b.p, st));
    else CK(launch_filter_keys_mod(h->s_u32a.p, n, mod, rem, h->nlist, h->s_u32b.p, st));
    CK(h->s_perm.ensure(n, 0, st, &h->dev_bytes));
    CK(h->s_group.ensure(stable_group_scratch_bytes(n, h->nlist), 0, st, &h->dev_bytes));
    CK(h->s_u32c.ensure(h->nlist + 2, 0, st, &h->dev_bytes));
    CK(launch_stable_group(h->s_u32b.p, n, h->nlist, h->s_u32c.p, h->s_perm.p, h->s_group.p, st));
    uint32_t kept = 0;
    CK(cudaMemcpyAsync(&kept, h->s_u32c.p + h->nlist, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (kept) {
        CK(h->pend_rows.ensure((h->pend_n + kept) * D, h->pend_n * D, st, &h->dev_bytes));
        CK(h->pend_ids.ensure(h->pend_n + kept, h->pend_n, st, &h->dev_bytes));
        CK(h->pend_list.ensure(h->pend_n + kept, h->pend_n, st, &h->dev_bytes));
        CK(launch_gather_rows(d_x, n, nullptr, h->s_perm.p, kept, D, h->pend_rows.p + h->pend_n * D, st));
        CK(launch_gather_u32(d_ids, n, nullptr, h->s_perm.p, kept, h->pend_ids.p + h->pend_n, st));
        CK(launch_gather_u32(h->s_u32b.p, n, nullptr, h->s_perm.p, kept, h->pend_list.p + h->pend_n, st));
        CK(cudaStreamSynchronize(st));
        h->pend_n += kept;
    }
    if (kept_out) *kept_out = kept;
    return FVDB_OK;
}

int flat_add_device_impl(fvdb_index* h, const float* d_x, const uint32_t* d_ids, uint64_t n) {
    if (n == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    RET(check_nan_device(h, d_x, n * D, st));
    if (h->flat_n + n >= 0xFFFFFFF0ull) return h->fail(FVDB_ERR_INVALID_ARG, "flat tier exceeds u32 rows");
    CK(h->flat_rows.ensure((h->flat_n + n) * D, h->flat_n * D, st, &h->dev_bytes));
    CK(h->flat_ids.ensure(h->flat_n + n, h->flat_n, st, &h->dev_bytes));
    CK(cudaMemcpyAsync(h->flat_rows.p + h->flat_n * D, d_x, n * D * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->flat_ids.p + h->flat_n, d_ids, n * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    h->flat_n += n;
    h->scratch.tc.flat_dirty = true;
    return FVDB_OK;
}

// host-side duplicate screen + presence update (HybridIndex::insert dup check, src/hybrid/core.rs:368;
// InvertedList::insert, src/ivf/core.rs:128-134)
int track_insert(fvdb_index* h, const uint32_t* ids, uint64_t n, uint8_t tier) {
    if (!h->track_ids) return FVDB_OK;
    uint32_t mx = 0;
    for (uint64_t i = 0; i < n; ++i) {
        if (ids[i] == ID_NONE) return h->fail(FVDB_ERR_INVALID_ARG, "row id 0xFFFFFFFF is reserved");
        mx = std::max(mx, ids[i]);
    }
    if (h->id_state.size() <= mx) h->id_state.resize((size_t)mx + 1, 0);
    for (uint64_t i = 0; i < n; ++i) {
        if (h->id_state[ids[i]] & 3) {
            // roll back what this call marked
            for (uint64_t j = 0; j < i; ++j) h->id_state[ids[j]] = 0;
            return h->fail(FVDB_ERR_DUPLICATE, "Vector with row id " + std::to_string(ids[i]) + " already exists");
        }
        h->id_state[ids[i]] = tier;
    }
    return FVDB_OK;
}

void clear_lists(fvdb_index* h) {
    if (h->track_ids)
        for (auto& s : h->id_state) if ((s & 3) == 2) { if (s & 0x80) h->deleted_count--; s = 0; }
    h->ivf_n = 0;
    h->pend_n = 0;
    mark_arena_dirty(h);
}

// compute_error, src/ivf/core.rs:419-429: f32 left fold of dist*dist, then / n.  (The library is built with
// -ffp-contract=off and without fast-math: the compiler neither fuses nor re-associates this loop.)
float host_mean_sq(const float* dist, size_t n) {
    float total = 0.0f;
    for (size_t i = 0; i < n; ++i) {
        const float sq = dist[i] * dist[i];
        total = total + sq;
    }
    return total / (float)n;
}

int compute_error_device(fvdb_index* h, const float* d_data, uint64_t n, const uint32_t* d_assign,
                         float* out) {
    cudaStream_t st = h->stream;
    CK(h->s_f32a.ensure(n, 0, st, &h->dev_bytes));
    CK(launch_rowwise_dist(d_data, n, h->dim, h->centroids.p, d_assign, h->s_f32a.p, st));
    // the per-row distances come back into the handle's page-locked buffer and are folded where they land
    CK(h->ensure_pin(n * sizeof(float)));
    CK(cudaMemcpyAsync(h->pin, h->s_f32a.p, n * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *out = host_mean_sq(static_cast<const float*>(h->pin), n);
    return FVDB_OK;
}

// The k-means proper.  Runs on h->centroids / h->nlist (the assignment kernels read them there); the
// caller (train_device_impl) has moved the previous centroid table aside and puts it back if this fails.
int train_body(fvdb_index* h, const float* d_data, uint64_t n, uint32_t nlist, uint32_t max_iterations,
               const float* d_init, uint64_t seed, fvdb_train_result* out) {
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    CK(h->centroids.ensure((size_t)nlist * D, 0, st, &h->dev_bytes));
    h->nlist = nlist;
    h->trained = false;
    mark_centroids_dirty(h); ++h->centroids_version;
    if (d_init) {
        CK(cudaMemcpyAsync(h->centroids.p, d_init, (size_t)nlist * D * 4, cudaMemcpyDeviceToDevice, st));
    } else {
        // k-means++ (src/ivf/core.rs:336-371) on the reference's own random stream (StdRng08 above).
        // The distances are computed on the device in the reference's operation order (one launch per
        // new centroid; the minimum over all chosen centroids :346-354 is kept as a running minimum,
        // which is exact).  The pick itself is a SEQUENTIAL f32 prefix sum over the points (:357-367) —
        // a parallel scan would move low bits and with them the picked index — so it runs on the host:
        // one 4 n-byte read-back and two passes over n floats per centroid.
        StdRng08 rng(seed);
        DevBuf<uint32_t> zeros;                     // every point "assigned" to the newest centroid
        CK(zeros.ensure(n, 0, st, nullptr, true));
        CK(cudaMemsetAsync(zeros.p, 0, n * 4, st));
        CK(h->s_f32a.ensure(n, 0, st, &h->dev_bytes));
        std::vector<float> mind(n, INFINITY), dist(n);
        const uint64_t first = rng.gen_range(n);
        CK(cudaMemcpyAsync(h->centroids.p, d_data + first * D, (size_t)D * 4, cudaMemcpyDeviceToDevice, st));
        uint32_t count = 1;
        for (uint32_t i = 1; i < nlist; ++i) {
            CK(launch_rowwise_dist(d_data, n, D, h->centroids.p + (size_t)(count - 1) * D, zeros.p, h->s_f32a.p, st));
            RET(d2h(h, dist.data(), h->s_f32a.p, n * 4));
            volatile float total = 0.0f;            // left folds in f32, as `.sum::<f32>()` / `+=`
            for (uint64_t j = 0; j < n; ++j) {
                const float m = mind[j] < dist[j] ? mind[j] : dist[j];
                mind[j] = m;
                total = total + m * m;
            }
            const float threshold = rng.gen_f32() * total;
            volatile float cumulative = 0.0f;
            for (uint64_t j = 0; j < n; ++j) {
                cumulative = cumulative + mind[j] * mind[j];
                if (cumulative >= threshold) {
                    CK(cudaMemcpyAsync(h->centroids.p + (size_t)count * D, d_data + j * D, (size_t)D * 4,
                                       cudaMemcpyDeviceToDevice, st));
                    ++count;
                    break;
                }
            }
        }
        CK(cudaStreamSynchronize(st));
        // f32 rounding can leave the cumulative sum below the threshold: the reference then ends up with
        // fewer than n_clusters centroids and indexes out of range later (SURVEY App. A.10) — an error here
        if (count < nlist)
            return h->fail(FVDB_ERR_INVALID_CONFIG, "k-means++ produced " + std::to_string(count) + " of " +
                           std::to_string(nlist) + " centroids (the cumulative f32 sum never reached the threshold)");
    }

    // Lloyd loop (src/ivf/core.rs:279-322)
    DevBuf<uint32_t> assign;
    CK(assign.ensure(n, 0, st, nullptr, true));
    CK(cudaMemsetAsync(assign.p, 0, n * 4, st));  // vec![ClusterId(0); n]
    CK(h->scratch.misc.ensure(64, 0, st, &h->dev_bytes));
    uint32_t* d_changed = h->scratch.misc.p + 4;
    float prev_error = INFINITY;
    float initial_error = 0.f;
    RET(compute_error_device(h, d_data, n, assign.p, &initial_error));
    bool converged = false;
    uint32_t iterations = 0;
    for (uint32_t iter = 0; iter < max_iterations; ++iter) {
        iterations = iter + 1;
        CK(cudaMemsetAsync(d_changed, 0, 4, st));
        RET(assign_device(h, d_data, n, assign.p, nullptr, assign.p, d_changed, st));
        uint32_t changed = 0;
        CK(cudaMemcpyAsync(&changed, d_changed, 4, cudaMemcpyDeviceToHost, st));
        // update step: order-faithful per-cluster sums
        CK(h->s_perm.ensure(n, 0, st, &h->dev_bytes));
        CK(h->s_group.ensure(stable_group_scratch_bytes(n, nlist), 0, st, &h->dev_bytes));
        CK(h->s_u32c.ensure(nlist + 2, 0, st, &h->dev_bytes));
        CK(launch_stable_group(assign.p, n, nlist, h->s_u32c.p, h->s_perm.p, h->s_group.p, st));
        CK(launch_centroid_update(d_data, D, h->s_u32c.p, h->s_perm.p, nlist, h->centroids.p, st));
        CK(cudaStreamSynchronize(st));
        mark_centroids_dirty(h); ++h->centroids_version;
        if (iterations >= max_iterations) break;
        float current_error = 0.f;
        RET(compute_error_device(h, d_data, n, assign.p, &current_error));
        volatile float diff = std::fabs(prev_error - current_error);
        const float error_change = diff / prev_error;
        if (!changed || error_change < 1e-4f) {
            converged = true;
            if (max_iterations == 10 && n < 20) {  // src/ivf/core.rs:313-317
                prev_error = current_error;
                continue;
            }
            break;
        }
        prev_error = current_error;
    }
    float final_error = 0.f;
    RET(compute_error_device(h, d_data, n, assign.p, &final_error));
    CK(h->list_off.ensure(nlist + 2, 0, st, &h->dev_bytes));
    CK(cudaMemsetAsync(h->list_off.p, 0, (nlist + 2) * 4, st));
    CK(cudaStreamSynchronize(st));
    if (out) {
        out->iterations = iterations;
        out->converged = converged ? 1u : 0u;
        out->initial_error = initial_error;
        out->final_error = final_error;
    }
    return FVDB_OK;
}

// IVFIndex::train (src/ivf/core.rs:240-334).  Like the reference, every check comes before anything is
// touched (:242-262), and a training run that fails half-way (CUDA error, out of memory) leaves the
// index exactly as it was: the previous centroid table, nlist, trained flag and posting lists come back.
int train_device_impl(fvdb_index* h, const float* d_data, uint64_t n, uint32_t nlist,
                      uint32_t max_iterations, const float* d_init, uint64_t seed,
                      fvdb_train_result* out) {
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    if (nlist == 0 || max_iterations == 0) return h->fail(FVDB_ERR_INVALID_CONFIG, "Invalid IVFConfig");
    if (n == 0 || n < nlist)
        return h->fail(FVDB_ERR_INSUFFICIENT_TRAINING, "Insufficient training data: got " +
                       std::to_string(n) + ", need at least " + std::to_string(nlist));
    if (n >= 0xFFFFFFF0ull) return h->fail(FVDB_ERR_INVALID_ARG, "training set exceeds u32 rows");
    RET(check_nan_device(h, d_data, n * D, st));
    if (d_init) RET(check_nan_device(h, d_init, (size_t)nlist * D, st));
    DevBuf<float> old_centroids;
    old_centroids.swap(h->centroids);
    const uint32_t old_nlist = h->nlist;
    const bool old_trained = h->trained;
    const int r = train_body(h, d_data, n, nlist, max_iterations, d_init, seed, out);
    if (r != FVDB_OK) {
        h->dev_bytes -= h->centroids.cap * sizeof(float);
        h->centroids.swap(old_centroids);   // the failed run's table is freed with old_centroids
        h->nlist = old_nlist;
        h->trained = old_trained;
        mark_centroids_dirty(h); ++h->centroids_version;
        return r;
    }
    h->dev_bytes -= old_centroids.cap * sizeof(float);
    h->trained = true;
    clear_lists(h);   // src/ivf/core.rs:273-277
    return FVDB_OK;
}

// Exact IVF search of `nq` queries given their exact coarse ranking (src/ivf/core.rs:661-678):
// bucket (query, probe) pairs by list, scan every probed list once, merge per query.
int ivf_scan_exact(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t np,
                   const uint64_t* coarse, const uint64_t* tomb, const uint64_t* filt,
                   uint64_t filter_bits, uint64_t* out_keys, uint64_t* d_scanned, bool timed,
                   cudaStream_t st) {
    const uint32_t D = h->dim;
    const uint32_t tq = exact_scan_tq();
    const size_t n_pairs = (size_t)nq * np;
    uint32_t Ppad = np;
    if (np > 256) Ppad = (np + 255) / 256 * 256;
    CK(h->s_partial.ensure((size_t)nq * Ppad * k, 0, st, &h->dev_bytes));
    CK(cudaMemsetAsync(h->s_partial.p, 0xFF, (size_t)nq * Ppad * k * 8, st));
    // sparse batch (few queries per probed list): one warp per (query, list) pair instead of
    // 32-query tiles that would be mostly padding
    const bool sparse = n_pairs <= (size_t)4 * h->nlist && (size_t)4 * (D * 4 + k * 8) <= 200 * 1024;
    if (sparse) {
        if (timed) CK(cudaEventRecord(h->scratch.ev_s0, st));
        CK(launch_exact_pair_scan(coarse, nq, np, h->list_off.p, h->ivf_rows.p, h->ivf_ids.p, d_q, D, Ppad, k, tomb,
                                  h->tomb_bits, filt, filter_bits, h->s_partial.p, st));
        if (timed) CK(cudaEventRecord(h->scratch.ev_s1, st));
        h->stats.last_launches += 1;
        if (d_scanned) CK(cudaMemsetAsync(d_scanned, 0, 8, st));
    } else {
    const size_t max_items = (size_t)h->nlist + (n_pairs + tq - 1) / tq + 1;
    CK(h->s_list_cnt.ensure(h->nlist + 1, 0, st, &h->dev_bytes));
    CK(h->s_pair_off.ensure(h->nlist + 2, 0, st, &h->dev_bytes));
    CK(h->s_cursor.ensure(h->nlist + 1, 0, st, &h->dev_bytes));
    CK(h->s_pair_q.ensure(n_pairs, 0, st, &h->dev_bytes));
    CK(h->s_pair_slot.ensure(n_pairs, 0, st, &h->dev_bytes));
    CK(h->s_items.ensure(max_items, 0, st, &h->dev_bytes));
    uint32_t* d_n_items = h->scratch.misc.p + 6;
    CK(launch_probe_bucketing(coarse, nq, np, h->list_off.p, h->nlist, tq, h->s_list_cnt.p,
                              h->s_pair_off.p, h->s_cursor.p, h->s_pair_q.p, h->s_pair_slot.p,
                              h->s_items.p, d_n_items, d_scanned, st));
    h->stats.last_launches += 3;
    ExactScanArgs a{};
    a.X = h->ivf_rows.p; a.ids = h->ivf_ids.p; a.Q = d_q; a.D = D;
    a.items = h->s_items.p; a.item_count = d_n_items; a.n_items = 0;
    a.pair_q = h->s_pair_q.p; a.pair_slot = h->s_pair_slot.p;
    a.P = Ppad; a.k = k;
    a.tomb = tomb; a.tomb_bits = h->tomb_bits; a.filt = filt; a.filt_bits = filter_bits;
    a.partial = h->s_partial.p;
    if (timed) CK(cudaEventRecord(h->scratch.ev_s0, st));
    CK(launch_exact_scan(a, (uint32_t)max_items, st));
    if (timed) CK(cudaEventRecord(h->scratch.ev_s1, st));
    h->stats.last_launches += 1;
    }
    // sort + truncate(k) (src/ivf/core.rs:677-678)
    if (Ppad > 256) {
        CK(h->s_partial2.ensure((size_t)nq * (Ppad / 256) * k, 0, st, &h->dev_bytes));
        CK(launch_merge_partials(h->s_partial.p, nq * (Ppad / 256), 256, k, h->s_partial2.p, st));
        CK(launch_merge_partials(h->s_partial2.p, nq, Ppad / 256, k, out_keys, st));
        h->stats.last_launches += 2;
    } else {
        CK(launch_merge_partials(h->s_partial.p, nq, Ppad, k, out_keys, st));
        h->stats.last_launches += 1;
    }
    return FVDB_OK;
}

// The tensor-core IVF scan serves k <= 16 and up to 256 probed lists (np: nprobe clamped to nlist).
bool tc_ivf_scan(uint32_t scan_mode, uint32_t D, uint32_t k, uint32_t np) {
    return scan_mode == FVDB_SCAN_TC && tc_supported(D) && k <= TC_MAX_K && np <= TC_MAX_NPROBE;
}
// The tensor-core coarse step serves D <= 384 and up to 112 probed lists; else the exact CUDA-core scan ranks them.
bool tc_coarse_step(uint32_t scan_mode, uint32_t D, uint32_t np) {
    return scan_mode == FVDB_SCAN_TC && tc_supported(D) && D <= 384 && np <= TC_MAX_NPROBE_COARSE;
}

// A page-locked record of at least `words` u32: a recycled one from the pool, else a new one.
cudaError_t take_record(fvdb_index* h, size_t words, fvdb_index::Record* rec) {
    for (size_t i = 0; i < h->pending_pool.size(); ++i)
        if (h->pending_pool[i].second >= words) {
            *rec = h->pending_pool[i];
            h->pending_pool.erase(h->pending_pool.begin() + i);
            return cudaSuccess;
        }
    *rec = {nullptr, words};
    return cudaHostAlloc((void**)&rec->first, words * 4, cudaHostAllocDefault);
}

// Coarse ranking only (src/ivf/core.rs:646-656) for nq queries: keys [nq][np] (distance bits << 32 |
// list id), ascending, ties to the lower list id.  Tensor cores + exact verify when possible;
// queries whose proof fails are re-ranked by the exact kernel.
int coarse_device_impl(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t np, uint64_t* d_out_keys,
                       cudaStream_t st, bool deferred = false) {
    const uint32_t D = h->dim;
    if (nq == 0) return FVDB_OK;
    BatchScratch& b = h->scratch;
    CK(b.misc.ensure(64, 0, st, &h->dev_bytes));
    int* d_nan = reinterpret_cast<int*>(b.misc.p);
    uint32_t* d_fb_count = b.misc.p + 10;
    CK(cudaMemsetAsync(b.misc.p, 0, 64, st));
    CK(launch_nan_check(d_q, (size_t)nq * D, d_nan, st));
    const bool tc = tc_coarse_step(h->scan_mode, D, np);
    if (tc) {
        CK(b.fb_idx.ensure((size_t)2 * nq, 0, st, &h->dev_bytes));
        TcSearchArgs ta{};
        ta.nlist = h->nlist; ta.Q = d_q; ta.nq = nq; ta.D = D; ta.k = 1; ta.nprobe = np;
        ta.centroids = h->centroids.p; ta.coarse_keys = nullptr; ta.coarse_out = d_out_keys; ta.coarse_only = true;
        ta.d_fallback_count = d_fb_count; ta.d_fallback_idx = b.fb_idx.p;
        ta.sm_count = h->sm_count;
        uint32_t launches = 0;
        int r = tc_ivf_search(b.tc, ta, st, &h->dev_bytes, &launches, &h->err);
        if (r != FVDB_OK) return r;
    } else {
        RET(scan_all_exact(h, h->centroids.p, nullptr, h->nlist, d_q, nq, np, nullptr, 0, nullptr, 0, d_out_keys, st));
    }
    if (deferred) {
        // stream-ordered: the NaN flag and the number of queries whose tensor-core proof failed go to a
        // page-locked record that fvdb_search_device_finish looks at (it reports them; the caller re-runs
        // the batch through the synchronous entry, which repairs them)
        fvdb_index::Record rec;
        CK(take_record(h, 16, &rec));
        h->pending_coarse.push_back(rec);
        CK(cudaMemcpyAsync(rec.first, b.misc.p, 64, cudaMemcpyDeviceToHost, st));
        return FVDB_OK;
    }
    uint32_t host_misc[16] = {0};
    CK(cudaMemcpyAsync(host_misc, b.misc.p, sizeof(host_misc), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (host_misc[0])
        return h->fail(FVDB_ERR_NAN, "NaN in query (the reference panics on partial_cmp().unwrap())");
    const uint32_t n_fb = tc ? std::min(host_misc[10], 2 * nq) : 0;
    if (n_fb) {
        CK(h->s_fb_q.ensure((size_t)n_fb * D, 0, st, &h->dev_bytes));
        CK(h->s_fb_coarse.ensure((size_t)n_fb * np, 0, st, &h->dev_bytes));
        CK(launch_gather_rows(d_q, nq, nullptr, b.fb_idx.p, n_fb, D, h->s_fb_q.p, st));
        RET(scan_all_exact(h, h->centroids.p, nullptr, h->nlist, h->s_fb_q.p, n_fb, np, nullptr, 0, nullptr, 0,
                           h->s_fb_coarse.p, st));
        CK(launch_scatter_keys(h->s_fb_coarse.p, b.fb_idx.p, n_fb, np, d_out_keys, st));
        CK(cudaStreamSynchronize(st));
    }
    return FVDB_OK;
}

cudaError_t copy_out(const HostOut* ho, const uint32_t* d_ids, const float* d_dist, const uint32_t* d_cnt,
                     cudaStream_t st) {
    cudaError_t e = cudaMemcpyAsync(ho->ids, d_ids, ho->ob, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ho->dist, d_dist, ho->ob, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ho->cnt, d_cnt, ho->cb, cudaMemcpyDeviceToHost, st);
    return e;
}
// page-locked host memory (fvdb_host_alloc, cudaHostAlloc, cudaHostRegister): DMA without staging
bool is_pinned_host(const void* p) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

// The optional arguments of search_device_impl.
struct SearchOpts {
    const uint64_t* ext_coarse = nullptr;   // the batch's coarse keys [nq][nprobe], ranked by the caller
    const HostOut* ho = nullptr;            // pinned host destinations of the results
    bool deferred = false;                  // stream-ordered: finish_pending checks the batch (and repairs it)
    cudaEvent_t wait_first = nullptr;       // the batch starts behind this event
    bool split = false;                     // fvdb_search_device_tiers: each tier to its own part of a packed chunk
    bool exact = false;                     // the exact path whatever the scan mode (a proof-failure repair)
};

int repair_rows(fvdb_index* h, const fvdb_index::Pending& pb, const std::vector<uint32_t>& rows, cudaStream_t st);

// The figures of a finished batch into h->stats; `misc` is its counter words, read back.  Call it before anything
// records the batch's events again.
void set_batch_stats(fvdb_index* h, const fvdb_index::Pending& pb, const uint32_t* misc) {
    uint64_t scanned = 0;
    std::memcpy(&scanned, misc + 2, 8);
    const uint64_t rows = scanned + (pb.use_flat ? h->flat_n : 0);
    h->stats.last_nq = pb.nq;
    h->stats.last_scanned_rows = rows;
    h->stats.last_algorithmic_bytes = rows * h->dim * 4ull + (uint64_t)pb.nq * h->dim * 4ull + (uint64_t)pb.nq * pb.k * 8ull +
                                      (pb.use_ivf ? (uint64_t)h->nlist * h->dim * 4ull : 0ull) + (uint64_t)pb.n_bitmaps * (rows / 8);
    auto elapsed = [](cudaEvent_t a, cudaEvent_t b) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) { cudaGetLastError(); ms = 0.f; }
        return ms;
    };
    h->stats.last_device_ms = elapsed(pb.scratch->ev_a, pb.scratch->ev_b);
    h->stats.last_scan_ms = pb.use_ivf ? elapsed(pb.scratch->ev_s0, pb.scratch->ev_s1) : 0.f;   // the IVF scan is timed
}

// The queries of a batch to re-run: both tiers' proof-failure lists as one ascending list without repeats.
std::vector<uint32_t> failed_queries(const uint32_t* ivf, uint32_t n_ivf, const uint32_t* flat, uint32_t n_flat) {
    std::vector<uint32_t> q(ivf, ivf + n_ivf);
    q.insert(q.end(), flat, flat + n_flat);
    std::sort(q.begin(), q.end());
    q.erase(std::unique(q.begin(), q.end()), q.end());
    return q;
}

int search_device_impl(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                       uint32_t tiers, const uint64_t* d_filter, uint64_t filter_bits,
                       uint32_t* d_out_ids, float* d_out_dist, uint32_t* d_out_count,
                       cudaStream_t st, const SearchOpts& o = {}) {
    if (k == 0) return h->fail(FVDB_ERR_INVALID_ARG, "k must be >= 1");
    if (k > h->k_max) return h->fail(FVDB_ERR_K_TOO_LARGE, "k exceeds k_max given at fvdb_create");
    h->stats.last_nq = nq;
    h->stats.last_fallback_queries = 0;
    h->stats.last_scanned_rows = 0;
    h->stats.last_algorithmic_bytes = 0;
    h->stats.last_launches = 0;
    h->stats.last_device_ms = 0.f;
    h->stats.last_scan_ms = 0.f;
    if (nq == 0) return FVDB_OK;
    RET(seal(h));
    const uint32_t D = h->dim;
    const uint32_t mode = o.exact ? FVDB_SCAN_EXACT : h->scan_mode;
    // the IVF tier exists for L2 only (fvdb_ivf_* reject a similarity handle), so use_ivf implies L2
    const bool use_ivf = (tiers & FVDB_TIER_HISTORICAL) && h->trained && h->ivf_n > 0 && nprobe > 0;
    const bool use_flat = (tiers & FVDB_TIER_RECENT) && h->flat_n > 0;
    const uint64_t* tomb = h->deleted_count ? h->tomb.p : nullptr;
    const uint64_t* filt = d_filter;
    const uint32_t np = use_ivf ? std::min(nprobe, h->nlist) : 0;
    if (np > 512) return h->fail(FVDB_ERR_INVALID_ARG, "nprobe > 512 is not supported");
    // the tensor-core IVF path looks at every query element anyway (query norms): it raises the flag
    const bool tc_ivf = use_ivf && tc_ivf_scan(mode, D, k, np);
    // coarse step: all centroid distances, nearest np lists (src/ivf/core.rs:646-656); exact CUDA-core
    // scan, or tensor-core distances + exact verify (or handed in: the multi-GPU driver ranks a slice of
    // the batch per GPU and all-gathers)
    const bool tc_coarse = tc_ivf && !o.ext_coarse && tc_coarse_step(mode, D, np);

    // Pipeline slot (stream-ordered entries, IVF tier alone on the tensor-core path): this batch runs on
    // the slot's stream with the slot's scratch; `st` (the caller's stream) is only what its inputs are
    // ordered after.  Everything else runs on `st` with the handle's own scratch, after the slots drained.
    int slot = -1;
    if (o.deferred && h->pipeline && tc_ivf && (tc_coarse || o.ext_coarse) && !use_flat) {
        slot = (int)(h->slot_next++ % fvdb_index::N_SLOTS);
        fvdb_index::Slot& sl = h->slots[slot];
        if (!sl.stream) {
            CK(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
            CK(sl.b.create_events());
            CK(cudaEventCreateWithFlags(&sl.ev_in, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&sl.ev_scan_end, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
        }
        CK(cudaEventRecord(sl.ev_in, st));
        CK(cudaStreamWaitEvent(sl.stream, sl.ev_in, 0));
        if (o.wait_first) CK(cudaStreamWaitEvent(sl.stream, o.wait_first, 0));
        st = sl.stream;
        sl.busy = true;
    } else {
        quiesce_slots(h);
        if (o.wait_first) CK(cudaStreamWaitEvent(st, o.wait_first, 0));
    }
    fvdb_index::Slot* const sl = slot >= 0 ? &h->slots[slot] : nullptr;
    BatchScratch& b = sl ? sl->b : h->scratch;

    CK(cudaEventRecord(b.ev_a, st));
    CK(b.misc.ensure(64, 0, st, &h->dev_bytes));
    int* d_nan = reinterpret_cast<int*>(b.misc.p);
    uint64_t* d_scanned = reinterpret_cast<uint64_t*>(b.misc.p + 2);
    CK(cudaMemsetAsync(b.misc.p, 0, 64, st));
    if (!tc_ivf) {
        CK(launch_nan_check(d_q, (size_t)nq * D, d_nan, st));
        h->stats.last_launches += 1;
    }

    uint64_t* ivf_keys = nullptr;
    uint64_t* flat_keys = nullptr;
    // split (fvdb_search_device_tiers): the result arrays are the recent-tier part of a packed chunk
    // [ids nq*k | dist nq*k | count nq]; the IVF tier's part follows it, one part length further on
    const size_t part_words = (size_t)2 * nq * k + nq;
    uint32_t* const ivf_out_ids = o.split ? d_out_ids + part_words : nullptr;
    float* const ivf_out_dist = o.split ? d_out_dist + part_words : nullptr;
    uint32_t* const ivf_out_count = o.split ? d_out_count + part_words : nullptr;
    bool fused_finalize = false;

    if (use_ivf) {
        CK(b.ivf_keys.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
        ivf_keys = b.ivf_keys.p;
        const uint64_t* coarse_in = o.ext_coarse;
        if (!o.ext_coarse) {
            CK(b.coarse.ensure((size_t)nq * np, 0, st, &h->dev_bytes));
            coarse_in = b.coarse.p;
            if (!tc_coarse)
                RET(scan_all_exact(h, h->centroids.p, nullptr, h->nlist, d_q, nq, np, nullptr, 0, nullptr, 0,
                                   b.coarse.p, st));
        }
        if (tc_ivf) {
            CK(b.fb_idx.ensure((size_t)2 * nq, 0, st, &h->dev_bytes));
            TcSearchArgs ta{};
            ta.rows = h->ivf_rows.p; ta.ids = h->ivf_ids.p; ta.n_rows = h->ivf_n;
            ta.list_off = h->list_off.p; ta.nlist = h->nlist;
            ta.Q = d_q; ta.nq = nq; ta.D = D; ta.k = k; ta.nprobe = np;
            ta.centroids = h->centroids.p;
            ta.coarse_keys = tc_coarse ? nullptr : coarse_in;
            ta.coarse_out = nullptr;
            ta.tomb = tomb; ta.tomb_bits = h->tomb_bits; ta.filt = filt; ta.filt_bits = filter_bits;
            ta.out_keys = ivf_keys;
            ta.d_scanned_rows = d_scanned;
            ta.d_fallback_count = b.misc.p + 10; ta.d_fallback_idx = b.fb_idx.p;
            ta.ev_scan0 = b.ev_s0; ta.ev_scan1 = b.ev_s1;
            ta.sm_count = h->sm_count;
            ta.xmax_floor_sq = h->proof_xmax_sq;
            ta.scan_sms = sl ? h->scan_sms : 0;   // only pipelined batches have neighbours to leave room for
            ta.d_nan = d_nan;
            if (!use_flat && !o.split) {   // the only tier: the re-rank writes the result arrays itself
                ta.fin_ids = d_out_ids; ta.fin_dist = d_out_dist; ta.fin_count = d_out_count;
                fused_finalize = true;
            }
            if (h->bounds_armed_nq == nq && h->bounds) {   // fvdb_bounds_begin_batch was called for this batch
                ta.thr_ext = h->bounds + (size_t)h->bounds_parity * h->bounds_cap;
                ta.n_peers = (uint32_t)std::min<size_t>(h->peer_bounds.size(), TC_MAX_PEERS);
                for (uint32_t r = 0; r < ta.n_peers; ++r)
                    ta.thr_peers[r] = h->peer_bounds[r] + (size_t)h->bounds_parity * h->bounds_cap;
            }
            h->bounds_armed_nq = 0;
            uint32_t launches = 0;
            if (sl) {
                // one scan at a time: this one waits for the scan of the batch enqueued before it
                ta.wait_before_scan = h->prev_scan_end;
                ta.record_after_scan = sl->ev_scan_end;
            }
            int r = tc_ivf_search(b.tc, ta, st, &h->dev_bytes, &launches, &h->err);
            if (sl && r == FVDB_OK) h->prev_scan_end = sl->ev_scan_end;
            if (r != FVDB_OK) return r;
            h->stats.last_launches += launches;
        } else {
            RET(ivf_scan_exact(h, d_q, nq, k, np, coarse_in, tomb, filt, filter_bits, ivf_keys,
                               d_scanned, true, st));
        }
    }
    bool flat_tc = false;
    if (use_flat) {
        CK(h->s_flat_keys.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
        flat_keys = h->s_flat_keys.p;
        // recent tier: exhaustive scan instead of the HNSW walk (src/hnsw/core.rs:398-467); on the
        // tensor cores when the batch is large enough to amortise the item set-up
        flat_tc = mode == FVDB_SCAN_TC && tc_supported(D) && k <= TC_MAX_K &&
                  (uint64_t)h->flat_n * nq >= (4ull << 20) && (h->metric == FVDB_METRIC_L2 || D <= 384);
        if (flat_tc) {
            CK(h->s_fb_idx_flat.ensure((size_t)2 * nq, 0, st, &h->dev_bytes));
            TcFlatArgs fa{};
            fa.rows = h->flat_rows.p; fa.ids = h->flat_ids.p; fa.n_rows = h->flat_n;
            fa.Q = d_q; fa.nq = nq; fa.D = D; fa.k = k;
            fa.tomb = tomb; fa.tomb_bits = h->tomb_bits; fa.filt = filt; fa.filt_bits = filter_bits;
            fa.out_keys = flat_keys;
            fa.d_fallback_count = b.misc.p + 11; fa.d_fallback_idx = h->s_fb_idx_flat.p;
            fa.sm_count = h->sm_count;
            fa.metric = h->metric;
            uint32_t launches = 0;
            int r = tc_flat_search(h->scratch.tc, fa, st, &h->dev_bytes, &launches, &h->err);
            if (r != FVDB_OK) return r;
            h->stats.last_launches += launches;
        } else {
            RET(scan_all_exact(h, h->flat_rows.p, h->flat_ids.p, h->flat_n, d_q, nq, k, tomb, h->tomb_bits,
                               filt, filter_bits, flat_keys, st, h->metric));
        }
    }
    if (!fused_finalize) {
        CK(launch_finalize(flat_keys, ivf_keys, nq, k, d_out_ids, d_out_dist, d_out_count, st, h->metric,
                           ivf_out_ids, ivf_out_dist, ivf_out_count));
        h->stats.last_launches += 1;
    }
    CK(cudaEventRecord(b.ev_b, st));
    if (o.ho) CK(copy_out(o.ho, d_out_ids, d_out_dist, d_out_count, st));

    fvdb_index::Pending pb{d_q, nq, k, nprobe, tiers, d_filter, filter_bits, d_out_ids, d_out_dist, d_out_count,
                           o.ho ? *o.ho : HostOut{}, o.split, tc_ivf, flat_tc, use_ivf, use_flat,
                           (tomb ? 1u : 0u) + (filt ? 1u : 0u), slot, &b, {nullptr, 0}};
    if (o.deferred) {
        // stream-ordered variant: the counters and the fallback lists are copied to a page-locked
        // record in stream order; fvdb_search_device_finish looks at them after ONE synchronisation
        // for any number of batches (no GPU idle time between consecutive batches)
        CK(take_record(h, 16 + (size_t)4 * nq, &pb.rec));
        uint32_t* rec = pb.rec.first;
        CK(cudaMemcpyAsync(rec, b.misc.p, 64, cudaMemcpyDeviceToHost, st));
        if (tc_ivf) CK(cudaMemcpyAsync(rec + 16, b.fb_idx.p, (size_t)2 * nq * 4, cudaMemcpyDeviceToHost, st));
        if (flat_tc) CK(cudaMemcpyAsync(rec + 16 + 2 * nq, h->s_fb_idx_flat.p, (size_t)2 * nq * 4, cudaMemcpyDeviceToHost, st));
        if (sl) CK(cudaEventRecord(sl->ev_done, st));
        h->pending.push_back(pb);
        return FVDB_OK;
    }
    // one synchronisation point per batch: NaN flag + counters
    uint32_t host_misc[16] = {0};
    CK(cudaMemcpyAsync(host_misc, b.misc.p, sizeof(host_misc), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (host_misc[0])
        return h->fail(FVDB_ERR_NAN, "NaN in query (the reference panics on partial_cmp().unwrap())");
    set_batch_stats(h, pb, host_misc);
    const uint32_t n_ivf = tc_ivf ? std::min(host_misc[10], 2 * nq) : 0;
    const uint32_t n_flat = flat_tc ? std::min(host_misc[11], 2 * nq) : 0;
    if (n_ivf || n_flat) {
        // the tensor-core proof failed for some queries (rare: only near-duplicate-heavy neighbourhoods):
        // their lists come back, and the repair re-runs them on the exact path
        std::vector<uint32_t> lists(n_ivf + n_flat);
        if (n_ivf) CK(cudaMemcpyAsync(lists.data(), b.fb_idx.p, (size_t)n_ivf * 4, cudaMemcpyDeviceToHost, st));
        if (n_flat)
            CK(cudaMemcpyAsync(lists.data() + n_ivf, h->s_fb_idx_flat.p, (size_t)n_flat * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const std::vector<uint32_t> rows = failed_queries(lists.data(), n_ivf, lists.data() + n_ivf, n_flat);
        RET(repair_rows(h, pb, rows, st));
        h->stats.last_fallback_queries = (uint32_t)rows.size();
    }
    return FVDB_OK;
}

// Proof failures of a batch: the queries `rows` (ascending, distinct) are searched again on the exact path,
// every tier the batch asked for (a tier whose proof held returns the same bits there), and their result rows
// are replaced: in both parts of a split batch, and in the pinned host outputs when the batch has them.
// h->stats keep describing the batch; last_launches adds the repair's launches.
int repair_rows(fvdb_index* h, const fvdb_index::Pending& pb, const std::vector<uint32_t>& rows, cudaStream_t st) {
    const uint32_t m = (uint32_t)rows.size(), k = pb.k;
    // the row list, the gathered queries and the re-run results sit in buffers the nested search does not use
    CK(h->s_fb_rows.ensure(m, 0, st, &h->dev_bytes));
    CK(h->s_fb_q.ensure((size_t)m * h->dim, 0, st, &h->dev_bytes));
    CK(h->s_fb_keys.ensure((size_t)m * k * 2 + m, 0, st, &h->dev_bytes));   // ids | dist | counts, two parts
    CK(cudaMemcpyAsync(h->s_fb_rows.p, rows.data(), (size_t)m * 4, cudaMemcpyHostToDevice, st));
    CK(launch_gather_rows(pb.d_q, pb.nq, nullptr, h->s_fb_rows.p, m, h->dim, h->s_fb_q.p, st));
    uint32_t* t_ids = reinterpret_cast<uint32_t*>(h->s_fb_keys.p);
    float* t_dist = reinterpret_cast<float*>(t_ids + (size_t)m * k);
    uint32_t* t_cnt = t_ids + (size_t)2 * m * k;
    const fvdb_stats batch = h->stats;
    SearchOpts o; o.split = pb.split; o.exact = true;
    RET(search_device_impl(h, h->s_fb_q.p, m, k, pb.nprobe, pb.tiers, pb.d_filter, pb.filter_bits, t_ids, t_dist,
                           t_cnt, st, o));
    uint32_t launches = h->stats.last_launches + 2;   // and the gather and the scatter
    CK(launch_scatter_result_rows(t_ids, t_dist, t_cnt, h->s_fb_rows.p, m, k, pb.d_out_ids, pb.d_out_dist,
                                  pb.d_out_count, st));
    if (pb.split) {   // the IVF tier's part follows the recent tier's, one part length further on
        const size_t tp = (size_t)2 * m * k + m, bp = (size_t)2 * pb.nq * k + pb.nq;
        CK(launch_scatter_result_rows(t_ids + tp, t_dist + tp, t_cnt + tp, h->s_fb_rows.p, m, k, pb.d_out_ids + bp,
                                      pb.d_out_dist + bp, pb.d_out_count + bp, st));
        launches += 1;
    }
    if (pb.ho.ids) CK(copy_out(&pb.ho, pb.d_out_ids, pb.d_out_dist, pb.d_out_count, st));
    CK(cudaStreamSynchronize(st));
    h->stats = batch;
    h->stats.last_launches += launches;
    return FVDB_OK;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int fvdb_abi_version(void) { return FVDB_ABI_VERSION; }

const char* fvdb_last_error(const fvdb_index* h) {
    if (h) return h->err.c_str();
    std::lock_guard<std::mutex> g(g_err_mu);
    return g_create_err.c_str();
}

int fvdb_create(int device, uint32_t dim, int metric, uint32_t k_max, fvdb_index** out) {
    auto fail = [&](int code, const std::string& m) {
        std::lock_guard<std::mutex> g(g_err_mu);
        g_create_err = m;
        return code;
    };
    if (!out) return fail(FVDB_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (dim == 0) return fail(FVDB_ERR_INVALID_CONFIG, "dim must be > 0");
    if (metric != FVDB_METRIC_L2 && metric != FVDB_METRIC_COS && metric != FVDB_METRIC_DOT)
        return fail(FVDB_ERR_INVALID_CONFIG, "metric must be FVDB_METRIC_L2, FVDB_METRIC_COS or FVDB_METRIC_DOT");
    if (k_max == 0 || k_max > 512) return fail(FVDB_ERR_INVALID_CONFIG, "k_max must be in 1..512");
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(FVDB_ERR_NO_DEVICE, std::string("no CUDA device: ") +
                    (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                    " (libfvdb_b200 has no CPU fallback)");
    }
    if (device < 0 || device >= count) return fail(FVDB_ERR_NO_DEVICE, "device ordinal out of range");
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return fail(FVDB_ERR_NO_DEVICE, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail(FVDB_ERR_NO_DEVICE, std::string("device ") + prop.name +
                    " is not sm_100; libfvdb_b200 ships sm_100a code only");
    if (cudaSetDevice(device) != cudaSuccess) return fail(FVDB_ERR_NO_DEVICE, "cudaSetDevice failed");
    fvdb_index* h = new fvdb_index();
    h->device = device;
    h->dim = dim;
    h->metric = metric;
    h->k_max = k_max;
    h->sm_count = prop.multiProcessorCount;
    h->scan_mode = tc_supported(dim) ? FVDB_SCAN_TC : FVDB_SCAN_EXACT;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        h->scratch.create_events() != cudaSuccess) {
        delete h;
        return fail(FVDB_ERR_CUDA, "stream/event creation failed");
    }
    *out = h;
    return FVDB_OK;
}

void fvdb_destroy(fvdb_index* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto& sl : h->slots) {
        if (sl.stream) cudaStreamSynchronize(sl.stream);
        sl.b.release();
        for (cudaEvent_t e : {sl.ev_in, sl.ev_scan_end, sl.ev_done})
            if (e) cudaEventDestroy(e);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    h->scratch.release();
    if (h->pin) cudaFreeHost(h->pin);
    for (auto& pb : h->pending) cudaFreeHost(pb.rec.first);
    for (auto& pp : h->pending_pool) cudaFreeHost(pp.first);
    for (auto& pp : h->pending_coarse) cudaFreeHost(pp.first);
    for (auto& sl : h->host_slots) {
        if (sl.uploaded) cudaEventDestroy(sl.uploaded);
        if (sl.done) cudaEventDestroy(sl.done);
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (uint32_t* pb : h->peer_bounds) cudaIpcCloseMemHandle(pb);
    if (h->bounds) cudaFree(h->bounds);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

#define ENTER_PIPE(h)                                       \
    if (!(h)) return FVDB_ERR_INVALID_ARG;                  \
    std::lock_guard<std::mutex> guard__((h)->mu);           \
    (h)->err.clear();                                       \
    if (cudaSetDevice((h)->device) != cudaSuccess) return (h)->fail(FVDB_ERR_CUDA, "cudaSetDevice failed")
// every entry but the stream-ordered submits first lets the batches in the pipeline slots finish: nothing
// they read (arena, centroids, bitmaps) may move under them
#define ENTER(h)                                            \
    ENTER_PIPE(h);                                          \
    quiesce_slots(h)

int fvdb_set_option(fvdb_index* h, int option, uint64_t value) {
    ENTER(h);
    switch (option) {
        case FVDB_OPT_SCAN_MODE:
            if (value == FVDB_SCAN_TC && !tc_supported(h->dim))
                return h->fail(FVDB_ERR_INVALID_CONFIG, "tensor-core scan needs dim % 32 == 0 and dim <= 512");
            if (value > FVDB_SCAN_TC) return h->fail(FVDB_ERR_INVALID_ARG, "unknown scan mode");
            h->scan_mode = (uint32_t)value;
            return FVDB_OK;
        case FVDB_OPT_SHORTLIST:
            h->shortlist = (uint32_t)value;
            return FVDB_OK;
        case FVDB_OPT_KMEANS_TC:
            h->kmeans_tc = value ? 1u : 0u;
            return FVDB_OK;
        case FVDB_OPT_COALESCE:
            h->coalesce = value ? 1u : 0u;
            return FVDB_OK;
        case FVDB_OPT_SCAN_SMS:
            h->scan_sms = (uint32_t)value;
            return FVDB_OK;
        case FVDB_OPT_PIPELINE:
            h->pipeline = value ? 1u : 0u;
            return FVDB_OK;
        case FVDB_OPT_PROOF_XMAX: {
            const uint32_t b = (uint32_t)value;
            float f;
            std::memcpy(&f, &b, 4);
            if (!(f >= 0.f)) return h->fail(FVDB_ERR_INVALID_ARG, "FVDB_OPT_PROOF_XMAX takes the f32 bits of a value >= 0");
            h->proof_xmax_sq = f;
            return FVDB_OK;
        }
        default:
            return h->fail(FVDB_ERR_INVALID_ARG, "unknown option");
    }
}

int fvdb_get_stats(fvdb_index* h, fvdb_stats* out) {
    ENTER(h);
    if (!out) return h->fail(FVDB_ERR_INVALID_ARG, "out is NULL");
    h->stats.dim = h->dim;
    h->stats.nlist = h->nlist;
    h->stats.trained = h->trained ? 1u : 0u;
    h->stats.ivf_rows = h->ivf_n + h->pend_n;
    h->stats.flat_rows = h->flat_n;
    h->stats.deleted_rows = h->deleted_count;
    h->stats.device_bytes = h->dev_bytes;
    h->stats.last_batch_calls = h->last_batch_calls;
    *out = h->stats;
    return FVDB_OK;
}

int fvdb_ivf_set_centroids(fvdb_index* h, const float* centroids, uint32_t nlist) {
    ENTER(h);
    if (h->metric != FVDB_METRIC_L2)
        return h->fail(FVDB_ERR_INVALID_CONFIG, "the IVF tier is L2 only, like the reference's IVFIndex (src/ivf/core.rs:373-386, 646-678): "
                       "a cosine / dot handle serves the flat tier (batch_cosine_similarity + top_k_indices, src/core/vector_ops.rs:8-23)");
    if (!centroids || nlist == 0) return h->fail(FVDB_ERR_INVALID_CONFIG, "centroids empty");
    for (size_t i = 0; i < (size_t)nlist * h->dim; ++i)
        if (std::isnan(centroids[i])) return h->fail(FVDB_ERR_NAN, "NaN in centroids");
    CK(h->centroids.ensure((size_t)nlist * h->dim, 0, h->stream, &h->dev_bytes));
    RET(h2d(h, h->centroids.p, centroids, (size_t)nlist * h->dim * 4));
    h->nlist = nlist;
    h->trained = true;
    mark_centroids_dirty(h); ++h->centroids_version;
    clear_lists(h);
    CK(h->list_off.ensure(nlist + 2, 0, h->stream, &h->dev_bytes));
    CK(cudaMemsetAsync(h->list_off.p, 0, (nlist + 2) * 4, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FVDB_OK;
}

int fvdb_ivf_get_centroids(fvdb_index* h, float* out, uint32_t* nlist) {
    ENTER(h);
    if (nlist) *nlist = h->trained ? h->nlist : 0;
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained.");
    if (out) RET(d2h(h, out, h->centroids.p, (size_t)h->nlist * h->dim * 4));
    return FVDB_OK;
}

int fvdb_ivf_train_device(fvdb_index* h, const float* d_data, uint64_t n, uint32_t nlist,
                          uint32_t max_iterations, const float* d_init_centroids, uint64_t seed,
                          fvdb_train_result* out) {
    ENTER(h);
    if (h->metric != FVDB_METRIC_L2)
        return h->fail(FVDB_ERR_INVALID_CONFIG, "the IVF tier is L2 only, like the reference's IVFIndex (src/ivf/core.rs:373-386, 646-678): "
                       "a cosine / dot handle serves the flat tier (batch_cosine_similarity + top_k_indices, src/core/vector_ops.rs:8-23)");
    return train_device_impl(h, d_data, n, nlist, max_iterations, d_init_centroids, seed, out);
}

int fvdb_ivf_train(fvdb_index* h, const float* data, uint64_t n, uint32_t nlist,
                   uint32_t max_iterations, const float* init_centroids, uint64_t seed,
                   fvdb_train_result* out) {
    ENTER(h);
    if (h->metric != FVDB_METRIC_L2)
        return h->fail(FVDB_ERR_INVALID_CONFIG, "the IVF tier is L2 only, like the reference's IVFIndex (src/ivf/core.rs:373-386, 646-678): "
                       "a cosine / dot handle serves the flat tier (batch_cosine_similarity + top_k_indices, src/core/vector_ops.rs:8-23)");
    if (nlist == 0 || max_iterations == 0) return h->fail(FVDB_ERR_INVALID_CONFIG, "Invalid IVFConfig");
    if (n == 0 || n < nlist)
        return h->fail(FVDB_ERR_INSUFFICIENT_TRAINING, "Insufficient training data: got " +
                       std::to_string(n) + ", need at least " + std::to_string(nlist));
    if (!data) return h->fail(FVDB_ERR_INVALID_ARG, "data is NULL");
    DevBuf<float> d_data, d_init;
    CK(d_data.ensure(n * h->dim, 0, h->stream, nullptr, true));
    RET(h2d(h, d_data.p, data, n * h->dim * 4));
    if (init_centroids) {
        CK(d_init.ensure((size_t)nlist * h->dim, 0, h->stream, nullptr, true));
        RET(h2d(h, d_init.p, init_centroids, (size_t)nlist * h->dim * 4));
    }
    return train_device_impl(h, d_data.p, n, nlist, max_iterations, init_centroids ? d_init.p : nullptr,
                             seed, out);
}

int fvdb_ivf_retrain(fvdb_index* h, uint32_t nlist, uint32_t max_iterations, const float* init_centroids,
                     uint64_t seed, fvdb_train_result* out) {
    ENTER(h);
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (nlist == 0 || max_iterations == 0) return h->fail(FVDB_ERR_INVALID_CONFIG, "Invalid IVFConfig");
    RET(seal(h));
    const uint64_t n = h->ivf_n;
    if (n == 0 || n < nlist)
        return h->fail(FVDB_ERR_INSUFFICIENT_TRAINING, "Insufficient training data: got " + std::to_string(n) +
                       ", need at least " + std::to_string(nlist));
    DevBuf<float> d_init;
    if (init_centroids) {
        CK(d_init.ensure((size_t)nlist * h->dim, 0, h->stream, nullptr, true));
        RET(h2d(h, d_init.p, init_centroids, (size_t)nlist * h->dim * 4));
    }
    // the resident rows are the training set (arena order: by list, insertion order inside a list);
    // they never leave the device.  Row ids, tombstones and the id-state table are untouched.
    DevBuf<float> rows;
    DevBuf<uint32_t> ids;
    rows.swap(h->ivf_rows);
    ids.swap(h->ivf_ids);
    const bool track = h->track_ids;
    h->track_ids = false;   // clear_lists() must not forget the ids: the same rows come back below
    int r = train_device_impl(h, rows.p, n, nlist, max_iterations, init_centroids ? d_init.p : nullptr, seed, out);
    h->track_ids = track;
    if (r != FVDB_OK) {
        // a failed training run restored the centroid table: the rows go back where they were and the
        // index is what it was before the call
        h->ivf_rows.swap(rows);
        h->ivf_ids.swap(ids);
        mark_arena_dirty(h);
        return r;
    }
    r = ivf_add_device_impl(h, rows.p, ids.p, n, 1, 0, nullptr, nullptr);
    if (r == FVDB_OK) r = seal(h);
    if (r == FVDB_OK) h->dev_bytes -= rows.cap * sizeof(float) + ids.cap * sizeof(uint32_t);   // freed on return
    if (r != FVDB_OK) {
        // new centroids, rows still grouped by the old ones: keep the rows, report "not trained"
        h->ivf_rows.swap(rows);
        h->ivf_ids.swap(ids);
        h->ivf_n = n;
        h->pend_n = 0;
        h->trained = false;
        mark_arena_dirty(h);
    }
    return r;
}

int fvdb_ivf_dump_lists(fvdb_index* h, uint32_t* out_row_ids, uint32_t* out_lists, uint64_t cap, uint64_t* n_out) {
    ENTER(h);
    RET(seal(h));
    if (n_out) *n_out = h->ivf_n;
    if (!out_row_ids && !out_lists) return FVDB_OK;
    if (cap < h->ivf_n) return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_ivf_dump_lists: buffers too small");
    if (h->ivf_n == 0) return FVDB_OK;
    if (out_row_ids) RET(d2h(h, out_row_ids, h->ivf_ids.p, h->ivf_n * 4));
    if (out_lists) RET(d2h(h, out_lists, h->ivf_list.p, h->ivf_n * 4));
    return FVDB_OK;
}

int fvdb_assign(fvdb_index* h, const float* x, uint64_t n, uint32_t* out_list) {
    ENTER(h);
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (n == 0) return FVDB_OK;
    if (!x || !out_list) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t CH = 1u << 20;
    for (uint64_t off = 0; off < n; off += CH) {
        const uint64_t c = std::min(CH, n - off);
        CK(h->s_x.ensure(c * h->dim, 0, h->stream, &h->dev_bytes));
        CK(h->s_u32a.ensure(c, 0, h->stream, &h->dev_bytes));
        RET(h2d(h, h->s_x.p, x + off * h->dim, c * h->dim * 4));
        RET(check_nan_device(h, h->s_x.p, c * h->dim, h->stream));
        RET(assign_device(h, h->s_x.p, c, h->s_u32a.p, nullptr, nullptr, nullptr, h->stream));
        RET(d2h(h, out_list + off, h->s_u32a.p, c * 4));
    }
    return FVDB_OK;
}

int fvdb_ivf_add(fvdb_index* h, const float* x, const uint32_t* row_ids, uint64_t n, uint32_t* out_list) {
    ENTER(h);
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (n == 0) return FVDB_OK;
    if (!x || !row_ids) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    RET(track_insert(h, row_ids, n, 2));
    const uint64_t CH = 1u << 20;
    for (uint64_t off = 0; off < n; off += CH) {
        const uint64_t c = std::min(CH, n - off);
        CK(h->s_x.ensure(c * h->dim, 0, h->stream, &h->dev_bytes));
        CK(h->s_out_ids.ensure(c, 0, h->stream, &h->dev_bytes));
        RET(h2d(h, h->s_x.p, x + off * h->dim, c * h->dim * 4));
        RET(h2d(h, h->s_out_ids.p, row_ids + off, c * 4));
        int r = ivf_add_device_impl(h, h->s_x.p, h->s_out_ids.p, c, 1, 0, nullptr,
                                    out_list ? out_list + off : nullptr);
        if (r != FVDB_OK) {
            if (h->track_ids) for (uint64_t i = off; i < n; ++i) h->id_state[row_ids[i]] = 0;
            return r;
        }
    }
    return FVDB_OK;
}

int fvdb_ivf_add_device(fvdb_index* h, const float* d_x, const uint32_t* d_row_ids, uint64_t n,
                        uint32_t list_filter_mod, uint32_t list_filter_rem, uint64_t* kept) {
    ENTER(h);
    h->track_ids = false;  // ids never visit the host on this path
    return ivf_add_device_impl(h, d_x, d_row_ids, n, list_filter_mod, list_filter_rem, kept, nullptr);
}

int fvdb_ivf_add_device_owned(fvdb_index* h, const float* d_x, const uint32_t* d_row_ids, uint64_t n,
                              const uint32_t* d_owner, uint32_t my_rank, uint64_t* kept) {
    ENTER(h);
    if (!d_owner) return h->fail(FVDB_ERR_INVALID_ARG, "owner table is NULL");
    h->track_ids = false;
    return ivf_add_device_impl(h, d_x, d_row_ids, n, 2, my_rank, kept, nullptr, d_owner);
}

int fvdb_assign_device(fvdb_index* h, const float* d_x, uint64_t n, uint32_t* d_out_list, void* stream) {
    ENTER(h);
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (n == 0) return FVDB_OK;
    if (!d_x || !d_out_list) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    RET(check_nan_device(h, d_x, n * h->dim, st));
    return assign_device(h, d_x, n, d_out_list, nullptr, nullptr, nullptr, st);
}

int fvdb_flat_add(fvdb_index* h, const float* x, const uint32_t* row_ids, uint64_t n) {
    ENTER(h);
    if (n == 0) return FVDB_OK;
    if (!x || !row_ids) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    RET(track_insert(h, row_ids, n, 1));
    const uint64_t CH = 1u << 20;
    for (uint64_t off = 0; off < n; off += CH) {
        const uint64_t c = std::min(CH, n - off);
        CK(h->s_x.ensure(c * h->dim, 0, h->stream, &h->dev_bytes));
        CK(h->s_out_ids.ensure(c, 0, h->stream, &h->dev_bytes));
        RET(h2d(h, h->s_x.p, x + off * h->dim, c * h->dim * 4));
        RET(h2d(h, h->s_out_ids.p, row_ids + off, c * 4));
        int r = flat_add_device_impl(h, h->s_x.p, h->s_out_ids.p, c);
        if (r != FVDB_OK) {
            if (h->track_ids) for (uint64_t i = off; i < n; ++i) h->id_state[row_ids[i]] = 0;
            return r;
        }
    }
    return FVDB_OK;
}

int fvdb_flat_add_device(fvdb_index* h, const float* d_x, const uint32_t* d_row_ids, uint64_t n) {
    ENTER(h);
    h->track_ids = false;
    return flat_add_device_impl(h, d_x, d_row_ids, n);
}

int fvdb_set_deleted(fvdb_index* h, const uint32_t* row_ids, uint64_t n, int deleted) {
    ENTER(h);
    if (n == 0) return FVDB_OK;
    if (!row_ids) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    uint32_t mx = 0;
    for (uint64_t i = 0; i < n; ++i) mx = std::max(mx, row_ids[i]);
    if (h->track_ids) {
        for (uint64_t i = 0; i < n; ++i)
            if (row_ids[i] >= h->id_state.size() || (h->id_state[row_ids[i]] & 3) == 0)
                return h->fail(FVDB_ERR_NOT_FOUND, "Vector not found: row id " + std::to_string(row_ids[i]));
        for (uint64_t i = 0; i < n; ++i) {
            uint8_t& s = h->id_state[row_ids[i]];
            if (deleted && !(s & 0x80)) { s |= 0x80; h->deleted_count++; }
            else if (!deleted && (s & 0x80)) { s &= 0x7f; h->deleted_count--; }
        }
    } else {
        if (deleted) h->deleted_count += n;  // upper bound; only used as "any tombstones" flag
    }
    RET(ensure_tomb(h, (uint64_t)mx + 1));
    CK(h->s_out_ids.ensure(n, 0, h->stream, &h->dev_bytes));
    RET(h2d(h, h->s_out_ids.p, row_ids, n * 4));
    CK(launch_set_bits(h->tomb.p, h->tomb_bits, h->s_out_ids.p, n, deleted ? 1 : 0, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return FVDB_OK;
}

int fvdb_vacuum(fvdb_index* h, uint64_t* removed) {
    ENTER(h);
    if (removed) *removed = 0;
    RET(seal(h));
    if (h->deleted_count == 0 || h->tomb_bits == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    uint64_t gone = 0;
    if (h->ivf_n) {
        const uint64_t n = h->ivf_n;
        CK(h->s_keys32.ensure(n, 0, st, &h->dev_bytes));
        CK(launch_keys_from_bitmap(h->ivf_ids.p, n, h->tomb.p, h->tomb_bits, h->nlist, h->ivf_list.p, 0,
                                   h->s_keys32.p, st));
        CK(h->s_perm.ensure(n, 0, st, &h->dev_bytes));
        CK(h->s_group.ensure(stable_group_scratch_bytes(n, h->nlist), 0, st, &h->dev_bytes));
        CK(launch_stable_group(h->s_keys32.p, n, h->nlist, h->list_off.p, h->s_perm.p, h->s_group.p, st));
        uint32_t kept = 0;
        CK(cudaMemcpyAsync(&kept, h->list_off.p + h->nlist, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        DevBuf<float> nrows;
        DevBuf<uint32_t> nids, nl;
        CK(nrows.ensure((size_t)std::max<uint64_t>(kept, 1) * D, 0, st, &h->dev_bytes, true));
        CK(nids.ensure(std::max<uint64_t>(kept, 1), 0, st, &h->dev_bytes, true));
        CK(nl.ensure(std::max<uint64_t>(kept, 1), 0, st, &h->dev_bytes, true));
        CK(launch_gather_rows(h->ivf_rows.p, n, nullptr, h->s_perm.p, kept, D, nrows.p, st));
        CK(launch_gather_u32(h->ivf_ids.p, n, nullptr, h->s_perm.p, kept, nids.p, st));
        CK(launch_gather_u32(h->ivf_list.p, n, nullptr, h->s_perm.p, kept, nl.p, st));
        CK(cudaStreamSynchronize(st));
        h->dev_bytes -= h->ivf_rows.cap * 4 + (h->ivf_ids.cap + h->ivf_list.cap) * 4;
        h->ivf_rows.swap(nrows);
        h->ivf_ids.swap(nids);
        h->ivf_list.swap(nl);
        gone += n - kept;
        h->ivf_n = kept;
        mark_arena_dirty(h);
    }
    if (h->flat_n) {
        const uint64_t n = h->flat_n;
        CK(h->s_keys32.ensure(n, 0, st, &h->dev_bytes));
        CK(launch_keys_from_bitmap(h->flat_ids.p, n, h->tomb.p, h->tomb_bits, 1, nullptr, 0, h->s_keys32.p, st));
        CK(h->s_perm.ensure(n, 0, st, &h->dev_bytes));
        CK(h->s_group.ensure(stable_group_scratch_bytes(n, 1), 0, st, &h->dev_bytes));
        CK(h->s_u32c.ensure(8, 0, st, &h->dev_bytes));
        CK(launch_stable_group(h->s_keys32.p, n, 1, h->s_u32c.p, h->s_perm.p, h->s_group.p, st));
        uint32_t kept = 0;
        CK(cudaMemcpyAsync(&kept, h->s_u32c.p + 1, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        DevBuf<float> nrows;
        DevBuf<uint32_t> nids;
        CK(nrows.ensure((size_t)std::max<uint64_t>(kept, 1) * D, 0, st, &h->dev_bytes, true));
        CK(nids.ensure(std::max<uint64_t>(kept, 1), 0, st, &h->dev_bytes, true));
        CK(launch_gather_rows(h->flat_rows.p, n, nullptr, h->s_perm.p, kept, D, nrows.p, st));
        CK(launch_gather_u32(h->flat_ids.p, n, nullptr, h->s_perm.p, kept, nids.p, st));
        CK(cudaStreamSynchronize(st));
        h->dev_bytes -= h->flat_rows.cap * 4 + h->flat_ids.cap * 4;
        h->flat_rows.swap(nrows);
        h->flat_ids.swap(nids);
        gone += n - kept;
        h->flat_n = kept;
        h->scratch.tc.flat_dirty = true;
    }
    CK(cudaMemsetAsync(h->tomb.p, 0, (h->tomb_bits + 63) / 64 * 8, st));
    CK(cudaStreamSynchronize(st));
    if (h->track_ids)
        for (auto& s : h->id_state) if (s & 0x80) s = 0;
    h->deleted_count = 0;
    if (removed) *removed = gone;
    return FVDB_OK;
}

int fvdb_move_flat_to_ivf(fvdb_index* h, const uint32_t* row_ids, uint64_t n, uint64_t* moved) {
    ENTER(h);
    if (moved) *moved = 0;
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (n == 0 || h->flat_n == 0) return FVDB_OK;
    if (!row_ids) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    uint32_t mx = 0;
    for (uint64_t i = 0; i < n; ++i) mx = std::max(mx, row_ids[i]);
    const uint64_t nbits = ((uint64_t)mx + 64) / 64 * 64;
    CK(h->s_tmpbits.ensure(nbits / 64, 0, st, &h->dev_bytes));
    CK(cudaMemsetAsync(h->s_tmpbits.p, 0, nbits / 8, st));
    CK(h->s_out_ids.ensure(n, 0, st, &h->dev_bytes));
    RET(h2d(h, h->s_out_ids.p, row_ids, n * 4));
    CK(launch_set_bits(h->s_tmpbits.p, nbits, h->s_out_ids.p, n, 1, st));
    const uint64_t fn = h->flat_n;
    CK(h->s_keys32.ensure(fn, 0, st, &h->dev_bytes));
    CK(launch_keys_from_bitmap(h->flat_ids.p, fn, h->s_tmpbits.p, nbits, 1, nullptr, 0, h->s_keys32.p, st));
    CK(h->s_perm.ensure(fn, 0, st, &h->dev_bytes));
    CK(h->s_group.ensure(stable_group_scratch_bytes(fn, 2), 0, st, &h->dev_bytes));
    CK(h->s_u32c.ensure(8, 0, st, &h->dev_bytes));
    CK(launch_stable_group(h->s_keys32.p, fn, 2, h->s_u32c.p, h->s_perm.p, h->s_group.p, st));
    uint32_t offs[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(offs, h->s_u32c.p, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const uint64_t stay = offs[1], mv = offs[2] - offs[1];
    if (mv == 0) return FVDB_OK;
    DevBuf<float> nrows;
    DevBuf<uint32_t> nids;
    CK(nrows.ensure((size_t)fn * D, 0, st, &h->dev_bytes, true));
    CK(nids.ensure(fn, 0, st, &h->dev_bytes, true));
    CK(launch_gather_rows(h->flat_rows.p, fn, nullptr, h->s_perm.p, fn, D, nrows.p, st));
    CK(launch_gather_u32(h->flat_ids.p, fn, nullptr, h->s_perm.p, fn, nids.p, st));
    CK(cudaStreamSynchronize(st));
    // append the moved rows to the IVF tier FIRST (assignment or allocation may fail); only then does
    // the compacted array replace the flat tier — a failure leaves both tiers as they were
    {
        const int r = ivf_add_device_impl(h, nrows.p + stay * D, nids.p + stay, mv, 1, 0, nullptr, nullptr);
        if (r != FVDB_OK) {
            h->dev_bytes -= nrows.cap * 4 + nids.cap * 4;
            return r;
        }
    }
    h->dev_bytes -= h->flat_rows.cap * 4 + h->flat_ids.cap * 4;
    h->flat_rows.swap(nrows);
    h->flat_ids.swap(nids);
    h->flat_n = stay;
    h->scratch.tc.flat_dirty = true;
    if (h->track_ids)
        for (uint64_t i = 0; i < n; ++i)
            if (row_ids[i] < h->id_state.size() && (h->id_state[row_ids[i]] & 3) == 1)
                h->id_state[row_ids[i]] = (h->id_state[row_ids[i]] & 0x80) | 2;
    if (moved) *moved = mv;
    return FVDB_OK;
}

int fvdb_search_device(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                       uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                       uint32_t* d_out_ids, float* d_out_dist, uint32_t* d_out_count, void* stream) {
    ENTER(h);
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    return search_device_impl(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_out_ids,
                              d_out_dist, d_out_count, st);
}

int fvdb_search_device_submit(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                              uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                              uint32_t* d_out_ids, float* d_out_dist, uint32_t* d_out_count, void* stream) {
    ENTER_PIPE(h);
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (h->pending.size() >= 64) return h->fail(FVDB_ERR_INVALID_ARG, "64 batches are pending: call fvdb_search_device_finish");
    SearchOpts o; o.deferred = true;
    return search_device_impl(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_out_ids,
                              d_out_dist, d_out_count, st, o);
}

static int finish_pending(fvdb_index* h, cudaStream_t st);

int fvdb_search_device_finish(fvdb_index* h, void* stream) {
    ENTER(h);
    return finish_pending(h, stream ? (cudaStream_t)stream : h->stream);
}

// Page-locked host buffers, stream-ordered: the upload of this batch runs on a second stream while the
// previous batch is still being scanned; the result copies follow the batch on the handle's stream.
int fvdb_search_submit(fvdb_index* h, const float* q, uint32_t nq, uint32_t k, uint32_t nprobe, uint32_t tiers,
                       uint32_t* out_ids, float* out_dist, uint32_t* out_count) {
    ENTER_PIPE(h);
    if (!q || !out_ids || !out_dist || !out_count) return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_search_submit: null buffer");
    if (!is_pinned_host(q) || !is_pinned_host(out_ids) || !is_pinned_host(out_dist) || !is_pinned_host(out_count))
        return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_search_submit needs page-locked buffers (fvdb_host_alloc)");
    if (h->pending.size() >= (size_t)fvdb_index::HOST_SLOTS)
        return h->fail(FVDB_ERR_INVALID_ARG, "8 host-buffer batches are pending: call fvdb_search_finish");
    if (nq == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    if (!h->copy_stream) CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    fvdb_index::HostSlot& sl = h->host_slots[h->host_slot_next++ % fvdb_index::HOST_SLOTS];
    if (!sl.uploaded) {
        CK(cudaEventCreateWithFlags(&sl.uploaded, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    }
    // growing a buffer frees the old one: no batch of this slot may still be running (pending < 4 slots,
    // and every earlier batch of this slot was finished, so only the stream order has to be kept)
    CK(sl.q.ensure((size_t)nq * h->dim, 0, st, &h->dev_bytes));
    CK(sl.ids.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
    CK(sl.dist.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
    CK(sl.cnt.ensure(nq, 0, st, &h->dev_bytes));
    if (sl.used) CK(cudaStreamWaitEvent(h->copy_stream, sl.done, 0));   // the slot's previous batch has read its queries
    CK(cudaMemcpyAsync(sl.q.p, q, (size_t)nq * h->dim * 4, cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(sl.uploaded, h->copy_stream));
    const HostOut ho{out_ids, out_dist, out_count, (size_t)nq * k * 4, (size_t)nq * 4};
    // the batch (in a pipeline slot when it qualifies) starts once its queries are on the device
    SearchOpts o; o.ho = &ho; o.deferred = true; o.wait_first = sl.uploaded;
    const int rc = search_device_impl(h, sl.q.p, nq, k, nprobe, tiers, nullptr, 0, sl.ids.p, sl.dist.p, sl.cnt.p, st, o);
    if (rc == FVDB_OK && !h->pending.empty()) {
        const int ps = h->pending.back().slot;
        CK(cudaEventRecord(sl.done, ps >= 0 ? h->slots[ps].stream : st));
        sl.used = true;
    }
    return rc;
}

int fvdb_search_finish(fvdb_index* h) {
    ENTER(h);
    return finish_pending(h, h->stream);
}

static int finish_pending(fvdb_index* h, cudaStream_t st) {
    // results are valid "in stream order" on the caller's stream: it waits for the slots' batches
    for (const fvdb_index::Pending& pb : h->pending)
        if (pb.slot >= 0) cudaStreamWaitEvent(st, h->slots[pb.slot].ev_done, 0);
    bool bad = false;
    for (auto& sl : h->slots)
        if (sl.busy && sl.stream) { bad |= cudaStreamSynchronize(sl.stream) != cudaSuccess; sl.busy = false; }
    if (bad || cudaStreamSynchronize(st) != cudaSuccess) {
        cudaGetLastError();
        for (const fvdb_index::Pending& pb : h->pending) h->pending_pool.push_back(pb.rec);
        for (auto& rec : h->pending_coarse) h->pending_pool.push_back(rec);
        h->pending.clear();
        h->pending_coarse.clear();
        return h->fail(FVDB_ERR_CUDA, "stream synchronisation failed");
    }
    int rc = FVDB_OK;
    std::vector<fvdb_index::Pending> todo;
    todo.swap(h->pending);
    // the figures of the last batch, as the synchronous call reports them
    if (!todo.empty()) set_batch_stats(h, todo.back(), todo.back().rec.first);
    uint32_t fallbacks = 0;
    for (const fvdb_index::Pending& pb : todo) {
        const uint32_t* host = pb.rec.first;
        if (rc == FVDB_OK && host[0])
            rc = h->fail(FVDB_ERR_NAN, "NaN in query (the reference panics on partial_cmp().unwrap())");
        const uint32_t n_ivf = pb.used_tc ? std::min(host[10], 2 * pb.nq) : 0;
        const uint32_t n_flat = pb.flat_tc ? std::min(host[11], 2 * pb.nq) : 0;
        if (rc == FVDB_OK && (n_ivf || n_flat)) {
            const std::vector<uint32_t> rows = failed_queries(host + 16, n_ivf, host + 16 + 2 * pb.nq, n_flat);
            const int r = repair_rows(h, pb, rows, st);
            if (r != FVDB_OK) rc = r;
            fallbacks += (uint32_t)rows.size();
        }
    }
    for (const fvdb_index::Pending& pb : todo) h->pending_pool.push_back(pb.rec);
    for (auto& rec : h->pending_coarse) {
        if (rc == FVDB_OK && rec.first[0])
            rc = h->fail(FVDB_ERR_NAN, "NaN in query (the reference panics on partial_cmp().unwrap())");
        fallbacks += rec.first[10];   // unrepaired: the caller re-runs the batch through the synchronous entries
        h->pending_pool.push_back(rec);
    }
    h->pending_coarse.clear();
    h->stats.last_fallback_queries = fallbacks;
    return rc;
}

int fvdb_coarse_device(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t nprobe, uint64_t* d_out_keys,
                       void* stream) {
    ENTER_PIPE(h);   // touches nothing a batch in a pipeline slot reads: no drain
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (nprobe == 0 || nprobe > h->nlist || nprobe > 512)
        return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_coarse_device needs 1 <= nprobe <= min(nlist, 512)");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    return coarse_device_impl(h, d_q, nq, nprobe, d_out_keys, st);
}

int fvdb_coarse_device_submit(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t nprobe, uint64_t* d_out_keys,
                              void* stream) {
    ENTER_PIPE(h);
    if (!h->trained) return h->fail(FVDB_ERR_NOT_TRAINED, "Index not trained. Call train() before inserting or searching.");
    if (nprobe == 0 || nprobe > h->nlist || nprobe > 512)
        return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_coarse_device needs 1 <= nprobe <= min(nlist, 512)");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    return coarse_device_impl(h, d_q, nq, nprobe, d_out_keys, st, true);
}

int fvdb_search_device_coarse_submit(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                                     uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                                     const uint64_t* d_coarse_keys, uint32_t* d_out_ids, float* d_out_dist,
                                     uint32_t* d_out_count, void* stream) {
    ENTER_PIPE(h);
    if (d_coarse_keys && nprobe > h->nlist)
        return h->fail(FVDB_ERR_INVALID_ARG, "coarse keys are [nq x nprobe]: nprobe must not exceed nlist");
    if (h->pending.size() >= 64) return h->fail(FVDB_ERR_INVALID_ARG, "64 batches are pending: call fvdb_search_device_finish");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    SearchOpts o; o.ext_coarse = d_coarse_keys; o.deferred = true;
    return search_device_impl(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_out_ids,
                              d_out_dist, d_out_count, st, o);
}

// Device-side join: `stream` waits for the batch submitted `age` submits ago (0 = the latest).
int fvdb_search_device_wait(fvdb_index* h, uint32_t age, void* stream) {
    ENTER_PIPE(h);
    if (age >= h->pending.size()) return FVDB_OK;
    const fvdb_index::Pending& pb = h->pending[h->pending.size() - 1 - age];
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (pb.slot >= 0) CK(cudaStreamWaitEvent(st, h->slots[pb.slot].ev_done, 0));
    return FVDB_OK;
}

int fvdb_search_device_coarse(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                              uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                              const uint64_t* d_coarse_keys, uint32_t* d_out_ids, float* d_out_dist,
                              uint32_t* d_out_count, void* stream) {
    ENTER(h);
    if (d_coarse_keys && nprobe > h->nlist)
        return h->fail(FVDB_ERR_INVALID_ARG, "coarse keys are [nq x nprobe]: nprobe must not exceed nlist");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    SearchOpts o; o.ext_coarse = d_coarse_keys;
    return search_device_impl(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_out_ids,
                              d_out_dist, d_out_count, st, o);
}

// fvdb_search_device_coarse / _coarse_submit with the tiers kept apart: one flag through search_device_impl,
// whose final merge then writes the recent tier to the first part of d_out_pack and the IVF tier to the second.
static int search_device_tiers_common(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                                      uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                                      const uint64_t* d_coarse_keys, uint32_t* d_out_pack, void* stream, bool submit) {
    if (h->metric != FVDB_METRIC_L2)
        return h->fail(FVDB_ERR_INVALID_CONFIG, "fvdb_search_device_tiers serves L2 handles only");
    if (!d_out_pack) return h->fail(FVDB_ERR_INVALID_ARG, "d_out_pack is NULL");
    if (d_coarse_keys && nprobe > h->nlist)
        return h->fail(FVDB_ERR_INVALID_ARG, "coarse keys are [nq x nprobe]: nprobe must not exceed nlist");
    if (submit && h->pending.size() >= 64)
        return h->fail(FVDB_ERR_INVALID_ARG, "64 batches are pending: call fvdb_search_device_finish");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    const size_t nk = (size_t)nq * k;
    SearchOpts o; o.ext_coarse = d_coarse_keys; o.deferred = submit; o.split = true;
    return search_device_impl(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_out_pack,
                              reinterpret_cast<float*>(d_out_pack + nk), d_out_pack + 2 * nk, st, o);
}

int fvdb_search_device_tiers(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                             uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                             const uint64_t* d_coarse_keys, uint32_t* d_out_pack, void* stream) {
    ENTER(h);
    return search_device_tiers_common(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_coarse_keys,
                                      d_out_pack, stream, false);
}

int fvdb_search_device_tiers_submit(fvdb_index* h, const float* d_q, uint32_t nq, uint32_t k, uint32_t nprobe,
                                    uint32_t tiers, const uint64_t* d_filter_bits, uint64_t filter_nbits,
                                    const uint64_t* d_coarse_keys, uint32_t* d_out_pack, void* stream) {
    ENTER_PIPE(h);
    return search_device_tiers_common(h, d_q, nq, k, nprobe, tiers, d_filter_bits, filter_nbits, d_coarse_keys,
                                      d_out_pack, stream, true);
}

namespace {

// One host-buffer batch: queries in, results out, one async copy each way.  Page-locked caller
// buffers (fvdb_host_alloc) are handed to the copy engine as they are; pageable ones go through
// the handle's pinned staging.  Caller holds h->mu.
int search_host_locked(fvdb_index* h, const float* q, uint32_t nq, uint32_t k, uint32_t nprobe, uint32_t tiers,
                       const uint64_t* filter_bits, uint64_t filter_nbits, uint32_t* out_ids, float* out_dist,
                       uint32_t* out_count) {
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim;
    const size_t qb = (size_t)nq * D * 4, ob = (size_t)nq * k * 4, cb = (size_t)nq * 4;
    CK(h->s_q.ensure((size_t)nq * D, 0, st, &h->dev_bytes));
    CK(h->s_out_ids.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
    CK(h->s_out_dist.ensure((size_t)nq * k, 0, st, &h->dev_bytes));
    CK(h->s_out_cnt.ensure(nq, 0, st, &h->dev_bytes));
    const bool q_pinned = is_pinned_host(q);
    const bool out_pinned = is_pinned_host(out_ids) && is_pinned_host(out_dist) && is_pinned_host(out_count);
    CK(h->ensure_pin(std::max(q_pinned ? (size_t)0 : qb, out_pinned ? (size_t)0 : 2 * ob + cb)));
    if (!q_pinned) std::memcpy(h->pin, q, qb);
    CK(cudaMemcpyAsync(h->s_q.p, q_pinned ? (const void*)q : (const void*)h->pin, qb, cudaMemcpyHostToDevice, st));
    const uint64_t* d_filter = nullptr;
    if (filter_bits && filter_nbits) {
        const size_t words = (filter_nbits + 63) / 64;
        CK(h->s_filter.ensure(words, 0, st, &h->dev_bytes));
        CK(cudaStreamSynchronize(st));  // pin buffer is about to be reused
        RET(h2d(h, h->s_filter.p, filter_bits, words * 8));
        d_filter = h->s_filter.p;
    } else if (filter_bits) {
        // an empty bitmap filters everything out
        CK(h->s_filter.ensure(1, 0, st, &h->dev_bytes));
        CK(cudaMemsetAsync(h->s_filter.p, 0, 8, st));
        d_filter = h->s_filter.p;
        filter_nbits = 0;
    }
    if (!out_pinned) CK(h->ensure_pin(2 * ob + cb));
    char* pin = (char*)h->pin;
    HostOut ho{out_pinned ? (void*)out_ids : (void*)pin, out_pinned ? (void*)out_dist : (void*)(pin + ob),
               out_pinned ? (void*)out_count : (void*)(pin + 2 * ob), ob, cb};
    // the result copies are enqueued in front of the batch's one synchronisation point
    SearchOpts o; o.ho = &ho;
    RET(search_device_impl(h, h->s_q.p, nq, k, nprobe, tiers, d_filter, filter_nbits, h->s_out_ids.p,
                           h->s_out_dist.p, h->s_out_cnt.p, st, o));
    if (!out_pinned) {
        std::memcpy(out_ids, pin, ob);
        std::memcpy(out_dist, pin + ob, ob);
        std::memcpy(out_count, pin + 2 * ob, cb);
    }
    return FVDB_OK;
}

// Several queued calls with the same (k, nprobe, tiers) as ONE device batch: the queries are
// concatenated in the pinned staging buffer, the results scattered back to each caller's buffers.
// A NaN anywhere fails the whole device batch; then every call is run on its own so that only
// the offending caller sees the error.  Caller holds h->mu.
void run_coalesced(fvdb_index* h, std::vector<SearchReq*>& batch) {
    h->last_batch_calls = (uint32_t)batch.size();
    if (batch.size() == 1) {
        SearchReq* r = batch[0];
        r->rc = search_host_locked(h, r->q, r->nq, r->k, r->nprobe, r->tiers, nullptr, 0, r->out_ids, r->out_dist,
                                   r->out_count);
        return;
    }
    const uint32_t D = h->dim, k = batch[0]->k;
    uint64_t total = 0;
    for (SearchReq* r : batch) total += r->nq;
    const size_t qb = (size_t)total * D * 4, ob = (size_t)total * k * 4, cb = (size_t)total * 4;
    int rc = FVDB_OK;
    cudaStream_t st = h->stream;
    auto stage = [&]() -> int {
        CK(h->s_q.ensure((size_t)total * D, 0, st, &h->dev_bytes));
        CK(h->s_out_ids.ensure((size_t)total * k, 0, st, &h->dev_bytes));
        CK(h->s_out_dist.ensure((size_t)total * k, 0, st, &h->dev_bytes));
        CK(h->s_out_cnt.ensure(total, 0, st, &h->dev_bytes));
        CK(h->ensure_pin(std::max(qb, 2 * ob + cb)));
        size_t off = 0;
        for (SearchReq* r : batch) {
            std::memcpy((char*)h->pin + off, r->q, (size_t)r->nq * D * 4);
            off += (size_t)r->nq * D * 4;
        }
        CK(cudaMemcpyAsync(h->s_q.p, h->pin, qb, cudaMemcpyHostToDevice, st));
        char* pin = (char*)h->pin;
        HostOut ho{pin, pin + ob, pin + 2 * ob, ob, cb};
        SearchOpts o; o.ho = &ho;
        RET(search_device_impl(h, h->s_q.p, (uint32_t)total, k, batch[0]->nprobe, batch[0]->tiers, nullptr, 0,
                               h->s_out_ids.p, h->s_out_dist.p, h->s_out_cnt.p, st, o));
        size_t row = 0;
        for (SearchReq* r : batch) {
            std::memcpy(r->out_ids, pin + row * k * 4, (size_t)r->nq * k * 4);
            std::memcpy(r->out_dist, pin + ob + row * k * 4, (size_t)r->nq * k * 4);
            std::memcpy(r->out_count, pin + 2 * ob + row * 4, (size_t)r->nq * 4);
            row += r->nq;
        }
        return FVDB_OK;
    };
    rc = stage();
    if (rc == FVDB_ERR_NAN) {
        for (SearchReq* r : batch)
            r->rc = search_host_locked(h, r->q, r->nq, r->k, r->nprobe, r->tiers, nullptr, 0, r->out_ids, r->out_dist,
                                       r->out_count);
        return;
    }
    for (SearchReq* r : batch) r->rc = rc;
}

constexpr uint64_t COALESCE_MAX_QUERIES = 8192;   // one device batch of coalesced calls

}  // namespace

int fvdb_search(fvdb_index* h, const float* q, uint32_t nq, uint32_t k, uint32_t nprobe, uint32_t tiers,
                const uint64_t* filter_bits, uint64_t filter_nbits, uint32_t* out_ids, float* out_dist,
                uint32_t* out_count) {
    if (!h) return FVDB_ERR_INVALID_ARG;
    if (filter_bits || !h->coalesce) {
        // a filter bitmap belongs to one call: no coalescing
        ENTER(h);
        if (k == 0) return h->fail(FVDB_ERR_INVALID_ARG, "k must be >= 1");
        if (k > h->k_max) return h->fail(FVDB_ERR_K_TOO_LARGE, "k exceeds k_max given at fvdb_create");
        if (nq == 0) return FVDB_OK;
        if (!q || !out_ids || !out_dist || !out_count) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
        h->last_batch_calls = 1;
        return search_host_locked(h, q, nq, k, nprobe, tiers, filter_bits, filter_nbits, out_ids, out_dist, out_count);
    }
    // Submission queue (the reference allows many concurrent `&self` searches, src/hybrid/core.rs:
    // 202-213, and its callers search one query at a time, src/ivf/operations.rs:139): a call
    // queues its request; the first caller becomes the leader, takes every queued request with its
    // own (k, nprobe, tiers) and runs them as ONE device batch, then hands the lead to the next
    // waiting caller.  Without concurrency this is exactly one call = one batch.
    SearchReq r{q, nq, k, nprobe, tiers, out_ids, out_dist, out_count};
    std::unique_lock<std::mutex> ql(h->qmu);
    h->queue.push_back(&r);
    if (h->leader_active) {
        r.cv.wait(ql, [&] { return r.state != SearchReq::WAITING; });
        if (r.state == SearchReq::DONE) return r.rc;
    } else {
        h->leader_active = true;
    }
    ql.unlock();
    {
        std::lock_guard<std::mutex> guard(h->mu);
        h->err.clear();
        std::vector<SearchReq*> batch;
        ql.lock();
        {
            // own request first, then every compatible one in arrival order
            uint64_t total = r.nq;
            batch.push_back(&r);
            for (auto it = h->queue.begin(); it != h->queue.end();) {
                SearchReq* o = *it;
                if (o == &r) { it = h->queue.erase(it); continue; }
                if (o->k == r.k && o->nprobe == r.nprobe && o->tiers == r.tiers && total + o->nq <= COALESCE_MAX_QUERIES) {
                    total += o->nq;
                    batch.push_back(o);
                    it = h->queue.erase(it);
                } else {
                    ++it;
                }
            }
        }
        ql.unlock();
        int early = FVDB_OK;
        if (cudaSetDevice(h->device) != cudaSuccess) early = h->fail(FVDB_ERR_CUDA, "cudaSetDevice failed");
        // per-call argument checks (a bad call must not fail the calls it was batched with)
        std::vector<SearchReq*> good;
        for (SearchReq* o : batch) {
            if (early != FVDB_OK) o->rc = early;
            else if (o->k == 0) o->rc = h->fail(FVDB_ERR_INVALID_ARG, "k must be >= 1");
            else if (o->k > h->k_max) o->rc = h->fail(FVDB_ERR_K_TOO_LARGE, "k exceeds k_max given at fvdb_create");
            else if (o->nq == 0) o->rc = FVDB_OK;
            else if (!o->q || !o->out_ids || !o->out_dist || !o->out_count) o->rc = h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
            else good.push_back(o);
        }
        if (!good.empty()) run_coalesced(h, good);
        ql.lock();
        for (SearchReq* o : batch)
            if (o != &r) { o->state = SearchReq::DONE; o->cv.notify_one(); }
        if (!h->queue.empty()) {
            SearchReq* nx = h->queue.front();
            nx->state = SearchReq::LEAD;
            nx->cv.notify_one();
        } else {
            h->leader_active = false;
        }
        ql.unlock();
    }
    return r.rc;
}

// HybridIndex::search_with_filter (src/hybrid/core.rs:513-549): search(3k), keep what matches, truncate(k).
// The oversampled search and the compaction both run on the device; `keep_bits` is the host's
// evaluation of the filter (one bit per row id; rows without metadata are 0, :536-541).
int fvdb_search_postfilter(fvdb_index* h, const float* q, uint32_t nq, uint32_t k, uint32_t nprobe, uint32_t tiers,
                           const uint64_t* keep_bits, uint64_t keep_nbits, uint32_t* out_ids, float* out_dist,
                           uint32_t* out_count) {
    ENTER(h);
    if (k == 0) return h->fail(FVDB_ERR_INVALID_ARG, "k must be >= 1");
    if ((uint64_t)k * 3 > h->k_max)
        return h->fail(FVDB_ERR_K_TOO_LARGE, "the 3x post-filter searches 3k candidates: 3k exceeds k_max given at fvdb_create");
    if (nq == 0) return FVDB_OK;
    if (!q || !out_ids || !out_dist || !out_count || !keep_bits) return h->fail(FVDB_ERR_INVALID_ARG, "NULL buffer");
    cudaStream_t st = h->stream;
    const uint32_t D = h->dim, k3 = 3 * k;
    const size_t words = std::max<uint64_t>((keep_nbits + 63) / 64, 1);
    CK(h->s_q.ensure((size_t)nq * D, 0, st, &h->dev_bytes));
    CK(h->s_filter.ensure(words, 0, st, &h->dev_bytes));
    CK(h->s_out_ids.ensure((size_t)nq * (k3 + k), 0, st, &h->dev_bytes));
    CK(h->s_out_dist.ensure((size_t)nq * (k3 + k), 0, st, &h->dev_bytes));
    CK(h->s_out_cnt.ensure((size_t)2 * nq, 0, st, &h->dev_bytes));
    RET(h2d(h, h->s_q.p, q, (size_t)nq * D * 4));
    if (keep_nbits) RET(h2d(h, h->s_filter.p, keep_bits, (keep_nbits + 63) / 64 * 8));
    uint32_t* c_ids = h->s_out_ids.p;
    float* c_dist = h->s_out_dist.p;
    uint32_t* c_cnt = h->s_out_cnt.p;
    uint32_t* f_ids = c_ids + (size_t)nq * k3;
    float* f_dist = c_dist + (size_t)nq * k3;
    uint32_t* f_cnt = c_cnt + nq;
    RET(search_device_impl(h, h->s_q.p, nq, k3, nprobe, tiers, nullptr, 0, c_ids, c_dist, c_cnt, st));
    CK(launch_postfilter_rows(c_ids, c_dist, c_cnt, nq, k3, k, h->s_filter.p, keep_nbits, f_ids, f_dist, f_cnt, st));
    h->stats.last_launches += 1;
    RET(d2h(h, out_ids, f_ids, (size_t)nq * k * 4));
    RET(d2h(h, out_dist, f_dist, (size_t)nq * k * 4));
    RET(d2h(h, out_count, f_cnt, (size_t)nq * 4));
    return FVDB_OK;
}

int fvdb_host_alloc(size_t bytes, void** out) {
    if (!out) return FVDB_ERR_INVALID_ARG;
    *out = nullptr;
    if (bytes == 0) return FVDB_OK;
    if (cudaHostAlloc(out, bytes, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        *out = nullptr;
        return FVDB_ERR_OOM;
    }
    return FVDB_OK;
}

void fvdb_host_free(void* p) {
    if (p && cudaFreeHost(p) != cudaSuccess) cudaGetLastError();
}

int fvdb_ivf_max_sqnorm(fvdb_index* h, float* out) {
    ENTER(h);
    if (!out) return h->fail(FVDB_ERR_INVALID_ARG, "out is NULL");
    *out = 0.f;
    RET(seal(h));
    if (h->ivf_n == 0) return FVDB_OK;
    cudaStream_t st = h->stream;
    CK(h->s_f32a.ensure(h->ivf_n, 0, st, &h->dev_bytes));
    CK(h->scratch.misc.ensure(64, 0, st, &h->dev_bytes));
    uint32_t* d_max = h->scratch.misc.p + 13;
    CK(cudaMemsetAsync(d_max, 0, 4, st));
    CK(launch_max_sqnorm(h->ivf_rows.p, h->ivf_n, h->dim, h->s_f32a.p, d_max, st));
    uint32_t bits = 0;
    CK(cudaMemcpyAsync(&bits, d_max, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    std::memcpy(out, &bits, 4);
    return FVDB_OK;
}

int fvdb_bounds_export(fvdb_index* h, uint32_t nq_cap, void* handle_out) {
    ENTER(h);
    if (!handle_out || nq_cap == 0) return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_bounds_export needs a handle buffer and nq_cap > 0");
    for (uint32_t* pb : h->peer_bounds) cudaIpcCloseMemHandle(pb);
    h->peer_bounds.clear();
    if (h->bounds) { CK(cudaStreamSynchronize(h->stream)); cudaFree(h->bounds); h->bounds = nullptr; }
    CK(cudaMalloc(&h->bounds, (size_t)2 * nq_cap * sizeof(uint32_t)));
    CK(cudaMemset(h->bounds, 0x7f, (size_t)2 * nq_cap * sizeof(uint32_t)));
    h->bounds_cap = nq_cap;
    h->bounds_parity = 0;
    h->bounds_armed_nq = 0;
    cudaIpcMemHandle_t ih;
    CK(cudaIpcGetMemHandle(&ih, h->bounds));
    static_assert(sizeof(cudaIpcMemHandle_t) == FVDB_BOUNDS_HANDLE_BYTES, "handle size");
    std::memcpy(handle_out, &ih, sizeof(ih));
    return FVDB_OK;
}

int fvdb_bounds_import(fvdb_index* h, const void* handles, uint32_t n_ranks, uint32_t my_rank) {
    ENTER(h);
    if (n_ranks == 0) {   // close every imported array (before a peer re-exports a larger one)
        for (uint32_t* pb : h->peer_bounds) cudaIpcCloseMemHandle(pb);
        h->peer_bounds.clear();
        return FVDB_OK;
    }
    if (!h->bounds) return h->fail(FVDB_ERR_INVALID_ARG, "call fvdb_bounds_export first");
    if (!handles || my_rank >= n_ranks || n_ranks - 1 > TC_MAX_PEERS)
        return h->fail(FVDB_ERR_INVALID_ARG, "fvdb_bounds_import: 2..8 ranks, my_rank < n_ranks");
    for (uint32_t* pb : h->peer_bounds) cudaIpcCloseMemHandle(pb);
    h->peer_bounds.clear();
    for (uint32_t r = 0; r < n_ranks; ++r) {
        if (r == my_rank) continue;
        cudaIpcMemHandle_t ih;
        std::memcpy(&ih, (const char*)handles + (size_t)r * sizeof(ih), sizeof(ih));
        void* ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess));
        h->peer_bounds.push_back(static_cast<uint32_t*>(ptr));
    }
    return FVDB_OK;
}

int fvdb_bounds_begin_batch(fvdb_index* h, uint32_t nq, void* stream) {
    ENTER_PIPE(h);   // touches nothing a batch in a pipeline slot reads: no drain
    if (!h->bounds || nq > h->bounds_cap) { h->bounds_armed_nq = 0; return FVDB_OK; }   // not shared: the scan uses its own array
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    h->bounds_parity ^= 1u;
    // +inf bits 0x7f800000: two passes of memset cannot write it, so a tiny fill kernel
    CK(launch_fill_u32(h->bounds + (size_t)h->bounds_parity * h->bounds_cap, nq, 0x7f800000u, st));
    h->bounds_armed_nq = nq;
    return FVDB_OK;
}

int fvdb_merge_topk_packed_device(fvdb_index* h, const uint32_t* d_pack, uint32_t parts, uint32_t nq, uint32_t k,
                                  uint32_t* d_out_ids, float* d_out_dist, uint32_t* d_out_count, void* stream) {
    ENTER_PIPE(h);   // touches nothing a batch in a pipeline slot reads: no drain
    if (parts == 0 || parts > 64) return h->fail(FVDB_ERR_INVALID_ARG, "parts must be in 1..64");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    const size_t nk = (size_t)nq * k, chunk = 2 * nk + nq;
    CK(launch_merge_parts(d_pack, reinterpret_cast<const float*>(d_pack + nk), d_pack + 2 * nk, parts, nq, k,
                          d_out_ids, d_out_dist, d_out_count, st, chunk, chunk));
    return FVDB_OK;
}

int fvdb_merge_topk_tiers_packed_device(fvdb_index* h, const uint32_t* d_pack, uint32_t ranks, uint32_t nq,
                                        uint32_t k, uint32_t* d_out_ids, float* d_out_dist, uint32_t* d_out_count,
                                        void* stream) {
    ENTER_PIPE(h);   // touches nothing a batch in a pipeline slot reads: no drain
    if (h->metric != FVDB_METRIC_L2)
        return h->fail(FVDB_ERR_INVALID_CONFIG, "the tiered merge is ascending L2: L2 handles only");
    if (ranks == 0 || ranks > 32) return h->fail(FVDB_ERR_INVALID_ARG, "ranks must be in 1..32");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    // a rank's chunk is two packed parts (recent, IVF) back to back: 2 * ranks parts of one part length each
    const size_t nk = (size_t)nq * k, part = 2 * nk + nq;
    CK(launch_merge_parts(d_pack, reinterpret_cast<const float*>(d_pack + nk), d_pack + 2 * nk, 2 * ranks, nq, k,
                          d_out_ids, d_out_dist, d_out_count, st, part, part, true));
    return FVDB_OK;
}

int fvdb_merge_topk_device(fvdb_index* h, const uint32_t* d_ids, const float* d_dist, const uint32_t* d_count,
                           uint32_t parts, uint32_t nq, uint32_t k, uint32_t* d_out_ids, float* d_out_dist,
                           uint32_t* d_out_count, void* stream) {
    ENTER_PIPE(h);   // touches nothing a batch in a pipeline slot reads: no drain
    if (parts == 0 || parts > 64) return h->fail(FVDB_ERR_INVALID_ARG, "parts must be in 1..64");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    CK(launch_merge_parts(d_ids, d_dist, d_count, parts, nq, k, d_out_ids, d_out_dist, d_out_count, st));
    return FVDB_OK;
}

int fvdb_kmeans_accumulate_device(fvdb_index* h, const float* d_data, uint64_t n, float* d_sums,
                                  uint32_t* d_counts, double* d_sqerr, uint32_t* d_assign,
                                  uint32_t* d_changed, void* stream) {
    ENTER(h);
    if (!h->nlist || !h->centroids.p) return h->fail(FVDB_ERR_NOT_TRAINED, "centroids not set");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (n == 0) return FVDB_OK;
    CK(h->s_f32a.ensure(n, 0, st, &h->dev_bytes));
    RET(assign_device(h, d_data, n, d_assign, h->s_f32a.p, d_assign, d_changed, st));
    CK(launch_accumulate_sums(d_data, n, h->dim, d_assign, h->s_f32a.p, d_sums, d_counts, d_sqerr, st));
    return FVDB_OK;
}

int fvdb_kmeans_apply_device(fvdb_index* h, const float* d_sums, const uint32_t* d_counts, void* stream) {
    ENTER(h);
    if (!h->nlist || !h->centroids.p) return h->fail(FVDB_ERR_NOT_TRAINED, "centroids not set");
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    CK(launch_apply_means(d_sums, d_counts, h->nlist, h->dim, h->centroids.p, st));
    mark_centroids_dirty(h); ++h->centroids_version;
    return FVDB_OK;
}

}  // extern "C"
