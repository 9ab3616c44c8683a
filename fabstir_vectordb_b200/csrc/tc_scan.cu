// tc_scan.cu — the Blackwell-native posting-list scan (SURVEY §2a K3):
//   TMA (cp.async.bulk.tensor, 128B swizzle)  ->  shared-memory ring
//   tcgen05.mma kind::tf32 (fp32 accumulate)  ->  TMEM accumulators, double buffered
//   tcgen05.ld epilogue: d2 = |x|^2 + |q|^2 - 2 x.q, threshold filter, per-query shortlist
// followed by an exact fp32 re-rank of the shortlist in the reference's operation order
// (euclidean_distance_scalar, src/core/vector_ops.rs:51-57) and a proof that no row outside the
// shortlist can belong to the exact top-k; queries whose proof fails are handed back to the
// exact path.  Replaces the loop of IVFIndex::search_with_config (src/ivf/core.rs:661-678).
//
// Tile orientation: the 128 database rows of a tile sit on the MMA M dimension (= the 128 TMEM
// lanes = one epilogue thread per row), the <= 64 queries that probe the list on N.  Every list
// is streamed from HBM once per batch; the query tile stays resident in shared memory.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner,
// warps 2-5 = epilogue.  Persistent CTAs, one per SM, static round-robin over work items.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../../include/fvdb.h"
#include "kernels.cuh"
#include "tc_ptx.cuh"
#include "tc_scan.cuh"

namespace fvdb {

namespace {

constexpr int TC_ROWS = 128;                     // rows per tile of kernel R (MMA M)
constexpr int TC_KB_FLOATS = 32;                 // one 128-byte swizzle atom
constexpr int TC_KP = 32;                        // shortlist entries per (query, item)
constexpr int TC_THREADS = 192;                  // kernel Q

struct TcScanParams {
    const ScanItem* items;
    const uint32_t* item_count;
    const uint32_t* pair_q;
    const uint32_t* pair_slot;
    const float* Q;
    const float* qnorm;
    uint32_t D;
    uint32_t KB;
    const float* xnorm;
    const uint32_t* ids;
    const uint64_t* tomb;
    uint64_t tomb_bits;
    const uint64_t* filt;
    uint64_t filt_bits;
    uint32_t P;
    uint64_t* partial;  // [nq][P][S][TC_KP] approx keys: (approx d2 bits << 32) | arena row
    uint32_t S;         // shortlist slots per (query, probe): row ranges a long list is split into (0 = 1)
    uint32_t* row_stamp; // [nq][P][S]: a shortlist row written by THIS launch carries `stamp` (rows that no item
    uint32_t stamp;      // touched keep an older one and are skipped by the merge: no memset of `partial`)
    uint32_t* thr_g;    // [nq] running upper bound of the query's TC_KP-th approx d2 (f32 bits)
    uint32_t* thr_peer[TC_MAX_PEERS];  // the same array on the peer GPUs (NVLink peer memory)
    uint32_t n_peer;
    uint32_t* work_counter;  // dynamic tile scheduler: next unclaimed work item
    uint32_t stages;
    uint32_t kbs;            // kernel Q: k-blocks (128 B each) per pipeline stage
    const float* rows_raw;   // read by no kernel; kept because removing it would move the fields below in kernel R and W
    uint64_t rows_bytes;
    float* dense_out;        // kernel Q dense mode (coarse step): out[q * dense_ld + row] = approx d2
    uint32_t dense_ld;
    uint32_t debug;          // timing experiments. bit 0: skip the epilogue math; 3: no MMAs; 4: a quarter of the MMAs; 5: N = 16
    unsigned long long* prof; // debug bit 7: [grid][3 roles][8] cycle counters (stopwatch laps per role)
    uint32_t scan_sms;        // host side: CTAs of the IVF scan kernels (0 = one per SM)
    uint32_t small_list;      // host side: kernel W keeps 8 candidates per thread in registers (assignment: k = 1)
    int metric;               // kernel W only: METRIC_L2 | METRIC_COS | METRIC_DOT (kernel R and Q are L2)
    const uint32_t* xmax_bits; // kernel W, METRIC_DOT: max |x|^2 of the row set (f32 bits, device)
};
constexpr int TC_SCHED = 4;          // depth of the in-CTA work-item ring
constexpr uint32_t ITEM_END = 0xFFFFFFFFu;

using namespace tcx;

// ================================================================================================
// Kernel R ("rows on lanes"): the scan kernel.  A 128-row tile of a posting list is the MMA A
// operand (TMA -> 128B-swizzled shared-memory ring, one 16 KB stage per 128-byte k-block), the
// <= 64 queries probing the list are the B operand (resident in shared memory for the whole
// item), accumulators [128 rows x ncols] rotate through EIGHT 64-column TMEM buffers so the
// MMA/TMA stream runs up to a whole list ahead of the epilogue.
//
// Warp roles (320 threads):
//   warp 0      TMA producer + dynamic tile scheduler + per-tile |x|^2 strips (masked rows = +inf)
//   warp 1      MMA issuer (one elected lane), TMEM owner
//   warps 2-5   epilogue, one thread per row: v = |x|^2 - 2 x.q against the per-query threshold
//               (shared memory, broadcast reads); the rare passing candidate is appended to the
//               query's pending list with a shared-memory atomic.  After every tile the four warps
//               meet at a named barrier; a query with > 16 pending candidates is merged into its
//               sorted 32-entry shortlist by the warp that owns it, which tightens its threshold
//               (also published to / refreshed from the global per-query bound thr_g that CTAs
//               scanning other lists of the same query share).  A pending list that overflowed
//               is replayed for exactly the rows that could not be stored.
//   warps 6-9   query loaders: stage the NEXT item's query tile (coalesced reads, swizzled
//               stores) as soon as the MMA warp has retired the current item.
// ================================================================================================
constexpr int R2_ROWS = 128;                     // rows per tile (MMA M = TMEM lanes)
constexpr int R2_STAGE_BYTES = R2_ROWS * 128;    // 16 KB: 128 rows x one 128-byte k-block
// Queries per item (the kernel's template parameter NQ, MMA N max) by dimension: the query tile,
// KB x NQ x 128 B, stays resident for the whole item, so the width halves as D doubles past 512 and
// the tile never exceeds the 128 KB it takes at D = 512 (a 64-query tile of D = 1024 would need 256 KB)
constexpr uint32_t r2_tile_q(uint32_t D) { return D <= 512 ? TC_TILE_Q : D <= 1024 ? 32u : 16u; }
constexpr int R2_CAP = 32;                       // pending candidates per query (<= 32: one sorting network)
constexpr int R2_FLUSH = R2_CAP / 2;             // merge a query once it holds more pending than this
constexpr int R2_NBUF = 8;                       // accumulator buffers of NQ columns
constexpr int R2_NSLOT = 16;                     // |x|^2 strips in flight
constexpr int R2_SLACK = 1024;                   // bytes reserved for aligning the dynamic shared memory to 1024 (0: trap if it is not)
static_assert(R2_CAP <= 32 && R2_FLUSH < R2_CAP && R2_NSLOT > R2_NBUF + 2, "kernel R pools");
constexpr int R2_THREADS = 320;
constexpr uint32_t TC_SPLIT_MAX = 4;          // row ranges a long posting list is split into, at most
constexpr uint32_t TC_SPLIT_MIN_ROWS = 2048;  // lists up to this length are never split

struct R2Smem {
    unsigned char* q_tile;    // KB x NQ x 128 B, 128B-swizzled K-major [query][32 floats]
    unsigned char* ring;      // STAGES x 16 KB
    uint64_t* sorted;         // [NQ][TC_KP]  ascending approx keys of this item
    uint64_t* pend;           // [NQ][R2_CAP] unsorted pending candidates
    float* xn_ring;           // [R2_NSLOT][R2_ROWS]
    float* thrp;              // [NQ] threshold - |q|^2   (-inf for padded columns)
    uint32_t* pcnt;           // [2][NQ] pending count (may exceed the capacity: overflow marker)
    uint32_t* qidx;           // [2][NQ]
    uint32_t* qslot;          // [2][NQ]
    float* qn;                // [2][NQ]
    uint32_t* redo;           // [8] bitmask of queries to replay ([half][round parity][2] with offloaded merges)
    uint64_t* bars;
    uint32_t* tmem_ptr;
    uint32_t* sched;          // [TC_SCHED]
};

template <int NQ>
__device__ __forceinline__ R2Smem r2_carve(unsigned char* smem, uint32_t KB, uint32_t STAGES) {
    R2Smem m;
    m.q_tile = smem;
    m.ring = m.q_tile + (size_t)KB * NQ * 128;
    m.sorted = reinterpret_cast<uint64_t*>(m.ring + (size_t)STAGES * R2_STAGE_BYTES);
    m.pend = m.sorted + NQ * TC_KP;
    m.xn_ring = reinterpret_cast<float*>(m.pend + NQ * R2_CAP);
    m.thrp = m.xn_ring + R2_NSLOT * R2_ROWS;
    m.pcnt = reinterpret_cast<uint32_t*>(m.thrp + NQ);
    m.qidx = m.pcnt + 2 * NQ;
    m.qslot = m.qidx + 2 * NQ;
    m.qn = reinterpret_cast<float*>(m.qslot + 2 * NQ);
    m.redo = reinterpret_cast<uint32_t*>(m.qn + 2 * NQ);
    m.bars = reinterpret_cast<uint64_t*>(m.redo + 8);
    m.tmem_ptr = reinterpret_cast<uint32_t*>(m.bars + 2 * STAGES + 2 * R2_NBUF + R2_NSLOT + 2 * TC_SCHED + 8);
    m.sched = m.tmem_ptr + 1;
    return m;
}

size_t tc_scan_smem_bytes(uint32_t KB, uint32_t stages, uint32_t NQ) {
    return (size_t)KB * NQ * 128 + (size_t)stages * R2_STAGE_BYTES + (size_t)NQ * TC_KP * 8 +
           (size_t)NQ * R2_CAP * 8 + (size_t)R2_NSLOT * R2_ROWS * 4 + (size_t)NQ * 9 * 4 + 32 +
           (size_t)(2 * stages + 2 * R2_NBUF + R2_NSLOT + 2 * TC_SCHED + 8) * 8 + 16 + (size_t)TC_SCHED * 4;
}

__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t& r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr));
}
__device__ __forceinline__ void epi_bar_n(int id) { asm volatile("bar.sync %0, 128;" ::"r"(id) : "memory"); }

// Merge the pending candidates of up to four queries (owned by this warp) into their sorted
// shortlists; lane i holds entry i.  n[g] pending entries (already clamped to R2_CAP).
__device__ __forceinline__ void r2_merge4(const R2Smem& sm, const uint32_t (&qs)[4], const uint32_t (&n)[4],
                                          const bool (&act)[4], uint64_t (&lst)[4], int lane,
                                          const uint64_t* pend = nullptr, uint32_t cap = R2_CAP) {
    if (!pend) pend = sm.pend;
    uint64_t nw[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        lst[g] = KEY_NONE;
        nw[g] = KEY_NONE;
        if (act[g]) {
            lst[g] = sm.sorted[qs[g] * TC_KP + lane];
            if ((uint32_t)lane < n[g]) nw[g] = pend[qs[g] * cap + lane];
        }
    }
#pragma unroll
    for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            const bool keep_min = (((lane & k) == 0) == ((lane & j) == 0));
            uint64_t o[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) o[g] = shfl_xor64(nw[g], j);
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const uint64_t mn = nw[g] < o[g] ? nw[g] : o[g], mx = nw[g] < o[g] ? o[g] : nw[g];
                nw[g] = keep_min ? mn : mx;
            }
        }
    }
    warp_merge32x4(lst, nw, lane);
}

// Publish a tightened bound of query qi: a fire-and-forget reduction on the local array, and —
// when it beats what this lane last sent by ~1 % (2^16 in the bit pattern of a positive float) —
// on the peer GPUs' arrays over NVLink.
__device__ __forceinline__ void publish_bound(const TcScanParams& p, uint32_t qi, uint32_t bits, uint32_t& peer_sent) {
    atomicMin(p.thr_g + qi, bits);
    if (p.n_peer && bits + 0x10000u < peer_sent) {
        peer_sent = bits;
        for (uint32_t r = 0; r < p.n_peer; ++r) atomicMin(p.thr_peer[r] + qi, bits);
    }
}

// stopwatch lap: the cycles since the previous lap of this role are charged to category i
#define Q1_LAP(i) do { if (p.prof) { const long long n_ = clock64(); lap[i] += (unsigned long long)(n_ - tl); tl = n_; } } while (0)
#define Q1_LAP_DUMP(role) do { if (p.prof && lane == 0) { for (int i_ = 0; i_ < 8; ++i_) p.prof[((size_t)blockIdx.x * 6 + (role)) * 8 + i_] = lap[i_]; } } while (0)

template <int NQ>   // queries per item: r2_tile_q(D)
__global__ void __launch_bounds__(R2_THREADS, 1)
tc_scan_kernel(const __grid_constant__ CUtensorMap tmap, const TcScanParams p) {
    static_assert(NQ == 16 || NQ == 32 || NQ == 64, "kind::tf32 with M = 128 and one 16-column epilogue chunk");
    constexpr int QBLK_BYTES = NQ * 128;          // one k-block of the query tile (a multiple of the 1 KB swizzle atom)
    constexpr uint32_t TMEM_COLS = R2_NBUF * NQ;  // a power of two >= 32, as tcgen05.alloc needs
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment; the launch reserves 1 KB of slack for this
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    if (R2_SLACK < 1024 && smem != smem_raw) __trap();   // built without slack: the declared alignment must hold
    const uint32_t KB = p.KB;
    const uint32_t STAGES = p.stages;
    const R2Smem sm = r2_carve<NQ>(smem, KB, STAGES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_full = smem_u32(sm.bars);
    const uint32_t bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * STAGES;
    const uint32_t bar_tempty = bar_tfull + 8 * R2_NBUF;
    const uint32_t bar_nfull = bar_tempty + 8 * R2_NBUF;
    const uint32_t bar_sfull = bar_nfull + 8 * R2_NSLOT;
    const uint32_t bar_sempty = bar_sfull + 8 * TC_SCHED;
    const uint32_t bar_qready = bar_sempty + 8 * TC_SCHED;  // query tile + item metadata staged
    const uint32_t bar_qfree = bar_qready + 8;              // every MMA of the item has retired
    const uint32_t bar_mfree = bar_qfree + 8;               // epilogue is done with an item's metadata

    if (threadIdx.x == 0) {
        for (int i = 0; i < 8; ++i) sm.redo[i] = 0;
        for (uint32_t s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int i = 0; i < R2_NBUF; ++i) {
            mbar_init(bar_tfull + 8 * i, 1);
            mbar_init(bar_tempty + 8 * i, 4);
        }
        for (int i = 0; i < R2_NSLOT; ++i) mbar_init(bar_nfull + 8 * i, 1);
        for (int i = 0; i < TC_SCHED; ++i) {
            mbar_init(bar_sfull + 8 * i, 1);
            mbar_init(bar_sempty + 8 * i, 9);  // MMA lane + one lane of each epilogue and loader warp
        }
        mbar_init(bar_qready, 128);
        mbar_init(bar_qfree, 1);
        mbar_init(bar_mfree, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sm.tmem_ptr)),
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *sm.tmem_ptr;
    const uint32_t n_items = *p.item_count;
    unsigned long long lap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tl = clock64();
    if (p.prof && threadIdx.x == 0) {  // wall-clock window of this CTA (role 3, slots 4..6)
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 4] = gt;
        p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 6] = (unsigned long long)tl;
    }

    if (warp == 0) {
        // ============ TMA producer + tile scheduler (whole warp converged, one lane issues) ============
        // Norm-strip slots need no "free" barrier: while this warp fills tile T the MMA warp has
        // started a tile >= T - 1 - ceil(STAGES / KB), hence the epilogue has released a tile
        // >= T - 1 - ceil(STAGES / KB) - R2_NBUF; the launcher keeps that window below R2_NSLOT.
        uint32_t stage = 0, phase = 0, ss = 0, sphase = 0, tcount = 0;
        const uint64_t hint_first = 0x12F0000000000000ull;   // L2 evict-first: rows read once
        const uint64_t hint_normal = 0x1000000000000000ull;  // list shared by several items
        const uint32_t ring_base = smem_u32(sm.ring);
        while (true) {
            Q1_LAP(3);
            mbar_wait(bar_sempty + 8 * ss, sphase ^ 1);
            uint32_t item = 0;
            if (lane == 0) {
                item = atomicAdd(p.work_counter, 1u);
                if (item >= n_items) item = ITEM_END;
                sm.sched[ss] = item;
                mbar_arrive(bar_sfull + 8 * ss);
            }
            item = __shfl_sync(0xffffffffu, item, 0);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            lap[6] += 1;
            Q1_LAP(1);
            // rows shared by several items (a list with > 64 probing queries, a flat-tier chunk) stay in L2
            const uint64_t hint = (it.identity == 2 || (!it.identity && it.slot > 1)) ? hint_normal : hint_first;
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += R2_ROWS) {
                float xnv[4];
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const uint32_t pos = rt + h * 32 + lane;
                    float xn = __uint_as_float(F32_INF_BITS);
                    if (pos < it.row_end) {
                        bool live = true;
                        if (p.tomb || p.filt) {
                            const uint32_t id = p.ids[pos];
                            if (p.tomb && bit_test(p.tomb, p.tomb_bits, id)) live = false;
                            else if (p.filt && !bit_test(p.filt, p.filt_bits, id)) live = false;
                        }
                        if (live) xn = __ldg(p.xnorm + pos);
                    }
                    xnv[h] = xn;
                }
                __syncwarp();
                lap[7] += 1;
                for (uint32_t kb = 0; kb < KB; ++kb) {
                    Q1_LAP(3);
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    Q1_LAP(2);
                    if (elect_one()) {
                        const uint32_t fb = bar_full + 8 * stage;
                        mbar_expect_tx(fb, R2_STAGE_BYTES);
                        tma_load_2d(ring_base + stage * R2_STAGE_BYTES, &tmap, fb, (int)(kb * TC_KB_FLOATS), (int)rt, hint);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                const uint32_t slot = tcount % R2_NSLOT;
#pragma unroll
                for (int h = 0; h < 4; ++h) sm.xn_ring[slot * R2_ROWS + h * 32 + lane] = xnv[h];
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_nfull + 8 * slot);
                ++tcount;
            }
        }
        Q1_LAP_DUMP(0);
    } else if (warp == 1) {
        // ============ MMA issuer (whole warp converged, one elected lane issues) ============
        uint32_t stage = 0, phase = 0, ss = 0, sphase = 0, tile = 0, nit = 0;
        const uint32_t q_base = smem_u32(sm.q_tile);
        const uint32_t ring_base = smem_u32(sm.ring);
        while (true) {
            Q1_LAP(4);
            mbar_wait(bar_sfull + 8 * ss, sphase);
            const uint32_t item = sm.sched[ss];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sempty + 8 * ss);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            const uint32_t ncols = (it.pair_count + 15u) & ~15u;
            const uint32_t idesc = umma_idesc_tf32(R2_ROWS, (p.debug & 32u) ? 16u : ncols);   // debug: narrow MMAs (timing only)
            Q1_LAP(4);
            mbar_wait(bar_qready, nit & 1u);
            tc_fence_after();
            Q1_LAP(1);
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += R2_ROWS) {
                const uint32_t buf = tile & (R2_NBUF - 1);
                Q1_LAP(4);
                mbar_wait(bar_tempty + 8 * buf, ((tile / R2_NBUF) & 1u) ^ 1u);
                tc_fence_after();
                Q1_LAP(2);
                const uint32_t d_tmem = tmem_base + buf * NQ;
                const bool last_tile = rt + R2_ROWS >= it.row_end;
                for (uint32_t kb = 0; kb < KB; ++kb) {
                    Q1_LAP(4);
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    Q1_LAP(3);
                    if (elect_one()) {
                        const uint64_t a0 = umma_desc_sw128(ring_base + stage * R2_STAGE_BYTES);
                        const uint64_t b0 = umma_desc_sw128(q_base + kb * QBLK_BYTES);
#pragma unroll
                        for (uint32_t k4 = 0; k4 < 4; ++k4)  // UMMA_K = 8 tf32 = 32 bytes = +2 in the descriptor
                            if (!(p.debug & 8u) && (!(p.debug & 16u) || k4 == 0))   // timing experiments: no / a quarter of the MMAs
                                umma_tf32(d_tmem, a0 + 2 * k4, b0 + 2 * k4, idesc, (kb | k4) != 0 ? 1u : 0u);
                        umma_commit(bar_empty + 8 * stage);  // frees the ring slot once these MMAs retire
                        if (kb + 1 == KB) {
                            umma_commit(bar_tfull + 8 * buf);   // accumulator ready for the epilogue
                            if (last_tile) umma_commit(bar_qfree);  // query tile may be replaced
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                ++tile;
            }
            ++nit;
        }
        Q1_LAP_DUMP(1);
    } else if (warp >= 6) {
        // ============ query loaders (128 threads) ============
        const int lw = warp - 6;
        const int lt = lw * 32 + lane;
        const uint32_t D = p.D;
        uint32_t ss = 0, sphase = 0, nit = 0;
        while (true) {
            Q1_LAP(3);
            mbar_wait(bar_sfull + 8 * ss, sphase);
            const uint32_t item = sm.sched[ss];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sempty + 8 * ss);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            const uint32_t cnt = it.pair_count;
            const uint32_t ncols = (cnt + 15u) & ~15u;
            // query indices of the item: lane l holds queries l and l + 32
            uint32_t qi0 = ID_NONE, qi1 = ID_NONE, sl0 = 0, sl1 = 0;
            if ((uint32_t)lane < cnt) {
                if (it.identity) { qi0 = it.pair_begin + lane; sl0 = it.slot; }
                else { qi0 = p.pair_q[it.pair_begin + lane]; sl0 = p.pair_slot[it.pair_begin + lane]; }
            }
            if ((uint32_t)lane + 32 < cnt) {
                if (it.identity) { qi1 = it.pair_begin + lane + 32; sl1 = it.slot; }
                else { qi1 = p.pair_q[it.pair_begin + lane + 32]; sl1 = p.pair_slot[it.pair_begin + lane + 32]; }
            }
            // metadata buffer (nit & 1) was last used by item nit - 2
            Q1_LAP(3);
            if (nit >= 2) mbar_wait(bar_mfree, nit & 1u);
            Q1_LAP(1);
            if (lw == 0) {
                const uint32_t mb = (nit & 1u) * NQ;
                if (lane < NQ) {
                    sm.qidx[mb + lane] = qi0;
                    sm.qslot[mb + lane] = sl0;
                    sm.qn[mb + lane] = (qi0 != ID_NONE) ? p.qnorm[qi0] : 0.f;
                }
                if (NQ > 32) {
                    sm.qidx[mb + 32 + lane] = qi1;
                    sm.qslot[mb + 32 + lane] = sl1;
                    sm.qn[mb + 32 + lane] = (qi1 != ID_NONE) ? p.qnorm[qi1] : 0.f;
                }
            }
            // the query tile may be overwritten once every MMA of the previous item has retired
            Q1_LAP(3);
            if (nit >= 1) mbar_wait(bar_qfree, (nit - 1) & 1u);
            Q1_LAP(2);
            {
                // warp lw stages queries lw, lw+4, ...; a lane moves float4 columns lane, lane+32, ...
                // Loads of four query rows are issued before any store (12 LDG.128 per lane in flight).
                const uint32_t f4_per_row = KB * 8;
                for (uint32_t q0 = lw; q0 < ncols; q0 += 16) {
                    const float4* src[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        const uint32_t q = q0 + 4 * g;
                        const uint32_t qa = __shfl_sync(0xffffffffu, qi0, q & 31), qb = __shfl_sync(0xffffffffu, qi1, q & 31);
                        const uint32_t qi = (q < 32) ? qa : qb;
                        src[g] = (q < ncols && qi != ID_NONE) ? reinterpret_cast<const float4*>(p.Q + (size_t)qi * D) : nullptr;
                    }
                    // three float4 columns x four query rows = 12 independent 16-byte loads per lane
                    for (uint32_t c = lane; c < f4_per_row; c += 96) {
                        float4 v[3][4];
#pragma unroll
                        for (int u = 0; u < 3; ++u)
#pragma unroll
                            for (int g = 0; g < 4; ++g)
                                v[u][g] = (src[g] && c + 32 * u < f4_per_row) ? __ldg(src[g] + c + 32 * u)
                                                                               : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                        for (int u = 0; u < 3; ++u) {
                            const uint32_t cc = c + 32 * u;
                            if (cc >= f4_per_row) break;
                            const uint32_t kb = cc >> 3, ch = cc & 7;
#pragma unroll
                            for (int g = 0; g < 4; ++g) {
                                const uint32_t q = q0 + 4 * g;
                                if (q < ncols)
                                    *reinterpret_cast<float4*>(sm.q_tile + (size_t)kb * QBLK_BYTES + q * 128 +
                                                               ((ch ^ (q & 7)) << 4)) = v[u][g];
                            }
                        }
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> async proxy (UMMA)
            mbar_arrive(bar_qready);
            ++nit;
            (void)lt;
        }
        if (warp == 6 && p.prof && lane == 0) {
            for (int i_ = 0; i_ < 4; ++i_) p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + i_] = lap[i_];
            p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 7] = lap[7];
        }
    } else {
        // ================= epilogue (warps 2-5): one thread = one row of the tile =================
        const int ew = warp - 2;                 // owner stripe: this warp merges queries j with j % 4 == ew
        const int quarter = warp & 3;            // TMEM lane quarter this warp may read
        const int trow = quarter * 32 + lane;    // row within the tile == TMEM lane
        const int et = ew * 32 + lane;           // 0..127
        const uint32_t lane_taddr = (uint32_t)(quarter * 32) << 16;
        uint32_t ss = 0, sphase = 0, tile = 0, nit = 0;
        uint32_t st_app = 0, st_ovf = 0, st_merge = 0, st_replay = 0, st_chunks = 0;
        // the query this lane owns in the merge phases (lanes 0..15): j = lane * 4 + ew
        const uint32_t jown = (uint32_t)lane * 4u + (uint32_t)ew;
        while (true) {
            Q1_LAP(6);
            mbar_wait(bar_sfull + 8 * ss, sphase);
            const uint32_t item = sm.sched[ss];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sempty + 8 * ss);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            const uint32_t cnt = it.pair_count;
            const uint32_t ncols = (cnt + 15u) & ~15u;
            const uint32_t mb = (nit & 1u) * NQ;
            mbar_wait(bar_qready, nit & 1u);           // metadata of this item is staged
            Q1_LAP(1);
            if (nit >= 1) {                            // ... and only now release the previous item's
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_mfree);
            }
            // ---- item prologue: empty shortlists, thresholds from the shared bounds ----
            if (et < NQ) {
                float thr = -__uint_as_float(F32_INF_BITS);  // padded columns never pass
                if ((uint32_t)et < cnt) {
                    const uint32_t g = p.thr_g ? *(volatile uint32_t*)(p.thr_g + sm.qidx[mb + et]) : (uint32_t)0x7f800000u;
                    thr = __uint_as_float(g) - sm.qn[mb + et];
                }
                sm.thrp[et] = thr;
                sm.pcnt[et] = 0;
            }
            if (et < 2) sm.redo[et] = 0;
            for (int i = et; i < NQ * TC_KP; i += 128) sm.sorted[i] = KEY_NONE;
            const bool own = lane < 16 && jown < cnt;
            const uint32_t qi_own = own ? sm.qidx[mb + jown] : 0u;
            const float qn_own = own ? sm.qn[mb + jown] : 0.f;
            uint32_t thr_pending = F32_INF_BITS;
            uint32_t peer_sent = F32_INF_BITS;   // last bound of the owned query pushed to the peer GPUs
            epi_bar_n(1);
            Q1_LAP(6);

            // merge every owned query selected by `need` (warp-uniform mask over lanes 0..15)
            auto merge_owned = [&](unsigned need) {
                st_merge += __popc(need);
                if (__popc(need) == 1) {
                    // the common case: one query to fold -> a single 32-lane network (a quarter of
                    // the instructions of the 4-way interleaved one)
                    const int src = __ffs(need) - 1;
                    const uint32_t q = (uint32_t)src * 4u + (uint32_t)ew;
                    const uint32_t c = sm.pcnt[q];
                    const uint32_t n = min(c, (uint32_t)R2_CAP);
                    uint64_t nw = ((uint32_t)lane < n) ? sm.pend[q * R2_CAP + lane] : KEY_NONE;
                    uint64_t lst = sm.sorted[q * TC_KP + lane];
                    nw = warp_sort32(nw, lane);
                    lst = warp_merge32(lst, nw, lane);
                    sm.sorted[q * TC_KP + lane] = lst;
                    const uint64_t last = shfl64(lst, 31);
                    if (lane == src) {
                        sm.pcnt[q] = 0;
                        if (last != KEY_NONE) {
                            sm.thrp[q] = fminf(sm.thrp[q], __uint_as_float((uint32_t)(last >> 32)) - qn_own);
                            if (p.thr_g) publish_bound(p, qi_own, (uint32_t)(last >> 32), peer_sent);
                        }
                        if (c > (uint32_t)R2_CAP) atomicOr(&sm.redo[q >> 5], 1u << (q & 31));
                    }
                    __syncwarp();
                    return;
                }
                while (need) {
                    uint32_t qs[4], nn[4], over = 0;
                    bool act[4];
                    int src[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        act[g] = need != 0;
                        src[g] = act[g] ? (__ffs(need) - 1) : 0;
                        if (act[g]) need &= need - 1;
                        qs[g] = (uint32_t)src[g] * 4u + (uint32_t)ew;
                        const uint32_t c = act[g] ? sm.pcnt[qs[g]] : 0u;
                        nn[g] = min(c, (uint32_t)R2_CAP);
                        if (c > (uint32_t)R2_CAP) over |= 1u << g;
                    }
                    uint64_t lst[4];
                    r2_merge4(sm, qs, nn, act, lst, lane);
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        if (!act[g]) continue;
                        sm.sorted[qs[g] * TC_KP + lane] = lst[g];
                        const uint64_t last = shfl64(lst[g], 31);
                        if (lane == src[g]) {
                            sm.pcnt[qs[g]] = 0;
                            if (last != KEY_NONE) {
                                sm.thrp[qs[g]] = fminf(sm.thrp[qs[g]], __uint_as_float((uint32_t)(last >> 32)) - qn_own);
                                // any 32 rows below a value bound the global 32nd: share it at once
                                if (p.thr_g) publish_bound(p, qi_own, (uint32_t)(last >> 32), peer_sent);
                            }
                            if (over & (1u << g)) atomicOr(&sm.redo[qs[g] >> 5], 1u << (qs[g] & 31));
                        }
                    }
                    __syncwarp();
                }
            };

            // ---- row tiles ----
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += R2_ROWS) {
                const uint32_t slot = tile % R2_NSLOT;
                Q1_LAP(4);
                mbar_wait(bar_nfull + 8 * slot, (tile / R2_NSLOT) & 1u);
                const float xn = sm.xn_ring[slot * R2_ROWS + trow];
                const uint32_t buf = tile & (R2_NBUF - 1);
                mbar_wait(bar_tfull + 8 * buf, (tile / R2_NBUF) & 1u);
                tc_fence_after();
                Q1_LAP(2);
                const uint32_t taddr = tmem_base + buf * NQ + lane_taddr;
                const uint32_t pos = rt + (uint32_t)trow;
                uint64_t ovf = 0;  // queries whose pending list was full when this row passed

                auto append = [&](uint32_t q, float v) {
                    const uint32_t s = atomicAdd(&sm.pcnt[q], 1u);
                    ++st_app;
                    if (s < (uint32_t)R2_CAP)
                        sm.pend[q * R2_CAP + s] =
                            ((uint64_t)__float_as_uint(fmaxf(v + sm.qn[mb + q], 0.0f)) << 32) | (uint64_t)pos;
                    else {
                        ovf |= 1ull << q;
                        ++st_ovf;
                    }
                };

                for (uint32_t c0 = 0; c0 < ((p.debug & 1u) ? 0u : ncols); c0 += 16) {
                    uint32_t acc[16];
                    ++st_chunks;
                    tmem_ld16(taddr + c0, acc);
                    float thr[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 t4 = *reinterpret_cast<const float4*>(sm.thrp + c0 + 4 * j4);
                        thr[4 * j4 + 0] = t4.x; thr[4 * j4 + 1] = t4.y; thr[4 * j4 + 2] = t4.z; thr[4 * j4 + 3] = t4.w;
                    }
                    tmem_ld_wait();
                    // branch-free compare of the 16 columns into a bit mask, then one divergent loop over
                    // the set bits: the warp pays max-over-lanes(passing columns) append latencies per
                    // chunk (2-3) instead of one per column in which ANY lane passes (~11 of 16)
                    uint32_t pass = 0;
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const float v = fmaf(-2.0f, __uint_as_float(acc[j]), xn);  // |x|^2 - 2 x.q
                        pass |= (v < thr[j]) ? (1u << j) : 0u;
                    }
                    while (pass) {
                        const uint32_t b = (uint32_t)__ffs((int)pass) - 1u;
                        pass &= pass - 1u;
                        uint32_t a = acc[0];
#pragma unroll
                        for (int j = 1; j < 16; ++j) a = (b == (uint32_t)j) ? acc[j] : a;
                        append(c0 + b, fmaf(-2.0f, __uint_as_float(a), xn));
                    }
                }
                Q1_LAP(3);
                epi_bar_n(2);  // every candidate of this tile is in the pending lists
                // ---- merge phase: owners fold long pending lists, refresh shared thresholds ----
                while (true) {
                    if (own) {
                        // bound tightened meanwhile by CTAs scanning other lists of the same query
                        // (loaded during the previous tile: no exposed latency)
                        sm.thrp[jown] = fminf(sm.thrp[jown], __uint_as_float(thr_pending) - qn_own);
                        if (p.thr_g) thr_pending = *(volatile uint32_t*)(p.thr_g + qi_own);
                    }
                    const uint32_t pc = own ? sm.pcnt[jown] : 0u;
                    merge_owned(__ballot_sync(0xffffffffu, pc > (uint32_t)R2_FLUSH));
                    epi_bar_n(1);  // thresholds / pending counters settled
                    const uint32_t r0 = sm.redo[0], r1 = sm.redo[1];
                    if ((r0 | r1) == 0) break;
                    ++st_replay;
                    // replay: rows that met a full pending list are tested against the new thresholds
                    epi_bar_n(2);
                    if (et < 2) sm.redo[et] = 0;
                    uint64_t rm = ((uint64_t)r1 << 32) | r0;
                    while (rm) {
                        const uint32_t q = (uint32_t)__ffsll((long long)rm) - 1u;
                        rm &= rm - 1;
                        uint32_t a;
                        tmem_ld1(taddr + q, a);
                        tmem_ld_wait();
                        if ((ovf >> q) & 1ull) {
                            ovf &= ~(1ull << q);
                            const float v = fmaf(-2.0f, __uint_as_float(a), xn);
                            if (v < sm.thrp[q]) append(q, v);
                        }
                    }
                    epi_bar_n(1);
                    // every replayed query is merged again (its pending list may have refilled)
                    {
                        const bool mine = own && (((jown < 32 ? r0 : r1) >> (jown & 31)) & 1u);
                        merge_owned(__ballot_sync(0xffffffffu, mine && sm.pcnt[jown] > 0));
                    }
                    epi_bar_n(2);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty + 8 * buf);  // accumulator may be overwritten
                ++tile;
            }
            // ---- item epilogue: fold what is pending, publish the shortlists ----
            Q1_LAP(4);
            {
                // a query that never merged in this item (the usual case away from its nearest
                // lists) publishes its few pending candidates UNSORTED; the shortlist merge that
                // follows the scan sorts such rows.  Only queries holding both a sorted list and
                // pending candidates need one more fold here.
                const uint32_t pc = own ? sm.pcnt[jown] : 0u;
                const bool has_sorted = own && sm.sorted[jown * TC_KP] != KEY_NONE;
                merge_owned(__ballot_sync(0xffffffffu, pc > 0 && has_sorted));
                __syncwarp();
                for (uint32_t j = (uint32_t)ew; j < cnt; j += 4) {
                    uint64_t mine = sm.sorted[j * TC_KP + lane];
                    if (__shfl_sync(0xffffffffu, mine == KEY_NONE ? 1 : 0, 0)) {   // no sorted list: pending, as is
                        const uint32_t n = sm.pcnt[j];
                        if (n == 0) continue;                                      // partial is pre-filled
                        mine = ((uint32_t)lane < n) ? sm.pend[j * R2_CAP + lane] : KEY_NONE;
                    }
                    const size_t prow = ((size_t)sm.qidx[mb + j] * p.P + sm.qslot[mb + j]) * (p.S ? p.S : 1u) + it.sub;
                    p.partial[prow * TC_KP + lane] = mine;
                    if (lane == 0) p.row_stamp[prow] = p.stamp;
                }
            }
            epi_bar_n(1);  // pools may be re-initialised for the next item
            ++nit;
            Q1_LAP(5);
        }
        if (warp == 2) Q1_LAP_DUMP(2);
        if (p.prof && warp == 2) {
            const uint32_t a = __reduce_add_sync(0xffffffffu, st_app), o = __reduce_add_sync(0xffffffffu, st_ovf);
            if (lane == 0) {
                unsigned long long* d = p.prof + ((size_t)blockIdx.x * 6 + 4) * 8;
                d[0] = a; d[1] = o; d[2] = st_merge; d[3] = st_replay; d[4] = tile; d[5] = st_chunks;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (p.prof && threadIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 5] = gt;
        p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 6] = (unsigned long long)clock64() - p.prof[((size_t)blockIdx.x * 6 + 3) * 8 + 6];
    }
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                     "r"(TMEM_COLS)
                     : "memory");
    }
}



// ================================================================================================
// Kernel Q ("queries on lanes"), dense form: the coarse step's distance matrix.  The query tile is
// the MMA A operand and lives in TENSOR MEMORY (128 TMEM lanes = 128 queries, D <= 384 columns),
// centroid rows stream through shared memory as the B operand (64 rows x 128 B per stage),
// accumulators double-buffered in the remaining 128 TMEM columns.  One epilogue thread owns one
// query and writes its approximate d2 to every centroid of the tile.  (The same orientation with
// CTA pairs, thread-private candidate heaps and a split row stream is kernel W, tc_scan_wide.cuh.)
// ================================================================================================
constexpr int Q1_M = 128;                       // queries per work item
constexpr int Q1_N = 64;                        // rows per tile
constexpr int Q1_STAGE_BYTES = Q1_N * 128;      // 8 KB
constexpr int Q1_TMEM_COLS = 512;
constexpr int Q1_ACC_COL = 384;                 // accumulators at columns 384..511
constexpr int Q1_NSLOT = 16;                    // ring of per-tile row-norm strips (see the producer)
constexpr int Q1_XP_LD = 36;                    // floats per query row of the prologue transposition buffer

__global__ void __launch_bounds__(TC_THREADS, 1)
tc_scan_q_kernel(const __grid_constant__ CUtensorMap tmap, const TcScanParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t KB = p.KB;
    const uint32_t KBS = p.kbs;                     // k-blocks per stage
    const uint32_t NST = KB / KBS;                  // stages per row tile
    const uint32_t STAGES = p.stages;
    const uint32_t STAGE_BYTES = KBS * Q1_STAGE_BYTES;
    unsigned char* ring = smem;                                                     // STAGES x KBS x 8 KB
    float* xpose = reinterpret_cast<float*>(ring + (size_t)STAGES * STAGE_BYTES);      // [2][Q1_M][Q1_XP_LD] prologue transposition
    float* xn_ring = xpose + 2 * Q1_M * Q1_XP_LD;                                    // [Q1_NSLOT][64] tile row norms
    uint64_t* bars = reinterpret_cast<uint64_t*>(xn_ring + Q1_NSLOT * Q1_N);
    uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 5 + 2 * TC_SCHED + Q1_NSLOT);
    uint32_t* sched_s = tmem_ptr_s + 1;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t bar_full = smem_u32(bars);
    const uint32_t bar_empty = bar_full + 8 * STAGES;
    const uint32_t bar_tfull = bar_empty + 8 * STAGES;
    const uint32_t bar_tempty = bar_tfull + 16;
    const uint32_t bar_qready = bar_tempty + 16;
    const uint32_t bar_sfull = bar_qready + 8;
    const uint32_t bar_sempty = bar_sfull + 8 * TC_SCHED;
    const uint32_t bar_nfull = bar_sempty + 8 * TC_SCHED;   // [Q1_NSLOT] norms of a tile are in shared memory

    if (threadIdx.x == 0) {
        for (uint32_t s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int i = 0; i < Q1_NSLOT; ++i) mbar_init(bar_nfull + 8 * i, 1);
        mbar_init(bar_tfull, 1);
        mbar_init(bar_tfull + 8, 1);
        mbar_init(bar_tempty, 4);
        mbar_init(bar_tempty + 8, 4);
        mbar_init(bar_qready, 4);  // one arrival per epilogue warp once its queries sit in TMEM
        for (int i = 0; i < TC_SCHED; ++i) {
            mbar_init(bar_sfull + 8 * i, 1);
            mbar_init(bar_sempty + 8 * i, 5);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_s)),
                     "r"((uint32_t)Q1_TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_s;
    const uint32_t n_items = *p.item_count;
    unsigned long long lap[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tl = clock64();

    if (warp == 0) {
        // ============ TMA producer + tile scheduler (whole warp converged, one lane issues) ============
        // It also stages the |x|^2 strip of every row tile (masked rows / rows past the list end
        // = +inf) in a shared-memory ring, so the epilogue never waits on a global load.  Slot
        // reuse needs no barrier: while this warp fills tile T the MMA warp has started a tile
        // >= T - ceil(STAGES/NST) - 1, hence the epilogue has finished tile >= T - ceil(..) - 3;
        // the launcher keeps ceil(STAGES/NST) + 3 < Q1_NSLOT.
        uint32_t stage = 0, phase = 0, ss = 0, sphase = 0, tcount = 0;
        const uint64_t hint_first = 0x12F0000000000000ull;
        const uint64_t hint_normal = 0x1000000000000000ull;
        const uint32_t ring_base = smem_u32(ring);
        while (true) {
            Q1_LAP(3);
            mbar_wait(bar_sempty + 8 * ss, sphase ^ 1);
            uint32_t item = 0;
            if (lane == 0) {
                item = atomicAdd(p.work_counter, 1u);
                if (item >= n_items) item = ITEM_END;
                sched_s[ss] = item;
                mbar_arrive(bar_sfull + 8 * ss);
            }
            item = __shfl_sync(0xffffffffu, item, 0);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            lap[6] += 1;
            Q1_LAP(1);
            const uint64_t hint = (!it.identity && it.slot > 1) ? hint_normal : hint_first;
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += Q1_N) {
                float xnv[2];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t pos = rt + h * 32 + lane;
                    float xn = __uint_as_float(F32_INF_BITS);
                    if (pos < it.row_end) {
                        bool live = true;
                        if (p.tomb || p.filt) {
                            const uint32_t id = p.ids[pos];
                            if (p.tomb && bit_test(p.tomb, p.tomb_bits, id)) live = false;
                            else if (p.filt && !bit_test(p.filt, p.filt_bits, id)) live = false;
                        }
                        if (live) xn = __ldg(p.xnorm + pos);
                    }
                    xnv[h] = xn;
                }
                __syncwarp();
                lap[7] += 1;
                for (uint32_t st = 0; st < NST; ++st) {
                    Q1_LAP(3);
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    Q1_LAP(2);
                    if (elect_one()) {
                        const uint32_t fb = bar_full + 8 * stage;
                        const uint32_t dst = ring_base + stage * STAGE_BYTES;
                        if (p.debug & 4u) {
                            mbar_arrive(fb);
                        } else {
                            mbar_expect_tx(fb, STAGE_BYTES);
                            for (uint32_t j = 0; j < KBS; ++j)
                                tma_load_2d(dst + j * Q1_STAGE_BYTES, &tmap, fb, (int)((st * KBS + j) * TC_KB_FLOATS),
                                            (int)rt, hint);
                        }
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                {
                    const uint32_t slot = tcount & (Q1_NSLOT - 1);
                    xn_ring[slot * Q1_N + lane] = xnv[0];
                    xn_ring[slot * Q1_N + 32 + lane] = xnv[1];
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_nfull + 8 * slot);
                    ++tcount;
                }
            }
        }
        Q1_LAP_DUMP(0);
    } else if (warp == 1) {
        // ============ MMA issuer (whole warp converged, one elected lane issues) ============
        uint32_t stage = 0, phase = 0, buf = 0, qphase = 0, ss = 0, sphase = 0, tph0 = 0, tph1 = 0;
        const uint32_t ring_base = smem_u32(ring);
        const uint32_t idesc = umma_idesc_tf32(Q1_M, (p.debug >> 8) ? (p.debug >> 8) : Q1_N);  // debug: MMA N override
        while (true) {
            Q1_LAP(4);
            mbar_wait(bar_sfull + 8 * ss, sphase);
            const uint32_t item = sched_s[ss];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sempty + 8 * ss);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            Q1_LAP(4);
            mbar_wait(bar_qready, qphase);
            qphase ^= 1;
            tc_fence_after();
            Q1_LAP(1);
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += Q1_N) {
                const uint32_t tph = buf ? tph1 : tph0;
                Q1_LAP(4);
                mbar_wait(bar_tempty + 8 * buf, tph ^ 1);
                tc_fence_after();
                Q1_LAP(2);
                const uint32_t d_tmem = tmem_base + Q1_ACC_COL + buf * Q1_N;
                for (uint32_t st = 0; st < NST; ++st) {
                    Q1_LAP(4);
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    Q1_LAP(3);
                    if (elect_one()) {
                        const uint32_t sbase = ring_base + stage * STAGE_BYTES;
                        if (!(p.debug & 8u)) {
                            for (uint32_t j = 0; j < KBS; ++j) {
                                const uint64_t b0 = umma_desc_sw128(sbase + j * Q1_STAGE_BYTES);
                                const uint32_t a0 = tmem_base + (st * KBS + j) * 32;
#pragma unroll
                                for (uint32_t k4 = 0; k4 < 4; ++k4) {  // A: 8 tf32 = 8 TMEM columns per step
                                    // debug bits 5/6 (timing experiments, garbage math): rotate the
                                    // accumulator per MMA to break the dependent-accumulate chain
                                    uint32_t d = d_tmem;
                                    if (p.debug & 32u) d = tmem_base + Q1_ACC_COL + (k4 & 1u) * 64u;
                                    if (p.debug & 64u) d = tmem_base + Q1_ACC_COL + k4 * 32u;
                                    umma_tf32_ts(d, a0 + k4 * 8, b0 + 2 * k4, idesc, (st | j | k4) != 0 ? 1u : 0u);
                                }
                            }
                        }
                        umma_commit(bar_empty + 8 * stage);
                        if (st + 1 == NST) umma_commit(bar_tfull + 8 * buf);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (buf) tph1 ^= 1; else tph0 ^= 1;
                buf ^= 1;
            }
        }
        Q1_LAP_DUMP(1);
    } else {
        // ================= epilogue: one thread = one query =================
        const int quarter = warp & 3;                 // TMEM lane quarter of this warp
        const uint32_t qslot_in_item = (uint32_t)lane * 4 + quarter;  // item query index held by this thread
        const uint32_t lane_taddr = (uint32_t)(quarter * 32) << 16;
        const uint32_t D = p.D;
        uint32_t buf = 0, ss = 0, sphase = 0, fph0 = 0, fph1 = 0, tcount = 0;
        // prologue transposition buffers of this warp
        float* xp0 = xpose + quarter * 32 * Q1_XP_LD;
        float* xp1 = xpose + (Q1_M + quarter * 32) * Q1_XP_LD;

        while (true) {
            Q1_LAP(4);
            mbar_wait(bar_sfull + 8 * ss, sphase);
            const uint32_t item = sched_s[ss];
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_sempty + 8 * ss);
            if (++ss == TC_SCHED) { ss = 0; sphase ^= 1; }
            Q1_LAP(0);
            if (item == ITEM_END) break;
            const ScanItem it = p.items[item];
            if (it.pair_count == 0 || it.row_begin >= it.row_end) continue;
            // ---- item prologue: the warp's 32 queries -> tensor memory ----
            // Rows are read coalesced (8 lanes x 16 B = one 128-byte k-block of one query, four
            // queries per load instruction), transposed through shared memory, and written by the
            // owning thread (TMEM lane = query) with one 32-column tcgen05.st per k-block.
            const bool have = qslot_in_item < it.pair_count;
            uint32_t qi = ID_NONE;
            float qn = 0.f;
            if (have) {
                qi = it.identity ? it.pair_begin + qslot_in_item : p.pair_q[it.pair_begin + qslot_in_item];
                qn = p.qnorm[qi];
            }
            {
                const float4* src[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t qs = __shfl_sync(0xffffffffu, qi, 4 * i + (lane >> 3));
                    src[i] = (qs == ID_NONE) ? nullptr : reinterpret_cast<const float4*>(p.Q + (size_t)qs * D) + (lane & 7);
                }
                auto ldq = [&](uint32_t kb, float4 (&v)[8]) {
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        v[i] = src[i] ? __ldg(src[i] + kb * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
                };
                float4 c0[8], c1[8], c2[8];
                ldq(0, c0);
                if (KB > 1) ldq(1, c1);
                for (uint32_t kb = 0; kb < KB; ++kb) {
                    if (kb + 2 < KB) ldq(kb + 2, c2);
                    float* xp = (kb & 1) ? xp1 : xp0;
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        *reinterpret_cast<float4*>(xp + (4 * i + (lane >> 3)) * Q1_XP_LD + (lane & 7) * 4) = c0[i];
                    __syncwarp();
                    uint32_t r[32];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float4 v = *reinterpret_cast<const float4*>(xp + lane * Q1_XP_LD + i * 4);
                        r[4 * i + 0] = __float_as_uint(v.x); r[4 * i + 1] = __float_as_uint(v.y);
                        r[4 * i + 2] = __float_as_uint(v.z); r[4 * i + 3] = __float_as_uint(v.w);
                    }
                    tmem_st32(tmem_base + lane_taddr + kb * 32, r);
#pragma unroll
                    for (int i = 0; i < 8; ++i) { c0[i] = c1[i]; c1[i] = c2[i]; }
                }
                tmem_st_wait();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_qready);
            Q1_LAP(1);

            // ---- row tiles ----
            for (uint32_t rt = it.row_begin; rt < it.row_end; rt += Q1_N) {
                const uint32_t slot = tcount & (Q1_NSLOT - 1);
                Q1_LAP(3);
                mbar_wait(bar_nfull + 8 * slot, (tcount / Q1_NSLOT) & 1u);
                const float* xs = xn_ring + slot * Q1_N;
                ++tcount;
                Q1_LAP(5);
                const uint32_t fph = buf ? fph1 : fph0;
                mbar_wait(bar_tfull + 8 * buf, fph);
                if (buf) fph1 ^= 1; else fph0 ^= 1;
                tc_fence_after();
                Q1_LAP(2);
                const uint32_t taddr = tmem_base + Q1_ACC_COL + buf * Q1_N + lane_taddr;
                for (uint32_t c0 = 0; c0 < ((p.debug & 1u) ? 0u : (uint32_t)Q1_N); c0 += 16) {
                    uint32_t acc[16];
                    tmem_ld16(taddr + c0, acc);
                    float xn[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 t4 = *reinterpret_cast<const float4*>(xs + c0 + 4 * j4);
                        xn[4 * j4 + 0] = t4.x; xn[4 * j4 + 1] = t4.y; xn[4 * j4 + 2] = t4.z; xn[4 * j4 + 3] = t4.w;
                    }
                    tmem_ld_wait();
                    // keep every approximate distance (rows = centroids)
                    if (have) {
                        float* dst = p.dense_out + (size_t)qi * p.dense_ld + (rt - it.row_begin + it.slot) + c0;
#pragma unroll
                        for (int j4 = 0; j4 < 4; ++j4) {
                            float4 o;
                            o.x = fmaf(-2.0f, __uint_as_float(acc[4 * j4 + 0]), xn[4 * j4 + 0]) + qn;
                            o.y = fmaf(-2.0f, __uint_as_float(acc[4 * j4 + 1]), xn[4 * j4 + 1]) + qn;
                            o.z = fmaf(-2.0f, __uint_as_float(acc[4 * j4 + 2]), xn[4 * j4 + 2]) + qn;
                            o.w = fmaf(-2.0f, __uint_as_float(acc[4 * j4 + 3]), xn[4 * j4 + 3]) + qn;
                            *reinterpret_cast<float4*>(dst + 4 * j4) = o;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty + 8 * buf);
                buf ^= 1;
            }
            Q1_LAP(6);
        }
        if (warp == 2) Q1_LAP_DUMP(2);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                     "r"((uint32_t)Q1_TMEM_COLS)
                     : "memory");
    }
}

size_t tc_scan_q_smem_bytes(uint32_t stages, uint32_t kbs) {
    return (size_t)stages * kbs * Q1_STAGE_BYTES + (size_t)2 * Q1_M * Q1_XP_LD * 4 + (size_t)Q1_NSLOT * Q1_N * 4 +
           (size_t)(2 * stages + 5 + 2 * TC_SCHED + Q1_NSLOT) * 8 + 16 + (size_t)TC_SCHED * 4;
}

// deepest ring that fits shared memory and keeps the norm-strip ring ahead of the epilogue
// (ceil(stages / stages-per-tile) + 3 < Q1_NSLOT, see the producer)
uint32_t q1_pick_stages(uint32_t KB, uint32_t kbs) {
    const uint32_t nst = KB / kbs;
    uint32_t stages = std::min<uint32_t>(18u, (uint32_t)(Q1_NSLOT - 4) * nst);
    while (stages > 2 && tc_scan_q_smem_bytes(stages, kbs) + 1024 > 232448) --stages;
    return stages;
}


#include "tc_scan_wide.cuh"

// ---- small support kernels ----------------------------------------------------------------------
// optional riders of the query-norm pass: fill[r] = fill_value (the per-query bound reset) and the
// NaN flag of the batch (a sum of squares is NaN exactly when an element is: no subtraction, and
// inf * inf = inf)
__global__ void row_norms_kernel(const float* __restrict__ x, uint64_t n, uint32_t D, float* __restrict__ out,
                                 uint32_t* __restrict__ max_bits, uint32_t* __restrict__ fill = nullptr,
                                 uint32_t fill_value = 0, int* __restrict__ nan_flag = nullptr) {
    const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const uint64_t nw = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    float mx = 0.f;
    for (uint64_t r = w; r < n; r += nw) {
        const float4* row = reinterpret_cast<const float4*>(x + (size_t)r * D);
        float s = 0.f;
        for (uint32_t c = lane; c < D / 4; c += 32) {
            const float4 v = __ldg(row + c);
            s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            out[r] = s;
            if (fill) fill[r] = fill_value;
            if (nan_flag && isnan(s)) *nan_flag = 1;
        }
        mx = fmaxf(mx, s);
    }
    if (max_bits && lane == 0 && mx > 0.f) atomicMax(max_bits, __float_as_uint(mx));
}

__global__ void fill_u32_kernel(uint32_t* __restrict__ p, uint64_t n, uint32_t v) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

// ---- row gather for the exact re-rank steps ------------------------------------------------------
// Each lane computes the exact distance of ITS OWN row (one candidate per lane), but the rows are
// fetched by the warp together.  A lane walking its own row makes every load instruction touch 32
// different cache lines, and the L1 tag stage (one line per cycle per SM) then bounds the kernel
// (ncu: 6.5 M sector requests, 47 us for 100 MB of centroid rows that sit in L2).  Here eight lanes
// fetch the 128-byte segment of one row (four lines per instruction) with cp.async into shared
// memory, up to GATHER_STAGES segments per row in flight and no registers held; 16-byte chunk c of
// row r sits at (c ^ (r & 7)), so both the cooperative writes and the lane-private reads are
// conflict-free.  The accumulation is the strictly sequential f32 chain of euclidean_distance_scalar
// (src/core/vector_ops.rs:51-57): same bits as exact_l2_lane.  All 32 lanes must call (row may be null).
constexpr int GATHER_STAGES_ROWS = 6;      // re-rank: rows come from HBM
constexpr int GATHER_STAGES_CENT = 4;      // coarse step: centroids come from L2
__host__ __device__ constexpr int gather_warp_bytes(int stages) { return stages * 32 * 128; }
// METRIC_DOT / METRIC_COS: the same walk with dot_product_scalar's arithmetic (x * y summed, sequential, no
// FMA, src/core/vector_ops.rs:35-37); for the cosine the row's own dot(x, x) is accumulated alongside and
// cosine_similarity_scalar's quotient is formed at the end from the caller's dot(q, q) (:39-49).
template <int GATHER_STAGES, int METRIC = METRIC_L2>
__device__ __forceinline__ float exact_l2_lane_gather(const float* __restrict__ q_s, const float* __restrict__ row,
                                                      uint32_t KB, uint32_t warp_stage_base, int lane, float qq = 0.0f) {
    // instruction j of a stage: this lane fetches chunk (lane & 7) of the row owned by lane 4 j + lane / 8
    const char* src[8];
    uint32_t dst[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int r = 4 * j + (lane >> 3);
        const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)row, r);
        src[j] = rp ? reinterpret_cast<const char*>((uintptr_t)rp) + (lane & 7) * 16 : nullptr;
        dst[j] = warp_stage_base + (uint32_t)r * 128u + ((uint32_t)((lane & 7) ^ (r & 7)) << 4);
    }
    auto issue = [&](uint32_t kb) {
        if (kb < KB) {
            const uint32_t so = (kb % GATHER_STAGES) * 4096u;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (src[j])
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst[j] + so), "l"(src[j] + (size_t)kb * 128) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
#pragma unroll
    for (uint32_t s2 = 0; s2 + 1 < GATHER_STAGES; ++s2) issue(s2);
    const float4* q4 = reinterpret_cast<const float4*>(q_s);
    const uint32_t mine = warp_stage_base + (uint32_t)lane * 128u;
    const uint32_t sw = (uint32_t)lane & 7u;
    float acc = 0.0f, xx = 0.0f;
    for (uint32_t kb = 0; kb < KB; ++kb) {
        issue(kb + GATHER_STAGES - 1);
        asm volatile("cp.async.wait_group %0;" ::"n"(GATHER_STAGES - 1) : "memory");
        __syncwarp();   // the segment of this lane's row was copied by eight other lanes
        if (row) {
            const uint32_t st = mine + (kb % GATHER_STAGES) * 4096u;
#pragma unroll
            for (uint32_t j = 0; j < 8; ++j) {
                float4 x;
                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                             : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                             : "r"(st + ((j ^ sw) << 4)));
                const float4 qv = q4[kb * 8 + j];
                if (METRIC == METRIC_L2) {
                    float t;
                    t = __fsub_rn(qv.x, x.x); acc = __fadd_rn(acc, __fmul_rn(t, t));
                    t = __fsub_rn(qv.y, x.y); acc = __fadd_rn(acc, __fmul_rn(t, t));
                    t = __fsub_rn(qv.z, x.z); acc = __fadd_rn(acc, __fmul_rn(t, t));
                    t = __fsub_rn(qv.w, x.w); acc = __fadd_rn(acc, __fmul_rn(t, t));
                } else {
                    acc = __fadd_rn(acc, __fmul_rn(qv.x, x.x)); acc = __fadd_rn(acc, __fmul_rn(qv.y, x.y));
                    acc = __fadd_rn(acc, __fmul_rn(qv.z, x.z)); acc = __fadd_rn(acc, __fmul_rn(qv.w, x.w));
                    if (METRIC == METRIC_COS) {
                        xx = __fadd_rn(xx, __fmul_rn(x.x, x.x)); xx = __fadd_rn(xx, __fmul_rn(x.y, x.y));
                        xx = __fadd_rn(xx, __fmul_rn(x.z, x.z)); xx = __fadd_rn(xx, __fmul_rn(x.w, x.w));
                    }
                }
            }
        }
        __syncwarp();   // the stage may be overwritten by the next iteration's copies
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if (METRIC == METRIC_L2) return __fsqrt_rn(acc);
    if (METRIC == METRIC_DOT) return acc;
    const float na = __fsqrt_rn(qq), nb = __fsqrt_rn(xx);
    return (na == 0.0f || nb == 0.0f) ? 0.0f : __fdiv_rn(acc, __fmul_rn(na, nb));
}

// Bound on |approximate d2 - exact d2| for a D-dimensional pair (DESIGN §3.1): qn = |q|, xmax = the largest |x|
// of the row set, a = the approximate d2.  The absolute term covers the TF32 operands (2^-10 relative each, 2^-8
// |q| |x| on 2 x.q) and the fp32 sums of D terms on the tensor cores and in the norms (2 D 2^-24 |q| |x|, within
// the 5 % margin up to D = 1638); the relative term covers the reference's sequential fp32 sum of D squared
// differences ((D + 2) 2^-24 relative, rounded up to D + 4).  For D <= 512 both are the constants
// 1.05 * 2^-8 and 3.1e-5, so the proofs of those shapes are unchanged bit for bit.
__device__ __forceinline__ float tc_proof_eps(uint32_t D, float qn, float xmax, float a) {
    const float c_abs = fmaxf(1.05f * 0.00390625f, 0.00390625f + (float)(2u * D) * 0x1p-24f);
    const float c_rel = fmaxf(3.1e-5f, (float)(D + 4u) * 0x1p-24f);
    return c_abs * qn * xmax + c_rel * a + 1e-30f;
}

// Exact re-rank + proof.  One warp per query, lane = shortlist entry.  Distances are recomputed
// as euclidean_distance_scalar does (sequential f32, (q - x)^2, no FMA, sqrt), so the returned
// keys are bit-identical to the exact path.  Proof: every row outside the shortlist has
// approx d2 >= a_last (the largest approx d2 kept), hence exact d2 >= a_last - eps, where eps
// bounds |approx - exact| for TF32 operands (2^-10 relative each) — if that is above the exact
// k-th d2 the shortlist provably contains the exact top-k.
// METRIC_COS / METRIC_DOT (flat tier of a similarity handle): the shortlist keys are the non-negative images
// kernel W builds (1 - cosine, B - dot); the candidates are re-scored with the scalar kernels' arithmetic,
// keyed by sim_to_key32 (descending similarity, ties to the lower id), and the proof compares in the
// approximate key's units: dot products of TF32 operands are off by at most ~2^-9 |q| |x|.
template <int METRIC = METRIC_L2>
__global__ void __launch_bounds__(128) rerank_kernel(const uint64_t* __restrict__ shortlist,  // [nq][KP]
                                                     const float* __restrict__ rows, const uint32_t* __restrict__ ids,
                                                     const float* __restrict__ Q, const float* __restrict__ qnorm,
                                                     const uint32_t* __restrict__ xmax_bits, uint32_t nq, uint32_t D,
                                                     uint32_t k, uint32_t R, float xmax_floor_sq, uint64_t* __restrict__ out_keys,
                                                     uint32_t* __restrict__ fb_count, uint32_t* __restrict__ fb_idx,
                                                     uint32_t* __restrict__ fin_ids = nullptr, float* __restrict__ fin_dist = nullptr,
                                                     uint32_t* __restrict__ fin_count = nullptr, uint32_t skip_separated = 0) {
    // R = shortlist entries that are re-ranked (TC_KP for search; a handful for nearest-centroid
    // assignment, where entry R — the best approximate value NOT re-ranked — is the proof bound)
    constexpr int GWB = gather_warp_bytes(GATHER_STAGES_ROWS);
    extern __shared__ __align__(128) unsigned char rr_sm[];  // [4] gather stages, then [4][D] queries
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t q = blockIdx.x * 4 + w;
    if (q >= nq) return;
    const uint64_t akey = shortlist[(size_t)q * TC_KP + lane];
    if (skip_separated && METRIC == METRIC_L2) {
        // nearest-centroid assignment where only the ARGMIN is wanted (k = 1, no distance): when the two best
        // approximate values are further apart than twice the TF32 bound, the best one is the exact argmin — no
        // row is fetched.  (Exact ties, e.g. duplicate centroids, are never separated: they take the exact path
        // and its lowest-id rule.)  The distance word of the key is then the approximate one.
        const uint64_t k0 = shfl64(akey, 0), k1 = shfl64(akey, 1);
        if (k0 != KEY_NONE) {
            const float a0 = __uint_as_float((uint32_t)(k0 >> 32));
            const float a1 = k1 != KEY_NONE ? __uint_as_float((uint32_t)(k1 >> 32)) : __uint_as_float(0x7f800000u);
            const float xmax = sqrtf(fmaxf(__uint_as_float(*xmax_bits), xmax_floor_sq));
            const float eps = tc_proof_eps(D, sqrtf(qnorm[q]), xmax, a1);
            if (a1 - a0 > 2.02f * eps) {
                const uint32_t pos0 = (uint32_t)k0;
                if (lane == 0) out_keys[(size_t)q * k] = make_key(sqrtf(a0), ids ? ids[pos0] : pos0);
                return;
            }
        }
    }
    float* q_s = reinterpret_cast<float*>(rr_sm + 4 * GWB) + (size_t)w * D;
    for (uint32_t d = lane; d < D; d += 32) q_s[d] = __ldg(Q + (size_t)q * D + d);
    __syncwarp();
    const bool have = akey != KEY_NONE && (uint32_t)lane < R;
    const uint32_t pos = have ? (uint32_t)akey : 0u;
    float qq = 0.0f;
    if (METRIC == METRIC_COS)      // dot(q, q) in the scalar kernel's order (every lane the same chain)
        for (uint32_t d = 0; d < D; ++d) qq = __fadd_rn(qq, __fmul_rn(q_s[d], q_s[d]));
    const float dist = exact_l2_lane_gather<GATHER_STAGES_ROWS, METRIC>(q_s, have ? rows + (size_t)pos * D : nullptr, D / 32,
                                                                        smem_u32(rr_sm) + (uint32_t)w * GWB, lane, qq);
    uint64_t ekey = KEY_NONE;
    if (have) ekey = METRIC == METRIC_L2 ? make_key(dist, ids ? ids[pos] : pos)
                                         : (((uint64_t)sim_to_key32(dist) << 32) | (ids ? ids[pos] : pos));
    ekey = warp_sort32(ekey, lane);
    if ((uint32_t)lane < k) out_keys[(size_t)q * k + lane] = ekey;
    if (fin_ids) {
        // the caller-facing arrays as finalize_kernel writes them when this tier is the only one
        if ((uint32_t)lane < k) {
            fin_ids[(size_t)q * k + lane] = ekey != KEY_NONE ? key_id(ekey) : ID_NONE;
            fin_dist[(size_t)q * k + lane] = ekey != KEY_NONE ? key_value(ekey, METRIC)
                                                              : __uint_as_float(METRIC == METRIC_L2 ? 0x7f800000u : 0xff800000u);
        }
        const uint32_t found = __popc(__ballot_sync(0xffffffffu, ekey != KEY_NONE && (uint32_t)lane < k));
        if (lane == 0) fin_count[q] = found;
    }
    // proof
    const uint64_t a_last_key = shfl64(akey, (int)min(R, 31u));
    const uint64_t kth = shfl64(ekey, (int)k - 1);
    if (lane == 0 && a_last_key != KEY_NONE) {
        const float a_last = __uint_as_float((uint32_t)(a_last_key >> 32));
        // xmax_floor_sq: list-sharded search with shared bounds — a row of THIS shard may have been
        // dropped by a bound a peer published, so every shard has to use the same (largest) norm term
        const float xmax = sqrtf(fmaxf(__uint_as_float(*xmax_bits), xmax_floor_sq));
        const float eps = tc_proof_eps(D, sqrtf(qnorm[q]), xmax, a_last);
        bool ok = false;
        if (kth != KEY_NONE) {
            if (METRIC == METRIC_L2) {
                const float dk = key_dist(kth);
                ok = (a_last - eps) > dk * dk * 1.000001f;
            } else {
                // the exact k-th similarity in the approximate key's units (see kernel W)
                const float sk = key32_to_sim((uint32_t)(kth >> 32));
                const float qn = sqrtf(qnorm[q]);
                const float scale = METRIC == METRIC_COS ? 1.0f : qn * xmax;
                const float ek = METRIC == METRIC_COS ? 1.0f - sk : 1.02f * qn * xmax - sk;
                const float eps_s = (1.05f * 0.001953125f + 1.0e-4f) * scale + 1e-30f;
                ok = (a_last - eps_s) > ek && (METRIC != METRIC_COS || qn > 0.0f);
            }
        }
        if (!ok) fb_idx[atomicAdd(fb_count, 1u)] = q;
    } else if (METRIC == METRIC_COS && lane == 0 && qnorm[q] == 0.0f) {
        fb_idx[atomicAdd(fb_count, 1u)] = q;   // a zero query passes nothing in the scan: the exact path scores it
    }
}


// ---- tensor-core coarse step (src/ivf/core.rs:646-656) ---------------------------------------
// 1. kernel Q in dense mode writes approx d2(query, centroid) for every pair   [nq][ld]
// 2. coarse_select_kernel: per query, the KC = nprobe + 8 approximately nearest centroids are
//    extracted, their distances recomputed exactly (reference operation order), sorted by
//    (distance, list id) and the first nprobe kept.  Proof: the next approximate value minus the
//    TF32 error bound must exceed the exact nprobe-th distance^2, else the query is handed to the
//    exact path (fallback list).

// identity work items for the dense pass: (query group of 128) x (row chunk); `slot` carries the
// row offset of the chunk so the kernel addresses the dense matrix with absolute centroid ids
__global__ void coarse_items_kernel(ScanItem* items, uint32_t nq, uint32_t nlist, uint32_t chunk_rows,
                                    uint32_t n_chunks, uint32_t* n_items) {
    const uint32_t n_qg = (nq + Q1_M - 1) / Q1_M;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_items = n_qg * n_chunks;
    if (i >= n_qg * n_chunks) return;
    const uint32_t g = i / n_chunks, c = i % n_chunks;
    ScanItem it;
    it.row_begin = c * chunk_rows;
    it.row_end = min(nlist, (c + 1) * chunk_rows);
    it.pair_begin = g * Q1_M;
    it.pair_count = min((uint32_t)Q1_M, nq - g * Q1_M);
    it.slot = it.row_begin;
    it.identity = 1;
    it.sub = 0;
    if (it.row_begin >= it.row_end) it.pair_count = 0;
    items[i] = it;
}

// identity work items of the flat-tier scan: (query group of tile_q) x (row chunk); `slot` = chunk
// index = the partial slot the item's shortlists are published to
__global__ void flat_items_kernel(ScanItem* items, uint32_t nq, uint32_t n_rows, uint32_t chunk_rows,
                                  uint32_t n_chunks, uint32_t* n_items, uint32_t tile_q) {
    const uint32_t n_qg = (nq + tile_q - 1) / tile_q;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_items = n_qg * n_chunks;
    if (i >= n_qg * n_chunks) return;
    // chunk-major order: the query groups of one chunk are adjacent, so its re-reads hit L2
    const uint32_t c = i / n_qg, g = i % n_qg;
    ScanItem it;
    it.row_begin = c * chunk_rows;
    it.row_end = min(n_rows, (c + 1) * chunk_rows);
    it.pair_begin = g * tile_q;
    it.pair_count = min(tile_q, nq - g * tile_q);
    it.slot = c;
    it.identity = n_qg > 1 ? 2 : 1;   // 2: the chunk is read by several query groups (keep it in L2)
    it.sub = 0;
    if (it.row_begin >= it.row_end) it.pair_count = 0;
    items[i] = it;
}

// One block (four warps) per query: at 1024 queries one warp per query leaves fewer than two warps per
// scheduler and the kernel runs at the latency of its ~10K dependent instructions (ncu: 8.5 cycles
// per issued instruction, 47 us).
template <int T>   // approximate values kept per thread
__global__ void __launch_bounds__(128) coarse_select_kernel(const float* __restrict__ dense, uint32_t ld,
                                                            const float* __restrict__ centroids,
                                                            const float* __restrict__ Q, const float* __restrict__ qnorm,
                                                            const uint32_t* __restrict__ cmax_bits, uint32_t nq,
                                                            uint32_t nlist, uint32_t D, uint32_t np, uint32_t KC,
                                                            uint64_t* __restrict__ out_keys,
                                                            uint32_t* __restrict__ fb_count, uint32_t* __restrict__ fb_idx) {
    constexpr int GWB = gather_warp_bytes(GATHER_STAGES_CENT);
    // [nw] gather stages (nw = warps that hold candidates), [D] query, [128] candidate ids, [32] scratch, [128] keys
    extern __shared__ __align__(128) unsigned char cs_sm[];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const uint32_t q = blockIdx.x;
    const uint32_t nw = (KC + 31) / 32;
    float* q_s = reinterpret_cast<float*>(cs_sm + (size_t)nw * GWB);
    uint32_t* cand_s = reinterpret_cast<uint32_t*>(q_s + D);
    uint32_t* red_s = cand_s + 128;
    uint64_t* key_s = reinterpret_cast<uint64_t*>(red_s + 32);
    for (uint32_t d = tid; d < D; d += 128) q_s[d] = __ldg(Q + (size_t)q * D + d);
    // thread-local sorted top-T of this thread's strided share: (approx d2 bits, list id) pairs; the
    // approximate distances are fetched eight per thread at a time BEFORE the insertions
    uint32_t ld2[T], lid[T];
#pragma unroll
    for (int i = 0; i < T; ++i) { ld2[i] = 0xFFFFFFFFu; lid[i] = 0xFFFFFFFFu; }
    const float* row = dense + (size_t)q * ld;
    for (uint32_t base = 0; base < nlist; base += 1024) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t c = base + (uint32_t)i * 128u + (uint32_t)tid;
            v[i] = (c < nlist) ? __ldg(row + c) : 0.0f;
        }
#pragma unroll
        for (int i2 = 0; i2 < 8; ++i2) {
            const uint32_t c = base + (uint32_t)i2 * 128u + (uint32_t)tid;
            uint32_t kd = __float_as_uint(fmaxf(v[i2], 0.0f)), ki = c;
            if (c < nlist && kd < ld2[T - 1]) {  // ids ascend within a thread, so equal d2 keeps the earlier (lower) id first
#pragma unroll
                for (int i = 0; i < T; ++i) {
                    const bool sw = kd < ld2[i];
                    const uint32_t td = sw ? ld2[i] : kd, ti = sw ? lid[i] : ki;
                    ld2[i] = sw ? kd : ld2[i];
                    lid[i] = sw ? ki : lid[i];
                    kd = td; ki = ti;
                }
            }
        }
    }
    // block-wide sum of one value per thread (scratch slots double-buffered, alternating from call to
    // call: one barrier per call)
    uint32_t sum_par = 0, excl_par = 0;
    auto block_sum = [&](uint32_t x) -> uint32_t {
        const uint32_t par = (sum_par ^= 1u);
        const uint32_t ws = __reduce_add_sync(0xffffffffu, x);
        if (lane == 0) red_s[par * 4 + w] = ws;
        __syncthreads();
        return red_s[par * 4] + red_s[par * 4 + 1] + red_s[par * 4 + 2] + red_s[par * 4 + 3];
    };
    // block-wide exclusive prefix (slots 8..15, one barrier per call)
    auto block_excl = [&](uint32_t x) -> uint32_t {
        const uint32_t par = (excl_par ^= 1u);
        uint32_t inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += up;
        }
        if (lane == 31) red_s[8 + par * 4 + w] = inc;
        __syncthreads();
        uint32_t before = 0;
        for (int i = 0; i < w; ++i) before += red_s[8 + par * 4 + i];
        return before + inc - x;
    };
    // the KC smallest over the block: bitwise search for the KC-th smallest d2 value t (the largest t with
    // fewer than KC entries below it); every entry below t plus as many entries equal to t as are still
    // needed (in thread order) are the candidates
    uint32_t n_valid = 0;
#pragma unroll
    for (int i = 0; i < T; ++i) n_valid += (ld2[i] != 0xFFFFFFFFu) ? 1u : 0u;
    uint32_t KCe = min(KC, block_sum(n_valid));
    uint32_t t = 0;
    for (int bit = 31; bit >= 0; --bit) {
        const uint32_t tc = t | (1u << bit);
        uint32_t below = 0;
#pragma unroll
        for (int i = 0; i < T; ++i) below += (ld2[i] < tc) ? 1u : 0u;
        if (block_sum(below) < KCe) t = tc;
    }
    uint32_t n_lt = 0, n_eq = 0;
#pragma unroll
    for (int i = 0; i < T; ++i) { n_lt += (ld2[i] < t) ? 1u : 0u; n_eq += (ld2[i] == t) ? 1u : 0u; }
    const uint32_t need_eq = KCe - block_sum(n_lt);
    const uint32_t eq_before = block_excl(n_eq);
    const uint32_t sel = n_lt + min(n_eq, need_eq > eq_before ? need_eq - eq_before : 0u);
    const uint32_t off = block_excl(sel);
    uint32_t my_next = 0xFFFFFFFFu;   // smallest approximate value this thread did NOT hand in
#pragma unroll
    for (int i = 0; i < T; ++i) {
        if ((uint32_t)i < sel) cand_s[off + i] = lid[i];
        if ((uint32_t)i == sel) my_next = ld2[i];
    }
    {
        const uint32_t wm = __reduce_min_sync(0xffffffffu, my_next);
        if (lane == 0) red_s[16 + w] = wm;
    }
    // a thread whose T local entries were all consumed may have dropped keys below next_d2
    bool uncertain = __syncthreads_or((sel == (uint32_t)T && nlist > (uint32_t)T * 128u) ? 1 : 0) != 0;
    uint32_t next_d2 = min(min(red_s[16], red_s[17]), min(red_s[18], red_s[19]));
    if (uncertain) {
        // Rare (centroids that are near-duplicates of one another AND share a residue mod 128 — e.g.
        // a k-means initialised from clumped seeds): select again straight from the dense row, without
        // the thread-local lists.  32 passes over the row (it sits in L2), exact for any nlist.
        KCe = min(KC, nlist);
        t = 0;
        for (int bit = 31; bit >= 0; --bit) {
            const uint32_t tc = t | (1u << bit);
            uint32_t below = 0;
            for (uint32_t c = tid; c < nlist; c += 128) below += (__float_as_uint(fmaxf(__ldg(row + c), 0.0f)) < tc) ? 1u : 0u;
            if (block_sum(below) < KCe) t = tc;
        }
        uint32_t lt = 0, eq = 0;
        for (uint32_t c = tid; c < nlist; c += 128) {
            const uint32_t b = __float_as_uint(fmaxf(__ldg(row + c), 0.0f));
            lt += (b < t) ? 1u : 0u;
            eq += (b == t) ? 1u : 0u;
        }
        const uint32_t need2 = KCe - block_sum(lt);
        const uint32_t eqb = block_excl(eq);
        uint32_t take = min(eq, need2 > eqb ? need2 - eqb : 0u);
        uint32_t o2 = block_excl(lt + take);
        uint32_t nx = 0xFFFFFFFFu;
        for (uint32_t c = tid; c < nlist; c += 128) {
            const uint32_t b = __float_as_uint(fmaxf(__ldg(row + c), 0.0f));
            bool pick = b < t;
            if (b == t && take) { pick = true; --take; }
            if (pick) cand_s[o2++] = c;
            else nx = min(nx, b);
        }
        nx = __reduce_min_sync(0xffffffffu, nx);
        if (lane == 0) red_s[20 + w] = nx;
        __syncthreads();
        next_d2 = min(min(red_s[20], red_s[21]), min(red_s[22], red_s[23]));
        uncertain = false;
    }
    // exact distances of the candidates (reference operation order): one candidate per thread
    {
        uint64_t key = KEY_NONE;
        if ((uint32_t)w < nw) {   // warp-uniform
            const bool h = (uint32_t)tid < KCe;
            const uint32_t c = h ? cand_s[tid] : 0u;
            const float d = exact_l2_lane_gather<GATHER_STAGES_CENT>(q_s, h ? centroids + (size_t)c * D : nullptr, D / 32,
                                                                     smem_u32(cs_sm) + (uint32_t)w * GWB, lane);
            if (h) key = make_key(d, c);
        }
        key_s[tid] = key;
    }
    __syncthreads();
    if (w != 0) return;
    // sort by (distance, id): four sorted 32-chunks, then merge-split passes
    uint64_t ex[4];
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
        ex[ch] = KEY_NONE;
        if ((uint32_t)ch * 32 < KC) ex[ch] = warp_sort32(key_s[ch * 32 + lane], lane);
    }
#pragma unroll
    for (int a2 = 0; a2 < 3; ++a2) {
#pragma unroll
        for (int b2 = 3; b2 > a2; --b2) {
            if ((uint32_t)b2 * 32 >= KC) continue;
            const uint64_t rev = shfl64(ex[b2], 31 - lane);
            uint64_t lo = ex[b2 - 1] < rev ? ex[b2 - 1] : rev;
            uint64_t hi = ex[b2 - 1] < rev ? rev : ex[b2 - 1];
#pragma unroll
            for (int j = 16; j > 0; j >>= 1) {
                const uint64_t ol = shfl_xor64(lo, j), oh = shfl_xor64(hi, j);
                const bool lower = (lane & j) == 0;
                lo = lower ? (lo < ol ? lo : ol) : (lo < ol ? ol : lo);
                hi = lower ? (hi < oh ? hi : oh) : (hi < oh ? oh : hi);
            }
            ex[b2 - 1] = lo;
            ex[b2] = hi;
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t o = i * 32 + lane;
        if (o < np) out_keys[(size_t)q * np + o] = ex[i];
    }
    // proof: every centroid outside the candidate set has approx d2 >= next_d2
    uint64_t kth = KEY_NONE;
#pragma unroll
    for (int i = 0; i < 4; ++i) if ((int)((np - 1) >> 5) == i) kth = shfl64(ex[i], (int)((np - 1) & 31));
    if (lane == 0) {
        bool ok = true;
        if (uncertain) ok = false;
        else if (next_d2 != 0xFFFFFFFFu) {
            const float a_next = __uint_as_float(next_d2);
            const float cmax = sqrtf(__uint_as_float(*cmax_bits));
            const float eps = tc_proof_eps(D, sqrtf(qnorm[q]), cmax, a_next);
            ok = false;
            if (kth != KEY_NONE) {
                const float dk = key_dist(kth);
                ok = (a_next - eps) > dk * dk * 1.000001f;
            }
        }
#ifdef FVDB_CS_DEBUG
        if (!ok) printf("coarse_select q %u uncertain %d next_d2 %08x (%f) kth %f KCe %u t %08x\n", q, (int)uncertain, next_d2,
                        __uint_as_float(next_d2), kth != KEY_NONE ? key_dist(kth) * key_dist(kth) : -1.f, KCe, t);
#endif
        if (!ok) fb_idx[atomicAdd(fb_count, 1u)] = q;
    }
}

// Shortlist merge after the scan: P rows of TC_KP approx keys per query (one per probed list), each
// either empty, sorted (a list that was merged during the scan) or unsorted (pending candidates
// published as they were).  One warp per query folds them into the query's best TC_KP.
__global__ void __launch_bounds__(128) merge_rows32_kernel(const uint64_t* __restrict__ in, uint32_t nq, uint32_t P,
                                                           uint64_t* __restrict__ out,
                                                           const uint32_t* __restrict__ row_stamp, uint32_t stamp) {
    // one block per query: warp w folds rows w, w + 4, ... (a chain of P / 4 dependent merges instead of
    // P, and four times the warps in flight), warp 0 folds the four results.
    // Only rows this launch wrote count (the others hold whatever an earlier batch left there).  The stamps of
    // 32 candidate rows are read by the 32 lanes at once and turned into a mask; only live rows are fetched,
    // four at a time.  On a list-sharded index 1 / world of a query's rows are live: the work follows the live
    // rows, not the nprobe x ranges slots.
    __shared__ uint64_t part[3][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t q = blockIdx.x;
    const uint64_t* base = in + (size_t)q * P * TC_KP;
    const uint32_t* st_q = row_stamp + (size_t)q * P;
    uint64_t best = KEY_NONE;
    for (uint32_t c0 = 0; c0 * 4 + (uint32_t)w < P; c0 += 32) {
        const uint32_t r_mine = (c0 + (uint32_t)lane) * 4 + (uint32_t)w;
        unsigned live = __ballot_sync(0xffffffffu, r_mine < P && __ldg(st_q + r_mine) == stamp);
        while (live) {
            uint64_t row[4];
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                row[g] = KEY_NONE;
                if (live) {
                    const uint32_t r = (c0 + (uint32_t)(__ffs((int)live) - 1)) * 4 + (uint32_t)w;
                    live &= live - 1;
                    row[g] = base[(size_t)r * TC_KP + lane];
                }
            }
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                if (__ballot_sync(0xffffffffu, row[g] != KEY_NONE) == 0) continue;
                const uint64_t up = shfl_up64(row[g], 1);
                if (__ballot_sync(0xffffffffu, lane > 0 && up > row[g])) row[g] = warp_sort32(row[g], lane);
                best = warp_merge32(best, row[g], lane);
            }
        }
    }
    if (w) part[w - 1][lane] = best;
    __syncthreads();
    if (w) return;
#pragma unroll
    for (int i = 0; i < 3; ++i) best = warp_merge32(best, part[i][lane], lane);
    out[(size_t)q * TC_KP + lane] = best;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
    return fn;
}

template <typename T>
struct Buf {
    T* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t n, size_t* bytes) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        const size_t ncap = std::max(n, cap + cap / 2);
        cudaError_t e = cudaMalloc(&p, ncap * sizeof(T));
        if (e != cudaSuccess) { cap = 0; return e; }
        if (bytes) *bytes += (ncap - cap) * sizeof(T);
        cap = ncap;
        return cudaSuccess;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace

// timing experiment only (FVDB_TC_DEBUG bit 7): per-role stopwatch laps, averaged over CTAs
static cudaError_t dump_prof(const unsigned long long* d_prof, uint32_t grid, cudaStream_t st) {
    std::vector<unsigned long long> hp((size_t)grid * 48);
    cudaError_t e = cudaMemcpyAsync(hp.data(), d_prof, hp.size() * 8, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return e;
    {
        unsigned long long t0 = ~0ull, t1 = 0;
        double dur_avg = 0, dur_max = 0, cyc_avg = 0, start_max = 0;
        for (uint32_t b = 0; b < grid; ++b) {
            const unsigned long long* r = &hp[((size_t)b * 6 + 3) * 8];
            if (r[4] == 0) continue;
            t0 = std::min(t0, r[4]); t1 = std::max(t1, r[5]);
        }
        for (uint32_t b = 0; b < grid; ++b) {
            const unsigned long long* r = &hp[((size_t)b * 6 + 3) * 8];
            if (r[4] == 0) continue;
            const double d = (double)(r[5] - r[4]);
            dur_avg += d / grid; dur_max = std::max(dur_max, d); cyc_avg += (double)r[6] / grid;
            start_max = std::max(start_max, (double)(r[4] - t0));
        }
        {
            std::vector<double> ends;
            for (uint32_t b = 0; b < grid; ++b) {
                const unsigned long long* r = &hp[((size_t)b * 6 + 3) * 8];
                if (r[4]) ends.push_back((double)(r[5] - t0) * 1e-3);
            }
            std::sort(ends.begin(), ends.end());
            if (!ends.empty()) {
                fprintf(stderr, "[tc prof] CTA end times (us), deciles:");
                for (int d = 0; d <= 10; ++d) fprintf(stderr, " %.0f", ends[std::min(ends.size() - 1, ends.size() * d / 10)]);
                fprintf(stderr, "\n");
            }
        }
        if (t1) fprintf(stderr, "[tc prof] wall: first start -> last end %.1f us; CTA duration avg %.1f max %.1f us; "
                        "latest start +%.1f us; avg cycles %.0f => %.3f GHz\n", (t1 - t0) * 1e-3, dur_avg * 1e-3,
                        dur_max * 1e-3, start_max * 1e-3, cyc_avg, cyc_avg / dur_avg);
    }
    static const char* names[5] = {"producer", "mma", "epilogue", "loader", "epistats"};
    for (int r = 0; r < 5; ++r) {
        double avg[8] = {0}, mx[8] = {0};
        for (uint32_t b = 0; b < grid; ++b)
            for (int i = 0; i < 8; ++i) {
                const double v = (double)hp[((size_t)b * 6 + r) * 8 + i];
                avg[i] += v / grid;
                mx[i] = std::max(mx[i], v);
            }
        fprintf(stderr, "[tc prof] %-8s avg:", names[r]);
        for (int i = 0; i < 8; ++i) fprintf(stderr, " %9.0f", avg[i]);
        fprintf(stderr, "  max:");
        for (int i = 0; i < 8; ++i) fprintf(stderr, " %9.0f", mx[i]);
        fprintf(stderr, "\n");
    }
    return cudaSuccess;
}

cudaError_t launch_max_sqnorm(const float* x, uint64_t n, uint32_t D, float* scratch_norms, uint32_t* max_bits,
                              cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((n * 32 + 255) / 256, (uint64_t)148 * 16);
    row_norms_kernel<<<blocks, 256, 0, stream>>>(x, n, D, scratch_norms, max_bits);
    return cudaGetLastError();
}

cudaError_t launch_fill_u32(uint32_t* p, uint64_t n, uint32_t v, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    fill_u32_kernel<<<(uint32_t)((n + 255) / 256), 256, 0, stream>>>(p, n, v);
    return cudaGetLastError();
}

cudaError_t launch_merge_rows32(const uint64_t* in, uint32_t nq, uint32_t P, uint64_t* out, cudaStream_t stream,
                                const uint32_t* row_stamp, uint32_t stamp) {
    if (nq == 0) return cudaSuccess;
    merge_rows32_kernel<<<nq, 128, 0, stream>>>(in, nq, P, out, row_stamp, stamp);
    return cudaGetLastError();
}

// A row matrix the scan kernels read, with what they need of it besides the rows: |x|^2 per row and the
// TMA descriptors.  Set s keeps its max |x|^2 (f32 bits) in misc[4 * s].
enum RowSetId : uint32_t { SET_ARENA, SET_CENTROIDS, SET_RECENT, SET_ASSIGN, N_ROW_SETS };
struct RowSet {
    Buf<float> xnorm;
    CUtensorMap tmap;      // box 32 floats x 128 rows (kernel R), or x 64 rows for the centroid table (kernel Q)
    CUtensorMap tmap_w;    // box 32 floats x W_NH rows (kernel W: each CTA of a pair streams half a tile)
    const float* rows = nullptr;
    uint64_t n = 0, version = ~0ull;
};

struct TcScratchImpl {
    Buf<float> qnorm;
    Buf<uint32_t> misc;  // [4 * s] = max |x|^2 bits of row set s
    Buf<unsigned long long> prof;
    Buf<uint32_t> list_order;  // lists by descending length (tile-scheduler order)
    Buf<uint32_t> live_ids;    // the non-empty lists, ascending (the bucketing pass walks only these)
    uint32_t n_live = 0;
    RowSet sets[N_ROW_SETS];
    Buf<ScanItem> fitems;
    uint32_t list_order_n = 0;
    uint32_t max_list_len = 0;
    Buf<uint32_t> thr_g, list_cnt, pair_off, cursor, pair_q, pair_slot, n_items;
    Buf<ScanItem> items, items_w;   // work items of kernel R / kernel W
    Buf<uint64_t> partial, shortlist;
    Buf<uint32_t> row_stamp;   // one stamp per shortlist row of `partial`
    uint32_t stamp = 0;        // launch counter; a fresh or wrapped counter clears the stamps
    // stamps for `rows` shortlist rows of the next scan launch: returns the launch's stamp
    cudaError_t next_stamp(size_t rows, size_t* dev_bytes, cudaStream_t st, uint32_t* out) {
        const size_t before = row_stamp.cap;
        cudaError_t e = row_stamp.ensure(rows, dev_bytes);
        if (e != cudaSuccess) return e;
        if (row_stamp.cap != before || stamp == 0xFFFFFFFFu) {
            e = cudaMemsetAsync(row_stamp.p, 0, row_stamp.cap * sizeof(uint32_t), st);
            if (e != cudaSuccess) return e;
            stamp = 0;
        }
        *out = ++stamp;
        return cudaSuccess;
    }
    Buf<float> dense;
    Buf<uint64_t> coarse;
    Buf<ScanItem> citems;
    uint32_t smem_attr_set_w = 0;   // bit per metric instantiation of kernel W
    bool smem_attr_set_q = false;
    uint32_t smem_attr_set_r = 0;   // bit per item width of kernel R
    bool smem_attr_set_rerank = false;
};

bool tc_supported(uint32_t D) { return D % 32 == 0 && D >= 32 && D <= TC_MAX_D; }

static size_t rerank_smem_bytes(uint32_t D) { return (size_t)4 * gather_warp_bytes(GATHER_STAGES_ROWS) + (size_t)4 * D * sizeof(float); }
static size_t coarse_select_smem_bytes(uint32_t D, uint32_t KC) {
    return (size_t)((KC + 31) / 32) * gather_warp_bytes(GATHER_STAGES_CENT) + (size_t)D * sizeof(float) + (128 + 32) * 4 + 128 * 8;
}
static cudaError_t rerank_prepare(TcScratchImpl* m) {
    if (m->smem_attr_set_rerank) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(rerank_kernel<METRIC_L2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rerank_smem_bytes(TC_MAX_D));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(rerank_kernel<METRIC_COS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rerank_smem_bytes(TC_MAX_D));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(rerank_kernel<METRIC_DOT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rerank_smem_bytes(TC_MAX_D));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(coarse_select_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coarse_select_smem_bytes(TC_MAX_D, 128));
    if (e == cudaSuccess) m->smem_attr_set_rerank = true;
    return e;
}

void tc_release(TcScratch& s) {
    if (!s.impl) return;
    TcScratchImpl* m = s.impl;
    m->qnorm.release(); m->misc.release(); m->thr_g.release(); m->list_cnt.release();
    m->pair_off.release(); m->cursor.release(); m->pair_q.release(); m->pair_slot.release(); m->n_items.release();
    m->items.release(); m->items_w.release(); m->partial.release(); m->shortlist.release(); m->row_stamp.release();
    m->prof.release(); m->list_order.release(); m->live_ids.release(); m->fitems.release();
    for (RowSet& rs : m->sets) rs.xnorm.release();
    m->dense.release(); m->coarse.release(); m->citems.release();
    delete m;
    s.impl = nullptr;
}

#define TCK(call)                                                                      \
    do {                                                                               \
        cudaError_t e__ = (call);                                                      \
        if (e__ != cudaSuccess) {                                                      \
            if (err) *err = std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #call; \
            cudaGetLastError();                                                        \
            return e__ == cudaErrorMemoryAllocation ? FVDB_ERR_OOM : FVDB_ERR_CUDA;    \
        }                                                                              \
    } while (0)

// Which scan kernel(s), as the least number of a batch's queries that puts a posting list on kernel W; 0 = kernel
// R alone.  Kernel W (query tile in tensor memory: D <= 384, on SM pairs) takes the heavily probed lists and the
// dense scans, kernel R the sparsely probed lists; above D = 384 kernel R scans alone.  Test hook, read on every
// call: FVDB_TC_KERNEL=R puts every list on kernel R, FVDB_TC_KERNEL=W every list on kernel W where it exists.
static uint32_t tc_kernel_choice(uint32_t D, int sm_count) {
    if (D > 384 || sm_count < 2) return 0;
    const char* e = getenv("FVDB_TC_KERNEL");
    if (e && e[0] == 'R') return 0;
    if (e && e[0] == 'W') return 1;
    return TC_WIDE_MIN_QUERIES;
}

// FVDB_TC_DEBUG: the scan kernels' timing-only modes and per-role stopwatch (bit 7, dump_prof), and bit 9: keep
// the previous batch's per-query bounds
static uint32_t tc_debug_bits() {
    const char* e = getenv("FVDB_TC_DEBUG");
    return e ? (uint32_t)atoi(e) : 0u;
}

static cudaError_t launch_wide(TcScratchImpl* m, const CUtensorMap& tmap, TcScanParams& p, uint32_t KB, int sm_count,
                               size_t* dev_bytes, cudaStream_t st, cudaEvent_t ev0) {
    const uint32_t kbs = wide_pick_kbs(KB);
    const uint32_t stages = wide_pick_stages(KB, kbs);
    p.kbs = kbs;
    p.stages = stages;
    const size_t smem = tc_scan_wide_smem_bytes(stages, kbs) + 1024;
    cudaError_t e;
    const bool small = p.small_list != 0 && p.metric == METRIC_L2;
    auto kern = small ? tc_scan_wide_kernel<METRIC_L2, true>
              : p.metric == METRIC_COS ? tc_scan_wide_kernel<METRIC_COS>
              : p.metric == METRIC_DOT ? tc_scan_wide_kernel<METRIC_DOT> : tc_scan_wide_kernel<METRIC_L2>;
    const uint32_t kbit = small ? 8u : (1u << p.metric);
    if (!(m->smem_attr_set_w & kbit)) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        m->smem_attr_set_w |= kbit;
    }
    uint32_t grid = (uint32_t)sm_count & ~1u;   // whole pairs; idle pairs exit at once
    if (p.scan_sms && p.scan_sms < grid) grid = p.scan_sms & ~1u;
    if (p.debug & 128u) {
        e = m->prof.ensure((size_t)grid * 48, dev_bytes);
        if (e != cudaSuccess) return e;
        e = cudaMemsetAsync(m->prof.p, 0, (size_t)grid * 48 * 8, st);
        if (e != cudaSuccess) return e;
        p.prof = m->prof.p;
    }
    if (ev0) { e = cudaEventRecord(ev0, st); if (e != cudaSuccess) return e; }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(W_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, kern, tmap, p);
    if (e != cudaSuccess) return e;
    if (p.prof) return dump_prof(m->prof.p, grid, st);
    return cudaSuccess;
}

// Kernel R at the item width of D, with the deepest ring that fits; the norm-strip window (see the producer)
// caps the ring at 6 tiles.  *smem = 0 when not even two stages fit.
static uint32_t r2_pick_stages(uint32_t D, size_t* smem) {
    const uint32_t KB = D / 32, nq = r2_tile_q(D);
    uint32_t stages = std::min<uint32_t>(12u, (uint32_t)(R2_NSLOT - 2 - R2_NBUF) * KB);
    while (stages > 2 && tc_scan_smem_bytes(KB, stages, nq) + R2_SLACK > 232448) --stages;
    *smem = tc_scan_smem_bytes(KB, stages, nq) + R2_SLACK;   // slack for the 1024-byte alignment
    if (*smem > 232448) *smem = 0;
    return stages;
}

static cudaError_t launch_r2(TcScratchImpl* m, const CUtensorMap& tmap, const TcScanParams& p, uint32_t grid, size_t smem,
                             cudaStream_t st) {
    const uint32_t nq = r2_tile_q(p.D);
    auto kern = nq == 64 ? tc_scan_kernel<64> : nq == 32 ? tc_scan_kernel<32> : tc_scan_kernel<16>;
    const uint32_t bit = nq / 16;
    if (!(m->smem_attr_set_r & bit)) {
        const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
        if (e != cudaSuccess) return e;
        m->smem_attr_set_r |= bit;
    }
    kern<<<grid, R2_THREADS, smem, st>>>(tmap, p);
    return cudaGetLastError();
}

static CUresult encode_rows_tmap(CUtensorMap* out, const float* rows, uint64_t n_rows, uint32_t D, uint32_t box_rows) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return CUDA_ERROR_NOT_SUPPORTED;
    const cuuint64_t gdim[2] = {D, n_rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)D * 4};
    const cuuint32_t box[2] = {TC_KB_FLOATS, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(rows), gdim, gstride, box, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
}

// Brings row set `id` up to date with `rows` when the caller marks it stale or the rows moved: zeroes its max word,
// launches row_norms_kernel once (|x|^2 per row and their max) and encodes its TMA descriptors.  *refreshed (when
// given) tells whether it did.
static int refresh_row_set(TcScratchImpl* m, RowSetId id, const float* rows, uint64_t n, uint32_t D, bool stale,
                           int sm_count, cudaStream_t st, size_t* dev_bytes, uint32_t* launches, std::string* err,
                           bool* refreshed = nullptr) {
    RowSet& rs = m->sets[id];
    if (refreshed) *refreshed = false;
    if (!stale && rs.rows == rows && rs.n == n) return FVDB_OK;
    uint32_t* max_bits = m->misc.p + 4 * id;
    TCK(rs.xnorm.ensure(n, dev_bytes));
    TCK(cudaMemsetAsync(max_bits, 0, 4, st));
    const uint32_t blocks = (uint32_t)std::min<uint64_t>((n * 32 + 255) / 256, (uint64_t)sm_count * 16);
    row_norms_kernel<<<blocks, 256, 0, st>>>(rows, n, D, rs.xnorm.p, max_bits);
    TCK(cudaGetLastError());
    (*launches)++;
    // kernel Q alone reads the centroid table; kernels R and W read the other sets
    CUresult r = encode_rows_tmap(&rs.tmap, rows, n, D, id == SET_CENTROIDS ? Q1_N : TC_ROWS);
    if (r == CUDA_SUCCESS && id != SET_CENTROIDS) r = encode_rows_tmap(&rs.tmap_w, rows, n, D, W_NH);
    if (r != CUDA_SUCCESS) {
        if (err) *err = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r);
        return FVDB_ERR_CUDA;
    }
    rs.rows = rows;
    rs.n = n;
    if (refreshed) *refreshed = true;
    return FVDB_OK;
}

int tc_ivf_search(TcScratch& s, const TcSearchArgs& a, cudaStream_t st, size_t* dev_bytes, uint32_t* launches,
                  std::string* err) {
    if (!s.impl) s.impl = new TcScratchImpl();
    TcScratchImpl* m = s.impl;
    const uint32_t D = a.D, KB = D / 32, nq = a.nq, np = a.nprobe;
    if (a.n_rows >= 0x7FFFFFFFull) { if (err) *err = "arena too large for the TC path"; return FVDB_ERR_INVALID_ARG; }
    const uint32_t debug = tc_debug_bits();

    TCK(m->misc.ensure(4 * N_ROW_SETS, dev_bytes));
    bool arena_refreshed = false;
    if (!a.coarse_only) {
        const int r = refresh_row_set(m, SET_ARENA, a.rows, a.n_rows, D, s.arena_dirty, a.sm_count, st, dev_bytes,
                                      launches, err, &arena_refreshed);
        if (r != FVDB_OK) return r;
        s.arena_dirty = false;
    }
    if (arena_refreshed) {
        // longest-list-first order for the dynamic tile scheduler (once per arena layout)
        std::vector<uint32_t> off(a.nlist + 1), order(a.nlist);
        TCK(cudaMemcpyAsync(off.data(), a.list_off, (size_t)(a.nlist + 1) * 4, cudaMemcpyDeviceToHost, st));
        TCK(cudaStreamSynchronize(st));
        m->max_list_len = 0;
        for (uint32_t l = 0; l < a.nlist; ++l) m->max_list_len = std::max(m->max_list_len, off[l + 1] - off[l]);
        for (uint32_t l = 0; l < a.nlist; ++l) order[l] = l;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
            return off[x + 1] - off[x] > off[y + 1] - off[y];
        });
        TCK(m->list_order.ensure(a.nlist, dev_bytes));
        TCK(cudaMemcpyAsync(m->list_order.p, order.data(), (size_t)a.nlist * 4, cudaMemcpyHostToDevice, st));
        // the non-empty lists in id order (a shard of a list-sharded index owns 1 / world of them)
        std::vector<uint32_t> live;
        for (uint32_t l = 0; l < a.nlist; ++l) if (off[l + 1] > off[l]) live.push_back(l);
        m->n_live = (uint32_t)live.size();
        TCK(m->live_ids.ensure(std::max<size_t>(live.size(), 1), dev_bytes));
        if (!live.empty()) TCK(cudaMemcpyAsync(m->live_ids.p, live.data(), live.size() * 4, cudaMemcpyHostToDevice, st));
        TCK(cudaStreamSynchronize(st));
        m->list_order_n = a.nlist;
    }

    // ---- per-batch state ----
    const size_t n_pairs = (size_t)nq * np;
    // Two scan kernels share a batch.  Kernel W (wide query tiles on CTA pairs, queries in tensor
    // memory: D <= 384) takes the lists probed by at least `wide_min` queries: a row enters one SM once
    // per 256 queries, and with many live queries per warp its thread-per-query epilogue runs lane-
    // parallel.  Kernel R (items of up to 64 queries, query tile in shared memory, rows on the accumulator lanes,
    // candidate handling shared by the 128 row threads) takes the sparsely probed lists, where its MMA
    // cost (proportional to the queries of the item) and its cooperative epilogue are the cheaper ones.
    const uint32_t wide_min = tc_kernel_choice(D, a.sm_count);   // 0: kernel R only
    const bool use_wide = wide_min != 0;
    const uint32_t tile_q = r2_tile_q(D);   // kernel R's items; a list probed by more queries becomes several
    // Long posting lists are cut into row ranges (one work item and one shortlist slot each): a hub
    // list of 9 K rows probed by 64 queries is otherwise ONE item of 71 tiles — a third of the whole
    // scan on one SM, and the tail every other SM waits for.  At most TC_SPLIT_MAX ranges per list.
    uint32_t n_split = 1, rows_cap = 0;
    if (m->max_list_len > TC_SPLIT_MIN_ROWS) {
        const uint32_t unit = (uint32_t)R2_ROWS;   // a multiple of both kernels' tile heights
        rows_cap = std::max<uint32_t>(TC_SPLIT_MIN_ROWS / 2,
                                      ((m->max_list_len + TC_SPLIT_MAX - 1) / TC_SPLIT_MAX + unit - 1) / unit * unit);
        n_split = (m->max_list_len + rows_cap - 1) / rows_cap;
        if (n_split <= 1) { n_split = 1; rows_cap = 0; }
    }
    // shortlist rows per (query, probe): one per row range, times two when kernel W takes part (each
    // half of its tiles publishes its own row; kernel R writes row `range` of the same block)
    const uint32_t prows = (use_wide ? (uint32_t)W_SUBROWS : 1u) * n_split;
    const size_t max_items = ((size_t)a.nlist + (n_pairs + tile_q - 1) / tile_q) * n_split + 1;
    const size_t max_items_w = use_wide ? ((size_t)a.nlist + (n_pairs + W_NQ - 1) / W_NQ) * n_split + 1 : 0;
    TCK(m->qnorm.ensure(nq, dev_bytes));
    TCK(m->thr_g.ensure(nq, dev_bytes));
    TCK(m->list_cnt.ensure(a.nlist + 1, dev_bytes));
    TCK(m->pair_off.ensure(a.nlist + 2, dev_bytes));
    TCK(m->cursor.ensure(a.nlist + 1, dev_bytes));
    TCK(m->pair_q.ensure(n_pairs, dev_bytes));
    TCK(m->pair_slot.ensure(n_pairs, dev_bytes));
    TCK(m->n_items.ensure(8, dev_bytes));   // [0] items R, [1] counter R, [2][3] coarse, [4][5] flat tier, [6] items W, [7] counter W
    TCK(m->items.ensure(max_items, dev_bytes));
    if (use_wide) TCK(m->items_w.ensure(max_items_w, dev_bytes));
    TCK(m->partial.ensure(n_pairs * prows * TC_KP, dev_bytes));
    TCK(m->shortlist.ensure((size_t)nq * TC_KP, dev_bytes));

    {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>(((uint64_t)nq * 32 + 255) / 256, (uint64_t)a.sm_count * 8);
        // query norms; the same pass resets the per-query bounds (unless the caller shares an array it
        // has reset itself) and raises the batch's NaN flag
        // experiment (FVDB_TC_DEBUG bit 9): keep the previous batch's bounds = perfectly seeded thresholds
        const bool reset_bounds = !(debug & 512u) && !a.thr_ext;
        row_norms_kernel<<<blocks, 256, 0, st>>>(a.Q, nq, D, m->qnorm.p, nullptr, reset_bounds ? m->thr_g.p : nullptr,
                                                 F32_INF_BITS, a.d_nan);
        TCK(cudaGetLastError());
        (*launches) += 1;
    }
    const uint64_t* coarse_keys = a.coarse_keys;
    if (!coarse_keys) {
        if (D > 384 || np > TC_MAX_NPROBE_COARSE) { if (err) *err = "TC coarse step unsupported for this shape"; return FVDB_ERR_INVALID_ARG; }
        {
            const int r = refresh_row_set(m, SET_CENTROIDS, a.centroids, a.nlist, D, s.centroids_dirty, a.sm_count, st,
                                          dev_bytes, launches, err);
            if (r != FVDB_OK) return r;
            s.centroids_dirty = false;
        }
        const uint32_t ld = (a.nlist + 63) / 64 * 64;
        const uint32_t n_qg = (nq + Q1_M - 1) / Q1_M;
        const uint32_t tiles = ld / 64;
        uint32_t n_chunks = std::max(1u, std::min(tiles, ((uint32_t)a.sm_count + n_qg - 1) / n_qg));
        const uint32_t chunk_rows = ((tiles + n_chunks - 1) / n_chunks) * 64;
        n_chunks = (ld + chunk_rows - 1) / chunk_rows;
        const uint32_t n_citems = n_qg * n_chunks;
        TCK(m->dense.ensure((size_t)nq * ld, dev_bytes));
        TCK(m->coarse.ensure((size_t)nq * np, dev_bytes));
        TCK(m->citems.ensure(n_citems, dev_bytes));
        coarse_items_kernel<<<(n_citems + 127) / 128, 128, 0, st>>>(m->citems.p, nq, a.nlist, chunk_rows, n_chunks,
                                                                     m->n_items.p + 2);
        TCK(cudaGetLastError());
        TcScanParams cp{};
        cp.items = m->citems.p; cp.item_count = m->n_items.p + 2; cp.Q = a.Q; cp.qnorm = m->qnorm.p; cp.D = D; cp.KB = KB;
        cp.xnorm = m->sets[SET_CENTROIDS].xnorm.p; cp.ids = nullptr; cp.P = 1; cp.partial = nullptr; cp.thr_g = nullptr;
        cp.work_counter = m->n_items.p + 3;
        TCK(cudaMemsetAsync(cp.work_counter, 0, 4, st));
        cp.dense_out = m->dense.p; cp.dense_ld = ld;
        uint32_t kbs = 1;
        for (uint32_t c : {4u, 3u, 2u}) if (KB % c == 0) { kbs = c; break; }
        uint32_t stages = q1_pick_stages(KB, kbs);
        cp.stages = stages; cp.kbs = kbs;
        if (!m->smem_attr_set_q) {
            TCK(cudaFuncSetAttribute(tc_scan_q_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448));
            m->smem_attr_set_q = true;
        }
        tc_scan_q_kernel<<<std::min<uint32_t>((uint32_t)a.sm_count, n_citems), TC_THREADS,
                           tc_scan_q_smem_bytes(stages, kbs) + 1024, st>>>(m->sets[SET_CENTROIDS].tmap, cp);
        TCK(cudaGetLastError());
        // candidate set: nprobe + 32 (the proof needs the next approx value to clear the exact
        // nprobe-th by the TF32 bound; centroid distances are dense, so a generous margin)
        const uint32_t KC = std::min(np + 32, 128u);
        const size_t sel_smem = coarse_select_smem_bytes(D, KC);
        TCK(rerank_prepare(m));
        // 8 local entries per thread: P(one thread holds >= 8 of the KC nearest) is negligible
        coarse_select_kernel<8><<<nq, 128, sel_smem, st>>>(m->dense.p, ld, a.centroids, a.Q, m->qnorm.p,
                                                          m->misc.p + 4 * SET_CENTROIDS, nq, a.nlist, D, np, KC,
                                                          m->coarse.p, a.d_fallback_count, a.d_fallback_idx);
        TCK(cudaGetLastError());
        (*launches) += 3;
        coarse_keys = m->coarse.p;
        if (a.coarse_out) TCK(cudaMemcpyAsync(a.coarse_out, m->coarse.p, (size_t)nq * np * 8, cudaMemcpyDeviceToDevice, st));
    }
    if (a.coarse_only) return FVDB_OK;
    TCK(launch_probe_bucketing(coarse_keys, nq, np, a.list_off, a.nlist, tile_q, m->list_cnt.p, m->pair_off.p,
                               m->cursor.p, m->pair_q.p, m->pair_slot.p, m->items.p, m->n_items.p, a.d_scanned_rows, st,
                               m->list_order_n == a.nlist ? m->list_order.p : nullptr, rows_cap, wide_min, (uint32_t)W_NQ,
                               use_wide ? m->items_w.p : nullptr, m->n_items.p + 6,
                               m->list_order_n == a.nlist ? m->live_ids.p : nullptr, m->n_live));
    (*launches) += 3;
    uint32_t stamp = 0;
    TCK(m->next_stamp(n_pairs * prows, dev_bytes, st, &stamp));

    // ---- the scan ----
    TcScanParams p{};
    p.items = m->items.p; p.item_count = m->n_items.p; p.pair_q = m->pair_q.p; p.pair_slot = m->pair_slot.p;
    p.Q = a.Q; p.qnorm = m->qnorm.p; p.D = D; p.KB = KB; p.xnorm = m->sets[SET_ARENA].xnorm.p; p.ids = a.ids;
    p.tomb = a.tomb; p.tomb_bits = a.tomb_bits; p.filt = a.filt; p.filt_bits = a.filt_bits;
    p.P = np; p.S = prows; p.partial = m->partial.p; p.thr_g = a.thr_ext ? a.thr_ext : m->thr_g.p;
    p.row_stamp = m->row_stamp.p; p.stamp = stamp;
    p.n_peer = a.thr_ext ? std::min(a.n_peers, TC_MAX_PEERS) : 0u;
    for (uint32_t r = 0; r < p.n_peer; ++r) p.thr_peer[r] = a.thr_peers[r];
    p.work_counter = m->n_items.p + 1;
    p.debug = debug;
    p.scan_sms = a.scan_sms;
    TCK(cudaMemsetAsync(p.work_counter, 0, 4, st));
    if (use_wide) TCK(cudaMemsetAsync(m->n_items.p + 7, 0, 4, st));   // kernel W's work counter
    if (a.wait_before_scan) TCK(cudaStreamWaitEvent(st, a.wait_before_scan, 0));
    if (a.ev_scan0) TCK(cudaEventRecord(a.ev_scan0, st));
    // Order: the sparsely probed lists first (kernel R), then the hub lists (kernel W).  Every query probes
    // mostly sparse lists; after their scan its bound is already close to final, so the hub items — where a
    // candidate is the expensive thing (one thread per query) — start warm.
    {
        size_t smem = 0;
        p.stages = r2_pick_stages(D, &smem);
        if (!smem) { if (err) *err = "TC scan does not fit shared memory for this dim"; return FVDB_ERR_INVALID_CONFIG; }
        uint32_t grid = (uint32_t)std::min<size_t>((size_t)a.sm_count, max_items);
        if (p.scan_sms && p.scan_sms < grid) grid = p.scan_sms;
        if (p.debug & 128u) {
            TCK(m->prof.ensure((size_t)grid * 48, dev_bytes));
            TCK(cudaMemsetAsync(m->prof.p, 0, (size_t)grid * 48 * 8, st));
            p.prof = m->prof.p;
        }
        TCK(launch_r2(m, m->sets[SET_ARENA].tmap, p, grid, smem, st));
        if (p.prof) TCK(dump_prof(m->prof.p, grid, st));
    }
    if (use_wide) {
        TcScanParams pw = p;
        pw.items = m->items_w.p; pw.item_count = m->n_items.p + 6; pw.work_counter = m->n_items.p + 7;
        TCK(launch_wide(m, m->sets[SET_ARENA].tmap_w, pw, KB, a.sm_count, dev_bytes, st, nullptr));
        (*launches)++;
    }
    if (a.ev_scan1) TCK(cudaEventRecord(a.ev_scan1, st));
    if (a.record_after_scan) TCK(cudaEventRecord(a.record_after_scan, st));
    (*launches)++;

    // ---- merge the per-(query, probe) shortlists, exact re-rank, proof ----
    TCK(launch_merge_rows32(m->partial.p, nq, np * prows, m->shortlist.p, st, m->row_stamp.p, stamp));
    TCK(rerank_prepare(m));
    rerank_kernel<METRIC_L2><<<(nq + 3) / 4, 128, rerank_smem_bytes(D), st>>>(m->shortlist.p, a.rows, a.ids, a.Q, m->qnorm.p, m->misc.p + 4 * SET_ARENA, nq, D, a.k, (uint32_t)TC_KP,
                                               a.xmax_floor_sq, a.out_keys, a.d_fallback_count, a.d_fallback_idx, a.fin_ids, a.fin_dist, a.fin_count);
    TCK(cudaGetLastError());
    (*launches) += 2;
    return FVDB_OK;
}

int tc_flat_search(TcScratch& s, const TcFlatArgs& a, cudaStream_t st, size_t* dev_bytes, uint32_t* launches,
                   std::string* err) {
    if (!s.impl) s.impl = new TcScratchImpl();
    TcScratchImpl* m = s.impl;
    const uint32_t D = a.D, KB = D / 32, nq = a.nq;
    if (a.n_rows >= 0x7FFFFFFFull) { if (err) *err = "flat tier too large for the TC path"; return FVDB_ERR_INVALID_ARG; }
    TCK(m->misc.ensure(4 * N_ROW_SETS, dev_bytes));
    const RowSetId id = a.state ? SET_ASSIGN : SET_RECENT;
    RowSet& rs = m->sets[id];
    uint32_t* xmax_bits = m->misc.p + 4 * id;
    {
        const bool stale = a.state ? (rs.version != a.version) : s.flat_dirty;
        const int r = refresh_row_set(m, id, a.rows, a.n_rows, D, stale, a.sm_count, st, dev_bytes, launches, err);
        if (r != FVDB_OK) return r;
        rs.version = a.version;
        if (!a.state) s.flat_dirty = false;
    }
    // ---- work items: every query group (256 queries for kernel W, 64 for kernel R) against every row chunk ----
    const bool use_wide = tc_kernel_choice(D, a.sm_count) != 0;
    if (a.metric != METRIC_L2 && !use_wide) { if (err) *err = "cosine / dot scans need kernel W (dim <= 384)"; return FVDB_ERR_INVALID_CONFIG; }
    const uint32_t tile_q = use_wide ? (uint32_t)W_NQ : r2_tile_q(D);
    const uint32_t tile_rows = use_wide ? (uint32_t)W_N : (uint32_t)TC_ROWS;
    const uint32_t n_qg = (nq + tile_q - 1) / tile_q;
    const uint32_t tiles = (uint32_t)((a.n_rows + tile_rows - 1) / tile_rows);
    // enough items to fill the machine a few times over (pairs for kernel W), never more than 128
    // shortlist slots per query
    const uint32_t workers = use_wide ? (uint32_t)a.sm_count / 2 : (uint32_t)a.sm_count;
    uint32_t n_chunks = std::max(1u, std::min(std::min(tiles, 128u), (workers * 4 + n_qg - 1) / n_qg));
    const uint32_t chunk_rows = ((tiles + n_chunks - 1) / n_chunks) * tile_rows;
    n_chunks = (uint32_t)((a.n_rows + chunk_rows - 1) / chunk_rows);
    const uint32_t n_items = n_qg * n_chunks;
    TCK(m->qnorm.ensure(nq, dev_bytes));
    TCK(m->thr_g.ensure(nq, dev_bytes));
    TCK(m->n_items.ensure(8, dev_bytes));
    TCK(m->fitems.ensure(n_items, dev_bytes));
    const uint32_t frows = use_wide ? (uint32_t)W_SUBROWS : 1u;   // shortlist rows per (query, chunk)
    TCK(m->partial.ensure((size_t)nq * n_chunks * frows * TC_KP, dev_bytes));
    TCK(m->shortlist.ensure((size_t)nq * TC_KP, dev_bytes));
    {
        const uint32_t blocks = (uint32_t)std::min<uint64_t>(((uint64_t)nq * 32 + 255) / 256, (uint64_t)a.sm_count * 8);
        // query norms; the same pass resets the per-query bounds
        row_norms_kernel<<<blocks, 256, 0, st>>>(a.Q, nq, D, m->qnorm.p, nullptr, m->thr_g.p, F32_INF_BITS);
        flat_items_kernel<<<(n_items + 127) / 128, 128, 0, st>>>(m->fitems.p, nq, (uint32_t)a.n_rows, chunk_rows, n_chunks,
                                                                m->n_items.p + 4, tile_q);
        TCK(cudaGetLastError());
        (*launches) += 2;
    }
    uint32_t stamp = 0;
    TCK(m->next_stamp((size_t)nq * n_chunks * frows, dev_bytes, st, &stamp));
    TcScanParams p{};
    p.items = m->fitems.p; p.item_count = m->n_items.p + 4; p.pair_q = nullptr; p.pair_slot = nullptr;
    p.Q = a.Q; p.qnorm = m->qnorm.p; p.D = D; p.KB = KB; p.xnorm = rs.xnorm.p; p.ids = a.ids;
    p.tomb = a.tomb; p.tomb_bits = a.tomb_bits; p.filt = a.filt; p.filt_bits = a.filt_bits;
    p.P = n_chunks; p.S = use_wide ? frows : 0u; p.partial = m->partial.p; p.thr_g = m->thr_g.p;
    p.row_stamp = m->row_stamp.p; p.stamp = stamp;
    p.metric = a.metric; p.xmax_bits = xmax_bits;
    p.small_list = (a.k == 1 && a.rerank_r && a.rerank_r + 1 <= (uint32_t)W_SMALL_N) ? 1u : 0u;
    p.work_counter = m->n_items.p + 5;
    p.debug = tc_debug_bits();
    TCK(cudaMemsetAsync(p.work_counter, 0, 4, st));
    if (a.ev_scan0 && !use_wide) TCK(cudaEventRecord(a.ev_scan0, st));
    if (use_wide) {
        TCK(launch_wide(m, rs.tmap_w, p, KB, a.sm_count, dev_bytes, st, a.ev_scan0));
    } else {
        size_t smem = 0;
        p.stages = r2_pick_stages(D, &smem);
        if (!smem) { if (err) *err = "TC scan does not fit shared memory for this dim"; return FVDB_ERR_INVALID_CONFIG; }
        TCK(launch_r2(m, rs.tmap, p, std::min<uint32_t>((uint32_t)a.sm_count, n_items), smem, st));
    }
    if (a.ev_scan1) TCK(cudaEventRecord(a.ev_scan1, st));
    TCK(launch_merge_rows32(m->partial.p, nq, n_chunks * frows, m->shortlist.p, st, m->row_stamp.p, stamp));
    TCK(rerank_prepare(m));
    auto rr = a.metric == METRIC_COS ? rerank_kernel<METRIC_COS> : a.metric == METRIC_DOT ? rerank_kernel<METRIC_DOT>
                                                                                            : rerank_kernel<METRIC_L2>;
    rr<<<(nq + 3) / 4, 128, rerank_smem_bytes(D), st>>>(m->shortlist.p, a.rows, a.ids, a.Q, m->qnorm.p, xmax_bits, nq, D, a.k,
                                                        a.rerank_r ? a.rerank_r : (uint32_t)TC_KP, 0.0f, a.out_keys,
                                                        a.d_fallback_count, a.d_fallback_idx, nullptr, nullptr, nullptr,
                                                        (a.argmin_only && a.k == 1) ? 1u : 0u);
    TCK(cudaGetLastError());
    (*launches) += 3;
    return FVDB_OK;
}

}  // namespace fvdb
