// exact_scan.cu — the fp32 CUDA-core scan: every (query,row) distance is accumulated in the
// reference's own operation order (euclidean_distance_scalar, src/core/vector_ops.rs:51-57:
// t = a-b; acc = acc + t*t, index order, no FMA; then sqrt), so distances are bit-identical to
// the Rust reference.  One kernel serves four callers, all as "rows of a matrix against a
// group of queries -> per-query sorted partial top-k of u64 keys":
//   * IVF coarse step        (rows = centroids, k = nprobe)     src/ivf/core.rs:646-656
//   * IVF posting-list scan  (rows = one list, queries = probers) src/ivf/core.rs:661-678
//   * recent-tier flat scan  (rows = flat tier)                 replaces src/hnsw/core.rs:398-467
//   * k-means assignment     (rows = centroids, queries = points, k = 1) src/ivf/core.rs:291-297
// It is also the fallback / re-rank arithmetic of the tensor-core mode (tc_scan.cu).
//
// Tiling: CTA = 256 threads = 32 queries x 128 rows per tile, each thread a 4x4 register
// tile; D is walked in 32-wide chunks staged transposed in shared memory so the inner loop is
// 2 x LDS.128 + 48 ALU ops per d.  Bounded by the fp32 pipe (3 instructions per element, no
// FMA allowed), not by HBM: this path is the parity anchor, the tensor-core path is the fast one.
#include "common.cuh"
#include "kernels.cuh"

namespace fvdb {

namespace {

constexpr int TQ = 32;    // queries per tile
constexpr int TR = 128;   // rows per tile
constexpr int DK = 32;    // d-chunk
constexpr int NT = 256;   // threads
constexpr int QS_LD = TQ + 4;
constexpr int XS_LD = TR + 4;

// Insert `cand` into the ascending list[0..k) held in shared memory, dropping the largest.
// Whole warp cooperates.  Precondition: cand < list[k-1].
__device__ __forceinline__ void warp_insert(uint64_t* list, int k, uint64_t cand, int lane) {
    // position = number of entries < cand (keys are unique per (dist,id); equal keys keep
    // the incumbent first)
    int cnt = 0;
    for (int i = lane; i < k; i += 32) cnt += (list[i] <= cand) ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const int pos = cnt;
    // shift [pos, k-1) up by one, chunk by chunk from the top
    for (int base = ((k - 1) / 32) * 32; base >= 0 && base + 31 > pos; base -= 32) {
        int i = base + lane;
        uint64_t tmp = 0;
        bool mv = (i > pos) && (i < k);
        if (mv) tmp = list[i - 1];
        __syncwarp();
        if (mv) list[i] = tmp;
        __syncwarp();
    }
    if (lane == 0) list[pos] = cand;
    __syncwarp();
}

// METRIC: how a pair is scored, always in the reference's operation order (strictly sequential f32, no FMA):
//   L2   sqrt(sum (q - x)^2)                      euclidean_distance_scalar  src/core/vector_ops.rs:51-57
//   DOT  sum q * x                                dot_product_scalar         :35-37
//   COS  dot / (sqrt(dot(q,q)) * sqrt(dot(x,x))), 0 if either norm is 0      cosine_similarity_scalar :39-49
template <bool VEC, int METRIC>
__global__ void __launch_bounds__(NT) exact_scan_kernel(ExactScanArgs a) {
    const uint32_t n_items = a.item_count ? *a.item_count : a.n_items;
    if (blockIdx.x >= n_items) return;
    const ScanItem it = a.items[blockIdx.x];
    if (it.pair_count == 0) return;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* Qs = reinterpret_cast<float*>(smem_raw);                 // [DK][QS_LD]
    float* Xs = Qs + DK * QS_LD;                                    // [DK][XS_LD]; later dist tile [TQ][XS_LD]
    uint32_t* rowid_s = reinterpret_cast<uint32_t*>(Xs + DK * XS_LD);  // [TR]
    uint32_t* qidx_s = rowid_s + TR;                                // [TQ]
    uint32_t* qslot_s = qidx_s + TQ;                                // [TQ]
    uint64_t* topk_s = reinterpret_cast<uint64_t*>(qslot_s + TQ);   // [TQ][k]

    const int t = threadIdx.x;
    const int lane = t & 31, warp = t >> 5;
    const int tq = t & 7;    // query sub-tile: queries tq*4..+3
    const int tr = t >> 3;   // row sub-tile: rows tr*4..+3
    const uint32_t D = a.D;
    const int k = a.k;

    if (t < TQ) {
        uint32_t qi = ID_NONE, sl = 0;
        if ((uint32_t)t < it.pair_count) {
            if (it.identity) { qi = it.pair_begin + t; sl = it.slot; }
            else { qi = a.pair_q[it.pair_begin + t]; sl = a.pair_slot[it.pair_begin + t]; }
        }
        qidx_s[t] = qi;
        qslot_s[t] = sl;
    }
    for (int i = t; i < TQ * k; i += NT) topk_s[i] = KEY_NONE;
    __syncthreads();

    // global-load coordinates of this thread for a chunk
    const int ld_c4 = t & 7;          // float4 column within the 32-wide chunk
    const int ld_row = t >> 3;        // 0..31 ; X rows ld_row + 32*i, Q row ld_row
    const uint32_t my_q = qidx_s[ld_row];
    const float* qptr = (my_q != ID_NONE) ? a.Q + (size_t)my_q * D : nullptr;

    for (uint32_t rt = it.row_begin; rt < it.row_end; rt += TR) {
        if (t < TR) {
            uint32_t r = rt + t;
            uint32_t id = ID_NONE;
            if (r < it.row_end) {
                id = a.ids ? a.ids[r] : r;
                if (a.tomb && bit_test(a.tomb, a.tomb_bits, id)) id = ID_NONE;
                else if (a.filt && !bit_test(a.filt, a.filt_bits, id)) id = ID_NONE;
            }
            rowid_s[t] = id;
        }

        float acc[4][4];
        float qq_acc[4] = {0.f, 0.f, 0.f, 0.f}, xx_acc[4] = {0.f, 0.f, 0.f, 0.f};   // COS: dot(q,q), dot(x,x)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

        float4 xv[4], qv;
        auto gload = [&](uint32_t kc) {
            const uint32_t c = kc + ld_c4 * 4;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t r = rt + ld_row + 32 * i;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r < it.row_end) {
                    const float* p = a.X + (size_t)r * D + c;
                    if (VEC) {
                        if (c < D) v = __ldg(reinterpret_cast<const float4*>(p));
                    } else {
                        if (c + 0 < D) v.x = __ldg(p + 0);
                        if (c + 1 < D) v.y = __ldg(p + 1);
                        if (c + 2 < D) v.z = __ldg(p + 2);
                        if (c + 3 < D) v.w = __ldg(p + 3);
                    }
                }
                xv[i] = v;
            }
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (qptr) {
                const float* p = qptr + c;
                if (VEC) {
                    if (c < D) v = __ldg(reinterpret_cast<const float4*>(p));
                } else {
                    if (c + 0 < D) v.x = __ldg(p + 0);
                    if (c + 1 < D) v.y = __ldg(p + 1);
                    if (c + 2 < D) v.z = __ldg(p + 2);
                    if (c + 3 < D) v.w = __ldg(p + 3);
                }
            }
            qv = v;
        };

        gload(0);
        for (uint32_t kc = 0; kc < D; kc += DK) {
            // registers -> transposed shared tiles
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int r = ld_row + 32 * i;
                Xs[(ld_c4 * 4 + 0) * XS_LD + r] = xv[i].x;
                Xs[(ld_c4 * 4 + 1) * XS_LD + r] = xv[i].y;
                Xs[(ld_c4 * 4 + 2) * XS_LD + r] = xv[i].z;
                Xs[(ld_c4 * 4 + 3) * XS_LD + r] = xv[i].w;
            }
            Qs[(ld_c4 * 4 + 0) * QS_LD + ld_row] = qv.x;
            Qs[(ld_c4 * 4 + 1) * QS_LD + ld_row] = qv.y;
            Qs[(ld_c4 * 4 + 2) * QS_LD + ld_row] = qv.z;
            Qs[(ld_c4 * 4 + 3) * QS_LD + ld_row] = qv.w;
            __syncthreads();
            if (kc + DK < D) gload(kc + DK);  // prefetch the next chunk behind the math
#pragma unroll 8
            for (int d = 0; d < DK; ++d) {
                const float4 q4 = *reinterpret_cast<const float4*>(&Qs[d * QS_LD + tq * 4]);
                const float4 x4 = *reinterpret_cast<const float4*>(&Xs[d * XS_LD + tr * 4]);
                const float qq[4] = {q4.x, q4.y, q4.z, q4.w};
                const float xx[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (METRIC == METRIC_L2) {
                            // reference order: (a - b), squared, added — never fused
                            const float df = __fsub_rn(qq[i], xx[j]);
                            acc[i][j] = __fadd_rn(acc[i][j], __fmul_rn(df, df));
                        } else {
                            acc[i][j] = __fadd_rn(acc[i][j], __fmul_rn(qq[i], xx[j]));   // x * y, summed
                        }
                    }
                if (METRIC == METRIC_COS) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        qq_acc[i] = __fadd_rn(qq_acc[i], __fmul_rn(qq[i], qq[i]));
                        xx_acc[i] = __fadd_rn(xx_acc[i], __fmul_rn(xx[i], xx[i]));
                    }
                }
            }
            __syncthreads();
        }

        // distances -> shared tile (aliases Xs; all reads of Xs are behind the barrier above)
        float* dist_s = Xs;  // [TQ][XS_LD]
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (METRIC == METRIC_L2) {
                    o[j] = __fsqrt_rn(acc[i][j]);
                } else if (METRIC == METRIC_DOT) {
                    o[j] = acc[i][j];
                } else {
                    const float na = __fsqrt_rn(qq_acc[i]), nb = __fsqrt_rn(xx_acc[j]);
                    o[j] = (na == 0.0f || nb == 0.0f) ? 0.0f : __fdiv_rn(acc[i][j], __fmul_rn(na, nb));
                }
            }
            *reinterpret_cast<float4*>(&dist_s[(tq * 4 + i) * XS_LD + tr * 4]) = make_float4(o[0], o[1], o[2], o[3]);
        }
        __syncthreads();

        // selection: warp w owns queries 4w..4w+3; running sorted top-k per query in smem
#pragma unroll 1
        for (int qi = 0; qi < 4; ++qi) {
            const int q = warp * 4 + qi;
            if ((uint32_t)q >= it.pair_count) break;
            uint64_t* list = topk_s + (size_t)q * k;
            uint64_t thr = list[k - 1];
#pragma unroll 1
            for (int c = 0; c < TR / 32; ++c) {
                const int r = lane + 32 * c;
                const uint32_t id = rowid_s[r];
                uint64_t key = KEY_NONE;
                if (id != ID_NONE) {
                    const float v = dist_s[q * XS_LD + r];
                    key = METRIC == METRIC_L2 ? make_key(v, id) : (((uint64_t)sim_to_key32(v) << 32) | id);
                }
                unsigned m = __ballot_sync(0xffffffffu, key < thr);
                while (m) {
                    const int src = __ffs(m) - 1;
                    const uint64_t cand = __shfl_sync(0xffffffffu, key, src);
                    warp_insert(list, k, cand, lane);
                    thr = list[k - 1];
                    if (lane == src) key = KEY_NONE;
                    m = __ballot_sync(0xffffffffu, key < thr);
                }
            }
        }
        __syncthreads();
    }

    // write the partial lists
    for (int q = warp; q < (int)it.pair_count; q += NT / 32) {
        const uint32_t qi = qidx_s[q];
        uint64_t* dst = a.partial + ((size_t)qi * a.P + qslot_s[q]) * k;
        const uint64_t* src = topk_s + (size_t)q * k;
        for (int i = lane; i < k; i += 32) dst[i] = src[i];
    }
}

}  // namespace

size_t exact_scan_smem_bytes(uint32_t k) {
    return (size_t)(DK * QS_LD + DK * XS_LD) * sizeof(float) + (TR + 2 * TQ) * sizeof(uint32_t) +
           (size_t)TQ * k * sizeof(uint64_t);
}

cudaError_t launch_exact_scan(const ExactScanArgs& a, uint32_t grid, cudaStream_t stream) {
    if (grid == 0) return cudaSuccess;
    const size_t smem = exact_scan_smem_bytes(a.k);
    const bool vec = (a.D % 4 == 0) && ((reinterpret_cast<uintptr_t>(a.X) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(a.Q) & 15) == 0);
    auto go = [&](auto kern) -> cudaError_t {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        kern<<<grid, NT, smem, stream>>>(a);
        return cudaSuccess;
    };
    cudaError_t e;
    if (a.metric == METRIC_COS) e = vec ? go(exact_scan_kernel<true, METRIC_COS>) : go(exact_scan_kernel<false, METRIC_COS>);
    else if (a.metric == METRIC_DOT) e = vec ? go(exact_scan_kernel<true, METRIC_DOT>) : go(exact_scan_kernel<false, METRIC_DOT>);
    else e = vec ? go(exact_scan_kernel<true, METRIC_L2>) : go(exact_scan_kernel<false, METRIC_L2>);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Item builders
// ---------------------------------------------------------------------------------------------

// identity items: every query against rows [row_begin,row_end) split into `nsplit` chunks.
__global__ void build_identity_items_kernel(ScanItem* items, uint32_t nq, uint32_t row_begin,
                                            uint32_t row_end, uint32_t nsplit) {
    const uint32_t n_qt = (nq + TQ - 1) / TQ;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_qt * nsplit) return;
    const uint32_t qt = i / nsplit, sp = i % nsplit;
    const uint32_t rows = row_end - row_begin;
    // chunk boundaries on multiples of TR so tiles stay aligned
    const uint32_t tiles = (rows + TR - 1) / TR;
    const uint32_t t0 = (uint32_t)(((uint64_t)tiles * sp) / nsplit);
    const uint32_t t1 = (uint32_t)(((uint64_t)tiles * (sp + 1)) / nsplit);
    ScanItem it;
    it.row_begin = row_begin + t0 * TR;
    it.row_end = min(row_end, row_begin + t1 * TR);
    it.pair_begin = qt * TQ;
    it.pair_count = min((uint32_t)TQ, nq - qt * TQ);
    it.slot = sp;
    it.identity = 1;
    it.sub = 0;
    if (it.row_begin >= it.row_end) it.pair_count = 0;
    items[i] = it;
}

cudaError_t launch_build_identity_items(ScanItem* items, uint32_t nq, uint32_t row_begin,
                                        uint32_t row_end, uint32_t nsplit, uint32_t* n_items_out,
                                        cudaStream_t stream) {
    const uint32_t n_qt = (nq + TQ - 1) / TQ;
    const uint32_t n = n_qt * nsplit;
    *n_items_out = n;
    if (n == 0) return cudaSuccess;
    build_identity_items_kernel<<<(n + 255) / 256, 256, 0, stream>>>(items, nq, row_begin, row_end,
                                                                    nsplit);
    return cudaGetLastError();
}

uint32_t exact_scan_tq() { return TQ; }
uint32_t exact_scan_tr() { return TR; }

// ---------------------------------------------------------------------------------------------
// Probe bucketing: (query, rank) pairs grouped by list  (builds the list -> queries CSR that
// lets each posting list be streamed once per batch instead of once per query)
// ---------------------------------------------------------------------------------------------

// coarse_keys [nq][nprobe]: low 32 bits = list id.  KEY_NONE entries (nprobe > nlist) skipped.
// list_cnt[l] += 1 per probing query; bit 31 of list_cnt[l] is set when l is some query's
// NEAREST list (rank 0) — those lists are scheduled first so per-query thresholds tighten early.
constexpr uint32_t NEAREST_BIT = 0x80000000u;
__global__ void probe_hist_kernel(const uint64_t* __restrict__ coarse_keys, uint32_t n_pairs,
                                  uint32_t nprobe, uint32_t* __restrict__ list_cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const uint64_t key = coarse_keys[i];
    if (key == KEY_NONE) return;
    atomicAdd(&list_cnt[key_id(key)], 1u);
    if (i % nprobe == 0) atomicOr(&list_cnt[key_id(key)], NEAREST_BIT);
}

// single-CTA exclusive scan over lists: pair offsets and work-item offsets; also emits the
// items.  tile_q = queries per item (TQ for the exact kernel, the query-tile of the TC kernel).
// Items of one list are adjacent so a list re-read by a second query tile hits L2.
// block-wide exclusive scan of a packed u64 (items << 32 | pairs) over 1024 threads;
// returns the exclusive prefix, *total receives the block total (all threads)
__device__ __forceinline__ uint64_t block_excl_scan_u64(uint64_t v, uint64_t* warp_tot, uint64_t* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint64_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t n = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) warp_tot[w] = inc;
    __syncthreads();
    if (w == 0) {
        uint64_t t = warp_tot[lane];
        uint64_t ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t n = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += n;
        }
        warp_tot[lane] = ti - t;       // exclusive warp offsets
        if (lane == 31) warp_tot[32] = ti;
    }
    __syncthreads();
    const uint64_t r = warp_tot[w] + inc - v;
    *total = warp_tot[32];
    __syncthreads();
    return r;
}

// One CTA: per-list pair offsets and the work-item table(s).  Lists that are the NEAREST list of
// at least one query come first in the item order (their scan tightens that query's threshold
// for every other list); items of one list stay adjacent so a re-read hits L2.
// Two tables when wide_min > 0: lists probed by at least wide_min queries go to `items_w` (query
// groups of tile_q_w: the wide-tile scan kernel), the others to `items` (groups of tile_q).
__global__ void __launch_bounds__(1024) probe_scan_kernel(const uint32_t* __restrict__ list_cnt,
                                  const uint32_t* __restrict__ list_off,
                                  const uint32_t* __restrict__ list_order, uint32_t nlist,
                                  uint32_t tile_q, uint32_t* __restrict__ pair_off,
                                  uint32_t* __restrict__ cursor, ScanItem* __restrict__ items,
                                  uint32_t* __restrict__ n_items, uint64_t* __restrict__ scanned_rows,
                                  bool order_near_in, uint32_t rows_cap, uint32_t wide_min, uint32_t tile_q_w,
                                  ScanItem* __restrict__ items_w, uint32_t* __restrict__ n_items_w, bool wide_longest_first,
                                  const uint32_t* __restrict__ live_ids, uint32_t n_live) {
    // live_ids (optional, with list_order): the n_live non-empty lists in ascending id order; list_order then
    // holds them first (longest first).  A list-sharded index owns 1 / world of the lists: walking only those
    // keeps this single-CTA pass as long as it is on one GPU instead of growing with the world size.
    const uint32_t n_walk = (live_ids && list_order) ? n_live : nlist;
    __shared__ uint64_t warp_tot[33];
    const int t = threadIdx.x;
    uint64_t my_rows = 0;
    uint64_t pair_carry = 0;   // pairs placed so far (both tables share the pair arrays)
    for (int tbl = 0; tbl < (wide_min ? 2 : 1); ++tbl) {
        // tbl 0 (when two tables): the wide table, so that its pairs come first
        const bool wide = wide_min && tbl == 0;
        const uint32_t tq = wide ? tile_q_w : tile_q;
        ScanItem* out = wide ? items_w : items;
        const bool order_near = order_near_in || (wide && wide_longest_first);
        // offsets and items.  g = 0: the nearest-first group in list order; g = 1: the other
        // lists, longest first when list_order is given — the dynamic tile scheduler then ends with
        // the cheapest items, which keeps the tail of the scan short.  (Ordering the nearest group by
        // length as well starts every CTA on the most popular lists with cold thresholds: measured
        // 20 % more work.)
        uint64_t carry = pair_carry;   // (items << 32) | pairs
        auto mine = [&](uint32_t l, uint32_t& c, uint32_t& len, bool& nearest) {
            c = 0; len = 0; nearest = false;
            if (l >= nlist) return;
            const uint32_t raw = list_cnt[l];
            len = list_off[l + 1] - list_off[l];
            c = len ? (raw & ~NEAREST_BIT) : 0u;
            nearest = (raw & NEAREST_BIT) != 0;
            if (wide_min && ((c >= wide_min) != wide)) c = 0;   // the other table's list
        };
        for (int g = 0; g < 2; ++g) {
            for (uint32_t base = 0; base < n_walk; base += 1024) {
                const uint32_t l = (base + t < n_walk) ? (((g || order_near) && list_order) ? list_order[base + t]
                                                          : (live_ids && list_order) ? live_ids[base + t] : base + t) : nlist;
                uint32_t c, len;
                bool nearest;
                mine(l, c, len, nearest);
                if (nearest != (g == 0)) c = 0;   // not this group's list
                const uint32_t ni = (c + tq - 1) / tq;
                // a long list is cut into ns row ranges of at most rows_cap rows: ns items per query group,
                // each with its own shortlist slot (ScanItem::sub), so that no single item is a long tail.
                // Nearest-first group: only the FIRST range here, the others follow below.  Other lists
                // (bounds already tight when they start): all ranges, adjacent.
                const uint32_t ns = (rows_cap && len > rows_cap) ? (len + rows_cap - 1) / rows_cap : 1u;
                const uint32_t ns_here = g ? ns : 1u;
                const uint64_t v = ((uint64_t)(ni * ns_here) << 32) | c;
                uint64_t tot;
                const uint64_t ex = block_excl_scan_u64(v, warp_tot, &tot);
                if (c > 0) {
                    const uint64_t off = carry + ex;
                    const uint32_t p_excl = (uint32_t)off, i_excl = (uint32_t)(off >> 32);
                    pair_off[l] = p_excl;
                    cursor[l] = p_excl;
                    for (uint32_t j = 0; j < ni; ++j) {
                        for (uint32_t sb = 0; sb < ns_here; ++sb) {
                            ScanItem it;
                            it.row_begin = list_off[l] + (ns > 1 ? sb * rows_cap : 0u);
                            it.row_end = (ns > 1) ? min(list_off[l + 1], it.row_begin + rows_cap) : list_off[l + 1];
                            it.pair_begin = p_excl + j * tq;
                            it.pair_count = min(tq, c - j * tq);
                            it.slot = ni;  // query groups sharing this list (the TC scan keeps such lists in L2)
                            it.identity = 0;
                            it.sub = sb;
                            out[i_excl + j * ns_here + sb] = it;
                        }
                    }
                    my_rows += len;
                }
                carry += tot;
            }
            if (g == 0 && rows_cap) {
                // the further row ranges of the nearest-first lists, range by range, behind every first
                // range: by the time range s of a list starts, its range s - 1 has been scanned for a while
                // and has published the queries' bounds (ranges that start together all start cold:
                // measured 5 % more work).  The cheap far lists still come last.
                for (uint32_t sb = 1; sb < 64; ++sb) {
                    uint32_t any = 0;
                    for (uint32_t base = 0; base < n_walk; base += 1024) {
                        const uint32_t l = (base + t < n_walk) ? ((order_near && list_order) ? list_order[base + t]
                                                                  : (live_ids && list_order) ? live_ids[base + t] : base + t) : nlist;
                        uint32_t c, len;
                        bool nearest;
                        mine(l, c, len, nearest);
                        if (!nearest) c = 0;
                        const uint32_t ns = (len > rows_cap) ? (len + rows_cap - 1) / rows_cap : 1u;
                        const uint32_t ni = (c && sb < ns) ? (c + tq - 1) / tq : 0u;
                        uint64_t tot;
                        const uint64_t ex = block_excl_scan_u64(ni, warp_tot, &tot);
                        if (ni) {
                            const uint32_t p_excl = pair_off[l];
                            const uint32_t i0 = (uint32_t)(carry >> 32) + (uint32_t)ex;
                            for (uint32_t j = 0; j < ni; ++j) {
                                ScanItem it;
                                it.row_begin = list_off[l] + sb * rows_cap;
                                it.row_end = min(list_off[l + 1], it.row_begin + rows_cap);
                                it.pair_begin = p_excl + j * tq;
                                it.pair_count = min(tq, c - j * tq);
                                it.slot = ni;
                                it.identity = 0;
                                it.sub = sb;
                                out[i0 + j] = it;
                            }
                        }
                        carry += tot << 32;
                        any += (uint32_t)tot;
                    }
                    if (any == 0) break;   // block-uniform: no list has this many ranges
                }
            }
        }
        if (t == 0) *(wide ? n_items_w : n_items) = (uint32_t)(carry >> 32);
        pair_carry = carry & 0xFFFFFFFFull;
    }
    uint64_t rows_total;
    block_excl_scan_u64(my_rows, warp_tot, &rows_total);
    if (t == 0) {
        pair_off[nlist] = (uint32_t)pair_carry;
        if (scanned_rows) *scanned_rows = rows_total;
    }
}

__global__ void probe_scatter_kernel(const uint64_t* __restrict__ coarse_keys, uint32_t n_pairs,
                                     uint32_t nprobe, const uint32_t* __restrict__ list_off,
                                     uint32_t* __restrict__ cursor, uint32_t* __restrict__ pair_q,
                                     uint32_t* __restrict__ pair_slot) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const uint64_t key = coarse_keys[i];
    if (key == KEY_NONE) return;
    const uint32_t l = key_id(key);
    if (list_off[l + 1] == list_off[l]) return;
    const uint32_t p = atomicAdd(&cursor[l], 1u);
    pair_q[p] = i / nprobe;
    pair_slot[p] = i % nprobe;
}

cudaError_t launch_probe_bucketing(const uint64_t* coarse_keys, uint32_t nq, uint32_t nprobe,
                                   const uint32_t* list_off, uint32_t nlist, uint32_t tile_q,
                                   uint32_t* list_cnt, uint32_t* pair_off, uint32_t* cursor,
                                   uint32_t* pair_q, uint32_t* pair_slot, ScanItem* items,
                                   uint32_t* n_items, uint64_t* scanned_rows, cudaStream_t stream,
                                   const uint32_t* list_order, bool order_near, uint32_t rows_cap,
                                   uint32_t wide_min, uint32_t tile_q_w, ScanItem* items_w, uint32_t* n_items_w,
                                   bool wide_longest_first, const uint32_t* live_ids, uint32_t n_live) {
    const uint32_t n_pairs = nq * nprobe;
    cudaError_t e = cudaMemsetAsync(list_cnt, 0, sizeof(uint32_t) * nlist, stream);
    if (e != cudaSuccess) return e;
    if (n_pairs == 0) {
        if (wide_min) { e = cudaMemsetAsync(n_items_w, 0, sizeof(uint32_t), stream); if (e != cudaSuccess) return e; }
        return cudaMemsetAsync(n_items, 0, sizeof(uint32_t), stream);
    }
    probe_hist_kernel<<<(n_pairs + 255) / 256, 256, 0, stream>>>(coarse_keys, n_pairs, nprobe, list_cnt);
    probe_scan_kernel<<<1, 1024, 0, stream>>>(list_cnt, list_off, list_order, nlist, tile_q, pair_off, cursor,
                                              items, n_items, scanned_rows, order_near, rows_cap, wide_min, tile_q_w,
                                              items_w, n_items_w, wide_longest_first, live_ids, n_live);
    probe_scatter_kernel<<<(n_pairs + 255) / 256, 256, 0, stream>>>(coarse_keys, n_pairs, nprobe,
                                                                   list_off, cursor, pair_q,
                                                                   pair_slot);
    return cudaGetLastError();
}

// Sparse exact scan: one CTA (4 warps) per (query, probed list) pair — for small batches
// (single-query search, the fallback queries of the tensor-core mode) where a 32-query tile would
// be mostly padding.  Lane = row; every lane walks its own row in the reference's operation
// order with eight 16-byte loads in flight; each warp keeps a sorted top-k, warp 0 merges them.
__global__ void __launch_bounds__(128) exact_pair_scan_kernel(const uint64_t* __restrict__ coarse_keys, uint32_t n_pairs,
                                                              const uint32_t* __restrict__ list_off,
                                                              const float* __restrict__ X, const uint32_t* __restrict__ ids,
                                                              const float* __restrict__ Q, uint32_t D, uint32_t nprobe,
                                                              uint32_t P, uint32_t k, const uint64_t* __restrict__ tomb,
                                                              uint64_t tomb_bits, const uint64_t* __restrict__ filt,
                                                              uint64_t filt_bits, uint64_t* __restrict__ partial) {
    extern __shared__ __align__(16) unsigned char pair_smem[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t pair = blockIdx.x;
    float* q_s = reinterpret_cast<float*>(pair_smem);
    uint64_t* list = reinterpret_cast<uint64_t*>(pair_smem + (((size_t)D * sizeof(float) + 15) & ~(size_t)15)) + (size_t)w * k;
    const uint32_t q = pair / nprobe, slot = pair % nprobe;
    const uint64_t ck = coarse_keys[pair];
    if (ck == KEY_NONE) return;  // partial pre-filled with KEY_NONE
    const uint32_t l = key_id(ck);
    const uint32_t b = list_off[l], e = list_off[l + 1];
    for (uint32_t d = threadIdx.x; d < D; d += 128) q_s[d] = __ldg(Q + (size_t)q * D + d);
    for (uint32_t i = lane; i < k; i += 32) list[i] = KEY_NONE;
    __syncthreads();
    uint64_t thr = KEY_NONE;
    for (uint32_t r0 = b + w * 32; r0 < e; r0 += 128) {
        const uint32_t r = r0 + lane;
        uint64_t key = KEY_NONE;
        if (r < e) {
            const uint32_t id = ids ? ids[r] : r;
            bool live = true;
            if (tomb && bit_test(tomb, tomb_bits, id)) live = false;
            else if (filt && !bit_test(filt, filt_bits, id)) live = false;
            if (live) {
                float dist;
                if ((D & 3) == 0) {
                    dist = exact_l2_lane(q_s, X + (size_t)r * D, D);
                } else {
                    const float* xr = X + (size_t)r * D;
                    float acc = 0.0f;
                    for (uint32_t i = 0; i < D; ++i) {
                        const float t = __fsub_rn(q_s[i], __ldg(xr + i));
                        acc = __fadd_rn(acc, __fmul_rn(t, t));
                    }
                    dist = __fsqrt_rn(acc);
                }
                key = make_key(dist, id);
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, key < thr);
        while (m) {
            const int src = __ffs(m) - 1;
            const uint64_t cand = __shfl_sync(0xffffffffu, key, src);
            warp_insert(list, (int)k, cand, lane);
            thr = list[k - 1];
            if (lane == src) key = KEY_NONE;
            m = __ballot_sync(0xffffffffu, key < thr);
        }
    }
    __syncthreads();
    if (w == 0) {
        // fold the other warps' lists into mine (ascending lists: stop at the first non-improving key)
        uint64_t* base = reinterpret_cast<uint64_t*>(pair_smem + (((size_t)D * sizeof(float) + 15) & ~(size_t)15));
        for (int ow = 1; ow < 4; ++ow) {
            const uint64_t* other = base + (size_t)ow * k;
            for (uint32_t i = 0; i < k; ++i) {
                const uint64_t cand = other[i];
                if (cand >= list[k - 1]) break;
                warp_insert(list, (int)k, cand, lane);
            }
        }
        uint64_t* dst = partial + ((size_t)q * P + slot) * k;
        for (uint32_t i = lane; i < k; i += 32) dst[i] = list[i];
    }
}

cudaError_t launch_exact_pair_scan(const uint64_t* coarse_keys, uint32_t nq, uint32_t nprobe, const uint32_t* list_off,
                                   const float* X, const uint32_t* ids, const float* Q, uint32_t D, uint32_t P,
                                   uint32_t k, const uint64_t* tomb, uint64_t tomb_bits, const uint64_t* filt,
                                   uint64_t filt_bits, uint64_t* partial, cudaStream_t stream) {
    const uint32_t n_pairs = nq * nprobe;
    if (n_pairs == 0) return cudaSuccess;
    const size_t smem = (((size_t)D * sizeof(float) + 15) & ~(size_t)15) + (size_t)4 * k * sizeof(uint64_t);
    cudaError_t e = cudaFuncSetAttribute(exact_pair_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    exact_pair_scan_kernel<<<n_pairs, 128, smem, stream>>>(coarse_keys, n_pairs, list_off, X, ids, Q, D, nprobe,
                                                                     P, k, tomb, tomb_bits, filt, filt_bits, partial);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Merging sorted partial lists
// ---------------------------------------------------------------------------------------------

// One warp per query: P ascending lists of k keys -> the k smallest, ascending.
// in [nq][P][k], out [nq][k_out stride]; KEY_NONE pads.
__global__ void merge_partials_kernel(const uint64_t* __restrict__ in, uint32_t nq, uint32_t P,
                                      uint32_t k, uint64_t* __restrict__ out) {
    const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (q >= nq) return;
    const uint64_t* base = in + (size_t)q * P * k;
    // each lane walks lists lane, lane+32, ... keeping the smallest current head among them
    // (per-lane: index of the list with the smallest head, found by a linear pass — P/32 small)
    constexpr int MAXL = 8;  // lists per lane handled in registers => P <= 256 per pass
    uint32_t pos[MAXL];
#pragma unroll
    for (int j = 0; j < MAXL; ++j) pos[j] = 0;
    for (uint32_t o = 0; o < k; ++o) {
        uint64_t best = KEY_NONE;
        int bj = -1;
#pragma unroll
        for (int j = 0; j < MAXL; ++j) {
            const uint32_t p = lane + 32 * j;
            if (p < P && pos[j] < k) {
                const uint64_t v = base[(size_t)p * k + pos[j]];
                if (v < best) { best = v; bj = j; }
            }
        }
        // warp argmin on (key, lane) — keys with equal value can only be KEY_NONE or true
        // duplicates (same id twice); either choice gives the same output value
        uint64_t wbest = best;
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) {
            const uint64_t other = __shfl_xor_sync(0xffffffffu, wbest, s);
            wbest = other < wbest ? other : wbest;
        }
        const unsigned who = __ballot_sync(0xffffffffu, best == wbest && bj >= 0);
        if (wbest == KEY_NONE || who == 0) {
            for (uint32_t r = o + lane; r < k; r += 32) out[(size_t)q * k + r] = KEY_NONE;
            return;
        }
        const int winner = __ffs(who) - 1;
        if (lane == winner) {
#pragma unroll
            for (int j = 0; j < MAXL; ++j) if (j == bj) pos[j]++;
        }
        if (lane == 0) out[(size_t)q * k + o] = wbest;
    }
}

cudaError_t launch_merge_partials(const uint64_t* in, uint32_t nq, uint32_t P, uint32_t k,
                                  uint64_t* out, cudaStream_t stream) {
    if (nq == 0) return cudaSuccess;
    if (P > 256) return cudaErrorInvalidValue;
    const uint32_t threads = 128;
    const uint32_t blocks = (nq * 32 + threads - 1) / threads;
    merge_partials_kernel<<<blocks, threads, 0, stream>>>(in, nq, P, k, out);
    return cudaGetLastError();
}

// Final hybrid merge (src/hybrid/core.rs:482-483): recent-tier keys and IVF keys, each sorted,
// two-pointer merged by distance with the recent tier first on ties, truncated to k, split
// into ids / distances / count.  Either input may be null.
__device__ __forceinline__ void finalize_row(const uint64_t* a, const uint64_t* b, uint32_t q, uint32_t k,
                                             uint32_t* __restrict__ out_ids, float* __restrict__ out_dist,
                                             uint32_t* __restrict__ out_count, int metric) {
    uint32_t ia = 0, ib = 0, o = 0;
    while (o < k) {
        const uint64_t ka = (a && ia < k) ? a[ia] : KEY_NONE;
        const uint64_t kb = (b && ib < k) ? b[ib] : KEY_NONE;
        if (ka == KEY_NONE && kb == KEY_NONE) break;
        uint64_t pick;
        // compare distances only; recent wins ties (stable sort, recent results pushed first)
        if (kb == KEY_NONE || (ka != KEY_NONE && (uint32_t)(ka >> 32) <= (uint32_t)(kb >> 32))) { pick = ka; ++ia; }
        else { pick = kb; ++ib; }
        out_ids[(size_t)q * k + o] = key_id(pick);
        out_dist[(size_t)q * k + o] = key_value(pick, metric);
        ++o;
    }
    out_count[q] = o;
    for (; o < k; ++o) {
        out_ids[(size_t)q * k + o] = ID_NONE;
        out_dist[(size_t)q * k + o] = __uint_as_float(metric == METRIC_L2 ? 0x7f800000u : 0xff800000u);   // worst value
    }
}

// Without a second output set the two tiers are merged into the first; with one (fvdb_search_device_tiers)
// the recent tier goes to the first set and the IVF tier to the second, each as finalize writes a lone tier.
__global__ void finalize_kernel(const uint64_t* __restrict__ recent, const uint64_t* __restrict__ ivf,
                                uint32_t nq, uint32_t k, uint32_t* __restrict__ out_ids,
                                float* __restrict__ out_dist, uint32_t* __restrict__ out_count, int metric,
                                uint32_t* __restrict__ ivf_ids, float* __restrict__ ivf_dist,
                                uint32_t* __restrict__ ivf_count) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint64_t* a = recent ? recent + (size_t)q * k : nullptr;
    const uint64_t* b = ivf ? ivf + (size_t)q * k : nullptr;
    if (ivf_ids) {
        finalize_row(a, nullptr, q, k, out_ids, out_dist, out_count, metric);
        finalize_row(nullptr, b, q, k, ivf_ids, ivf_dist, ivf_count, metric);
    } else {
        finalize_row(a, b, q, k, out_ids, out_dist, out_count, metric);
    }
}

cudaError_t launch_finalize(const uint64_t* recent, const uint64_t* ivf, uint32_t nq, uint32_t k,
                            uint32_t* out_ids, float* out_dist, uint32_t* out_count,
                            cudaStream_t stream, int metric, uint32_t* ivf_ids, float* ivf_dist,
                            uint32_t* ivf_count) {
    if (nq == 0) return cudaSuccess;
    finalize_kernel<<<(nq + 127) / 128, 128, 0, stream>>>(recent, ivf, nq, k, out_ids, out_dist,
                                                         out_count, metric, ivf_ids, ivf_dist, ivf_count);
    return cudaGetLastError();
}

// Cross-GPU merge after the all-gather (fvdb_merge_topk_device): parts x [nq][k] (ids, dist,
// count) -> [nq][k].  Order: (distance, row id), the ABI's tie rule — each part is already sorted
// that way and the parts hold disjoint rows, so the head of every part is compared by distance and,
// on equal distances, by id.  TIERED (fvdb_merge_topk_tiers_packed_device): part p holds rows of tier
// p & 1 (0 = recent, 1 = IVF) and the order is (distance, tier, row id), the recent-first rule of
// finalize_kernel.  One thread per query (k and parts are small).
// part p's block starts at p * stride_kv (ids, dist; elements) and p * stride_c (counts).
template <bool TIERED>
__global__ void merge_parts_kernel(const uint32_t* __restrict__ ids, const float* __restrict__ dist,
                                   const uint32_t* __restrict__ cnt, uint32_t parts, uint32_t nq,
                                   uint32_t k, size_t stride_kv, size_t stride_c, uint32_t* __restrict__ out_ids,
                                   float* __restrict__ out_dist, uint32_t* __restrict__ out_count) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    constexpr int MAXP = 64;
    uint16_t pos[MAXP];
    for (uint32_t p = 0; p < parts; ++p) pos[p] = 0;
    uint32_t o = 0;
    for (; o < k; ++o) {
        float best = 0.f;
        uint32_t best_id = 0;
        int bp = -1;
        for (uint32_t p = 0; p < parts; ++p) {
            const uint32_t c = min(cnt[(size_t)p * stride_c + q], k);
            if (pos[p] < c) {
                const size_t at = (size_t)p * stride_kv + (size_t)q * k + pos[p];
                const float d = dist[at];
                const uint32_t id = ids[at];
                bool take = bp < 0 || d < best;
                if (!take && d == best) {
                    const uint32_t tp = TIERED ? (p & 1u) : 0u, tb = TIERED ? ((uint32_t)bp & 1u) : 0u;
                    take = tp < tb || (tp == tb && id < best_id);
                }
                if (take) { best = d; best_id = id; bp = (int)p; }
            }
        }
        if (bp < 0) break;
        out_ids[(size_t)q * k + o] = best_id;
        out_dist[(size_t)q * k + o] = best;
        pos[bp]++;
    }
    out_count[q] = o;
    for (; o < k; ++o) {
        out_ids[(size_t)q * k + o] = ID_NONE;
        out_dist[(size_t)q * k + o] = __uint_as_float(0x7f800000u);
    }
}

cudaError_t launch_merge_parts(const uint32_t* ids, const float* dist, const uint32_t* cnt,
                               uint32_t parts, uint32_t nq, uint32_t k, uint32_t* out_ids,
                               float* out_dist, uint32_t* out_count, cudaStream_t stream,
                               size_t stride_kv, size_t stride_c, bool tiered) {
    if (nq == 0) return cudaSuccess;
    if (parts > 64) return cudaErrorInvalidValue;
    if (stride_kv == 0) stride_kv = (size_t)nq * k;
    if (stride_c == 0) stride_c = nq;
    if (tiered)
        merge_parts_kernel<true><<<(nq + 127) / 128, 128, 0, stream>>>(ids, dist, cnt, parts, nq, k, stride_kv, stride_c,
                                                                      out_ids, out_dist, out_count);
    else
        merge_parts_kernel<false><<<(nq + 127) / 128, 128, 0, stream>>>(ids, dist, cnt, parts, nq, k, stride_kv, stride_c,
                                                                       out_ids, out_dist, out_count);
    return cudaGetLastError();
}

__global__ void scatter_keys_kernel(const uint64_t* __restrict__ src, const uint32_t* __restrict__ idx,
                                    uint32_t n, uint32_t k, uint64_t* __restrict__ dst) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * k) return;
    dst[(size_t)idx[i / k] * k + (i % k)] = src[i];
}

cudaError_t launch_scatter_keys(const uint64_t* src, const uint32_t* idx, uint32_t n, uint32_t k,
                                uint64_t* dst, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    scatter_keys_kernel<<<(n * k + 255) / 256, 256, 0, stream>>>(src, idx, n, k, dst);
    return cudaGetLastError();
}

// Result rows of re-run queries back into the batch's result arrays (deferred proof failures of
// fvdb_search_device_submit): row i of the sources goes to row idx[i] of the destinations.
__global__ void scatter_result_rows_kernel(const uint32_t* __restrict__ ids, const float* __restrict__ dist,
                                           const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ idx,
                                           uint32_t n, uint32_t k, uint32_t* __restrict__ out_ids,
                                           float* __restrict__ out_dist, uint32_t* __restrict__ out_cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * k) return;
    const uint32_t r = i / k, c = i % k;
    out_ids[(size_t)idx[r] * k + c] = ids[i];
    out_dist[(size_t)idx[r] * k + c] = dist[i];
    if (c == 0) out_cnt[idx[r]] = cnt[r];
}

cudaError_t launch_scatter_result_rows(const uint32_t* ids, const float* dist, const uint32_t* cnt,
                                       const uint32_t* idx, uint32_t n, uint32_t k, uint32_t* out_ids,
                                       float* out_dist, uint32_t* out_cnt, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    scatter_result_rows_kernel<<<(n * k + 255) / 256, 256, 0, stream>>>(ids, dist, cnt, idx, n, k, out_ids, out_dist, out_cnt);
    return cudaGetLastError();
}

// The reference's 3x POST-filter (HybridIndex::search_with_filter, src/hybrid/core.rs:529-546) on the
// device: of a query's k3 = 3k candidates (already ascending) keep, in order, those whose row id has
// its bit set in `keep` (bit = "metadata present and filter.matches", evaluated once per row by the
// host), and truncate to k.  One thread per query: k3 <= 3 * k_max entries, a sequential compaction.
__global__ void postfilter_rows_kernel(const uint32_t* __restrict__ ids, const float* __restrict__ dist,
                                       const uint32_t* __restrict__ cnt, uint32_t nq, uint32_t k3, uint32_t k,
                                       const uint64_t* __restrict__ keep, uint64_t keep_bits,
                                       uint32_t* __restrict__ out_ids, float* __restrict__ out_dist,
                                       uint32_t* __restrict__ out_cnt) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    const uint32_t n = min(cnt[q], k3);
    uint32_t r = 0;
    for (uint32_t i = 0; i < n && r < k; ++i) {
        const uint32_t id = ids[(size_t)q * k3 + i];
        if (bit_test(keep, keep_bits, id)) {
            out_ids[(size_t)q * k + r] = id;
            out_dist[(size_t)q * k + r] = dist[(size_t)q * k3 + i];
            ++r;
        }
    }
    out_cnt[q] = r;
    for (; r < k; ++r) {
        out_ids[(size_t)q * k + r] = ID_NONE;
        out_dist[(size_t)q * k + r] = __uint_as_float(0x7f800000u);
    }
}

cudaError_t launch_postfilter_rows(const uint32_t* ids, const float* dist, const uint32_t* cnt, uint32_t nq,
                                   uint32_t k3, uint32_t k, const uint64_t* keep, uint64_t keep_bits,
                                   uint32_t* out_ids, float* out_dist, uint32_t* out_cnt, cudaStream_t stream) {
    if (nq == 0) return cudaSuccess;
    postfilter_rows_kernel<<<(nq + 127) / 128, 128, 0, stream>>>(ids, dist, cnt, nq, k3, k, keep, keep_bits, out_ids,
                                                                out_dist, out_cnt);
    return cudaGetLastError();
}

// NaN screen over a float matrix (the reference panics on NaN: src/ivf/core.rs:655,677).
__global__ void nan_check_kernel(const float* __restrict__ x, size_t n, int* __restrict__ flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    bool bad = false;
    for (; i < n; i += stride) bad |= isnan(x[i]);
    if (bad) *flag = 1;
}

cudaError_t launch_nan_check(const float* x, size_t n, int* flag, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    const uint32_t blocks = (uint32_t)min((size_t)148 * 8, (n + 255) / 256);
    nan_check_kernel<<<blocks, 256, 0, stream>>>(x, n, flag);
    return cudaGetLastError();
}

}  // namespace fvdb
