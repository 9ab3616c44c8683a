// layout.cu — HBM layout maintenance: stable grouping of rows by posting list, row gathers,
// id bitmaps.  The device layout replaces the reference's
// HashMap<ClusterId, InvertedList{HashMap<VectorId, Vec<f32>>}> (src/ivf/core.rs:112-118,157)
// with one row-major arena whose lists are contiguous row ranges (SURVEY Appendix C).
#include "common.cuh"
#include "kernels.cuh"

namespace fvdb {

namespace {

constexpr uint32_t MAX_UNITS = 2048;

struct GroupPlan {
    uint32_t unit;     // elements per warp-unit (multiple of 32)
    uint32_t n_units;
    uint32_t nk;       // nkeys + 1 (drop group)
};

GroupPlan plan_group(uint64_t n, uint32_t nkeys) {
    GroupPlan p;
    uint64_t u = (n + MAX_UNITS - 1) / MAX_UNITS;
    if (u < 256) u = 256;
    u = (u + 31) / 32 * 32;
    p.unit = (uint32_t)u;
    p.n_units = (uint32_t)((n + u - 1) / u);
    if (p.n_units == 0) p.n_units = 1;
    p.nk = nkeys + 1;
    return p;
}

__global__ void group_hist_kernel(const uint32_t* __restrict__ keys, uint64_t n, GroupPlan p,
                                  uint32_t* __restrict__ H) {
    const uint32_t unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (unit >= p.n_units) return;
    const uint64_t b = (uint64_t)unit * p.unit;
    const uint64_t e = min(n, b + p.unit);
    uint32_t* row = H + (size_t)unit * p.nk;
    for (uint64_t i = b + lane; i < e; i += 32) {
        uint32_t key = keys[i];
        if (key >= p.nk) key = p.nk - 1;
        atomicAdd(&row[key], 1u);
    }
}

// per key: exclusive scan down the unit axis; totals[key] = column sum
__global__ void group_colscan_kernel(uint32_t* __restrict__ H, GroupPlan p,
                                     uint32_t* __restrict__ totals) {
    const uint32_t key = blockIdx.x * blockDim.x + threadIdx.x;
    if (key >= p.nk) return;
    uint32_t run = 0;
    for (uint32_t u = 0; u < p.n_units; ++u) {
        const uint32_t v = H[(size_t)u * p.nk + key];
        H[(size_t)u * p.nk + key] = run;
        run += v;
    }
    totals[key] = run;
}

// single CTA: offsets[0..nk] = exclusive scan of totals; offsets[nk] = n
__global__ void group_offsets_kernel(const uint32_t* __restrict__ totals, uint32_t nk,
                                     uint32_t* __restrict__ offsets) {
    __shared__ uint32_t s[1024];
    __shared__ uint32_t carry;
    const int t = threadIdx.x;
    if (t == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < nk; base += 1024) {
        const uint32_t i = base + t;
        const uint32_t v = (i < nk) ? totals[i] : 0;
        s[t] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            uint32_t a = (t >= o) ? s[t - o] : 0;
            __syncthreads();
            s[t] += a;
            __syncthreads();
        }
        if (i < nk) offsets[i] = carry + s[t] - v;
        __syncthreads();
        if (t == 1023) carry += s[1023];
        __syncthreads();
    }
    if (t == 0) offsets[nk] = carry;
}

__global__ void group_rank_kernel(const uint32_t* __restrict__ keys, uint64_t n, GroupPlan p,
                                  uint32_t* __restrict__ H, const uint32_t* __restrict__ offsets,
                                  uint32_t* __restrict__ perm) {
    const uint32_t unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (unit >= p.n_units) return;
    const uint64_t b = (uint64_t)unit * p.unit;
    const uint64_t e = min(n, b + p.unit);
    uint32_t* row = H + (size_t)unit * p.nk;
    for (uint64_t c = b; c < e; c += 32) {
        const uint64_t i = c + lane;
        const bool valid = i < e;
        uint32_t key = valid ? keys[i] : 0xFFFFFFFFu;
        if (valid && key >= p.nk) key = p.nk - 1;
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        const unsigned lt = (1u << lane) - 1u;
        const uint32_t rank = __popc(peers & lt);
        uint32_t base = 0;
        if (valid) base = row[key];
        __syncwarp();
        if (valid) {
            perm[offsets[key] + base + rank] = (uint32_t)i;
            if (rank == 0) row[key] = base + __popc(peers);
        }
        __syncwarp();
    }
}

__global__ void gather_rows_kernel(const float* __restrict__ src0, uint64_t n0,
                                   const float* __restrict__ src1, const uint32_t* __restrict__ perm,
                                   uint64_t n, uint32_t D, float* __restrict__ dst) {
    // one warp per destination row: coalesced both ways
    const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = warp; r < n; r += nwarps) {
        const uint32_t s = perm[r];
        const float* src = (s < n0) ? src0 + (size_t)s * D : src1 + (size_t)(s - n0) * D;
        float* d = dst + (size_t)r * D;
        if ((D & 3) == 0) {
            const float4* s4 = reinterpret_cast<const float4*>(src);
            float4* d4 = reinterpret_cast<float4*>(d);
            for (uint32_t c = lane; c < D / 4; c += 32) d4[c] = s4[c];
        } else {
            for (uint32_t c = lane; c < D; c += 32) d[c] = src[c];
        }
    }
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ src0, uint64_t n0,
                                  const uint32_t* __restrict__ src1, const uint32_t* __restrict__ perm,
                                  uint64_t n, uint32_t* __restrict__ dst) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const uint32_t s = perm[i];
        dst[i] = (s < n0) ? src0[s] : src1[s - n0];
    }
}

__global__ void keys_from_bitmap_kernel(const uint32_t* __restrict__ ids, uint64_t n,
                                        const uint64_t* __restrict__ bits, uint64_t nbits,
                                        uint32_t key_if_set, const uint32_t* __restrict__ keys_else,
                                        uint32_t key_if_clear, uint32_t* __restrict__ keys) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const bool set = bits && bit_test(bits, nbits, ids[i]);
        keys[i] = set ? key_if_set : (keys_else ? keys_else[i] : key_if_clear);
    }
}

__global__ void set_bits_kernel(uint64_t* __restrict__ bits, uint64_t nbits,
                                const uint32_t* __restrict__ ids, uint64_t n, int value) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const uint32_t id = ids[i];
        if (id >= nbits) continue;
        const unsigned long long m = 1ull << (id & 63);
        if (value) atomicOr(reinterpret_cast<unsigned long long*>(bits + (id >> 6)), m);
        else atomicAnd(reinterpret_cast<unsigned long long*>(bits + (id >> 6)), ~m);
    }
}

__global__ void filter_keys_mod_kernel(const uint32_t* __restrict__ keys, uint64_t n, uint32_t mod,
                                       uint32_t rem, uint32_t drop, uint32_t* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const uint32_t k = keys[i];
        out[i] = (k % mod == rem) ? k : drop;
    }
}

// re-placement after a sharded retrain: a row of a list this rank owns keeps its list as key (group l), a
// row of another rank's list gets nlist + that rank; an owner >= world goes to the drop group
__global__ void owner_keys_kernel(const uint32_t* __restrict__ lists, uint64_t n,
                                  const uint32_t* __restrict__ owner, uint32_t rank, uint32_t world,
                                  uint32_t nlist, uint32_t* __restrict__ keys) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const uint32_t l = lists[i];
        const uint32_t o = __ldg(owner + l);
        keys[i] = o == rank ? l : (o < world ? nlist + o : nlist + world);
    }
}

__global__ void extract_assign_kernel(const uint64_t* __restrict__ keys, uint64_t n,
                                      uint32_t* __restrict__ assign, float* __restrict__ dist,
                                      const uint32_t* __restrict__ prev, uint32_t* __restrict__ changed) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    bool ch = false;
    for (; i < n; i += stride) {
        const uint64_t k = keys[i];
        const uint32_t a = key_id(k);
        if (prev && prev[i] != a) ch = true;
        assign[i] = a;
        if (dist) dist[i] = key_dist(k);
    }
    if (ch && changed) *changed = 1u;
}

inline uint32_t grid_for(uint64_t n, uint32_t threads = 256) {
    uint64_t b = (n + threads - 1) / threads;
    const uint64_t cap = 148ull * 16;
    if (b > cap) b = cap;
    if (b == 0) b = 1;
    return (uint32_t)b;
}

}  // namespace

size_t stable_group_scratch_bytes(uint64_t n, uint32_t nkeys) {
    const GroupPlan p = plan_group(n, nkeys);
    return ((size_t)p.n_units * p.nk + p.nk + 16) * sizeof(uint32_t);
}

cudaError_t launch_stable_group(const uint32_t* keys, uint64_t n, uint32_t nkeys, uint32_t* offsets,
                                uint32_t* perm, void* scratch, cudaStream_t stream) {
    const GroupPlan p = plan_group(n, nkeys);
    uint32_t* H = reinterpret_cast<uint32_t*>(scratch);
    uint32_t* totals = H + (size_t)p.n_units * p.nk;
    cudaError_t e = cudaMemsetAsync(H, 0, (size_t)p.n_units * p.nk * sizeof(uint32_t), stream);
    if (e != cudaSuccess) return e;
    const uint32_t wblocks = (p.n_units * 32 + 255) / 256;
    if (n > 0) group_hist_kernel<<<wblocks, 256, 0, stream>>>(keys, n, p, H);
    group_colscan_kernel<<<(p.nk + 127) / 128, 128, 0, stream>>>(H, p, totals);
    group_offsets_kernel<<<1, 1024, 0, stream>>>(totals, p.nk, offsets);
    if (n > 0) group_rank_kernel<<<wblocks, 256, 0, stream>>>(keys, n, p, H, offsets, perm);
    return cudaGetLastError();
}

cudaError_t launch_gather_rows(const float* src0, uint64_t n0, const float* src1, const uint32_t* perm,
                               uint64_t n, uint32_t D, float* dst, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    gather_rows_kernel<<<grid_for(n * 32), 256, 0, stream>>>(src0, n0, src1, perm, n, D, dst);
    return cudaGetLastError();
}

cudaError_t launch_gather_u32(const uint32_t* src0, uint64_t n0, const uint32_t* src1,
                              const uint32_t* perm, uint64_t n, uint32_t* dst, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    gather_u32_kernel<<<grid_for(n), 256, 0, stream>>>(src0, n0, src1, perm, n, dst);
    return cudaGetLastError();
}

cudaError_t launch_keys_from_bitmap(const uint32_t* ids, uint64_t n, const uint64_t* bits,
                                    uint64_t nbits, uint32_t key_if_set, const uint32_t* keys_else,
                                    uint32_t key_if_clear, uint32_t* keys, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    keys_from_bitmap_kernel<<<grid_for(n), 256, 0, stream>>>(ids, n, bits, nbits, key_if_set,
                                                            keys_else, key_if_clear, keys);
    return cudaGetLastError();
}

cudaError_t launch_set_bits(uint64_t* bits, uint64_t nbits, const uint32_t* ids, uint64_t n, int value,
                            cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    set_bits_kernel<<<grid_for(n), 256, 0, stream>>>(bits, nbits, ids, n, value);
    return cudaGetLastError();
}

cudaError_t launch_filter_keys_mod(const uint32_t* keys, uint64_t n, uint32_t mod, uint32_t rem,
                                   uint32_t drop, uint32_t* keys_out, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    filter_keys_mod_kernel<<<grid_for(n), 256, 0, stream>>>(keys, n, mod, rem, drop, keys_out);
    return cudaGetLastError();
}

cudaError_t launch_owner_keys(const uint32_t* lists, uint64_t n, const uint32_t* owner, uint32_t rank,
                              uint32_t world, uint32_t nlist, uint32_t* keys, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    owner_keys_kernel<<<grid_for(n), 256, 0, stream>>>(lists, n, owner, rank, world, nlist, keys);
    return cudaGetLastError();
}

cudaError_t launch_extract_assign(const uint64_t* keys, uint64_t n, uint32_t* assign, float* dist,
                                  const uint32_t* prev_assign, uint32_t* changed, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    extract_assign_kernel<<<grid_for(n), 256, 0, stream>>>(keys, n, assign, dist, prev_assign, changed);
    return cudaGetLastError();
}

}  // namespace fvdb
