// Selection primitives of the search kernels (flat_search.cu, seq_match.cu, ivfpq.cu, ivfpq_lm.cu): the 64-bit sort keys,
// the block sorts, the warp / block reductions and the top-k merge.  Every search orders its results through these, so
// the key layouts and the tie rules -- lower row / list / label first -- are defined here once.
#pragma once
#include <cstdint>

#include "ptx.cuh"

namespace nafp {

// ---- descending score key: larger score first, equal scores to the lower row.  0 is below every real key.
__device__ __forceinline__ uint64_t score_key(float s, uint32_t row) {
    return (static_cast<uint64_t>(static_cast<uint32_t>(f2ord(s)) ^ 0x80000000u) << 32) | (0xFFFFFFFFu - row);
}
__device__ __forceinline__ float key_score(uint64_t key) {
    return ord2f(static_cast<int>(static_cast<uint32_t>(key >> 32) ^ 0x80000000u));
}
__device__ __forceinline__ uint32_t key_row(uint64_t key) { return 0xFFFFFFFFu - static_cast<uint32_t>(key); }

// ---- ascending distance key (distances >= 0): smaller distance first, equal distances to the lower id.  ~0 is past
// every real key.
__device__ __forceinline__ uint64_t dist_key(float d, uint32_t id) {
    return (static_cast<uint64_t>(__float_as_uint(d)) << 32) | id;
}
__device__ __forceinline__ float key_dist(uint64_t key) { return __uint_as_float(static_cast<uint32_t>(key >> 32)); }
__device__ __forceinline__ uint32_t key_id(uint64_t key) { return static_cast<uint32_t>(key); }

// the first k of ascending distance keys -> one row of D / I, +inf / -1 past the last real key (whole block)
__device__ __forceinline__ void store_topk(const uint64_t* keys, int k, int64_t label_offset, float* D, int64_t* I) {
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        const uint64_t key = keys[j];
        const bool real = key != ~0ull;
        D[j] = real ? key_dist(key) : INFINITY;
        I[j] = real ? static_cast<int64_t>(key_id(key)) + label_offset : -1;
    }
}

// ---- bitonic sorts of n (a power of two) entries in shared memory by the whole block
template <bool Ascending>
__device__ __forceinline__ void block_sort_u64(uint64_t* keys, int n) {
    for (int k = 2; k <= n; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint64_t a = keys[i], b = keys[ixj];
                    const bool up = ((i & k) == 0) == Ascending;
                    if (up ? (a > b) : (a < b)) { keys[i] = b; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
}
// (distance, label) pairs, ascending by distance, then label
__device__ __forceinline__ void block_sort_dist_label(float* d, int64_t* id, int n) {
    for (int k = 2; k <= n; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const float da = d[i], db = d[ixj];
                    const int64_t ia = id[i], ib = id[ixj];
                    const bool a_after_b = (da > db) || (da == db && ia > ib);
                    if (((i & k) == 0) ? a_after_b : !a_after_b) {
                        d[i] = db; d[ixj] = da;
                        id[i] = ib; id[ixj] = ia;
                    }
                }
            }
            __syncthreads();
        }
}

// ---- 128-bit entries of the device-wide sorts of the clip matcher (seq_match.cu): ascending by (hi, lo); all ones is
// past every real entry
struct SortKV {
    uint64_t hi, lo;
};
__device__ __forceinline__ bool kv_greater(const SortKV& a, const SortKV& b) {
    return a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo);
}
// s[i] <= s[j] afterwards
__device__ __forceinline__ void kv_order(SortKV* s, int64_t i, int64_t j) {
    const SortKV a = s[i], b = s[j];
    if (kv_greater(a, b)) { s[i] = b; s[j] = a; }
}
// the lower index of compare pair p at stride j (a power of two): pairs (i, i + j) with bit j of i clear
__device__ __forceinline__ int64_t pair_lo(int64_t p, int64_t j) { return ((p & ~(j - 1)) << 1) | (p & (j - 1)); }
// ascending bitonic sort of n (a power of two) entries in shared memory by the whole block
__device__ __forceinline__ void block_sort_kv(SortKV* s, int n) {
    for (int k = 2; k <= n; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int p = threadIdx.x; p < (n >> 1); p += blockDim.x) {
                const int i = static_cast<int>(pair_lo(p, j));
                if ((i & k) == 0) kv_order(s, i, i + j);
                else kv_order(s, i + j, i);
            }
            __syncthreads();
        }
}
// the closing steps (strides n/2 .. 1) of an ascending bitonic merge whose larger strides are done
__device__ __forceinline__ void block_merge_kv(SortKV* s, int n) {
    for (int j = n >> 1; j > 0; j >>= 1) {
        for (int p = threadIdx.x; p < (n >> 1); p += blockDim.x) {
            const int i = static_cast<int>(pair_lo(p, j));
            kv_order(s, i, i + j);
        }
        __syncthreads();
    }
}

// ---- reductions
// arg-min over the warp, ties to the lower index; every lane returns the winner
__device__ __forceinline__ void warp_argmin(float& best, int& idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ob < best || (ob == best && oi < idx)) { best = ob; idx = oi; }
    }
}
__device__ __forceinline__ uint64_t warp_max_u64(uint64_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint64_t other = __shfl_xor_sync(0xffffffffu, v, o);
        v = other > v ? other : v;
    }
    return v;
}
// max over a block of 8 warps; every thread returns it.  red[8] is shared; the caller separates two calls by a barrier.
__device__ __forceinline__ uint64_t block_max_u64(uint64_t v, uint64_t* red) {
    v = warp_max_u64(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    uint64_t b = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) b = red[w] > b ? red[w] : b;
    return b;
}

// ---- merge of W top-k lists of (distance, label) into one (seq_match.cu): one block of 128 threads per query row sorts
// all W * k entries in shared memory
constexpr int TOPK_MERGE_KEYS = 4096;     // 16 + 32 KB: the static shared-memory limit
__global__ void __launch_bounds__(128)
topk_merge_kernel(const float* __restrict__ D_all, const int64_t* __restrict__ I_all, int W, int64_t nq, int k,
                  float* __restrict__ D_out, int64_t* __restrict__ I_out);

}  // namespace nafp
