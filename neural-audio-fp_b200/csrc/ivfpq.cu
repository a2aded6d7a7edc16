// IVF-PQ index (SURVEY §8 a6): faiss.IndexIVFPQ(IndexFlatL2(d), d, nlist=256, M=64, nbits=8) as the
// reference builds it (eval/utils/get_index_faiss.py:69-74), trained by k-means (:105-117), searched
// with nprobe = 40 (:120).  L2 metric, residual encoding, dsub = d / M.
//
//   train   k-means (Lloyd, 25 iterations, <= 256 points per centroid, seeded) for the coarse
//           quantizer, then one k-means per sub-space on the residuals; deterministic (fixed-order sums)
//   add     ivfpq_encode_kernel: nearest coarse centroid + 64 one-byte codes per row; the inverted
//           lists are a stable counting sort of (list, row) rebuilt lazily before the next search
//   search  by default the list-major tensor-core scan of the compressed lists (ivfpq_lm.cu).  The LUT kernel
//           below is the reference formulation: it answers the query rows and shapes the list-major scan cannot
//           (and every search of an index created with NAFP_IVFPQ_PATH=lut):
//           ivfpq_probe_kernel (nprobe nearest lists per query row) ->
//           ivfpq_scan_kernel  (one CTA per (query row, probed list): 64 x 256 fp32 look-up table in
//                               shared memory, ADC scan of the list's codes, block top-k) ->
//           topk merge of the nprobe partial lists.
//
// IVF-Flat ('ivf', faiss.IndexIVFFlat(IndexFlatL2(d), d, nlist=400), get_index_faiss.py:63-66) shares the coarse
// quantizer and the probe: the exact flat scan of the index's own rows gives the 64 nearest rows, the filter drops
// the ones outside the probed lists; rows left with fewer than k answers get an exact scan of their probed lists
// (ivfflat_scan_kernel).
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <random>
#include <vector>

#include "ivfpq.h"
#include "ptx.cuh"

namespace nafp {

// ------------------------------------------------------------------------------------------ k-means
// nearest centroid of `dim`-dimensional points (row stride `ld` floats); one warp per point, lane l
// scans centroids l, l+32, ...; ties go to the lower centroid id
__global__ void kmeans_assign_kernel(const float* __restrict__ x, int64_t n, int ld, int dim,
                                     const float* __restrict__ cent, int k, int32_t* __restrict__ assign,
                                     float* __restrict__ dist_out) {
    extern __shared__ float xs[];      // [warps][dim]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (i >= n) return;
    float* xr = xs + w * dim;
    for (int j = lane; j < dim; j += 32) xr[j] = x[i * ld + j];
    __syncwarp();
    float best = FLT_MAX;
    int bi = INT_MAX;
    for (int c = lane; c < k; c += 32) {
        const float* cr = cent + static_cast<int64_t>(c) * dim;
        float d = 0.f;
        for (int j = 0; j < dim; ++j) {        // d = fma(t, t, d), j ascending: the oracle's k-means (oracle.c) rounds identically
            const float t = xr[j] - __ldg(cr + j);
            d = fmaf(t, t, d);
        }
        if (d < best) { best = d; bi = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) {
        assign[i] = bi;
        if (dist_out) dist_out[i] = best;
    }
}

// new centroid c = mean of its points; one block per centroid, fixed summation order; empty clusters keep
// their previous centroid
__global__ void kmeans_update_kernel(const float* __restrict__ x, int64_t n, int ld, int dim,
                                     const int32_t* __restrict__ assign, float* __restrict__ cent) {
    __shared__ double red[256];
    __shared__ int cnt_s[256];
    const int c = blockIdx.x;
    const int tid = threadIdx.x;
    // every thread scans a strided share of the points; dims are looped (dim <= 128)
    int cnt = 0;
    for (int64_t i = tid; i < n; i += blockDim.x) cnt += assign[i] == c ? 1 : 0;
    cnt_s[tid] = cnt;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (tid < s) cnt_s[tid] += cnt_s[tid + s];
        __syncthreads();
    }
    const int total = cnt_s[0];
    __syncthreads();
    if (total == 0) return;
    for (int j = 0; j < dim; ++j) {
        double acc = 0.0;
        for (int64_t i = tid; i < n; i += blockDim.x)
            if (assign[i] == c) acc += x[i * ld + j];
        red[tid] = acc;
        __syncthreads();
        for (int s = blockDim.x / 2; s > 0; s >>= 1) {
            if (tid < s) red[tid] += red[tid + s];
            __syncthreads();
        }
        if (tid == 0) cent[static_cast<int64_t>(c) * dim + j] = static_cast<float>(red[0] / total);
        __syncthreads();
    }
}

__global__ void residual_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ coarse,
                                const int32_t* __restrict__ assign, float* __restrict__ r) {
    const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= n * D128) return;
    const int64_t i = idx / D128;
    const int j = static_cast<int>(idx % D128);
    r[idx] = x[idx] - coarse[static_cast<int64_t>(assign[i]) * D128 + j];
}

__global__ void gather_rows_kernel(const float* __restrict__ x, int ld, int dim, const int32_t* __restrict__ rows,
                                   int k, float* __restrict__ out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= k * dim) return;
    out[idx] = x[static_cast<int64_t>(rows[idx / dim]) * ld + idx % dim];
}

// Seeded choice of `cnt` of n rows, defined so that any implementation can reproduce it (the oracle does, in numpy:
// oracle/ivfpq_index.py select_rows): row i gets the key splitmix64(seed * 0xD1342543DE82EF95 + i); the cnt rows with
// the smallest (key, i) are chosen and returned in ascending row order.
static inline uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
static std::vector<int64_t> select_rows(int64_t n, int64_t cnt, uint64_t seed) {
    std::vector<std::pair<uint64_t, int64_t>> keyed(static_cast<size_t>(n));
    const uint64_t base = seed * 0xD1342543DE82EF95ull;
    for (int64_t i = 0; i < n; ++i) keyed[i] = {splitmix64(base + static_cast<uint64_t>(i)), i};
    if (cnt > n) cnt = n;
    std::nth_element(keyed.begin(), keyed.begin() + cnt, keyed.end());
    std::vector<int64_t> rows(static_cast<size_t>(cnt));
    for (int64_t i = 0; i < cnt; ++i) rows[i] = keyed[i].second;
    std::sort(rows.begin(), rows.end());
    return rows;
}

static int run_kmeans(nafp_ctx* ctx, const float* x_dev, int64_t n, int ld, int dim, int k, float* cent_dev,
                      int32_t* assign_dev, int niter, uint64_t seed) {
    // initial centroids: k distinct training points (select_rows), in ascending row order
    const std::vector<int64_t> rows = select_rows(n, k, seed);
    int32_t* rows_dev = nullptr;
    NAFP_CUDA(cudaMalloc(&rows_dev, k * sizeof(int32_t)));
    std::vector<int32_t> first(k);
    for (int i = 0; i < k; ++i) first[i] = static_cast<int32_t>(rows[i % std::max<size_t>(rows.size(), 1)]);
    NAFP_CUDA(cudaMemcpyAsync(rows_dev, first.data(), k * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    gather_rows_kernel<<<(k * dim + 255) / 256, 256, 0, ctx->stream>>>(x_dev, ld, dim, rows_dev, k, cent_dev);
    const int threads = 256, warps = threads / 32;
    const unsigned blocks = static_cast<unsigned>((n + warps - 1) / warps);
    for (int it = 0; it < niter; ++it) {
        kmeans_assign_kernel<<<blocks, threads, warps * dim * sizeof(float), ctx->stream>>>(x_dev, n, ld, dim, cent_dev, k,
                                                                                         assign_dev, nullptr);
        kmeans_update_kernel<<<k, 256, 0, ctx->stream>>>(x_dev, n, ld, dim, assign_dev, cent_dev);
        ctx->launches += 2;
    }
    NAFP_CUDA(cudaGetLastError());
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    cudaFree(rows_dev);
    return NAFP_OK;
}

// ------------------------------------------------------------------------------------------ add
// one warp per row: nearest coarse centroid, residual, then lane l encodes sub-spaces l and l + 32
__global__ void __launch_bounds__(256)
ivfpq_encode_kernel(const float* __restrict__ x32, int64_t row0, int64_t n, const float* __restrict__ coarse,
                    int nlist, const float* __restrict__ pq, int m, int dsub, int32_t* __restrict__ assign,
                    uint8_t* __restrict__ codes) {
    __shared__ float xs[8][D128];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    for (int64_t r = ((static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5); r < n; r += nwarps) {
        const int64_t row = row0 + r;
        float* xr = xs[w];
        reinterpret_cast<float4*>(xr)[lane] = reinterpret_cast<const float4*>(x32 + row * D128)[lane];
        __syncwarp();
        float best = FLT_MAX;
        int bi = INT_MAX;
        for (int c = lane; c < nlist; c += 32) {
            const float* cr = coarse + static_cast<int64_t>(c) * D128;
            float d = 0.f;
#pragma unroll 8
            for (int j = 0; j < D128; ++j) {
                const float t = xr[j] - __ldg(cr + j);
                d += t * t;
            }
            if (d < best) { best = d; bi = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (lane == 0) assign[row] = bi;
        // residual in place
        {
            const float4 cv = reinterpret_cast<const float4*>(coarse + static_cast<int64_t>(bi) * D128)[lane];
            float4 v = reinterpret_cast<float4*>(xr)[lane];
            v.x -= cv.x; v.y -= cv.y; v.z -= cv.z; v.w -= cv.w;
            __syncwarp();
            reinterpret_cast<float4*>(xr)[lane] = v;
        }
        __syncwarp();
        for (int sub = lane; sub < m; sub += 32) {
            const float* pc = pq + static_cast<int64_t>(sub) * PQ_KSUB * dsub;
            float bd = FLT_MAX;
            int bc = 0;
            for (int c = 0; c < PQ_KSUB; ++c) {
                float d = 0.f;
                for (int j = 0; j < dsub; ++j) {
                    const float t = xr[sub * dsub + j] - __ldg(pc + c * dsub + j);
                    d += t * t;
                }
                if (d < bd) { bd = d; bc = c; }
            }
            codes[row * m + sub] = static_cast<uint8_t>(bc);
        }
        __syncwarp();
    }
}

// The same two steps for the reference's shape (nlist <= 256, M = 64, dsub = 2) with the tables in shared memory: the
// 56 M-row build spent 13.5 s in the kernel above, whose 128 KB codebook thrashes L1.  Arithmetic and tie-breaking are
// the kernel's above (fma chains, dimensions ascending, first minimum wins), so assignments and codes are identical.
constexpr int ENC_NLIST = 256;
constexpr int ENC_ASSIGN_SMEM = (D128 * ENC_NLIST + 8 * D128) * 4;          // transposed centroids + 8 rows
constexpr int ENC_CODE_SMEM = PQ_KSUB * 64 * 8 + 8 * D128 * 4;              // [code][sub] float2 + 8 residual rows
__global__ void __launch_bounds__(256)
ivfpq_assign_smem_kernel(const float* __restrict__ x32, int64_t row0, int64_t n, const float* __restrict__ coarse, int nlist,
                         int32_t* __restrict__ assign) {
    extern __shared__ float esm[];
    float* cs = esm;                                   // [dim][256 centroids]
    float* xs = esm + D128 * ENC_NLIST;                // [8 warps][128]
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < D128 * ENC_NLIST; e += blockDim.x) {
        const int j = e / ENC_NLIST, c = e % ENC_NLIST;
        cs[e] = c < nlist ? __ldg(coarse + static_cast<int64_t>(c) * D128 + j) : 0.f;
    }
    __syncthreads();
    float* xr = xs + w * D128;
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + w; r < n; r += static_cast<int64_t>(gridDim.x) * 8) {
        __syncwarp();
        reinterpret_cast<float4*>(xr)[lane] = reinterpret_cast<const float4*>(x32 + (row0 + r) * D128)[lane];
        __syncwarp();
        float d[ENC_NLIST / 32];
#pragma unroll
        for (int t = 0; t < ENC_NLIST / 32; ++t) d[t] = 0.f;
#pragma unroll 4
        for (int j = 0; j < D128; ++j) {
            const float xj = xr[j];
            const float* cr = cs + j * ENC_NLIST + lane;
#pragma unroll
            for (int t = 0; t < ENC_NLIST / 32; ++t) {
                const float v = xj - cr[32 * t];
                d[t] = fmaf(v, v, d[t]);
            }
        }
        float best = FLT_MAX;
        int bi = INT_MAX;
#pragma unroll
        for (int t = 0; t < ENC_NLIST / 32; ++t)              // centroid lane + 32 t, ascending: the first minimum wins
            if (lane + 32 * t < nlist && d[t] < best) { best = d[t]; bi = lane + 32 * t; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (lane == 0) assign[row0 + r] = bi;
    }
}
__global__ void __launch_bounds__(256)
ivfpq_code_smem_kernel(const float* __restrict__ x32, int64_t row0, int64_t n, const float* __restrict__ coarse,
                       const float* __restrict__ pq, const int32_t* __restrict__ assign, uint8_t* __restrict__ codes) {
    extern __shared__ float esm[];
    float2* pqs = reinterpret_cast<float2*>(esm);      // [code][sub]: lane = sub-quantizer reads consecutive 8 bytes
    float* xs = esm + PQ_KSUB * 64 * 2;                // [8 warps][128] residuals
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int e = threadIdx.x; e < PQ_KSUB * 64; e += blockDim.x) {
        const int c = e >> 6, sub = e & 63;
        pqs[e] = __ldg(reinterpret_cast<const float2*>(pq) + sub * PQ_KSUB + c);
    }
    __syncthreads();
    float* xr = xs + w * D128;
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + w; r < n; r += static_cast<int64_t>(gridDim.x) * 8) {
        const int64_t row = row0 + r;
        const float4 cv = reinterpret_cast<const float4*>(coarse + static_cast<int64_t>(assign[row]) * D128)[lane];
        float4 v = reinterpret_cast<const float4*>(x32 + row * D128)[lane];
        v.x -= cv.x; v.y -= cv.y; v.z -= cv.z; v.w -= cv.w;
        __syncwarp();
        reinterpret_cast<float4*>(xr)[lane] = v;
        __syncwarp();
        const float a0 = xr[2 * lane], a1 = xr[2 * lane + 1];                 // sub-quantizer lane
        const float b0 = xr[2 * (lane + 32)], b1 = xr[2 * (lane + 32) + 1];   // sub-quantizer lane + 32
        float bda = FLT_MAX, bdb = FLT_MAX;
        int bca = 0, bcb = 0;
#pragma unroll 4
        for (int c = 0; c < PQ_KSUB; ++c) {
            const float2 pa = pqs[c * 64 + lane], pb = pqs[c * 64 + 32 + lane];
            const float ta0 = a0 - pa.x, ta1 = a1 - pa.y, tb0 = b0 - pb.x, tb1 = b1 - pb.y;
            const float da = fmaf(ta1, ta1, ta0 * ta0), db = fmaf(tb1, tb1, tb0 * tb0);
            if (da < bda) { bda = da; bca = c; }
            if (db < bdb) { bdb = db; bcb = c; }
        }
        codes[row * 64 + lane] = static_cast<uint8_t>(bca);
        codes[row * 64 + 32 + lane] = static_cast<uint8_t>(bcb);
    }
}

// ------------------------------------------------------------------------------------------ inverted lists
constexpr int SORT_CHUNK = 4096;     // rows per (single-warp) block of the stable counting sort

__global__ void ivf_hist_kernel(const int32_t* __restrict__ assign, int64_t n, int nlist, int32_t* __restrict__ hist) {
    // hist[list][chunk]; one warp per chunk
    __shared__ int h[IVF_MAX_NLIST];
    const int chunk = blockIdx.x, nchunks = gridDim.x;
    for (int l = threadIdx.x; l < nlist; l += 32) h[l] = 0;
    __syncwarp();
    const int64_t lo = static_cast<int64_t>(chunk) * SORT_CHUNK;
    const int64_t hi = lo + SORT_CHUNK < n ? lo + SORT_CHUNK : n;
    for (int64_t i = lo + threadIdx.x; i < hi; i += 32) atomicAdd(&h[assign[i]], 1);
    __syncwarp();
    for (int l = threadIdx.x; l < nlist; l += 32) hist[static_cast<int64_t>(l) * nchunks + chunk] = h[l];
}

__global__ void ivf_scatter_kernel(const int32_t* __restrict__ assign, const uint8_t* __restrict__ codes, int64_t n,
                                   int nlist, int m, const int64_t* __restrict__ base, uint8_t* __restrict__ lcodes,
                                   int32_t* __restrict__ lids) {
    // base[list][chunk] = first slot of this chunk's rows inside the list; rows keep their order (stable)
    __shared__ int64_t run[IVF_MAX_NLIST];
    const int chunk = blockIdx.x, nchunks = gridDim.x, lane = threadIdx.x;
    for (int l = lane; l < nlist; l += 32) run[l] = base[static_cast<int64_t>(l) * nchunks + chunk];
    __syncwarp();
    const int64_t lo = static_cast<int64_t>(chunk) * SORT_CHUNK;
    const int64_t hi = lo + SORT_CHUNK < n ? lo + SORT_CHUNK : n;
    for (int64_t i0 = lo; i0 < hi; i0 += 32) {
        const int64_t i = i0 + lane;
        const bool ok = i < hi;
        const int l = ok ? assign[i] : -1 - lane;
        const unsigned peers = __match_any_sync(0xffffffffu, l);
        const int rank = __popc(peers & ((1u << lane) - 1));
        int64_t pos = 0;
        if (ok) pos = run[l] + rank;
        __syncwarp();
        if (ok && rank == __popc(peers) - 1) run[l] += __popc(peers);     // last peer advances the list cursor
        __syncwarp();
        if (ok) {
            lids[pos] = static_cast<int32_t>(i);
            if (codes) {                          // IVF-Flat lists carry row ids only
                const uint4* src = reinterpret_cast<const uint4*>(codes + i * m);
                for (int v = 0; v < m / 16; ++v) {
                    const uint4 cw = src[v];
                    const uint32_t wds[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                    for (int t = 0; t < 4; ++t)
#pragma unroll
                        for (int b = 0; b < 4; ++b)
                            lcodes[lcode_off(pos, v * 16 + t * 4 + b, m)] = static_cast<uint8_t>(wds[t] >> (8 * b));
                }
            }
        }
    }
}

// the inverse of the scatter: row-order codes from the lists (one thread per list position)
__global__ void ivf_unscatter_kernel(const uint8_t* __restrict__ lcodes, const int32_t* __restrict__ lids, int64_t n_pos, int m,
                                     uint8_t* __restrict__ codes) {
    const int64_t pos = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (pos >= n_pos) return;
    const int32_t row = lids[pos];
    if (row < 0) return;
    for (int sub = 0; sub < m; ++sub) codes[static_cast<int64_t>(row) * m + sub] = lcodes[lcode_off(pos, sub, m)];
}

// ------------------------------------------------------------------------------------------ search
// one warp per query row: the nprobe nearest coarse centroids, ascending (ties -> lower list id)
__global__ void ivfpq_probe_kernel(const float* __restrict__ q, int64_t nq, const float* __restrict__ coarse,
                                   int nlist, int nprobe, int32_t* __restrict__ probes) {
    __shared__ float qs[8][D128];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (i >= nq) return;
    reinterpret_cast<float4*>(qs[w])[lane] = reinterpret_cast<const float4*>(q + i * D128)[lane];
    __syncwarp();
    float d[IVF_MAX_NLIST / 32];
#pragma unroll
    for (int t = 0; t < IVF_MAX_NLIST / 32; ++t) {
        const int c = lane + 32 * t;
        float acc = FLT_MAX;
        if (c < nlist) {
            acc = 0.f;
            const float* cr = coarse + static_cast<int64_t>(c) * D128;
            for (int j = 0; j < D128; ++j) {
                const float v = qs[w][j] - __ldg(cr + j);
                acc = fmaf(v, v, acc);
            }
        }
        d[t] = acc;
    }
    for (int p = 0; p < nprobe; ++p) {
        float best = FLT_MAX;
        int bi = INT_MAX;
#pragma unroll
        for (int t = 0; t < IVF_MAX_NLIST / 32; ++t)
            if (d[t] < best) { best = d[t]; bi = lane + 32 * t; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (lane == 0) probes[i * nprobe + p] = bi == INT_MAX ? -1 : bi;
#pragma unroll
        for (int t = 0; t < IVF_MAX_NLIST / 32; ++t)
            if (lane + 32 * t == bi) d[t] = FLT_MAX;
    }
}

// CTA (probe p, query row i): LUT T[m][c] = |(q - c_l)_m - pq_m[c]|^2 in shared memory, ADC scan of list l
__global__ void __launch_bounds__(256)
ivfpq_scan_kernel(const float* __restrict__ q, int64_t nq, const float* __restrict__ coarse,
                  const float* __restrict__ pq, int m, int dsub, const int32_t* __restrict__ probes, int nprobe,
                  const uint8_t* __restrict__ lcodes, const int32_t* __restrict__ lids, const int32_t* __restrict__ loff,
                  const int32_t* __restrict__ lend, int k, int64_t label_offset, int64_t n_search, float* __restrict__ partD,
                  int64_t* __restrict__ partI) {
    extern __shared__ float lut[];                          // [m][256]
    __shared__ uint64_t buf[IVF_SCAN_CAP];
    __shared__ int cnt_s;
    __shared__ unsigned long long thr_s;
    const int p = blockIdx.x;
    const int64_t i = blockIdx.y;
    const int tid = threadIdx.x;
    const int l = probes[i * nprobe + p];
    float* outD = partD + (static_cast<int64_t>(p) * nq + i) * k;
    int64_t* outI = partI + (static_cast<int64_t>(p) * nq + i) * k;
    const int64_t lo = l >= 0 ? loff[l] : 0, hi = l >= 0 ? lend[l] : 0;
    if (hi <= lo) {
        for (int j = tid; j < k; j += blockDim.x) { outD[j] = INFINITY; outI[j] = -1; }
        return;
    }
    for (int e = tid; e < m * PQ_KSUB; e += blockDim.x) {
        const int sub = e >> 8, c = e & 255;
        float d = 0.f;
        for (int j = 0; j < dsub; ++j) {
            const int dim = sub * dsub + j;
            const float r = q[i * D128 + dim] - coarse[static_cast<int64_t>(l) * D128 + dim];
            const float t = r - pq[(static_cast<int64_t>(sub) * PQ_KSUB + c) * dsub + j];
            d = fmaf(t, t, d);            // (what the compiler contracts `d += t * t` to; spelled out because ivfpq_lm.cu's
                                          // exact re-rank must round identically)
        }
        lut[e] = d;
    }
    for (int e = tid; e < IVF_SCAN_CAP; e += blockDim.x) buf[e] = ~0ull;
    if (tid == 0) { cnt_s = 0; thr_s = ~0ull; }
    __syncthreads();
    for (int64_t base = lo; base < hi; base += blockDim.x) {
        const int64_t pos = base + tid;
        if (pos < hi && lids[pos] < n_search) {          // rows past n_search are the halo of a row-sharded index
            // (the codes are stored tile-transposed for the list-major scan, lcode_off: the position's byte of every
            // 4-byte word of its 4 * mlo-byte segment, one segment per group of 32 sub-quantizers)
            const int mlo = m < 32 ? m : 32;
            const uint8_t* seg = lcodes + lcode_off(pos & ~static_cast<int64_t>(3), 0, m);
            const int sh = static_cast<int>(pos & 3) * 8;
            float d = 0.f;
            for (int kb = 0; kb < m / mlo; ++kb) {
                const uint4* lp = reinterpret_cast<const uint4*>(seg + kb * (LIST_TILE * mlo));
                for (int v = 0; v < mlo / 4; ++v) {
                    const uint4 cw = lp[v];
                    const uint32_t wds[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                    for (int b = 0; b < 4; ++b) d += lut[(kb * mlo + 4 * v + b) * PQ_KSUB + ((wds[b] >> sh) & 255u)];
                }
            }
            const uint64_t key = (static_cast<uint64_t>(__float_as_uint(d)) << 32) | static_cast<uint32_t>(lids[pos]);
            if (key < thr_s) {
                const int slot = atomicAdd(&cnt_s, 1);
                buf[slot] = key;         // slot < CAP: the buffer is pruned whenever fewer than 256 slots remain
            }
        }
        // block-uniform decision: every thread reads the counter between two barriers, so that a warp that is
        // already inserting the next iteration's keys cannot make a slower warp take the branch alone
        __syncthreads();
        const int filled = cnt_s;
        __syncthreads();
        if (filled > IVF_SCAN_CAP - 256) {
            block_sort_asc_u64(buf, IVF_SCAN_CAP);
            for (int e = k + tid; e < IVF_SCAN_CAP; e += blockDim.x) buf[e] = ~0ull;
            if (tid == 0) { cnt_s = k; thr_s = buf[k - 1]; }
            __syncthreads();
        }
    }
    block_sort_asc_u64(buf, IVF_SCAN_CAP);
    for (int j = tid; j < k; j += blockDim.x) {
        const uint64_t key = buf[j];
        if (key != ~0ull) {
            outD[j] = __uint_as_float(static_cast<uint32_t>(key >> 32));
            outI[j] = static_cast<int64_t>(static_cast<uint32_t>(key)) + label_offset;
        } else {
            outD[j] = INFINITY;
            outI[j] = -1;
        }
    }
}

// IVF-Flat: CTA (probe p, query row i) scans the stored rows of list l exactly (fp32), a warp per row
__global__ void __launch_bounds__(256)
ivfflat_scan_kernel(const float* __restrict__ q, int64_t nq, const int32_t* __restrict__ probes, int nprobe,
                    const float* __restrict__ x32, const int32_t* __restrict__ lids, const int32_t* __restrict__ loff,
                    const int32_t* __restrict__ lend, int k, int64_t label_offset, int64_t n_search, float* __restrict__ partD, int64_t* __restrict__ partI) {
    __shared__ uint64_t buf[IVF_SCAN_CAP];
    __shared__ int cnt_s;
    __shared__ unsigned long long thr_s;
    const int p = blockIdx.x;
    const int64_t i = blockIdx.y;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int l = probes[i * nprobe + p];
    float* outD = partD + (static_cast<int64_t>(p) * nq + i) * k;
    int64_t* outI = partI + (static_cast<int64_t>(p) * nq + i) * k;
    const int64_t lo = l >= 0 ? loff[l] : 0, hi = l >= 0 ? lend[l] : 0;
    if (hi <= lo) {
        for (int j = tid; j < k; j += blockDim.x) { outD[j] = INFINITY; outI[j] = -1; }
        return;
    }
    const float4 qv = reinterpret_cast<const float4*>(q + i * D128)[lane];
    for (int e = tid; e < IVF_SCAN_CAP; e += blockDim.x) buf[e] = ~0ull;
    if (tid == 0) { cnt_s = 0; thr_s = ~0ull; }
    __syncthreads();
    constexpr int ROWS_PER_WARP = 8;          // 64 rows per block iteration: <= 64 new keys between two prune checks
    for (int64_t base = lo; base < hi; base += 8 * ROWS_PER_WARP) {
#pragma unroll 4
        for (int r = 0; r < ROWS_PER_WARP; ++r) {
            const int64_t pos = base + warp * ROWS_PER_WARP + r;
            const int32_t row = pos < hi ? lids[pos] : INT_MAX;
            if (row < n_search) {                        // (rows past n_search: halo of a row-sharded index)
                const float4 xv = reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(row) * D128)[lane];
                const float d0 = qv.x - xv.x, d1 = qv.y - xv.y, d2 = qv.z - xv.z, d3 = qv.w - xv.w;
                float d = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
                if (lane == 0) {
                    const uint64_t key = (static_cast<uint64_t>(__float_as_uint(d)) << 32) | static_cast<uint32_t>(row);
                    if (key < thr_s) buf[atomicAdd(&cnt_s, 1)] = key;      // slot < CAP: pruned below before it can fill
                }
            }
        }
        __syncthreads();
        const int filled = cnt_s;           // block-uniform (see ivfpq_scan_kernel)
        __syncthreads();
        if (filled > IVF_SCAN_CAP - 8 * ROWS_PER_WARP) {
            block_sort_asc_u64(buf, IVF_SCAN_CAP);
            for (int e = k + tid; e < IVF_SCAN_CAP; e += blockDim.x) buf[e] = ~0ull;
            if (tid == 0) { cnt_s = k; thr_s = buf[k - 1]; }
            __syncthreads();
        }
    }
    block_sort_asc_u64(buf, IVF_SCAN_CAP);
    for (int j = tid; j < k; j += blockDim.x) {
        const uint64_t key = buf[j];
        if (key != ~0ull) {
            outD[j] = __uint_as_float(static_cast<uint32_t>(key >> 32));
            outI[j] = static_cast<int64_t>(static_cast<uint32_t>(key)) + label_offset;
        } else {
            outD[j] = INFINITY;
            outI[j] = -1;
        }
    }
}

// IVF-Flat, one warp per query row: keep the flat scan's candidates whose list is probed, in order.  k of them (or
// all stored rows of the probed lists) ARE the restricted top-k; otherwise the row goes to ivfflat_scan_kernel.
__global__ void ivfpq_filter_kernel(const float* __restrict__ candD, const int64_t* __restrict__ candI, int64_t nq, int k,
                                    const int32_t* __restrict__ probes, int nprobe, const int32_t* __restrict__ assign,
                                    int64_t label_offset, float* __restrict__ D, int64_t* __restrict__ I,
                                    int32_t* __restrict__ redo_rows, int32_t* __restrict__ redo_count) {
    const int lane = threadIdx.x & 31;
    const int64_t q = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (q >= nq) return;
    int kept = 0;
    bool exhausted = false;            // fewer than IVFFLAT_K rows exist at all: the candidate list is complete
    for (int c0 = 0; c0 < IVFFLAT_K && kept < k; c0 += 32) {
        const int c = c0 + lane;
        const int64_t id = candI[q * IVFFLAT_K + c];
        bool in = false;
        if (id >= 0) {
            const int l = assign[id];
            for (int p = 0; p < nprobe; ++p) in = in || (probes[q * nprobe + p] == l);
        }
        if (__any_sync(0xffffffffu, id < 0)) exhausted = true;
        const unsigned mask = __ballot_sync(0xffffffffu, in);
        const int pos = kept + __popc(mask & ((1u << lane) - 1));
        if (in && pos < k) {
            D[q * k + pos] = candD[q * IVFFLAT_K + c];
            I[q * k + pos] = id + label_offset;
        }
        kept += __popc(mask);
    }
    if (kept >= k) return;
    if (exhausted) {                   // everything that exists was looked at: pad like faiss
        for (int j = kept + lane; j < k; j += 32) {
            D[q * k + j] = INFINITY;
            I[q * k + j] = -1;
        }
        return;
    }
    if (lane == 0) redo_rows[atomicAdd(redo_count, 1)] = static_cast<int32_t>(q);
}

__global__ void ivfpq_gather_q_kernel(const float* __restrict__ q, const int32_t* __restrict__ rows, int64_t n, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (w >= n) return;
    reinterpret_cast<float4*>(out + w * D128)[lane] = reinterpret_cast<const float4*>(q + static_cast<int64_t>(rows[w]) * D128)[lane];
}
__global__ void ivfpq_scatter_kernel(const float* __restrict__ Ds, const int64_t* __restrict__ Is, const int32_t* __restrict__ rows,
                                     int64_t n, int k, float* __restrict__ D, int64_t* __restrict__ I) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n * k) return;
    const int64_t w = i / k, j = i - w * k;
    D[static_cast<int64_t>(rows[w]) * k + j] = Ds[i];
    I[static_cast<int64_t>(rows[w]) * k + j] = Is[i];
}

// ------------------------------------------------------------------------------------------ IVFPQR
// xhat of a row from its list and PQ code: lane owns dims 4 lane .. 4 lane + 3 (two dsub = 2 sub-spaces, or one of 4, ...)
__device__ __forceinline__ float4 pq_reconstruct_lane(const float* __restrict__ coarse, const float* __restrict__ pq, int m,
                                                      int dsub, int list, const uint8_t* __restrict__ code, int lane) {
    float4 v = reinterpret_cast<const float4*>(coarse + static_cast<int64_t>(list) * D128)[lane];
    float* vv = reinterpret_cast<float*>(&v);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int dim = 4 * lane + j, sub = dim / dsub;
        vv[j] += pq[(static_cast<int64_t>(sub) * PQ_KSUB + code[sub]) * dsub + (dim - sub * dsub)];
    }
    return v;
}
// nearest of the 16 refinement codewords of sub-space (lane / 8) for the 32-dim residual slice spread over 8 lanes
// (4 dims each); every lane of the group returns the code.  Ties go to the lower code.
__device__ __forceinline__ int refine_encode_group(const float4 r, const float* __restrict__ rpq, int lane) {
    const int sub = lane >> 3, part = lane & 7;
    float best = FLT_MAX;
    int bi = 0;
    for (int c = 0; c < REFINE_KSUB; ++c) {
        const float4 w = reinterpret_cast<const float4*>(rpq + (static_cast<int64_t>(sub) * REFINE_KSUB + c) * REFINE_DSUB)[part];
        const float d0 = r.x - w.x, d1 = r.y - w.y, d2 = r.z - w.z, d3 = r.w - w.w;
        float d = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        d += __shfl_xor_sync(0xffffffffu, d, 1);
        d += __shfl_xor_sync(0xffffffffu, d, 2);
        d += __shfl_xor_sync(0xffffffffu, d, 4);
        if (d < best) { best = d; bi = c; }
    }
    return bi;
}
// second-level residual of rows whose first-level residual r1 = x - coarse[list] is given (training): for every PQ
// sub-space the nearest codeword is subtracted.  One thread per (row, sub-space).
__global__ void ivfpqr_residual2_kernel(const float* __restrict__ r1, int64_t n, const float* __restrict__ pq, int m, int dsub,
                                        float* __restrict__ r2) {
    const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n * m) return;
    const int64_t row = t / m;
    const int sub = static_cast<int>(t - row * m);
    const float* rr = r1 + row * D128 + sub * dsub;
    float best = FLT_MAX;
    int bi = 0;
    for (int c = 0; c < PQ_KSUB; ++c) {
        const float* w = pq + (static_cast<int64_t>(sub) * PQ_KSUB + c) * dsub;
        float d = 0.f;
        for (int j = 0; j < dsub; ++j) {
            const float e = rr[j] - w[j];
            d = fmaf(e, e, d);
        }
        if (d < best) { best = d; bi = c; }
    }
    const float* w = pq + (static_cast<int64_t>(sub) * PQ_KSUB + bi) * dsub;
    for (int j = 0; j < dsub; ++j) r2[row * D128 + sub * dsub + j] = rr[j] - w[j];
}
// add: refinement code of rows [row0, row0 + n): r2 = x - xhat, 4 nibbles.  One warp per row.
__global__ void __launch_bounds__(256)
ivfpqr_encode_kernel(const float* __restrict__ x32, const int32_t* __restrict__ assign, const uint8_t* __restrict__ codes,
                     int64_t row0, int64_t n, const float* __restrict__ coarse, const float* __restrict__ pq, int m, int dsub,
                     const float* __restrict__ rpq, uint8_t* __restrict__ rcodes) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (r >= n) return;
    const int64_t row = row0 + r;
    const float4 xh = pq_reconstruct_lane(coarse, pq, m, dsub, assign[row], codes + row * m, lane);
    const float4 xv = reinterpret_cast<const float4*>(x32 + row * D128)[lane];
    const int code = refine_encode_group(make_float4(xv.x - xh.x, xv.y - xh.y, xv.z - xh.z, xv.w - xh.w), rpq, lane);
    const int c0 = __shfl_sync(0xffffffffu, code, 0), c1 = __shfl_sync(0xffffffffu, code, 8);
    const int c2 = __shfl_sync(0xffffffffu, code, 16), c3 = __shfl_sync(0xffffffffu, code, 24);
    if (lane == 0) {
        rcodes[row * 2] = static_cast<uint8_t>(c0 | (c1 << 4));
        rcodes[row * 2 + 1] = static_cast<uint8_t>(c2 | (c3 << 4));
    }
}
// search: block = query row; its kc first-level candidates are re-scored as |q - (xhat + rhat)|^2 (a warp per candidate),
// sorted by (distance, label), the k best are returned (IndexIVFPQR::search_preassigned).  Only labels of the index's
// searched rows [label_offset, label_offset + n_search) are re-scored: a shard of a row-sharded index re-ranks the
// candidates it owns out of the global first-level top kc.
__global__ void __launch_bounds__(128)
ivfpqr_rerank_kernel(const float* __restrict__ q, const int64_t* __restrict__ candI, int kc, int k, int64_t n_search,
                     const int32_t* __restrict__ assign, const uint8_t* __restrict__ codes, const uint8_t* __restrict__ rcodes,
                     const float* __restrict__ coarse, const float* __restrict__ pq, int m, int dsub, const float* __restrict__ rpq,
                     int64_t label_offset, float* __restrict__ D, int64_t* __restrict__ I) {
    __shared__ float d_s[128];
    __shared__ int64_t i_s[128];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t qi = blockIdx.x;
    const float4 qv = reinterpret_cast<const float4*>(q + qi * D128)[lane];
    for (int e = threadIdx.x; e < 128; e += blockDim.x) { d_s[e] = INFINITY; i_s[e] = LLONG_MAX; }
    __syncthreads();
    for (int c = warp; c < kc; c += 4) {
        const int64_t id = candI[qi * kc + c];
        const int64_t row = id - label_offset;
        if (id < 0 || row < 0 || row >= n_search) continue;
        float4 xh = pq_reconstruct_lane(coarse, pq, m, dsub, assign[row], codes + row * m, lane);
        const int sub = lane >> 3;
        const int code = (rcodes[row * 2 + (sub >> 1)] >> (4 * (sub & 1))) & 15;
        const float4 w = reinterpret_cast<const float4*>(rpq + (static_cast<int64_t>(sub) * REFINE_KSUB + code) * REFINE_DSUB)[lane & 7];
        const float d0 = qv.x - (xh.x + w.x), d1 = qv.y - (xh.y + w.y), d2 = qv.z - (xh.z + w.z), d3 = qv.w - (xh.w + w.w);
        float d = d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        if (lane == 0) { d_s[c] = d; i_s[c] = id; }
    }
    __syncthreads();
    for (int kk = 2; kk <= 128; kk <<= 1) {
        for (int j = kk >> 1; j > 0; j >>= 1) {
            const int i = threadIdx.x, ixj = i ^ j;
            if (ixj > i) {
                const float da = d_s[i], db = d_s[ixj];
                const int64_t ia = i_s[i], ib = i_s[ixj];
                const bool a_after_b = (da > db) || (da == db && ia > ib);
                const bool asc = (i & kk) == 0;
                if (asc ? a_after_b : !a_after_b) {
                    d_s[i] = db; d_s[ixj] = da;
                    i_s[i] = ib; i_s[ixj] = ia;
                }
            }
            __syncthreads();
        }
    }
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        const int64_t id = i_s[j];
        D[qi * k + j] = id == LLONG_MAX ? INFINITY : d_s[j];
        I[qi * k + j] = id == LLONG_MAX ? -1 : id;
    }
}

// ------------------------------------------------------------------------------------------ host
int ivfpqr_enable(nafp_index* idx) {
    IvfPq* s = idx->ivf;
    NAFP_REQUIRE(s && !s->flat_lists && D128 == REFINE_M * REFINE_DSUB, NAFP_ERR_INVALID, "ivfpq-rr: needs an IVF-PQ state");
    NAFP_CUDA(cudaMalloc(&s->rpq, static_cast<size_t>(REFINE_M) * REFINE_KSUB * REFINE_DSUB * sizeof(float)));
    s->refine = true;
    return NAFP_OK;
}

int ivfflat_create(nafp_index* idx, int nlist) {
    NAFP_REQUIRE(nlist >= 1 && nlist <= IVF_MAX_NLIST, NAFP_ERR_INVALID, "ivf: nlist=%d outside [1,%d]", nlist, IVF_MAX_NLIST);
    IvfPq* s = new IvfPq();
    s->flat_lists = true;
    s->nlist = nlist;
    s->m = 0;
    s->dsub = 0;
    idx->ivf = s;                  // before the first fallible call: nafp_index_destroy releases it
    NAFP_CUDA(cudaMalloc(&s->coarse, static_cast<size_t>(nlist) * D128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->loff, (nlist + 1) * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&s->lend, nlist * sizeof(int32_t)));
    return NAFP_OK;
}

int ivfpq_create(nafp_index* idx, int nlist, int m, int nbits) {
    NAFP_REQUIRE(nbits == 8, NAFP_ERR_UNSUPPORTED, "ivfpq: nbits=%d (only 8, as in the reference)", nbits);
    NAFP_REQUIRE(nlist >= 1 && nlist <= IVF_MAX_NLIST, NAFP_ERR_INVALID, "ivfpq: nlist=%d outside [1,%d]", nlist, IVF_MAX_NLIST);
    NAFP_REQUIRE(m >= 16 && m <= PQ_MAX_M && D128 % m == 0 && m % 16 == 0, NAFP_ERR_INVALID,
                 "ivfpq: M=%d must divide 128 and be a multiple of 16 (<= 64)", m);
    IvfPq* s = new IvfPq();
    s->nlist = nlist;
    s->m = m;
    s->dsub = D128 / m;
    idx->ivf = s;                  // before the first fallible call: nafp_index_destroy releases it
    NAFP_CUDA(cudaMalloc(&s->coarse, static_cast<size_t>(nlist) * D128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->pq, static_cast<size_t>(m) * PQ_KSUB * s->dsub * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->loff, (nlist + 1) * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&s->lend, nlist * sizeof(int32_t)));
    // search path: the list-major compressed-domain scan (ivfpq_lm.cu) unless NAFP_IVFPQ_PATH=lut asks for the LUT kernel
    const char* e = getenv("NAFP_IVFPQ_PATH");
    s->lut_only = e && !strcmp(e, "lut");
    return NAFP_OK;
}

void ivfpq_destroy(nafp_index* idx) {
    IvfPq* s = idx->ivf;
    if (!s) return;
    ivfpq_lm_destroy(s);
    void* bufs[] = {s->coarse, s->pq, s->assign, s->codes, s->lcodes, s->lids, s->loff, s->lend, s->probes, s->partD, s->partI,
                    s->candD, s->candI, s->probes_all, s->redo_rows, s->redo_q, s->redo_D, s->redo_I,
                    s->rpq, s->rcodes, s->refD, s->refI};
    for (void* b : bufs) if (b) cudaFree(b);
    delete s;
    idx->ivf = nullptr;
}

int ivfpq_train(nafp_index* idx, const float* x_host, int64_t n, int64_t seed) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    // faiss-style subsampling: at most 256 training points per centroid
    const int64_t max_pts = 256ll * (s->flat_lists ? s->nlist : std::max(s->nlist, PQ_KSUB));
    const std::vector<int64_t> rows = select_rows(n, n > max_pts ? max_pts : n, static_cast<uint64_t>(seed));
    const int64_t nt = static_cast<int64_t>(rows.size());
    std::vector<float> xt(static_cast<size_t>(nt) * D128);
    for (int64_t i = 0; i < nt; ++i) memcpy(&xt[i * D128], x_host + rows[i] * D128, D128 * sizeof(float));
    float *x_dev = nullptr, *r_dev = nullptr;
    int32_t* a_dev = nullptr;
    struct Guard {                 // the temporaries (several hundred MB) are released on every return path
        float **x, **r;
        int32_t** a;
        ~Guard() { cudaFree(*x); cudaFree(*r); cudaFree(*a); }
    } guard{&x_dev, &r_dev, &a_dev};
    NAFP_CUDA(cudaMalloc(&x_dev, xt.size() * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&r_dev, xt.size() * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&a_dev, nt * sizeof(int32_t)));
    NAFP_CUDA(cudaMemcpy(x_dev, xt.data(), xt.size() * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_TRY(run_kmeans(ctx, x_dev, nt, D128, D128, s->nlist, s->coarse, a_dev, 25, static_cast<uint64_t>(seed) + 1));
    if (s->flat_lists) {
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        s->trained = true;
        return NAFP_OK;
    }
    // final assignment with the final centroids, then residuals
    kmeans_assign_kernel<<<static_cast<unsigned>((nt + 7) / 8), 256, 8 * D128 * sizeof(float), ctx->stream>>>(
        x_dev, nt, D128, D128, s->coarse, s->nlist, a_dev, nullptr);
    residual_kernel<<<static_cast<unsigned>((nt * D128 + 255) / 256), 256, 0, ctx->stream>>>(x_dev, nt, s->coarse, a_dev, r_dev);
    ctx->launches += 2;
    for (int sub = 0; sub < s->m; ++sub)
        NAFP_TRY(run_kmeans(ctx, r_dev + sub * s->dsub, nt, D128, s->dsub, PQ_KSUB,
                            s->pq + static_cast<size_t>(sub) * PQ_KSUB * s->dsub, a_dev, 25,
                            static_cast<uint64_t>(seed) + 2 + sub));
    if (s->refine) {
        // second level: residual of the first level on the training rows (r_dev -> x_dev), one k-means per 32-dim slice
        ivfpqr_residual2_kernel<<<static_cast<unsigned>((nt * s->m + 255) / 256), 256, 0, ctx->stream>>>(r_dev, nt, s->pq, s->m,
                                                                                                       s->dsub, x_dev);
        ctx->launches++;
        for (int sub = 0; sub < REFINE_M; ++sub)
            NAFP_TRY(run_kmeans(ctx, x_dev + sub * REFINE_DSUB, nt, D128, REFINE_DSUB, REFINE_KSUB,
                                s->rpq + static_cast<size_t>(sub) * REFINE_KSUB * REFINE_DSUB, a_dev, 25,
                                static_cast<uint64_t>(seed) + 100 + sub));
    }
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    s->trained = true;
    return NAFP_OK;
}

int ivfpq_add_rows(nafp_index* idx, int64_t row0, int64_t n) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    if (n == 0) return NAFP_OK;
    // The row-order copy of the codes is only the staging area of `add` (the lists are rebuilt from it): build_lists
    // releases it (64 of the index's 140 B per row), the next add regenerates it from the lists.
    const bool regen = !s->flat_lists && !s->codes && row0 > 0;
    if (idx->cap > s->cap || regen) {
        int32_t* a = nullptr;
        uint8_t* c = nullptr;
        NAFP_CUDA(cudaMalloc(&a, static_cast<size_t>(idx->cap) * sizeof(int32_t)));
        if (!s->flat_lists) NAFP_CUDA(cudaMalloc(&c, static_cast<size_t>(idx->cap) * s->m));
        if (row0 > 0) {
            NAFP_CUDA(cudaMemcpyAsync(a, s->assign, static_cast<size_t>(row0) * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
            if (regen) {
                const int64_t n_pos = s->h_loff[s->nlist];
                ivf_unscatter_kernel<<<static_cast<unsigned>((n_pos + 255) / 256), 256, 0, ctx->stream>>>(s->lcodes, s->lids, n_pos, s->m, c);
                ctx->launches++;
            } else if (!s->flat_lists) {
                NAFP_CUDA(cudaMemcpyAsync(c, s->codes, static_cast<size_t>(row0) * s->m, cudaMemcpyDeviceToDevice, ctx->stream));
            }
            NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        if (s->refine) {
            uint8_t* rc = nullptr;
            NAFP_CUDA(cudaMalloc(&rc, static_cast<size_t>(idx->cap) * 2));
            if (row0 > 0) {
                NAFP_CUDA(cudaMemcpyAsync(rc, s->rcodes, static_cast<size_t>(row0) * 2, cudaMemcpyDeviceToDevice, ctx->stream));
                NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
            }
            if (s->rcodes) cudaFree(s->rcodes);
            s->rcodes = rc;
        }
        if (s->assign) cudaFree(s->assign);
        if (s->codes) cudaFree(s->codes);
        s->assign = a;
        s->codes = c;
        s->cap = idx->cap;
    }
    if (s->flat_lists) {               // list of every new row = its nearest coarse centroid (ties -> lower id)
        kmeans_assign_kernel<<<static_cast<unsigned>((n + 7) / 8), 256, 8 * D128 * sizeof(float), ctx->stream>>>(
            idx->x32 + row0 * D128, n, D128, D128, s->coarse, s->nlist, s->assign + row0, nullptr);
        ctx->launches++;
        NAFP_CUDA(cudaGetLastError());
        s->dirty = true;
        return NAFP_OK;
    }
    int64_t blocks = (n + 7) / 8;
    if (s->nlist <= ENC_NLIST && s->m == 64 && s->dsub == 2) {
        if (blocks > ctx->sm_count) blocks = ctx->sm_count;          // one block per SM: each loads its table once
        NAFP_CUDA(cudaFuncSetAttribute(ivfpq_assign_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ENC_ASSIGN_SMEM));
        NAFP_CUDA(cudaFuncSetAttribute(ivfpq_code_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ENC_CODE_SMEM));
        ivfpq_assign_smem_kernel<<<static_cast<unsigned>(blocks), 256, ENC_ASSIGN_SMEM, ctx->stream>>>(idx->x32, row0, n, s->coarse,
                                                                                                     s->nlist, s->assign);
        ivfpq_code_smem_kernel<<<static_cast<unsigned>(blocks), 256, ENC_CODE_SMEM, ctx->stream>>>(idx->x32, row0, n, s->coarse, s->pq,
                                                                                                 s->assign, s->codes);
        ctx->launches++;
    } else {
        if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
        ivfpq_encode_kernel<<<static_cast<unsigned>(blocks), 256, 0, ctx->stream>>>(idx->x32, row0, n, s->coarse, s->nlist, s->pq,
                                                                                  s->m, s->dsub, s->assign, s->codes);
    }
    ctx->launches++;
    if (s->refine) {
        ivfpqr_encode_kernel<<<static_cast<unsigned>((n * 32 + 255) / 256), 256, 0, ctx->stream>>>(
            idx->x32, s->assign, s->codes, row0, n, s->coarse, s->pq, s->m, s->dsub, s->rpq, s->rcodes);
        ctx->launches++;
    }
    NAFP_CUDA(cudaGetLastError());
    s->dirty = true;
    return NAFP_OK;
}

int build_lists(nafp_index* idx) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    const int64_t n = idx->n;
    if (!s->dirty) return NAFP_OK;
    const int64_t need = idx->cap + static_cast<int64_t>(LIST_TILE) * s->nlist;      // every list is padded to whole tiles
    if (s->sorted_cap < need) {
        if (s->lcodes) cudaFree(s->lcodes);
        if (s->lids) cudaFree(s->lids);
        s->lcodes = nullptr; s->lids = nullptr; s->sorted_cap = 0;
        if (!s->flat_lists) NAFP_CUDA(cudaMalloc(&s->lcodes, static_cast<size_t>(need) * s->m));
        NAFP_CUDA(cudaMalloc(&s->lids, static_cast<size_t>(need) * sizeof(int32_t)));
        s->sorted_cap = need;
    }
    const int nchunks = static_cast<int>((n + SORT_CHUNK - 1) / SORT_CHUNK);
    std::vector<int32_t> off(s->nlist + 1, 0), end(s->nlist, 0);
    if (nchunks > 0) {
        int32_t* hist = nullptr;
        int64_t* base = nullptr;
        struct Guard {             // released on every return path
            int32_t** h;
            int64_t** b;
            ~Guard() { cudaFree(*h); cudaFree(*b); }
        } guard{&hist, &base};
        NAFP_CUDA(cudaMalloc(&hist, static_cast<size_t>(s->nlist) * nchunks * sizeof(int32_t)));
        NAFP_CUDA(cudaMalloc(&base, static_cast<size_t>(s->nlist) * nchunks * sizeof(int64_t)));
        ivf_hist_kernel<<<nchunks, 32, 0, ctx->stream>>>(s->assign, n, s->nlist, hist);
        std::vector<int32_t> h(static_cast<size_t>(s->nlist) * nchunks);
        NAFP_CUDA(cudaMemcpyAsync(h.data(), hist, h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        std::vector<int64_t> b(h.size());
        int64_t run = 0;
        for (int l = 0; l < s->nlist; ++l) {
            off[l] = static_cast<int32_t>(run);
            for (int c = 0; c < nchunks; ++c) {
                b[static_cast<size_t>(l) * nchunks + c] = run;
                run += h[static_cast<size_t>(l) * nchunks + c];
            }
            end[l] = static_cast<int32_t>(run);
            run = (run + LIST_TILE - 1) / LIST_TILE * LIST_TILE;
        }
        off[s->nlist] = static_cast<int32_t>(run);
        NAFP_REQUIRE(run <= s->sorted_cap && run < (1ll << 31), NAFP_ERR_UNSUPPORTED, "ivf lists: %lld padded positions", static_cast<long long>(run));
        // padding positions: row id -1, code 0
        NAFP_CUDA(cudaMemsetAsync(s->lids, 0xFF, static_cast<size_t>(run) * sizeof(int32_t), ctx->stream));
        if (!s->flat_lists) NAFP_CUDA(cudaMemsetAsync(s->lcodes, 0, static_cast<size_t>(run) * s->m, ctx->stream));
        NAFP_CUDA(cudaMemcpyAsync(base, b.data(), b.size() * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
        ivf_scatter_kernel<<<nchunks, 32, 0, ctx->stream>>>(s->assign, s->codes, n, s->nlist, s->m, base, s->lcodes, s->lids);
        ctx->launches += 2;
        NAFP_CUDA(cudaGetLastError());
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    NAFP_CUDA(cudaMemcpy(s->loff, off.data(), off.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->lend, end.data(), end.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    s->h_loff = off;
    s->h_lend = end;
    s->lists_version++;
    s->dirty = false;
    if (!s->flat_lists && !s->refine && s->codes) {      // (IVFPQR re-ranks by row)
        cudaFree(s->codes);
        s->codes = nullptr;
    }
    return NAFP_OK;
}

__global__ void topk_merge_kernel(const float* __restrict__ D_all, const int64_t* __restrict__ I_all, int W, int64_t nq,
                                  int k, float* __restrict__ D_out, int64_t* __restrict__ I_out);
constexpr int TOPK_MERGE_KEYS = 4096;     // keys one topk_merge_kernel block sorts (seq_match.cu)
// merge blocks per query row of the LUT scan: 1 when the nprobe * k partial keys fit one block, else the number of
// groups of floor(4096 / k) probes merged in a first round
static int lut_merge_groups(int nprobe, int k) {
    if (nprobe * k <= TOPK_MERGE_KEYS) return 1;
    const int G = TOPK_MERGE_KEYS / k;
    return (nprobe + G - 1) / G;
}

// the reference formulation: per (query row, probed list) LUT + ADC scan of the list's codes
int ivfpq_search_lut(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    if (nq == 0) return NAFP_OK;
    const int nprobe = idx->nprobe < s->nlist ? idx->nprobe : s->nlist;
    NAFP_REQUIRE(k >= 1 && k <= MAX_K && lut_merge_groups(nprobe, k) * k <= TOPK_MERGE_KEYS, NAFP_ERR_INVALID,
                 "ivfpq search: need k <= %d and ceil(nprobe / floor(%d / k)) * k <= %d (nprobe %d, k %d)", MAX_K, TOPK_MERGE_KEYS,
                 TOPK_MERGE_KEYS, nprobe, k);
    NAFP_TRY(build_lists(idx));
    const int64_t n_search = (idx->search_rows >= 0 && idx->search_rows < idx->n) ? idx->search_rows : idx->n;
    const int64_t chunk = 4096;       // query rows per launch group (bounds the partial buffers)
    if (s->scratch_nq < std::min(nq, chunk) || s->scratch_nprobe < nprobe || s->scratch_k < k) {
        if (s->probes) cudaFree(s->probes);
        if (s->partD) cudaFree(s->partD);
        if (s->partI) cudaFree(s->partI);
        s->probes = nullptr; s->partD = nullptr; s->partI = nullptr;
        const int64_t cq = std::min(nq, chunk) > s->scratch_nq ? std::min(nq, chunk) : s->scratch_nq;
        const int cp = nprobe > s->scratch_nprobe ? nprobe : s->scratch_nprobe;
        const int ck = k > s->scratch_k ? k : s->scratch_k;
        NAFP_CUDA(cudaMalloc(&s->probes, static_cast<size_t>(cq) * cp * sizeof(int32_t)));
        NAFP_CUDA(cudaMalloc(&s->partD, static_cast<size_t>(cq) * cp * ck * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->partI, static_cast<size_t>(cq) * cp * ck * sizeof(int64_t)));
        s->scratch_nq = cq; s->scratch_nprobe = cp; s->scratch_k = ck;
    }
    const size_t lut_bytes = static_cast<size_t>(s->m) * PQ_KSUB * sizeof(float);
    if (!s->flat_lists)
        NAFP_CUDA(cudaFuncSetAttribute(ivfpq_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(lut_bytes)));
    for (int64_t q0 = 0; q0 < nq; q0 += chunk) {
        const int64_t nc = nq - q0 < chunk ? nq - q0 : chunk;
        const float* qp = q_dev + q0 * D128;
        ivfpq_probe_kernel<<<static_cast<unsigned>((nc + 7) / 8), 256, 0, ctx->stream>>>(qp, nc, s->coarse, s->nlist, nprobe, s->probes);
        if (s->flat_lists)
            ivfflat_scan_kernel<<<dim3(nprobe, static_cast<unsigned>(nc)), 256, 0, ctx->stream>>>(
                qp, nc, s->probes, nprobe, idx->x32, s->lids, s->loff, s->lend, k, idx->label_offset, n_search, s->partD, s->partI);
        else
            ivfpq_scan_kernel<<<dim3(nprobe, static_cast<unsigned>(nc)), 256, lut_bytes, ctx->stream>>>(
                qp, nc, s->coarse, s->pq, s->m, s->dsub, s->probes, nprobe, s->lcodes, s->lids, s->loff, s->lend, k, idx->label_offset,
                n_search, s->partD, s->partI);
        const int groups = lut_merge_groups(nprobe, k);
        if (groups > 1) {
            // nprobe * k keys exceed one merge block: merge groups of G probes first.  The result of group g lands in the
            // partials of probe g of the same row, which group 0 (g < G) has already consumed; every block reads all its
            // inputs before it writes, so group 0 may overwrite its own probe 0.  Then merge the `groups` partial lists.
            const int G = TOPK_MERGE_KEYS / k;
            for (int g = 0; g < groups; ++g) {
                const int64_t in = static_cast<int64_t>(g) * G * nc * k, out = static_cast<int64_t>(g) * nc * k;
                topk_merge_kernel<<<static_cast<unsigned>(nc), 128, 0, ctx->stream>>>(
                    s->partD + in, s->partI + in, std::min(G, nprobe - g * G), nc, k, s->partD + out, s->partI + out);
            }
            ctx->launches += groups;
        }
        topk_merge_kernel<<<static_cast<unsigned>(nc), 128, 0, ctx->stream>>>(s->partD, s->partI, groups > 1 ? groups : nprobe, nc, k,
                                                                              D_dev + q0 * k, I_dev + q0 * k);
        ctx->launches += 3;
    }
    NAFP_CUDA(cudaGetLastError());
    s->lut_rows += static_cast<unsigned long long>(nq);
    return NAFP_OK;
}

void ivfpq_take_stats(nafp_index* idx, int64_t* out8) {
    IvfPq* s = idx->ivf;
    out8[0] = idx->host_rows;
    out8[1] = static_cast<int64_t>(s->lut_rows);
    ivfpq_lm_take_stats(s, &out8[2], &out8[3]);
    idx->host_rows = idx->host_passes = 0;
    s->lut_rows = 0;
}

// query rows a fast path could not answer: redo_rows[0 .. n) + the counter at redo_rows[redo_cap]
int ivfpq_reserve_redo(nafp_index* idx, int64_t nq) {
    IvfPq* s = idx->ivf;
    if (s->redo_cap < nq) {
        void* old[] = {s->redo_rows, s->redo_q, s->redo_D, s->redo_I};
        for (void* b : old) if (b) cudaFree(b);
        s->redo_rows = nullptr; s->redo_q = nullptr; s->redo_D = nullptr; s->redo_I = nullptr; s->redo_cap = 0;
        NAFP_CUDA(cudaMalloc(&s->redo_rows, static_cast<size_t>(nq + 1) * sizeof(int32_t)));
        s->redo_cap = nq;
    }
    return NAFP_OK;
}
// ... answered by the LUT scan of their probed lists, scattered back into D / I
int ivfpq_redo_rows(nafp_index* idx, const float* q_dev, int32_t n_redo, int k, float* D_dev, int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    if (!s->redo_q) {
        NAFP_CUDA(cudaMalloc(&s->redo_q, static_cast<size_t>(s->redo_cap) * D128 * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->redo_D, static_cast<size_t>(s->redo_cap) * MAX_K * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->redo_I, static_cast<size_t>(s->redo_cap) * MAX_K * sizeof(int64_t)));
    }
    ivfpq_gather_q_kernel<<<static_cast<unsigned>((static_cast<int64_t>(n_redo) * 32 + 255) / 256), 256, 0, ctx->stream>>>(
        q_dev, s->redo_rows, n_redo, s->redo_q);
    NAFP_TRY(ivfpq_search_lut(idx, s->redo_q, n_redo, k, s->redo_D, s->redo_I));
    ivfpq_scatter_kernel<<<static_cast<unsigned>((static_cast<int64_t>(n_redo) * k + 255) / 256), 256, 0, ctx->stream>>>(
        s->redo_D, s->redo_I, s->redo_rows, n_redo, k, D_dev, I_dev);
    ctx->launches += 2;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

static int ivfpq_search_first_level(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev);
static int ivfpqr_rerank(nafp_index* idx, const float* q_dev, int64_t nq, const int64_t* candI_dev, int kc, int k, float* D_dev,
                         int64_t* I_dev);

int ivfpq_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    if (!s->refine) return ivfpq_search_first_level(idx, q_dev, nq, k, D_dev, I_dev);
    // IVFPQR: k * k_factor first-level candidates (faiss default k_factor 4), re-ranked with the refinement codes
    nafp_ctx* ctx = idx->ctx;
    NAFP_REQUIRE(s->trained, NAFP_ERR_STATE, "ivfpq-rr search: index is not trained");
    const int kc = k * REFINE_KFACTOR;
    NAFP_REQUIRE(k >= 1 && kc <= MAX_K, NAFP_ERR_INVALID, "ivfpq-rr search: k=%d (k * %d candidates must be <= %d)", k, REFINE_KFACTOR, MAX_K);
    NAFP_CUDA(cudaSetDevice(ctx->device));
    if (nq == 0) return NAFP_OK;
    if (s->ref_nq < nq) {
        if (s->refD) cudaFree(s->refD);
        if (s->refI) cudaFree(s->refI);
        s->refD = nullptr; s->refI = nullptr; s->ref_nq = 0;
        NAFP_CUDA(cudaMalloc(&s->refD, static_cast<size_t>(nq) * MAX_K * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->refI, static_cast<size_t>(nq) * MAX_K * sizeof(int64_t)));
        s->ref_nq = nq;
    }
    NAFP_TRY(ivfpq_search_first_level(idx, q_dev, nq, kc, s->refD, s->refI));
    return ivfpqr_rerank(idx, q_dev, nq, s->refI, kc, k, D_dev, I_dev);
}

static int ivfpqr_rerank(nafp_index* idx, const float* q_dev, int64_t nq, const int64_t* candI_dev, int kc, int k, float* D_dev,
                         int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    NAFP_REQUIRE(k >= 1 && k <= kc && kc <= MAX_K, NAFP_ERR_INVALID, "ivfpq-rr re-rank: need 1 <= k <= kc <= %d (k %d, kc %d)", MAX_K, k, kc);
    if (nq == 0) return NAFP_OK;
    const int64_t n_search = (idx->search_rows >= 0 && idx->search_rows < idx->n) ? idx->search_rows : idx->n;
    ivfpqr_rerank_kernel<<<static_cast<unsigned>(nq), 128, 0, ctx->stream>>>(q_dev, candI_dev, kc, k, n_search, s->assign, s->codes,
                                                                             s->rcodes, s->coarse, s->pq, s->m, s->dsub, s->rpq,
                                                                             idx->label_offset, D_dev, I_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

static int ivfpq_search_first_level(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    NAFP_REQUIRE(s->trained, NAFP_ERR_STATE, "ivfpq search: index is not trained");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    if (nq == 0) return NAFP_OK;
    const int nprobe = idx->nprobe < s->nlist ? idx->nprobe : s->nlist;
    NAFP_REQUIRE(k >= 1 && k <= MAX_K && lut_merge_groups(nprobe, k) * k <= TOPK_MERGE_KEYS, NAFP_ERR_INVALID,
                 "ivfpq search: need k <= %d and ceil(nprobe / floor(%d / k)) * k <= %d (nprobe %d, k %d)", MAX_K, TOPK_MERGE_KEYS,
                 TOPK_MERGE_KEYS, nprobe, k);
    if (!s->flat_lists) idx->host_rows += nq;          // (the flat scan of an IVF-Flat index counts its own rows)
    if (nq >= (1ll << 31)) return ivfpq_search_lut(idx, q_dev, nq, k, D_dev, I_dev);
    if (!s->flat_lists) {
        if (!s->lut_only && ivfpq_lm_supported(idx, k)) return ivfpq_search_lm(idx, q_dev, nq, k, D_dev, I_dev);
        return ivfpq_search_lut(idx, q_dev, nq, k, D_dev, I_dev);
    }

    // IVF-Flat
    if (k > IVFFLAT_K / 2) return ivfpq_search_lut(idx, q_dev, nq, k, D_dev, I_dev);
    // 1. exact top-IVFFLAT_K over the stored rows (tensor-core scan + fp32 re-rank)
    if (s->cand_nq < nq) {
        if (s->candD) cudaFree(s->candD);
        if (s->candI) cudaFree(s->candI);
        s->candD = nullptr; s->candI = nullptr; s->cand_nq = 0;
        NAFP_CUDA(cudaMalloc(&s->candD, static_cast<size_t>(nq) * IVFFLAT_K * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->candI, static_cast<size_t>(nq) * IVFFLAT_K * sizeof(int64_t)));
        s->cand_nq = nq;
    }
    if (s->probes_all_elems < nq * nprobe) {
        if (s->probes_all) cudaFree(s->probes_all);
        s->probes_all = nullptr; s->probes_all_elems = 0;
        NAFP_CUDA(cudaMalloc(&s->probes_all, static_cast<size_t>(nq) * nprobe * sizeof(int32_t)));
        s->probes_all_elems = nq * nprobe;
    }
    int32_t* probes_all = s->probes_all;
    NAFP_TRY(ivfpq_reserve_redo(idx, nq));
    int32_t* redo_count = s->redo_rows + s->redo_cap;
    NAFP_CUDA(cudaMemsetAsync(redo_count, 0, sizeof(int32_t), ctx->stream));
    const int64_t off = idx->label_offset;      // the filter wants local rows and adds the offset itself
    idx->label_offset = 0;
    const int st = flat_search_dev(idx, q_dev, nq, IVFFLAT_K, s->candD, s->candI);
    idx->label_offset = off;
    NAFP_TRY(st);
    // 2. the nprobe nearest lists of every row, 3. keep the candidates that live in them
    ivfpq_probe_kernel<<<static_cast<unsigned>((nq + 7) / 8), 256, 0, ctx->stream>>>(q_dev, nq, s->coarse, s->nlist, nprobe, probes_all);
    ivfpq_filter_kernel<<<static_cast<unsigned>((nq + 7) / 8), 256, 0, ctx->stream>>>(s->candD, s->candI, nq, k, probes_all, nprobe,
                                                                                     s->assign, idx->label_offset, D_dev, I_dev,
                                                                                     s->redo_rows, redo_count);
    ctx->launches += 2;
    NAFP_CUDA(cudaGetLastError());
    int32_t n_redo = 0;
    NAFP_CUDA(cudaMemcpyAsync(&n_redo, redo_count, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    // 4. rows with fewer than k probed rows among their IVFFLAT_K nearest: the exact scan of their lists
    if (n_redo > 0) NAFP_TRY(ivfpq_redo_rows(idx, q_dev, n_redo, k, D_dev, I_dev));
    return NAFP_OK;
}

}  // namespace nafp

using namespace nafp;

extern "C" {

int nafp_index_is_trained(nafp_index* idx) {
    if (!idx) return 0;
    if (idx->type == NAFP_INDEX_FLAT_L2) return 1;
    return idx->ivf && idx->ivf->trained ? 1 : 0;
}

int nafp_index_ivf_get_coarse(nafp_index* idx, float* coarse_host) {
    NAFP_RANGE("nafp_index_ivf_get_coarse");
    NAFP_REQUIRE(idx && idx->ivf && coarse_host, NAFP_ERR_INVALID, "nafp_index_ivf_get_coarse: not an IVF index");
    IvfPq* s = idx->ivf;
    NAFP_REQUIRE(s->trained, NAFP_ERR_STATE, "nafp_index_ivf_get_coarse: index is not trained");
    NAFP_CUDA(cudaStreamSynchronize(idx->ctx->stream));
    NAFP_CUDA(cudaMemcpy(coarse_host, s->coarse, static_cast<size_t>(s->nlist) * D128 * sizeof(float), cudaMemcpyDeviceToHost));
    return NAFP_OK;
}

int nafp_index_ivf_set_coarse(nafp_index* idx, const float* coarse_host) {
    NAFP_RANGE("nafp_index_ivf_set_coarse");
    NAFP_REQUIRE(idx && idx->ivf && coarse_host, NAFP_ERR_INVALID, "nafp_index_ivf_set_coarse: not an IVF index");
    NAFP_REQUIRE(idx->n == 0, NAFP_ERR_STATE, "nafp_index_ivf_set_coarse: index already holds rows");
    IvfPq* s = idx->ivf;
    NAFP_CUDA(cudaMemcpy(s->coarse, coarse_host, static_cast<size_t>(s->nlist) * D128 * sizeof(float), cudaMemcpyHostToDevice));
    if (s->flat_lists) s->trained = true;
    return NAFP_OK;
}

int nafp_index_ivfpq_get_params(nafp_index* idx, float* coarse_host, float* pq_host) {
    NAFP_RANGE("nafp_index_ivfpq_get_params");
    NAFP_REQUIRE(idx && idx->ivf && !idx->ivf->flat_lists && coarse_host && pq_host, NAFP_ERR_INVALID,
                 "nafp_index_ivfpq_get_params: not an IVF-PQ index");
    IvfPq* s = idx->ivf;
    NAFP_REQUIRE(s->trained, NAFP_ERR_STATE, "nafp_index_ivfpq_get_params: index is not trained");
    NAFP_CUDA(cudaStreamSynchronize(idx->ctx->stream));
    NAFP_CUDA(cudaMemcpy(coarse_host, s->coarse, static_cast<size_t>(s->nlist) * D128 * sizeof(float), cudaMemcpyDeviceToHost));
    NAFP_CUDA(cudaMemcpy(pq_host, s->pq, static_cast<size_t>(s->m) * PQ_KSUB * s->dsub * sizeof(float), cudaMemcpyDeviceToHost));
    return NAFP_OK;
}

int nafp_index_ivfpq_set_params(nafp_index* idx, const float* coarse_host, const float* pq_host) {
    NAFP_RANGE("nafp_index_ivfpq_set_params");
    NAFP_REQUIRE(idx && idx->ivf && !idx->ivf->flat_lists && coarse_host && pq_host, NAFP_ERR_INVALID,
                 "nafp_index_ivfpq_set_params: not an IVF-PQ index");
    NAFP_REQUIRE(idx->n == 0, NAFP_ERR_STATE, "nafp_index_ivfpq_set_params: index already holds rows");
    IvfPq* s = idx->ivf;
    NAFP_CUDA(cudaMemcpy(s->coarse, coarse_host, static_cast<size_t>(s->nlist) * D128 * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->pq, pq_host, static_cast<size_t>(s->m) * PQ_KSUB * s->dsub * sizeof(float), cudaMemcpyHostToDevice));
    s->trained = true;
    return NAFP_OK;
}

int nafp_index_ivfpqr_get_refine(nafp_index* idx, float* refine_pq_host) {
    NAFP_RANGE("nafp_index_ivfpqr_get_refine");
    NAFP_REQUIRE(idx && idx->ivf && idx->ivf->refine && refine_pq_host, NAFP_ERR_INVALID, "nafp_index_ivfpqr_get_refine: not an IVFPQR index");
    NAFP_REQUIRE(idx->ivf->trained, NAFP_ERR_STATE, "nafp_index_ivfpqr_get_refine: index is not trained");
    NAFP_CUDA(cudaStreamSynchronize(idx->ctx->stream));
    NAFP_CUDA(cudaMemcpy(refine_pq_host, idx->ivf->rpq, static_cast<size_t>(REFINE_M) * REFINE_KSUB * REFINE_DSUB * sizeof(float),
                         cudaMemcpyDeviceToHost));
    return NAFP_OK;
}

int nafp_index_ivfpqr_set_refine(nafp_index* idx, const float* refine_pq_host) {
    NAFP_RANGE("nafp_index_ivfpqr_set_refine");
    NAFP_REQUIRE(idx && idx->ivf && idx->ivf->refine && refine_pq_host, NAFP_ERR_INVALID, "nafp_index_ivfpqr_set_refine: not an IVFPQR index");
    NAFP_REQUIRE(idx->n == 0, NAFP_ERR_STATE, "nafp_index_ivfpqr_set_refine: index already holds rows");
    NAFP_CUDA(cudaMemcpy(idx->ivf->rpq, refine_pq_host, static_cast<size_t>(REFINE_M) * REFINE_KSUB * REFINE_DSUB * sizeof(float),
                         cudaMemcpyHostToDevice));
    return NAFP_OK;
}

int nafp_index_ivfpqr_first_level_dev(nafp_index* idx, const float* q_dev, int64_t nq, int kc, float* D_dev, int64_t* I_dev) {
    NAFP_RANGE("nafp_index_ivfpqr_first_level_dev");
    NAFP_REQUIRE(idx && idx->ivf && idx->ivf->refine && nq >= 0 && (nq == 0 || (q_dev && D_dev && I_dev)), NAFP_ERR_INVALID,
                 "nafp_index_ivfpqr_first_level_dev: not an IVFPQR index, or bad arguments");
    return ivfpq_search_first_level(idx, q_dev, nq, kc, D_dev, I_dev);
}

int nafp_index_ivfpqr_rerank_dev(nafp_index* idx, const float* q_dev, int64_t nq, const int64_t* candI_dev, int kc, int k,
                                 float* D_dev, int64_t* I_dev) {
    NAFP_RANGE("nafp_index_ivfpqr_rerank_dev");
    NAFP_REQUIRE(idx && idx->ivf && idx->ivf->refine && nq >= 0 && (nq == 0 || (q_dev && candI_dev && D_dev && I_dev)),
                 NAFP_ERR_INVALID, "nafp_index_ivfpqr_rerank_dev: not an IVFPQR index, or bad arguments");
    NAFP_REQUIRE(idx->ivf->trained, NAFP_ERR_STATE, "nafp_index_ivfpqr_rerank_dev: index is not trained");
    NAFP_CUDA(cudaSetDevice(idx->ctx->device));
    return ivfpqr_rerank(idx, q_dev, nq, candI_dev, kc, k, D_dev, I_dev);
}

}  // extern "C"
