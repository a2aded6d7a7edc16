// Sequence-offset matcher (SURVEY §8 a7): the body of the reference's evaluation hot loop
// eval/eval_faiss.py:204-232, batched over test ids.
//
//   seq_mark/scan/rowmap the UNIQUE query rows needed by the test ids (id .. id+L-1, truncated at the end
//                       of the query set, :208): overlapping sequences share rows, each is searched once
//   <segment search>    one top-k_probe search of the unique rows (:211); rows of a shorter sequence
//                       length are a prefix of the longest one, so one search serves all lengths
//   seq_cand_kernel     offset compensation (:215-216), sorted unique candidates >= 0 (:219) and,
//                       per candidate, the running mean of q[j].recon[c+j] (:222-229) for every
//                       requested length -- a gather/reduce over the fp32 rows
//   seq_top_kernel      the 10 best candidates per (test id, length), ties to the lower id (:232)
// Candidates this shard does not own score -inf, so that a row-sharded database can combine the
// per-rank score tables with a max-reduce between the two kernels.
#include <algorithm>
#include <climits>

#include "index.h"
#include "ptx.cuh"
#include "topk.cuh"

namespace nafp {

constexpr int SEQ_MAXC = 1024;     // k_probe * max_len upper bound
constexpr int SEQ_MAXL = 32;
constexpr int SEQ_NPRED = 10;

// ---- unique query rows: many test ids share rows (id .. id+L-1 overlap), each row is searched once
__global__ void seq_mark_kernel(const int64_t* __restrict__ test_ids, int64_t n_test, int L, int64_t n_query_rows,
                                int32_t* __restrict__ flags) {
    const int64_t w = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= n_test * L) return;
    const int64_t id = test_ids[w / L];
    if (id < 0 || id >= n_query_rows) return;
    int64_t r = id + static_cast<int>(w % L);
    if (r >= n_query_rows) return;              // rows past the end are never used (eval_faiss.py:208 truncates)
    flags[r] = 1;
}
// exclusive prefix sum of flags (single block, chunked); pos[r] = rank of row r among the marked rows
__global__ void __launch_bounds__(1024)
seq_scan_kernel(const int32_t* __restrict__ flags, int64_t n, int32_t* __restrict__ pos, int32_t* __restrict__ uniq_rows,
                int32_t* __restrict__ n_uniq) {
    __shared__ int warp_sums[32];
    __shared__ int carry_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += 1024) {
        const int64_t i = base + tid;
        const int f = i < n ? flags[i] : 0;
        int x = f;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int s = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, s, o);
                if (lane >= o) s += y;
            }
            warp_sums[lane] = s;
        }
        __syncthreads();
        const int carry = carry_s;
        const int excl = carry + (warp > 0 ? warp_sums[warp - 1] : 0) + x - f;
        if (i < n) {
            pos[i] = f ? excl : -1;
            if (f) uniq_rows[excl] = static_cast<int32_t>(i);
        }
        __syncthreads();
        if (tid == 0) carry_s = carry + warp_sums[31];
        __syncthreads();
    }
    if (tid == 0) *n_uniq = carry_s;
}
__global__ void seq_rowmap_kernel(const int64_t* __restrict__ test_ids, int64_t n_test, int L, int64_t n_query_rows,
                                  const int32_t* __restrict__ pos, int32_t* __restrict__ rowmap) {
    const int64_t w = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= n_test * L) return;
    const int64_t id = test_ids[w / L];
    const int64_t r = id + static_cast<int>(w % L);
    rowmap[w] = (id >= 0 && r < n_query_rows) ? pos[r] : -1;
}
__global__ void seq_gather_rows_kernel(const float* __restrict__ qall, const int32_t* __restrict__ rows, int64_t n,
                                       float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (w >= n) return;
    reinterpret_cast<float4*>(out + w * D128)[lane] = reinterpret_cast<const float4*>(qall + static_cast<int64_t>(rows[w]) * D128)[lane];
}

__global__ void __launch_bounds__(256)
seq_cand_kernel(const float* __restrict__ qall, int64_t n_query_rows, const int64_t* __restrict__ test_ids,
                const int32_t* __restrict__ seq_lens, int n_len, int L, int k_probe,
                const int64_t* __restrict__ I, const int32_t* __restrict__ rowmap, const float* __restrict__ x32,
                int64_t n_rows_local,
                int64_t n_rows_global, int64_t label_offset, int64_t owned_lo, int64_t owned_hi,
                int64_t* __restrict__ cand_ids, float* __restrict__ cand_scores, int32_t* __restrict__ n_cand) {
    __shared__ uint64_t keys[SEQ_MAXC];
    __shared__ int64_t uniq_c[SEQ_MAXC];
    __shared__ uint8_t uniq_j[SEQ_MAXC];
    __shared__ int wsum[8];
    __shared__ float prefix[8][SEQ_MAXL + 1];
    const int64_t t = blockIdx.x;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t id = test_ids[t];
    int lq = 0;
    if (id >= 0 && id < n_query_rows) lq = static_cast<int>(n_query_rows - id < L ? n_query_rows - id : L);

    for (int e = tid; e < SEQ_MAXC; e += blockDim.x) {
        uint64_t key = ~0ull;
        if (e < L * k_probe) {
            const int j = e / k_probe, m = e % k_probe;
            if (j < lq) {
                const int64_t irow = rowmap ? rowmap[t * L + j] : t * L + j;      // row of the search result table
                const int64_t lab = I[irow * k_probe + m];
                const int64_t c = lab - j;
                if (lab >= 0 && c >= 0) key = (static_cast<uint64_t>(c) << 6) | static_cast<uint64_t>(j);
            }
        }
        keys[e] = key;
    }
    __syncthreads();
    block_sort_u64<true>(keys, SEQ_MAXC);

    // compaction of first occurrences (sorted by candidate, then by j => first has the minimal j)
    int base = 0;
    for (int e0 = 0; e0 < SEQ_MAXC; e0 += blockDim.x) {
        const int e = e0 + tid;
        const uint64_t key = keys[e];
        const bool head = key != ~0ull && (e == 0 || (keys[e - 1] >> 6) != (key >> 6));
        const unsigned bal = __ballot_sync(0xffffffffu, head);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int off = base;
        for (int w = 0; w < warp; ++w) off += wsum[w];
        int tot = 0;
        for (int w = 0; w < 8; ++w) tot += wsum[w];
        if (head) {
            const int pos = off + __popc(bal & ((1u << lane) - 1));
            uniq_c[pos] = static_cast<int64_t>(key >> 6);
            uniq_j[pos] = static_cast<uint8_t>(key & 63);
        }
        base += tot;
        __syncthreads();
    }
    const int nu = base;
    if (tid == 0) n_cand[t] = nu;
    for (int u = tid; u < SEQ_MAXC; u += blockDim.x) cand_ids[t * SEQ_MAXC + u] = u < nu ? uniq_c[u] : -1;

    // gather / reduce: per candidate the prefix sums of q[j] . recon[c + j]
    const float* qt = qall + (lq > 0 ? id : 0) * D128;      // rows id .. id+lq-1 of the query set
    for (int u = warp; u < nu; u += 8) {
        const int64_t c = uniq_c[u];
        const bool owned = c >= owned_lo && c < owned_hi;
        const int64_t row = c - label_offset;
        int avail = 0;     // rows of recon that exist at c, c+1, ... (global extent, :224 slice clamps)
        if (owned) {
            const int64_t left = n_rows_global - c;
            avail = static_cast<int>(left < L ? left : L);
            const int64_t loc = n_rows_local - row;
            if (loc < avail) avail = static_cast<int>(loc < 0 ? 0 : loc);
        }
        const int terms = avail < lq ? avail : lq;
        float sum = 0.f;
        if (lane == 0) prefix[warp][0] = 0.f;
        for (int j = 0; j < terms; ++j) {
            const float4 qv = reinterpret_cast<const float4*>(qt + j * D128)[lane];
            sum += warp_dot128(qv, x32 + (row + j) * D128, lane);
            if (lane == 0) prefix[warp][j + 1] = sum;
        }
        __syncwarp();
        for (int li = lane; li < n_len; li += 32) {
            const int sl = seq_lens[li];
            const int lq_sl = sl < lq ? sl : lq;
            int m = sl < terms ? sl : terms;
            float sc = -INFINITY;
            if (owned && m > 0 && uniq_j[u] < lq_sl) sc = prefix[warp][m] / static_cast<float>(m);
            cand_scores[(t * n_len + li) * SEQ_MAXC + u] = sc;
        }
        __syncwarp();
    }
    for (int li = 0; li < n_len; ++li)
        for (int u = nu + tid; u < SEQ_MAXC; u += blockDim.x) cand_scores[(t * n_len + li) * SEQ_MAXC + u] = -INFINITY;
}

__global__ void __launch_bounds__(256)
seq_top_kernel(int n_len, const int64_t* __restrict__ cand_ids, const float* __restrict__ cand_scores,
               const int32_t* __restrict__ n_cand, int64_t* __restrict__ pred_ids, float* __restrict__ pred_scores) {
    __shared__ uint64_t red[8];
    const int64_t t = blockIdx.x / n_len;
    const int li = blockIdx.x % n_len;
    const int tid = threadIdx.x;
    const int nu = n_cand[t];
    const float* sc = cand_scores + (t * n_len + li) * SEQ_MAXC;
    uint64_t mine[SEQ_MAXC / 256];
#pragma unroll
    for (int r = 0; r < SEQ_MAXC / 256; ++r) {
        const int u = r * 256 + tid;
        uint64_t key = 0;
        if (u < nu) {
            const float s = sc[u];
            if (s > -INFINITY) key = score_key(s, static_cast<uint32_t>(u));
        }
        mine[r] = key;
    }
    for (int p = 0; p < SEQ_NPRED; ++p) {
        uint64_t best = 0;
#pragma unroll
        for (int r = 0; r < SEQ_MAXC / 256; ++r) best = mine[r] > best ? mine[r] : best;
        const uint64_t w = block_max_u64(best, red);
        if (tid == 0) {
            const int64_t o = (t * n_len + li) * SEQ_NPRED + p;
            if (w != 0) {
                pred_ids[o] = cand_ids[t * SEQ_MAXC + key_row(w)];
                if (pred_scores) pred_scores[o] = key_score(w);
            } else {
                pred_ids[o] = -1;
                if (pred_scores) pred_scores[o] = -INFINITY;
            }
        }
#pragma unroll
        for (int r = 0; r < SEQ_MAXC / 256; ++r)
            if (mine[r] == w) mine[r] = 0;
        __syncthreads();
    }
}


// merge W per-shard top-k lists (already holding global labels) into one: order by (distance, label)
__global__ void topk_merge_kernel(const float* __restrict__ D_all, const int64_t* __restrict__ I_all, int W, int64_t nq, int k,
                                  float* __restrict__ D_out, int64_t* __restrict__ I_out) {
    __shared__ float d_s[TOPK_MERGE_KEYS];
    __shared__ int64_t i_s[TOPK_MERGE_KEYS];
    const int64_t q = blockIdx.x;
    const int n = W * k;
    int npow = 1;
    while (npow < n) npow <<= 1;
    for (int e = threadIdx.x; e < npow; e += blockDim.x) {
        float d = INFINITY;
        int64_t id = -1;
        if (e < n) {
            const int w = e / k, j = e % k;
            d = D_all[(static_cast<int64_t>(w) * nq + q) * k + j];
            id = I_all[(static_cast<int64_t>(w) * nq + q) * k + j];
        }
        if (id < 0) d = INFINITY;
        d_s[e] = d;
        i_s[e] = id < 0 ? LLONG_MAX : id;
    }
    __syncthreads();
    block_sort_dist_label(d_s, i_s, npow);
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        const int64_t id = i_s[j];
        D_out[q * k + j] = d_s[j];
        I_out[q * k + j] = id == LLONG_MAX ? -1 : id;
    }
}

// ---- clip matcher: one sequence of L (<= CLIP_MAXL) consecutive query rows per clip, any number of candidates.
//   clip_offsets_kernel  the device-side check of the clip offsets: any clip out of order or out of range -> flag
//   clip_cand_kernel     offset compensation c = label - j of every (row, neighbour) -> entry (clip << 32 | c)
//   clip_sort_*          device-wide ascending bitonic sort of those entries: candidates grouped by clip, ascending
//   clip_score_kernel    one warp per first occurrence: the running mean of q[j] . x32[c + j] (seq_cand_kernel's
//                        arithmetic), re-keyed as (clip, score descending, position) -- the position orders equal
//                        scores by candidate id
//   clip_sort_*          the same sort of the scored entries
//   clip_top_kernel      the first n_top entries of every clip
constexpr int CLIP_MAXL = 4096;
constexpr int CLIP_NTOP = 100;
constexpr int CLIP_SORT_TILE = 2048;      // entries one block sorts in shared memory (32 KB)
constexpr uint64_t CLIP_NONE = ~0ull;

// bad != 0 afterwards (it is zeroed before) unless 0 <= clip_off[0], every clip holds 1..CLIP_MAXL rows and
// clip_off[n_clips] <= n_rows
__global__ void __launch_bounds__(256)
clip_offsets_kernel(const int64_t* __restrict__ clip_off, int64_t n_clips, int64_t n_rows, int32_t* __restrict__ bad) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_clips;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t off = clip_off[i], L = clip_off[i + 1] - off;
        if (off < 0 || L < 1 || L > CLIP_MAXL || clip_off[i + 1] > n_rows) *bad = 1;
    }
}

// with bad offsets no (row, neighbour) becomes a candidate: every clip then reports -1 / -inf, and no query row
// outside [0, n_rows) is ever read
__global__ void __launch_bounds__(256)
clip_cand_kernel(const int64_t* __restrict__ I, int64_t n_keys, int k_probe, const int64_t* __restrict__ clip_off,
                 int64_t n_clips, const int32_t* __restrict__ bad, int64_t owned_lo, int64_t owned_hi, int64_t n_pad,
                 SortKV* __restrict__ out) {
    const bool ok = *bad == 0;
    for (int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; t < n_pad;
         t += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        SortKV v{CLIP_NONE, CLIP_NONE};
        if (ok && t < n_keys) {
            const int64_t g = t / k_probe;        // query row
            int64_t lo = 0, hi = n_clips;         // the last clip starting at or before g
            while (hi - lo > 1) {
                const int64_t mid = (lo + hi) >> 1;
                if (clip_off[mid] <= g) lo = mid;
                else hi = mid;
            }
            const int64_t off = clip_off[lo], L = clip_off[lo + 1] - off, j = g - off;
            const int64_t lab = I[t];
            const int64_t c = lab - j;
            if (L >= 1 && L <= CLIP_MAXL && j >= 0 && j < L && lab >= 0 && c >= 0 && c >= owned_lo && c < owned_hi)
                v = SortKV{(static_cast<uint64_t>(lo) << 32) | static_cast<uint64_t>(c), 0};
        }
        out[t] = v;
    }
}

__global__ void __launch_bounds__(1024) clip_sort_tiles_kernel(SortKV* __restrict__ a) {
    __shared__ SortKV s[CLIP_SORT_TILE];
    SortKV* g = a + static_cast<int64_t>(blockIdx.x) * CLIP_SORT_TILE;
    for (int i = threadIdx.x; i < CLIP_SORT_TILE; i += blockDim.x) s[i] = g[i];
    __syncthreads();
    block_sort_kv(s, CLIP_SORT_TILE);
    for (int i = threadIdx.x; i < CLIP_SORT_TILE; i += blockDim.x) g[i] = s[i];
}
__global__ void __launch_bounds__(1024) clip_merge_tiles_kernel(SortKV* __restrict__ a) {
    __shared__ SortKV s[CLIP_SORT_TILE];
    SortKV* g = a + static_cast<int64_t>(blockIdx.x) * CLIP_SORT_TILE;
    for (int i = threadIdx.x; i < CLIP_SORT_TILE; i += blockDim.x) s[i] = g[i];
    __syncthreads();
    block_merge_kv(s, CLIP_SORT_TILE);
    for (int i = threadIdx.x; i < CLIP_SORT_TILE; i += blockDim.x) g[i] = s[i];
}
// one global step of the merge at stride j >= CLIP_SORT_TILE; the first step of a merge of two sorted runs of j
// entries compares mirrored positions (i, 2j-1-i), which makes the pair one bitonic sequence
template <bool First>
__global__ void __launch_bounds__(256) clip_merge_step_kernel(SortKV* __restrict__ a, int64_t n_pairs, int64_t j) {
    for (int64_t p = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; p < n_pairs;
         p += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t i = pair_lo(p, j);
        kv_order(a, i, First ? (i | (j - 1)) + j - (i & (j - 1)) : i + j);
    }
}

__global__ void __launch_bounds__(256)
clip_score_kernel(const float* __restrict__ q, const int64_t* __restrict__ clip_off, const SortKV* __restrict__ cand,
                  int64_t n_pad, const float* __restrict__ x32, int64_t n_rows_local, int64_t label_offset,
                  SortKV* __restrict__ ranked, float* __restrict__ scores) {
    const int lane = threadIdx.x & 31;
    const int64_t n_warps = static_cast<int64_t>(gridDim.x) * (blockDim.x >> 5);
    for (int64_t e = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; e < n_pad; e += n_warps) {
        const uint64_t key = cand[e].hi;
        SortKV o{CLIP_NONE, CLIP_NONE};
        if (key != CLIP_NONE && (e == 0 || cand[e - 1].hi != key)) {      // first occurrence of (clip, c)
            const int64_t clip = static_cast<int64_t>(key >> 32), c = static_cast<int64_t>(key & 0xFFFFFFFFull);
            const int64_t off = clip_off[clip], L = clip_off[clip + 1] - off;
            const int64_t row = c - label_offset;
            const int64_t left = n_rows_local - row;             // rows of x32 that exist at c, c+1, ... (clamp)
            const int m = static_cast<int>(left < L ? left : L);
            const float* qc = q + off * D128;
            const float* xc = x32 + row * D128;
            float sum = 0.f;
            int j = 0;
            // four rows in flight per step; the running sum still adds them one by one in ascending j
            for (; j + 4 <= m; j += 4) {
                float4 qv[4], xv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    qv[u] = reinterpret_cast<const float4*>(qc + (j + u) * D128)[lane];
                    xv[u] = reinterpret_cast<const float4*>(xc + (j + u) * D128)[lane];
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) sum += warp_dot128_f4(qv[u], xv[u]);
            }
            for (; j < m; ++j) sum += warp_dot128(reinterpret_cast<const float4*>(qc + j * D128)[lane], xc + j * D128, lane);
            const float sc = sum / static_cast<float>(m);
            if (sc > -INFINITY) {
                const uint64_t desc = 0xFFFFFFFFull - (score_key(sc, 0) >> 32);
                o = SortKV{(static_cast<uint64_t>(clip) << 32) | desc, static_cast<uint64_t>(e)};
            }
            if (lane == 0) scores[e] = sc;
        }
        if (lane == 0) ranked[e] = o;
    }
}

// first entry of ranked[0, n) whose hi is >= v
__device__ __forceinline__ int64_t kv_lower_bound(const SortKV* __restrict__ a, int64_t n, uint64_t v) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (a[mid].hi < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
__global__ void __launch_bounds__(128)
clip_top_kernel(const SortKV* __restrict__ ranked, int64_t n_pad, const SortKV* __restrict__ cand,
                const float* __restrict__ scores, int64_t n_clips, int n_top, int64_t* __restrict__ pred_ids,
                float* __restrict__ pred_scores) {
    const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n_clips * n_top) return;
    const uint64_t clip = static_cast<uint64_t>(t / n_top);
    const int64_t r = t % n_top;
    const int64_t first = kv_lower_bound(ranked, n_pad, clip << 32);
    const int64_t end = kv_lower_bound(ranked, n_pad, (clip + 1) << 32);
    int64_t id = -1;
    float sc = -INFINITY;
    if (first + r < end) {
        const int64_t e = static_cast<int64_t>(ranked[first + r].lo);
        id = static_cast<int64_t>(cand[e].hi & 0xFFFFFFFFull);
        sc = scores[e];
    }
    pred_ids[t] = id;
    if (pred_scores) pred_scores[t] = sc;
}

// ascending sort of n_pad (a power of two >= CLIP_SORT_TILE) entries
static int clip_sort(nafp_ctx* ctx, SortKV* a, int64_t n_pad) {
    const unsigned tiles = static_cast<unsigned>(n_pad / CLIP_SORT_TILE);
    const int64_t n_pairs = n_pad / 2;
    const unsigned grid = static_cast<unsigned>(std::min<int64_t>((n_pairs + 255) / 256, int64_t(ctx->sm_count) * 16));
    clip_sort_tiles_kernel<<<tiles, 1024, 0, ctx->stream>>>(a);
    ctx->launches++;
    for (int64_t s = 2 * CLIP_SORT_TILE; s <= n_pad; s <<= 1) {
        clip_merge_step_kernel<true><<<grid, 256, 0, ctx->stream>>>(a, n_pairs, s >> 1);
        ctx->launches++;
        for (int64_t j = s >> 2; j >= CLIP_SORT_TILE; j >>= 1) {
            clip_merge_step_kernel<false><<<grid, 256, 0, ctx->stream>>>(a, n_pairs, j);
            ctx->launches++;
        }
        clip_merge_tiles_kernel<<<tiles, 1024, 0, ctx->stream>>>(a);
        ctx->launches++;
    }
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

static int64_t clip_pad(int64_t n_keys) {
    int64_t p = CLIP_SORT_TILE;
    while (p < n_keys) p <<= 1;
    return p;
}

// every checked argument of the clip matcher except the offsets, which only the host entry point can read
static int clip_check(nafp_index* idx, int64_t n_rows, int64_t n_clips, int32_t k_probe, int32_t n_top, const char* fn) {
    NAFP_REQUIRE(idx && n_rows >= 0 && n_clips >= 0, NAFP_ERR_INVALID, "%s: bad arguments", fn);
    NAFP_REQUIRE(k_probe >= 1 && k_probe <= MAX_K, NAFP_ERR_INVALID, "%s: k_probe %d outside [1,%d]", fn, k_probe, MAX_K);
    NAFP_REQUIRE(n_top >= 1 && n_top <= CLIP_NTOP, NAFP_ERR_INVALID, "%s: n_top %d outside [1,%d]", fn, n_top, CLIP_NTOP);
    NAFP_REQUIRE(n_rows * k_probe < (1ll << 31) && n_clips < (1ll << 31), NAFP_ERR_INVALID,
                 "%s: n_rows * k_probe must stay below 2^31 (split the clips over several calls)", fn);
    NAFP_REQUIRE(idx->label_offset + idx->n < (1ll << 32), NAFP_ERR_INVALID, "%s: labels must stay below 2^32", fn);
    NAFP_REQUIRE(idx->x32 != nullptr || idx->n == 0, NAFP_ERR_STATE, "%s: index holds no rows", fn);
    return NAFP_OK;
}

}  // namespace nafp

using namespace nafp;

extern "C" {

int nafp_seq_plan_dev(nafp_ctx* ctx, const int64_t* test_ids_dev, int64_t n_test, int32_t max_len,
                      int64_t n_query_rows, int32_t* scratch_dev, int32_t* rowmap_dev, int32_t* uniq_rows_dev,
                      int64_t* n_uniq_out) {
    NAFP_RANGE("nafp_seq_plan_dev");
    NAFP_REQUIRE(ctx && test_ids_dev && scratch_dev && rowmap_dev && uniq_rows_dev && n_uniq_out && n_test >= 0 &&
                     max_len >= 1 && max_len <= SEQ_MAXL && n_query_rows >= 0 && n_query_rows < (1ll << 31),
                 NAFP_ERR_INVALID, "nafp_seq_plan_dev: bad arguments (max_len <= %d)", SEQ_MAXL);
    *n_uniq_out = 0;
    if (n_test == 0 || n_query_rows == 0) return NAFP_OK;
    int32_t* flags = scratch_dev;                        // [n_query_rows]
    int32_t* pos = scratch_dev + n_query_rows;           // [n_query_rows]
    int32_t* count = scratch_dev + 2 * n_query_rows;     // [1]
    const int64_t pairs = n_test * max_len;
    NAFP_CUDA(cudaMemsetAsync(flags, 0, static_cast<size_t>(n_query_rows) * sizeof(int32_t), ctx->stream));
    seq_mark_kernel<<<static_cast<unsigned>((pairs + 255) / 256), 256, 0, ctx->stream>>>(test_ids_dev, n_test, max_len,
                                                                                       n_query_rows, flags);
    seq_scan_kernel<<<1, 1024, 0, ctx->stream>>>(flags, n_query_rows, pos, uniq_rows_dev, count);
    seq_rowmap_kernel<<<static_cast<unsigned>((pairs + 255) / 256), 256, 0, ctx->stream>>>(test_ids_dev, n_test, max_len,
                                                                                         n_query_rows, pos, rowmap_dev);
    ctx->launches += 3;
    NAFP_CUDA(cudaGetLastError());
    int32_t h = 0;
    NAFP_CUDA(cudaMemcpyAsync(&h, count, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    *n_uniq_out = h;
    return NAFP_OK;
}

int nafp_seq_gather_rows_dev(nafp_ctx* ctx, const float* q_dev, const int32_t* rows_dev, int64_t n_rows,
                             float* out_dev) {
    NAFP_RANGE("nafp_seq_gather_rows_dev");
    NAFP_REQUIRE(ctx && n_rows >= 0 && (n_rows == 0 || (q_dev && rows_dev && out_dev)), NAFP_ERR_INVALID,
                 "nafp_seq_gather_rows_dev: bad arguments");
    if (n_rows == 0) return NAFP_OK;
    seq_gather_rows_kernel<<<static_cast<unsigned>((n_rows * 32 + 255) / 256), 256, 0, ctx->stream>>>(q_dev, rows_dev, n_rows,
                                                                                                    out_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

int nafp_seq_cand_dev(nafp_index* idx, const float* q_dev, int64_t n_query_rows, const int64_t* test_ids_dev,
                      int64_t n_test, const int32_t* seq_lens_dev, int32_t n_len, int32_t max_len, int32_t k_probe,
                      const int64_t* I_dev, const int32_t* rowmap_dev, int64_t n_rows_global, int64_t owned_lo,
                      int64_t owned_hi, int64_t* cand_ids_dev, float* cand_scores_dev, int32_t* n_cand_dev) {
    NAFP_RANGE("nafp_seq_cand_dev");
    NAFP_REQUIRE(idx && q_dev && test_ids_dev && seq_lens_dev && I_dev && cand_ids_dev && cand_scores_dev &&
                     n_cand_dev, NAFP_ERR_INVALID, "nafp_seq_cand_dev: NULL argument");
    NAFP_REQUIRE(max_len >= 1 && max_len <= SEQ_MAXL && k_probe >= 1 && max_len * k_probe <= SEQ_MAXC &&
                     n_len >= 1 && n_len <= 32, NAFP_ERR_INVALID,
                 "nafp_seq_cand_dev: need max_len <= %d, n_len <= 32, max_len*k_probe <= %d", SEQ_MAXL, SEQ_MAXC);
    NAFP_REQUIRE(idx->x32 != nullptr || idx->n == 0, NAFP_ERR_STATE, "nafp_seq_cand_dev: index holds no rows");
    if (n_test == 0) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    seq_cand_kernel<<<static_cast<unsigned>(n_test), 256, 0, ctx->stream>>>(
        q_dev, n_query_rows, test_ids_dev, seq_lens_dev, n_len, max_len, k_probe, I_dev, rowmap_dev, idx->x32, idx->n,
        n_rows_global, idx->label_offset, owned_lo, owned_hi, cand_ids_dev, cand_scores_dev, n_cand_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

int nafp_seq_top_dev(nafp_ctx* ctx, int64_t n_test, int32_t n_len, const int64_t* cand_ids_dev,
                     const float* cand_scores_dev, const int32_t* n_cand_dev, int64_t* pred_ids_dev,
                     float* pred_scores_dev) {
    NAFP_RANGE("nafp_seq_top_dev");
    NAFP_REQUIRE(ctx && cand_ids_dev && cand_scores_dev && n_cand_dev && pred_ids_dev && n_len >= 1,
                 NAFP_ERR_INVALID, "nafp_seq_top_dev: bad arguments");
    if (n_test == 0) return NAFP_OK;
    seq_top_kernel<<<static_cast<unsigned>(n_test * n_len), 256, 0, ctx->stream>>>(
        n_len, cand_ids_dev, cand_scores_dev, n_cand_dev, pred_ids_dev, pred_scores_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

int nafp_topk_merge_dev(nafp_ctx* ctx, const float* D_all_dev, const int64_t* I_all_dev, int32_t n_shards,
                        int64_t nq, int32_t k, float* D_out_dev, int64_t* I_out_dev) {
    NAFP_RANGE("nafp_topk_merge_dev");
    NAFP_REQUIRE(ctx && D_all_dev && I_all_dev && D_out_dev && I_out_dev && n_shards >= 1 && k >= 1 &&
                     n_shards * k <= TOPK_MERGE_KEYS, NAFP_ERR_INVALID, "nafp_topk_merge_dev: need n_shards*k <= %d",
                 TOPK_MERGE_KEYS);
    if (nq == 0) return NAFP_OK;
    topk_merge_kernel<<<static_cast<unsigned>(nq), 128, 0, ctx->stream>>>(D_all_dev, I_all_dev, n_shards, nq, k,
                                                                          D_out_dev, I_out_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

int nafp_seq_match(nafp_index* idx, const float* q_host, int64_t n_query_rows, const int64_t* test_ids,
                   int64_t n_test, const int32_t* seq_lens, int32_t n_len, int32_t k_probe, int64_t* pred_ids_host,
                   float* pred_scores_host) {
    NAFP_RANGE("nafp_seq_match");
    NAFP_REQUIRE(idx && q_host && test_ids && seq_lens && pred_ids_host && n_test >= 0 && n_len >= 1 &&
                     n_query_rows >= 0, NAFP_ERR_INVALID, "nafp_seq_match: bad arguments");
    if (n_test == 0) return NAFP_OK;
    int L = 0;
    for (int i = 0; i < n_len; ++i) {
        NAFP_REQUIRE(seq_lens[i] >= 1 && seq_lens[i] <= SEQ_MAXL, NAFP_ERR_INVALID,
                     "nafp_seq_match: sequence length %d outside [1,%d]", seq_lens[i], SEQ_MAXL);
        if (seq_lens[i] > L) L = seq_lens[i];
    }
    NAFP_REQUIRE(k_probe >= 1 && k_probe * L <= SEQ_MAXC && k_probe <= MAX_K, NAFP_ERR_INVALID,
                 "nafp_seq_match: k_probe*max_len must be <= %d", SEQ_MAXC);
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    const int64_t pairs = n_test * L;
    const int64_t rows_cap = pairs < n_query_rows ? pairs : n_query_rows;      // unique query rows, at most
    // one arena for all temporaries
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_q = take(static_cast<size_t>(n_query_rows) * D128 * 4);
    const size_t o_ids = take(static_cast<size_t>(n_test) * 8);
    const size_t o_sl = take(static_cast<size_t>(n_len) * 4);
    const size_t o_scr = take(static_cast<size_t>(2 * n_query_rows + 1) * 4);
    const size_t o_map = take(static_cast<size_t>(pairs) * 4);
    const size_t o_uniq = take(static_cast<size_t>(pairs) * 4);
    const size_t o_qrows = take(static_cast<size_t>(rows_cap) * D128 * 4);
    const size_t o_D = take(static_cast<size_t>(rows_cap) * k_probe * 4);
    const size_t o_I = take(static_cast<size_t>(rows_cap) * k_probe * 8);
    const size_t o_cid = take(static_cast<size_t>(n_test) * SEQ_MAXC * 8);
    const size_t o_csc = take(static_cast<size_t>(n_test) * n_len * SEQ_MAXC * 4);
    const size_t o_nc = take(static_cast<size_t>(n_test) * 4);
    const size_t o_pid = take(static_cast<size_t>(n_test) * n_len * SEQ_NPRED * 8);
    const size_t o_psc = take(static_cast<size_t>(n_test) * n_len * SEQ_NPRED * 4);
    NAFP_TRY(ensure_dev(ctx, &ctx->stage_dev, &ctx->stage_dev_bytes, static_cast<int64_t>(off)));
    uint8_t* base = static_cast<uint8_t*>(ctx->stage_dev);
    float* q_dev = reinterpret_cast<float*>(base + o_q);
    int64_t* ids_dev = reinterpret_cast<int64_t*>(base + o_ids);
    int32_t* sl_dev = reinterpret_cast<int32_t*>(base + o_sl);
    int32_t* scr = reinterpret_cast<int32_t*>(base + o_scr);
    int32_t* rowmap = reinterpret_cast<int32_t*>(base + o_map);
    int32_t* uniq = reinterpret_cast<int32_t*>(base + o_uniq);
    float* qrows = reinterpret_cast<float*>(base + o_qrows);
    float* Dd = reinterpret_cast<float*>(base + o_D);
    int64_t* Id = reinterpret_cast<int64_t*>(base + o_I);
    int64_t* cid = reinterpret_cast<int64_t*>(base + o_cid);
    float* csc = reinterpret_cast<float*>(base + o_csc);
    int32_t* nc = reinterpret_cast<int32_t*>(base + o_nc);
    int64_t* pid = reinterpret_cast<int64_t*>(base + o_pid);
    float* psc = reinterpret_cast<float*>(base + o_psc);
    NAFP_CUDA(cudaMemcpyAsync(q_dev, q_host, static_cast<size_t>(n_query_rows) * D128 * 4, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(ids_dev, test_ids, static_cast<size_t>(n_test) * 8, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(sl_dev, seq_lens, static_cast<size_t>(n_len) * 4, cudaMemcpyHostToDevice, ctx->stream));
    // every query row that some (test id, offset) needs is searched ONCE
    int64_t n_uniq = 0;
    NAFP_TRY(nafp_seq_plan_dev(ctx, ids_dev, n_test, L, n_query_rows, scr, rowmap, uniq, &n_uniq));
    NAFP_TRY(nafp_seq_gather_rows_dev(ctx, q_dev, uniq, n_uniq, qrows));
    NAFP_TRY(nafp_index_search_dev(idx, qrows, n_uniq, k_probe, Dd, Id));
    const int64_t n_search = idx->search_rows >= 0 && idx->search_rows < idx->n ? idx->search_rows : idx->n;
    NAFP_TRY(nafp_seq_cand_dev(idx, q_dev, n_query_rows, ids_dev, n_test, sl_dev, n_len, L, k_probe, Id, rowmap,
                               idx->label_offset + idx->n, idx->label_offset, idx->label_offset + n_search, cid, csc, nc));
    NAFP_TRY(nafp_seq_top_dev(ctx, n_test, n_len, cid, csc, nc, pid, psc));
    NAFP_CUDA(cudaMemcpyAsync(pred_ids_host, pid, static_cast<size_t>(n_test) * n_len * SEQ_NPRED * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (pred_scores_host)
        NAFP_CUDA(cudaMemcpyAsync(pred_scores_host, psc, static_cast<size_t>(n_test) * n_len * SEQ_NPRED * 4, cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

int nafp_clip_match_dev(nafp_index* idx, const float* q_dev, int64_t n_rows, const int64_t* clip_off_dev,
                        int64_t n_clips, int32_t k_probe, int32_t n_top, int64_t* pred_ids_dev, float* pred_scores_dev) {
    NAFP_RANGE("nafp_clip_match_dev");
    NAFP_TRY(clip_check(idx, n_rows, n_clips, k_probe, n_top, "nafp_clip_match_dev"));
    NAFP_REQUIRE(n_clips == 0 || (q_dev && clip_off_dev && pred_ids_dev), NAFP_ERR_INVALID,
                 "nafp_clip_match_dev: NULL argument");
    if (n_clips == 0) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_keys = n_rows * k_probe;
    const int64_t n_pad = clip_pad(n_keys);
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_D = take(static_cast<size_t>(n_keys) * 4);
    const size_t o_I = take(static_cast<size_t>(n_keys) * 8);
    const size_t o_cand = take(static_cast<size_t>(n_pad) * sizeof(SortKV));
    const size_t o_rank = take(static_cast<size_t>(n_pad) * sizeof(SortKV));
    const size_t o_sc = take(static_cast<size_t>(n_pad) * 4);
    const size_t o_bad = take(4);
    NAFP_TRY(ensure_dev(ctx, &ctx->clip_ws, &ctx->clip_ws_bytes, static_cast<int64_t>(off)));
    uint8_t* base = static_cast<uint8_t*>(ctx->clip_ws);
    float* Dd = reinterpret_cast<float*>(base + o_D);
    int64_t* Id = reinterpret_cast<int64_t*>(base + o_I);
    SortKV* cand = reinterpret_cast<SortKV*>(base + o_cand);
    SortKV* ranked = reinterpret_cast<SortKV*>(base + o_rank);
    float* scores = reinterpret_cast<float*>(base + o_sc);
    int32_t* bad = reinterpret_cast<int32_t*>(base + o_bad);

    if (n_rows > 0) NAFP_TRY(nafp_index_search_dev(idx, q_dev, n_rows, k_probe, Dd, Id));
    const int64_t n_search = idx->search_rows >= 0 && idx->search_rows < idx->n ? idx->search_rows : idx->n;
    const unsigned grid = static_cast<unsigned>(std::min<int64_t>((n_pad + 255) / 256, int64_t(ctx->sm_count) * 16));
    NAFP_CUDA(cudaMemsetAsync(bad, 0, 4, ctx->stream));
    const unsigned grid_c = static_cast<unsigned>(std::min<int64_t>((n_clips + 255) / 256, int64_t(ctx->sm_count) * 4));
    clip_offsets_kernel<<<grid_c, 256, 0, ctx->stream>>>(clip_off_dev, n_clips, n_rows, bad);
    clip_cand_kernel<<<grid, 256, 0, ctx->stream>>>(Id, n_keys, k_probe, clip_off_dev, n_clips, bad, idx->label_offset,
                                                   idx->label_offset + n_search, n_pad, cand);
    ctx->launches += 2;
    NAFP_CUDA(cudaGetLastError());
    NAFP_TRY(clip_sort(ctx, cand, n_pad));
    // one warp per entry: 8 per block, enough blocks to fill every SM many times over
    const unsigned grid_w = static_cast<unsigned>(std::min<int64_t>((n_pad + 7) / 8, int64_t(ctx->sm_count) * 64));
    clip_score_kernel<<<grid_w, 256, 0, ctx->stream>>>(q_dev, clip_off_dev, cand, n_pad, idx->x32, idx->n,
                                                      idx->label_offset, ranked, scores);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    NAFP_TRY(clip_sort(ctx, ranked, n_pad));
    const int64_t n_out = n_clips * n_top;
    clip_top_kernel<<<static_cast<unsigned>((n_out + 127) / 128), 128, 0, ctx->stream>>>(
        ranked, n_pad, cand, scores, n_clips, n_top, pred_ids_dev, pred_scores_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

int nafp_clip_match(nafp_index* idx, const float* q_host, int64_t n_rows, const int64_t* clip_off_host,
                    int64_t n_clips, int32_t k_probe, int32_t n_top, int64_t* pred_ids_host, float* pred_scores_host) {
    NAFP_RANGE("nafp_clip_match");
    NAFP_TRY(clip_check(idx, n_rows, n_clips, k_probe, n_top, "nafp_clip_match"));
    NAFP_REQUIRE(clip_off_host && (n_clips == 0 || (q_host && pred_ids_host)), NAFP_ERR_INVALID,
                 "nafp_clip_match: NULL argument");
    NAFP_REQUIRE(clip_off_host[0] == 0 && clip_off_host[n_clips] == n_rows, NAFP_ERR_INVALID,
                 "nafp_clip_match: clip offsets must run from 0 to n_rows (%lld)", static_cast<long long>(n_rows));
    for (int64_t i = 0; i < n_clips; ++i) {
        const int64_t L = clip_off_host[i + 1] - clip_off_host[i];
        NAFP_REQUIRE(L >= 1 && L <= CLIP_MAXL, NAFP_ERR_INVALID,
                     "nafp_clip_match: clip %lld has %lld rows; clip offsets must ascend by 1..%d rows",
                     static_cast<long long>(i), static_cast<long long>(L), CLIP_MAXL);
    }
    if (n_clips == 0) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const size_t o_q = take(static_cast<size_t>(n_rows) * D128 * 4);
    const size_t o_off = take(static_cast<size_t>(n_clips + 1) * 8);
    const size_t o_pid = take(static_cast<size_t>(n_clips) * n_top * 8);
    const size_t o_psc = take(static_cast<size_t>(n_clips) * n_top * 4);
    NAFP_TRY(ensure_dev(ctx, &ctx->stage_dev, &ctx->stage_dev_bytes, static_cast<int64_t>(off)));
    uint8_t* base = static_cast<uint8_t*>(ctx->stage_dev);
    float* q_dev = reinterpret_cast<float*>(base + o_q);
    int64_t* off_dev = reinterpret_cast<int64_t*>(base + o_off);
    int64_t* pid = reinterpret_cast<int64_t*>(base + o_pid);
    float* psc = reinterpret_cast<float*>(base + o_psc);
    NAFP_CUDA(cudaMemcpyAsync(q_dev, q_host, static_cast<size_t>(n_rows) * D128 * 4, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(off_dev, clip_off_host, static_cast<size_t>(n_clips + 1) * 8, cudaMemcpyHostToDevice,
                              ctx->stream));
    NAFP_TRY(nafp_clip_match_dev(idx, q_dev, n_rows, off_dev, n_clips, k_probe, n_top, pid, psc));
    NAFP_CUDA(cudaMemcpyAsync(pred_ids_host, pid, static_cast<size_t>(n_clips) * n_top * 8, cudaMemcpyDeviceToHost,
                              ctx->stream));
    if (pred_scores_host)
        NAFP_CUDA(cudaMemcpyAsync(pred_scores_host, psc, static_cast<size_t>(n_clips) * n_top * 4,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

}  // extern "C"
