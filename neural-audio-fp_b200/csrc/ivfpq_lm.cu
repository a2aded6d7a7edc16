// List-major compressed-domain IVF-PQ search (SURVEY §8 a6; eval/utils/get_index_faiss.py:69-74,120).
//
// faiss scans, per (query, probed list), the list's 64-byte codes through a 64 x 256 look-up table.  On B200 the
// same sum is a tensor-core contraction:  with xhat = c_l + d (d = the decoded PQ residual of the row)
//
//     |q - xhat|^2 = |q - c_l|^2 - 2 (q . d - h),        h = 0.5 |d|^2 + c_l . d   (one fp32 per stored row)
//
// so ranking the rows of list l for query q means ranking  q . d - h.  The index stays compressed in HBM
// (64 B codes + 4 B h + 4 B row id per list position); a CTA works on one (list, block of <= 128 query rows that
// probe it) item at a time:
//
//   decoder warps   read 128 list positions of codes (stored tile-transposed so that a lane is a sub-quantizer), look the
//                   64 sub-vectors up in a bf16 copy of the PQ codebooks kept in shared memory (64 KB, one bank per
//                   sub-quantizer: conflict-free) and write them as a 128 x 128 bf16 K-major SWIZZLE_128B tile -- the
//                   layout TMA would have produced from a decoded copy of the rows -- into a 2-stage ring
//   MMA warp        tcgen05.mma  D[query][position] = Q (128 x 128 bf16, written to TENSOR MEMORY once per item) x tile^T
//                   - h: the row term rides a ninth K step -- the decoders write -h as three bf16 (hi + mid + lo, 24 bits)
//                   into a third K block of the stage, the query block has three columns of ones --; fp32 accumulators
//                   double-buffered in TMEM
//   epilogue warps  two groups of four, one query per thread, 64 of the tile's columns per group: the accumulator IS the
//                   score; it is compared with the query's threshold (one register); the rare hits are inserted
//                   warp-cooperatively into the group's sorted 32-entry candidate list of the query in shared memory
//
// Three launches per search.  Wave 0 scans every query's NEAREST list with an open threshold; the exact fp32 ADC
// distance of its k-th candidate bounds the answer (Dk).  Waves 1 (probe ranks 1-3) and 2 (the rest) start from the
// threshold  0.5 (|q - c_l|^2 - Dk) - E  (E = the bf16 rounding bound |q| max|d| 2^-8): rows below it cannot
// enter the top k, so almost nothing is inserted.  ivfpq_lm_merge_kernel re-scores the survivors with the LUT
// kernel's own fp32 arithmetic, sorts, and PROVES the answer (a full 32-entry list must end below the k-th exact
// distance by more than the rounding bound); unproven rows -- duplicates, ties -- go to the LUT kernel.
//
// k > 24 (up to 128, the 4 k first-level candidates of IVFPQR): every (query row, probed list) pair becomes S = ceil(k / 24)
// SLICES, each over a disjoint contiguous range of the list's tiles with its own two 32-entry lists; the waves, the bound
// and the proof walk S times as many lists.  Wave 0 then keeps S * 64 >= 2.6 k candidates of the nearest list.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cstring>
#include <vector>

#include "ivfpq.h"
#include "ptx.cuh"
#include "topk.cuh"

namespace nafp {

constexpr int LM_ROWS = 128;              // list positions per tile (MMA N, accumulator columns)
constexpr int LM_Q = 128;                 // query rows per work item (MMA M, TMEM lanes)
constexpr int LM_KP = 32;                 // entries of one warp-wide sorted candidate list
constexpr int LM_GROUPS = 2;              // epilogue warp groups: each keeps its own list per query for its half of a tile's columns
constexpr int LM_SLOT = LM_KP * LM_GROUPS; // candidates kept per (query row, probed list)
constexpr int LM_SLICE_K = 24;            // k one slice of a list answers (k + 8 spare candidates for the proof)
constexpr int LM_MAX_K = 128;             // k the path answers: ceil(k / LM_SLICE_K) slices per (query row, probed list)
constexpr int LM_MAX_NPROBE = 64;
constexpr int LM_MERGE_KEYS = LM_MAX_NPROBE * LM_SLOT;  // survivors one merge block sorts (every candidate when S = 1)
constexpr int LM_STAGES = 2;
constexpr int LM_WAVES = 3;               // launches per search: probe rank 0 | ranks 1 .. LM_WAVE1_END-1 | the rest
constexpr int LM_WAVE1_END = 4;
constexpr int LM_PF = 6;                  // tiles ahead whose codes are prefetched into L2
constexpr int LM_EPI_WARPS = 4 * LM_GROUPS, LM_DEC_WARPS = 8;
constexpr int LM_MMA_WARP = LM_EPI_WARPS + LM_DEC_WARPS;
constexpr int LM_THREADS = (LM_MMA_WARP + 1) * 32;      // 544
constexpr int LM_DEC_THREADS = LM_DEC_WARPS * 32;       // 256: (position, K block) per thread
constexpr int LM_KB_BYTES = LM_ROWS * 128;              // 16 KB: one 64-dim K block of a tile (= of the query block)
constexpr int LM_TMEM_A = 256;                          // TMEM columns [256, 320): the item's query block (A operand), after the two accumulators
constexpr int LM_B_BYTES = 3 * LM_KB_BYTES;             // 48 KB per stage: two K blocks of decoded rows + the K block of -h
constexpr int LM_TAB_BYTES = 64 * PQ_KSUB * 4;          // 64 KB: [sub-quantizer][code] -> two bf16
constexpr int LM_LIST_BYTES = LM_Q * LM_SLOT * 8;       // 64 KB
constexpr int LM_SMEM = 1024 + LM_STAGES * LM_B_BYTES + LM_TAB_BYTES + LM_LIST_BYTES + 512;
constexpr int64_t LM_CHUNK_Q = 32768;     // query rows per launch group at S = 1, LM_CHUNK_Q / S at S slices (bounds the
                                          // candidate buffer: 512 B per pair and slice)
static_assert(LM_ROWS == 128, "the epilogue reads four 32-column chunks per tile");
static_assert(LM_Q == LM_ROWS, "the query block and the tile share the K-block size");

__host__ __device__ __forceinline__ int lm_wave(int p) { return p == 0 ? 0 : (p < LM_WAVE1_END ? 1 : 2); }
static int lm_slices(int k) { return (k + LM_SLICE_K - 1) / LM_SLICE_K; }

struct LmItem {
    int32_t list, start, len, tiles;      // query pairs[start .. start + len) against tiles [t0, t0 + tiles) of list `list`
    int32_t t0, slice;                    // ... which are slice `slice` of the list
};

struct LmState {
    uint32_t* tab = nullptr;              // [64][256] bf16 pair of every codeword
    float* lh = nullptr;                  // [list position] 0.5 |d|^2 + c . d, +inf for rows outside the searched range
    int32_t* dmax2 = nullptr;             // device scalar: bits of max |d|^2
    int64_t lh_cap = 0;
    int64_t built_version = -1, built_n_search = -1;
    // per launch group
    int32_t* probes = nullptr;            // [nq][nprobe]
    float* gdist = nullptr;               // [nq][nprobe] |q - c_l|^2
    float* qE = nullptr;                  // [nq] rounding bound of the bf16 scores
    float* dkA = nullptr;                 // [nq] k-th exact distance inside the nearest list
    int32_t* pairs = nullptr;             // [nq * nprobe] (query, probe) pairs grouped by (phase, list)
    uint64_t* cand = nullptr;             // [nq * nprobe][S][LM_GROUPS][LM_KP]
    int64_t cap_pairs = 0, cap_q = 0, cap_cand = 0;
    int32_t* hist = nullptr;              // [LM_WAVES * nlist] bucket sizes, the same of scatter cursors, [LM_WAVES] item counters
    LmItem* items = nullptr;
    int64_t items_cap = 0;
    unsigned long long items_run = 0, tiles_run = 0;      // statistics (ivfpq_lm_take_stats)
};

void ivfpq_lm_destroy(IvfPq* s) {
    LmState* L = s->lm;
    if (!L) return;
    void* bufs[] = {L->tab, L->lh, L->dmax2, L->probes, L->gdist, L->qE, L->dkA, L->pairs, L->cand, L->hist, L->items};
    for (void* b : bufs) if (b) cudaFree(b);
    delete L;
    s->lm = nullptr;
}

void ivfpq_lm_take_stats(IvfPq* s, int64_t* items, int64_t* tiles) {
    *items = *tiles = 0;
    if (!s->lm) return;
    *items = static_cast<int64_t>(s->lm->items_run);
    *tiles = static_cast<int64_t>(s->lm->tiles_run);
    s->lm->items_run = s->lm->tiles_run = 0;
}

int ivfpq_lm_supported(const nafp_index* idx, int k) {
    const IvfPq* s = idx->ivf;
    const int nprobe = idx->nprobe < s->nlist ? idx->nprobe : s->nlist;
    return !s->flat_lists && s->m == 64 && s->dsub == 2 && k <= LM_MAX_K && nprobe <= LM_MAX_NPROBE && idx->n < (1ll << 31);
}

// ------------------------------------------------------------------------------------------ index-side tables
__global__ void lm_table_kernel(const float* __restrict__ pq, uint32_t* __restrict__ tab) {
    // tab[K block = sub / 32][code][sub % 32]: the 256 codewords of one sub-quantizer sit in ONE shared-memory bank
    const int e = blockIdx.x * blockDim.x + threadIdx.x;           // sub * 256 + code
    if (e >= 64 * PQ_KSUB) return;
    const int sub = e >> 8, code = e & 255;
    const __nv_bfloat162 v = __floats2bfloat162_rn(pq[2 * e], pq[2 * e + 1]);
    tab[(sub >> 5) * (PQ_KSUB * 32) + code * 32 + (sub & 31)] = *reinterpret_cast<const uint32_t*>(&v);
}

// one thread per (padded) list position: h = 0.5 |d|^2 + c . d of the stored row, max |d|^2 of the index
__global__ void lm_rowterm_kernel(const uint8_t* __restrict__ lcodes, const int32_t* __restrict__ lids, const int32_t* __restrict__ assign,
                                  int64_t n_pos, int64_t n_search, const float* __restrict__ coarse, const float* __restrict__ pq,
                                  float* __restrict__ lh, int32_t* __restrict__ dmax2) {
    const int64_t pos = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    float nn = 0.f;
    if (pos < n_pos) {
        const int32_t row = lids[pos];
        float h = INFINITY;                    // padding, and rows past n_search (halo of a row-sharded index): never candidates
        if (row >= 0 && row < n_search) {
            const float* c = coarse + static_cast<int64_t>(assign[row]) * D128;
            const uint8_t* cp = lcodes + lcode_off(pos, 0, 64);
            float cd = 0.f;
#pragma unroll 8
            for (int sub = 0; sub < 64; ++sub) {
                const uint32_t code = cp[(sub >> 5) * (LIST_TILE * 32) + 4 * (sub & 31)];
                const float2 p = *reinterpret_cast<const float2*>(pq + (static_cast<int64_t>(sub) * PQ_KSUB + code) * 2);
                const float2 cc = *reinterpret_cast<const float2*>(c + 2 * sub);
                nn = fmaf(p.x, p.x, fmaf(p.y, p.y, nn));
                cd = fmaf(cc.x, p.x, fmaf(cc.y, p.y, cd));
            }
            h = 0.5f * nn + cd;
        }
        lh[pos] = h;
    }
    nn = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(nn)));     // (non-negative floats order like their bits)
    if ((threadIdx.x & 31) == 0 && nn > 0.f) atomicMax(dmax2, __float_as_int(nn));
}

static int lm_prepare(nafp_index* idx, int64_t n_search) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    if (!s->lm) {
        s->lm = new LmState();
        NAFP_CUDA(cudaMalloc(&s->lm->tab, LM_TAB_BYTES));
        NAFP_CUDA(cudaMalloc(&s->lm->dmax2, sizeof(int32_t)));
        NAFP_CUDA(cudaMalloc(&s->lm->hist, (2 * LM_WAVES * IVF_MAX_NLIST + LM_WAVES) * sizeof(int32_t)));
    }
    LmState* L = s->lm;
    NAFP_TRY(build_lists(idx));
    if (L->built_version == s->lists_version && L->built_n_search == n_search) return NAFP_OK;
    const int64_t n_pos = s->h_loff[s->nlist];
    if (L->lh_cap < n_pos) {
        if (L->lh) cudaFree(L->lh);
        L->lh = nullptr; L->lh_cap = 0;
        NAFP_CUDA(cudaMalloc(&L->lh, static_cast<size_t>(s->sorted_cap) * sizeof(float)));
        L->lh_cap = s->sorted_cap;
    }
    lm_table_kernel<<<64, 256, 0, ctx->stream>>>(s->pq, L->tab);
    NAFP_CUDA(cudaMemsetAsync(L->dmax2, 0, sizeof(int32_t), ctx->stream));
    if (n_pos > 0)
        lm_rowterm_kernel<<<static_cast<unsigned>((n_pos + 255) / 256), 256, 0, ctx->stream>>>(s->lcodes, s->lids, s->assign, n_pos, n_search,
                                                                                             s->coarse, s->pq, L->lh, L->dmax2);
    ctx->launches += 2;
    NAFP_CUDA(cudaGetLastError());
    L->built_version = s->lists_version;
    L->built_n_search = n_search;
    return NAFP_OK;
}

// ------------------------------------------------------------------------------------------ per-search preparation
// (query, probe) pairs -> buckets: wave of the probe rank (0: the query's nearest list) * nlist + list
__global__ void lm_hist_kernel(const int32_t* __restrict__ probes, int64_t n_pairs, int nprobe, int nlist, int32_t* __restrict__ hist) {
    __shared__ int h[LM_WAVES * IVF_MAX_NLIST];
    for (int b = threadIdx.x; b < LM_WAVES * nlist; b += blockDim.x) h[b] = 0;
    __syncthreads();
    for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < n_pairs; e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int l = probes[e];
        if (l >= 0) atomicAdd(&h[lm_wave(static_cast<int>(e % nprobe)) * nlist + l], 1);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < LM_WAVES * nlist; b += blockDim.x)
        if (h[b]) atomicAdd(&hist[b], h[b]);
}
__global__ void lm_scatter_kernel(const int32_t* __restrict__ probes, int64_t n_pairs, int nprobe, int nlist, int32_t* __restrict__ cursor,
                                  int32_t* __restrict__ pairs) {
    const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= n_pairs) return;
    const int l = probes[e];
    if (l < 0) return;
    pairs[atomicAdd(&cursor[lm_wave(static_cast<int>(e % nprobe)) * nlist + l], 1)] = static_cast<int32_t>(e);
}

// ------------------------------------------------------------------------------------------ the scan
struct LmBars {
    uint64_t bfull[LM_STAGES];
    uint64_t bempty[LM_STAGES];
    uint64_t afull[2];
    uint64_t aempty[2];
    uint32_t tmem_base;
    int item;
};

__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T, kind::f16: the A operand read from tensor memory (row = lane, 16 bf16 = 8 columns per K step)
__device__ __forceinline__ void lm_mma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

__global__ void __launch_bounds__(LM_THREADS, 1)
ivfpq_lm_scan_kernel(const float* __restrict__ q, int nprobe, int S, const LmItem* __restrict__ items, int n_items,
                     int32_t* __restrict__ item_counter, const int32_t* __restrict__ pairs, const uint32_t* __restrict__ tab,
                     const uint8_t* __restrict__ lcodes, const float* __restrict__ lh, const int32_t* __restrict__ loff,
                     const float* __restrict__ gdist, const float* __restrict__ dkA, const float* __restrict__ qE,
                     uint64_t* __restrict__ cand) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* b_s = smem;                                             // [stage][kb 2][128 positions][128 B]
    uint32_t* tab_s = reinterpret_cast<uint32_t*>(b_s + LM_STAGES * LM_B_BYTES);
    uint64_t* lst_s = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(tab_s) + LM_TAB_BYTES);   // [group][128 queries][32] sorted, descending
    LmBars* bars = reinterpret_cast<LmBars*>(reinterpret_cast<uint8_t*>(lst_s) + LM_LIST_BYTES);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    for (int i = threadIdx.x; i < LM_TAB_BYTES / 16; i += LM_THREADS)
        reinterpret_cast<uint4*>(tab_s)[i] = __ldg(reinterpret_cast<const uint4*>(tab) + i);
    // the third K block of every stage carries -h of the tile's rows in its first three bf16 columns (below); the rest of
    // it stays zero for the life of the kernel
    for (int st = 0; st < LM_STAGES; ++st)
        for (int i = threadIdx.x; i < LM_KB_BYTES / 16; i += LM_THREADS)
            reinterpret_cast<uint4*>(b_s + st * LM_B_BYTES + 2 * LM_KB_BYTES)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (threadIdx.x == 0) {
        for (int s = 0; s < LM_STAGES; ++s) {
            mbar_init(&bars->bfull[s], LM_DEC_WARPS);
            mbar_init(&bars->bempty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bars->afull[a], 1);
            mbar_init(&bars->aempty[a], LM_EPI_WARPS);
        }
        mbar_fence_init();
    }
    if (warp == LM_MMA_WARP) {
        tmem_alloc(&bars->tmem_base, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, bars->tmem_base, 0);
    const bool mma_leader = warp == LM_MMA_WARP ? elect_one() : false;
    if (warp < 4) {             // the A columns that pick -h out of the third K block: (1, 1, 1, 0, ...) in bf16, every query lane
        uint32_t v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0u;
        v[0] = 0x3F803F80u;     // bf16 (1.0, 1.0)
        v[1] = 0x00003F80u;     // bf16 (1.0, 0.0)
        tmem_st_32x16(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + LM_TMEM_A + 64, v);
        tc_wait_st();
        tc_fence_before();
    }
    fence_proxy_async_smem();   // (the zeroed K blocks)

    uint32_t g = 0;                 // tiles this CTA has gone through (every role counts the same sequence)
    for (;;) {
        if (threadIdx.x == 0) bars->item = atomicAdd(item_counter, 1);
        __syncthreads();
        const int it = bars->item;
        if (it >= n_items) break;
        const LmItem item = items[it];
        const int lo = __ldg(loff + item.list) + item.t0 * LM_ROWS;      // first position of the slice
        const int T = item.tiles;
        // The item's query rows -> bf16 -> TENSOR MEMORY (columns [LM_TMEM_A, + 64) of the query's lane): the A operand of
        // every MMA of the item (no shared memory for it: the second set of candidate lists lives there instead).
        if (warp < 4) {
            const int r = warp * 32 + lane;
            const float4* src = nullptr;
            if (r < item.len) src = reinterpret_cast<const float4*>(q + static_cast<int64_t>(__ldg(pairs + item.start + r) / nprobe) * D128);
#pragma unroll
            for (int c = 0; c < 4; ++c) {                      // 32 dims = 16 words per store
                uint32_t v[16];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 x = src ? __ldg(src + c * 8 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                    const __nv_bfloat162 b0 = __floats2bfloat162_rn(x.x, x.y), b1 = __floats2bfloat162_rn(x.z, x.w);
                    v[2 * j] = *reinterpret_cast<const uint32_t*>(&b0);
                    v[2 * j + 1] = *reinterpret_cast<const uint32_t*>(&b1);
                }
                tmem_st_32x16(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + LM_TMEM_A + c * 16, v);
            }
            tc_wait_st();
            tc_fence_before();
        }
        for (int i = threadIdx.x; i < LM_Q * LM_SLOT; i += LM_THREADS) lst_s[i] = 0ull;
        __syncthreads();
        tc_fence_after();

        if (warp >= LM_EPI_WARPS && warp < LM_MMA_WARP) {
            // ------------------------------------------------------------ decoders: codes -> bf16 tile
            // Lane = sub-quantizer (32 per 64-dim K block).  One coalesced 128-byte load gives the warp the codes of 4
            // list positions (lcode_off); the lane looks its 4 codewords up in the table column of its own
            // sub-quantizer -- bank = lane, no conflicts for any codes -- and stores the 4-byte bf16 pairs: the 32 lanes
            // of a store cover one 128-byte swizzled row segment, one wavefront.  Warp dw takes K block dw & 1 and
            // the position groups (dw >> 1) + 4 j.
            const int dw = warp - LM_EPI_WARPS;                           // 0..7
            const int kb = dw & 1;
            const int rg0 = dw >> 1;
            const int dt = threadIdx.x - LM_EPI_WARPS * 32;               // 0..255
            const uint32_t tb = smem_u32(tab_s) + kb * (PQ_KSUB * 32 * 4) + lane * 4;
            const uint32_t dst_kb = smem_u32(b_s) + kb * LM_KB_BYTES + (lane & 3) * 4;
            const uint32_t chunk = static_cast<uint32_t>(lane >> 2);
            const uint8_t* tile0 = lcodes + static_cast<int64_t>(lo) * 64 + kb * (LIST_TILE * 32) + lane * 4;
            uint32_t nw[8];
            float nh = INFINITY;
            auto fetch = [&](int t) {
                const uint8_t* tp = tile0 + static_cast<int64_t>(t) * (LM_ROWS * 64);
#pragma unroll
                for (int j = 0; j < 8; ++j) nw[j] = __ldg(reinterpret_cast<const uint32_t*>(tp + (rg0 + 4 * j) * 128));
                if (dt < LM_ROWS) nh = __ldg(lh + lo + t * LM_ROWS + dt);     // (+inf for padding and halo rows)
            };
            // the loads of tile t + 1 are issued while tile t is decoded; one tile does not cover an HBM round trip, so
            // the lines of tile t + LM_PF are asked into L2 first
            auto prefetch = [&](int t) {
                if (dt < 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(lcodes + (static_cast<int64_t>(lo) + static_cast<int64_t>(t) * LM_ROWS) * 64 + dt * 128));
                else if (dt < 68) asm volatile("prefetch.global.L2 [%0];" ::"l"(lh + lo + t * LM_ROWS + (dt - 64) * 32));
            };
            for (int t = 1; t < LM_PF && t < T; ++t) prefetch(t);
            if (T > 0) fetch(0);
            for (int t = 0; t < T; ++t, ++g) {
                uint32_t w[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) w[j] = nw[j];
                const float hv = nh;
                if (t + LM_PF < T) prefetch(t + LM_PF);
                if (t + 1 < T) fetch(t + 1);
                const int s = g & 1;
                mbar_wait_parked(&bars->bempty[s], ((g >> 1) & 1) ^ 1);
                const uint32_t dst = dst_kb + s * LM_B_BYTES;
                uint32_t v[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {                              // word j: positions 4 (rg0 + 4 j) .. + 3
                    v[4 * j + 0] = lds32(tb + ((w[j] << 7) & 0x7F80u));
                    v[4 * j + 1] = lds32(tb + ((w[j] >> 1) & 0x7F80u));
                    v[4 * j + 2] = lds32(tb + ((w[j] >> 9) & 0x7F80u));
                    v[4 * j + 3] = lds32(tb + ((w[j] >> 17) & 0x7F80u));
                }
#pragma unroll
                for (int j = 0; j < 8; ++j)
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const uint32_t row = static_cast<uint32_t>(4 * (rg0 + 4 * j) + b);
                        asm volatile("st.shared.u32 [%0], %1;" ::"r"(dst + row * 128 + ((chunk ^ (row & 7u)) << 4)), "r"(v[4 * j + b]) : "memory");
                    }
                if (dt < LM_ROWS) {
                    // -h = hi + mid + lo in bf16 (24 significant bits): the MMA adds it to q . d through three columns of ones
                    uint32_t w0 = 0x0000FF80u, w1 = 0u;                            // h = +inf (padding, halo): -inf, 0, 0
                    if (hv < INFINITY) {
                        const float nhv = -hv;
                        const __nv_bfloat16 b_hi = __float2bfloat16_rn(nhv);
                        const float r1 = nhv - __bfloat162float(b_hi);
                        const __nv_bfloat16 b_mid = __float2bfloat16_rn(r1);
                        const __nv_bfloat16 b_lo = __float2bfloat16_rn(r1 - __bfloat162float(b_mid));
                        w0 = static_cast<uint32_t>(__bfloat16_as_ushort(b_hi)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b_mid)) << 16);
                        w1 = static_cast<uint32_t>(__bfloat16_as_ushort(b_lo));
                    }
                    sts128(smem_u32(b_s) + s * LM_B_BYTES + 2 * LM_KB_BYTES + dt * 128 + ((dt & 7) << 4), w0, w1, 0u, 0u);
                }
                fence_proxy_async_smem();          // this thread's tile bytes -> visible to the tensor core's (async) proxy
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&bars->bfull[s]);
                }
            }
        } else if (warp == LM_MMA_WARP) {
            // ------------------------------------------------------------ MMA issuer
            const uint32_t idesc = umma_idesc_f16(1u, 128u, static_cast<uint32_t>(LM_ROWS));
            const uint32_t a_tmem = tmem_base + LM_TMEM_A;          // 16 bf16 = 8 columns per K step
            const uint64_t bdesc0 = umma_desc_sw128(smem_u32(b_s));
            for (int t = 0; t < T; ++t, ++g) {
                const int s = g & 1;
                const uint32_t ph = (g >> 1) & 1;
                mbar_wait_parked(&bars->aempty[s], ph ^ 1);
                mbar_wait_parked(&bars->bfull[s], ph);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + s * LM_ROWS;
                const uint64_t b_kb0 = bdesc0 + static_cast<uint64_t>((s * LM_B_BYTES) >> 4);
                const uint64_t b_kb1 = b_kb0 + static_cast<uint64_t>(LM_KB_BYTES >> 4);
                if (mma_leader) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) lm_mma_ts(d_tmem, a_tmem + 8 * j, b_kb0 + 2 * j, idesc, j != 0 ? 1u : 0u);
#pragma unroll
                    for (int j = 0; j < 4; ++j) lm_mma_ts(d_tmem, a_tmem + 32 + 8 * j, b_kb1 + 2 * j, idesc, 1u);
                    lm_mma_ts(d_tmem, a_tmem + 64, b_kb1 + static_cast<uint64_t>(LM_KB_BYTES >> 4), idesc, 1u);       // ... - h
                    tc_commit(&bars->bempty[s]);
                    tc_commit(&bars->afull[s]);
                }
                __syncwarp();
            }
        } else {
            // ------------------------------------------------------------ epilogue: one query per thread
            // Warp e reads TMEM lane quadrant e & 3 (32 queries) and the 64 accumulator columns of half e >> 2 of every tile;
            // each half keeps its own sorted list and threshold per query (two TMEM round trips per tile and warp instead
            // of four: the epilogue, not the tensor pipe, sets the tile time).
            const int qd = warp & 3, half = warp >> 2;
            const int ql = qd * 32 + lane;
            const bool act = ql < item.len;
            const int pid = act ? __ldg(pairs + item.start + ql) : 0;
            float thr = INFINITY;                                       // padding lanes never fire
            if (act) {
                thr = -INFINITY;
                if (dkA) {
                    const int qrow = pid / nprobe;
                    // a row whose bf16 score is <= thr has an exact distance >= Dk: it cannot enter the top k
                    thr = 0.5f * (__ldg(gdist + pid) - __ldg(dkA + qrow)) - __ldg(qE + qrow);
                }
            }
            uint64_t* wl = lst_s + (half * LM_Q + qd * 32) * LM_KP;
            const uint32_t tlane = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + half * (LM_ROWS / 2);
            for (int t = 0; t < T; ++t, ++g) {
                const int acc = g & 1;
                mbar_wait_parked(&bars->afull[acc], (g >> 1) & 1);
                tc_fence_after();
                const uint32_t pos0 = static_cast<uint32_t>(lo + t * LM_ROWS + half * (LM_ROWS / 2));
#pragma unroll 1
                for (int c = 0; c < LM_ROWS / 64; ++c) {
                    uint32_t v[32];
                    tmem_ld_32x32(tlane + acc * LM_ROWS + c * 32, v);
                    tc_wait_ld();
                    float sc[32];                  // q . d - h: the accumulator already holds the score
#pragma unroll
                    for (int j = 0; j < 32; ++j) sc[j] = __uint_as_float(v[j]);
                    // one vote per chunk on the hot path (vote -> branch latency was half of the epilogue's time with one per
                    // 8 columns); the per-group votes run only inside the rare branch
                    float mg[4];
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) {
                        mg[g8] = fmaxf(fmaxf(sc[8 * g8], sc[8 * g8 + 1]), sc[8 * g8 + 2]);
                        mg[g8] = fmaxf(fmaxf(mg[g8], sc[8 * g8 + 3]), sc[8 * g8 + 4]);
                        mg[g8] = fmaxf(fmaxf(mg[g8], sc[8 * g8 + 5]), fmaxf(sc[8 * g8 + 6], sc[8 * g8 + 7]));
                    }
                    if (!__any_sync(0xffffffffu, fmaxf(fmaxf(mg[0], mg[1]), fmaxf(mg[2], mg[3])) > thr)) continue;
#pragma unroll
                    for (int g8 = 0; g8 < 4; ++g8) {
                        if (__any_sync(0xffffffffu, mg[g8] > thr)) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                const float sj = sc[8 * g8 + j];
                                unsigned mask = __ballot_sync(0xffffffffu, sj > thr);
                                while (mask) {
                                    // warp-cooperative insert into the sorted list of the query on lane qi
                                    const int qi = __ffs(mask) - 1;
                                    mask &= mask - 1;
                                    const float sv = __shfl_sync(0xffffffffu, sj, qi);
                                    const uint64_t key = (static_cast<uint64_t>(static_cast<uint32_t>(f2ord(sv)) ^ 0x80000000u) << 32) |
                                                         static_cast<uint64_t>(pos0 + c * 32 + 8 * g8 + j);
                                    uint64_t* lq = wl + qi * LM_KP;
                                    const uint64_t e = lq[lane];
                                    const int p = __popc(__ballot_sync(0xffffffffu, e > key));
                                    const uint64_t up = __shfl_up_sync(0xffffffffu, e, 1);
                                    const uint64_t ne = lane < p ? e : (lane == p ? key : up);
                                    lq[lane] = ne;
                                    const uint64_t last = __shfl_sync(0xffffffffu, ne, LM_KP - 1);
                                    if (lane == qi && last != 0ull) thr = fmaxf(thr, key_score(last));
                                    __syncwarp();
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&bars->aempty[acc]);
            }
        }
        __syncthreads();            // every accumulator of the item was consumed, every candidate list is final
        if (warp < LM_EPI_WARPS) {  // the item's candidate lists -> cand[pair][slice][group][32]
            const int qd = warp & 3, half = warp >> 2;
            const int ql = qd * 32 + lane;
            // (the lane's (pair, slice) row of cand, formed once so that the copy loop is the same as without slices)
            const int row = ql < item.len ? __ldg(pairs + item.start + ql) * S + item.slice : 0;
            const uint64_t* wl = lst_s + (half * LM_Q + qd * 32) * LM_KP;
            for (int qi = 0; qi < 32; ++qi) {
                const int cr = __shfl_sync(0xffffffffu, row, qi);
                if (qd * 32 + qi < item.len) cand[static_cast<int64_t>(cr) * LM_SLOT + half * LM_KP + lane] = wl[qi * LM_KP + lane];
            }
        }
    }
    __syncthreads();
    if (warp == LM_MMA_WARP) tmem_dealloc(tmem_base, 512);
}

// exact ADC distance of one list position for residual r = q - c_l, with ivfpq_scan_kernel's arithmetic: per
// sub-quantizer fma(t1, t1, t0 * t0), added sub-quantizer by sub-quantizer in ascending order
__device__ __forceinline__ float lm_exact_adc(const float* __restrict__ qs, const float* __restrict__ c, const float* __restrict__ pq,
                                              const uint8_t* __restrict__ lcodes, uint32_t pos) {
    // the position's 64 codes: byte (pos & 3) of the 32 words of its two 128-byte lines (lcode_off), read as 16-byte loads
    const uint4* lp = reinterpret_cast<const uint4*>(lcodes + static_cast<int64_t>(pos >> 7) * (LIST_TILE * 64) + ((pos & 127u) >> 2) * 128);
    const int sh = static_cast<int>(pos & 3u) * 8;
    float d = 0.f;
#pragma unroll
    for (int kb = 0; kb < 2; ++kb) {
#pragma unroll 4
        for (int j = 0; j < 8; ++j) {
            const uint4 cw = __ldg(lp + kb * (LIST_TILE * 32 / 16) + j);
            const uint32_t wds[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int sub = kb * 32 + 4 * j + b;
                const uint32_t code = (wds[b] >> sh) & 255u;
                const float2 p = __ldg(reinterpret_cast<const float2*>(pq + (static_cast<int64_t>(sub) * PQ_KSUB + code) * 2));
                const float2 cc = __ldg(reinterpret_cast<const float2*>(c + 2 * sub));
                const float r0 = qs[2 * sub] - cc.x, r1 = qs[2 * sub + 1] - cc.y;
                const float t0 = r0 - p.x, t1 = r1 - p.y;
                d += fmaf(t1, t1, fmaf(t0, t0, 0.f));
            }
        }
    }
    return d;
}

// one warp per query row: Dk = the k-th smallest exact distance among the candidates of the lists scanned so far
// (probe ranks [0, pend), pend <= LM_WAVE1_END; +inf if they gave fewer than k) -- the next wave's threshold.
// Dynamic shared memory: lm_bound_smem(S).  (S is a template parameter here and in the merge: at S = 1 their index
// arithmetic compiles to the same shifts as before slices existed.)
__host__ __device__ constexpr int lm_bound_smem(int S) { return 8 * (D128 + LM_WAVE1_END * S * LM_SLOT) * 4; }
template <int S>
__global__ void ivfpq_lm_bound_kernel(const float* __restrict__ q, int64_t nq, int nprobe, int pend, int k,
                                      const uint64_t* __restrict__ cand, const int32_t* __restrict__ probes,
                                      const float* __restrict__ gdist, const float* __restrict__ qE,
                                      const float* __restrict__ coarse, const float* __restrict__ pq,
                                      const uint8_t* __restrict__ lcodes, float* __restrict__ dkA) {
    extern __shared__ float bsm[];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float* qs = bsm + w * D128;                                       // [8 warps][128]
    float* ds = bsm + 8 * D128 + w * (LM_WAVE1_END * S * LM_SLOT);    // [8 warps][LM_WAVE1_END * S * LM_SLOT]
    const int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (i >= nq) return;
    reinterpret_cast<float4*>(qs)[lane] = reinterpret_cast<const float4*>(q + i * D128)[lane];
    __syncwarp();
    const float dk_prev = dkA[i];          // the previous wave's bound (3.4e38 before the first): what cannot beat it is not re-scored
    const float E = qE[i];
    constexpr int per_probe = S * LM_GROUPS;   // lists of one (query row, probe rank): slice p / LM_GROUPS % S, epilogue group p % LM_GROUPS
    for (int p = 0; p < pend * per_probe; ++p) {
        const uint64_t key = cand[(i * nprobe) * S * LM_SLOT + p * LM_KP + lane];
        const int l = probes[i * nprobe + p / per_probe];
        float d = INFINITY;
        // exact distance >= |q - c|^2 - 2 (bf16 score + E)
        if (key != 0ull && l >= 0 && gdist[i * nprobe + p / per_probe] - 2.f * (key_score(key) + E) <= dk_prev)
            d = lm_exact_adc(qs, coarse + static_cast<int64_t>(l) * D128, pq, lcodes, static_cast<uint32_t>(key));
        ds[p * LM_KP + lane] = d;
    }
    __syncwarp();
    // compact the re-scored distances (most slots were skipped), then rank them: the one of rank k - 1 is the bound
    int m = 0;
    for (int p = 0; p < pend * per_probe; ++p) {
        const float d = ds[p * LM_KP + lane];
        const bool fin = d < INFINITY;
        const unsigned mask = __ballot_sync(0xffffffffu, fin);
        __syncwarp();
        if (fin) ds[m + __popc(mask & ((1u << lane) - 1u))] = d;       // (target index <= source index: never an unread entry)
        m += __popc(mask);
        __syncwarp();
    }
    if (m < k) {
        if (lane == 0) dkA[i] = INFINITY;
        return;
    }
    for (int r = lane; r < m; r += 32) {
        const float d = ds[r];
        int rank = 0;
        for (int o = 0; o < m; ++o) {
            const float od = ds[o];
            rank += (od < d || (od == d && o < r)) ? 1 : 0;
        }
        if (rank == k - 1) dkA[i] = d;
    }
}

// one block per query row: exact re-rank of the survivors of all probed lists, top k, proof.  At S = 1 every candidate
// fits the key buffer; at S > 1 a row with more than LM_MERGE_KEYS survivors goes to the LUT kernel like an unproven one.
template <int S>
__global__ void __launch_bounds__(128)
ivfpq_lm_merge_kernel(const float* __restrict__ q, int64_t q0, int nprobe, int k, const uint64_t* __restrict__ cand,
                      const int32_t* __restrict__ probes, const float* __restrict__ gdist, const float* __restrict__ qE,
                      const float* __restrict__ dkA, const float* __restrict__ coarse, const float* __restrict__ pq,
                      const uint8_t* __restrict__ lcodes,
                      const int32_t* __restrict__ lids, int64_t label_offset, float* __restrict__ D, int64_t* __restrict__ I,
                      int32_t* __restrict__ redo_rows, int32_t* __restrict__ redo_count) {
    __shared__ float qs[D128];
    __shared__ uint64_t keys[LM_MERGE_KEYS];
    __shared__ int cnt_s, bound_s;
    const int64_t i = blockIdx.x;              // row inside the launch group
    const int tid = threadIdx.x;
    if (tid < 32) reinterpret_cast<float4*>(qs)[tid] = reinterpret_cast<const float4*>(q + i * D128)[tid];
    if (tid == 0) { cnt_s = 0; bound_s = INT_MAX; }
    __syncthreads();
    const float E = qE[i], dk = dkA[i];
    constexpr int per_probe = S * LM_SLOT;
    const int total = nprobe * per_probe;
    // 1. gather: compact (probe rank, list position) of every survivor; lower bound on the distance of what the
    //    full lists dropped: g - 2 (score of the list's last entry + E)
    for (int e = tid; e < total; e += blockDim.x) {
        const uint64_t key = cand[i * total + e];
        if (key != 0ull) {
            const int p = e / per_probe;
            // (a survivor whose distance cannot be below the last bound -- an upper bound of the k-th -- is not re-scored)
            if (gdist[i * nprobe + p] - 2.f * (key_score(key) + E) <= dk) {
                const int slot = atomicAdd(&cnt_s, 1);
                if (slot < LM_MERGE_KEYS) keys[slot] = (static_cast<uint64_t>(p) << 32) | static_cast<uint32_t>(key);
            }
            if ((e & (LM_KP - 1)) == LM_KP - 1)
                atomicMin(&bound_s, f2ord(gdist[i * nprobe + p] - 2.f * (key_score(key) + E)));
        }
    }
    __syncthreads();
    const int n = cnt_s;
    if (n > LM_MERGE_KEYS) {
        if (tid == 0) redo_rows[atomicAdd(redo_count, 1)] = static_cast<int32_t>(q0 + i);
        return;
    }
    int P = 32;
    while (P < n || P < k) P <<= 1;
    // 2. exact distances (the LUT kernel's arithmetic), key = (distance bits, row id): ascending order = faiss order,
    //    ties to the lower id
    for (int c = tid; c < P; c += blockDim.x) {
        uint64_t out = ~0ull;
        if (c < n) {
            const uint64_t pk = keys[c];
            const int p = static_cast<int>(pk >> 32);
            const uint32_t pos = static_cast<uint32_t>(pk);
            const int l = probes[i * nprobe + p];
            const float d = lm_exact_adc(qs, coarse + static_cast<int64_t>(l) * D128, pq, lcodes, pos);
            out = dist_key(d, static_cast<uint32_t>(lids[pos]));
        }
        __syncwarp();
        keys[c] = out;         // (slot c was read by this thread only)
    }
    __syncthreads();
    block_sort_u64<true>(keys, P);
    // 3. proof: nothing the full lists dropped can be closer than the k-th survivor
    const uint64_t kth = keys[k - 1];
    const float Dk = kth != ~0ull ? key_dist(kth) : INFINITY;
    const bool proven = bound_s == INT_MAX || Dk < ord2f(bound_s);
    if (!proven) {
        if (tid == 0) redo_rows[atomicAdd(redo_count, 1)] = static_cast<int32_t>(q0 + i);
        return;
    }
    store_topk(keys, k, label_offset, D + i * k, I + i * k);
}

// ------------------------------------------------------------------------------------------ host
constexpr int LM_MAX_S = (LM_MAX_K + LM_SLICE_K - 1) / LM_SLICE_K;
using LmBoundFn = decltype(&ivfpq_lm_bound_kernel<1>);
using LmMergeFn = decltype(&ivfpq_lm_merge_kernel<1>);
static const LmBoundFn lm_bound_fns[] = {ivfpq_lm_bound_kernel<1>, ivfpq_lm_bound_kernel<2>, ivfpq_lm_bound_kernel<3>,
                                         ivfpq_lm_bound_kernel<4>, ivfpq_lm_bound_kernel<5>, ivfpq_lm_bound_kernel<6>};
static const LmMergeFn lm_merge_fns[] = {ivfpq_lm_merge_kernel<1>, ivfpq_lm_merge_kernel<2>, ivfpq_lm_merge_kernel<3>,
                                         ivfpq_lm_merge_kernel<4>, ivfpq_lm_merge_kernel<5>, ivfpq_lm_merge_kernel<6>};
static_assert(sizeof(lm_bound_fns) / sizeof(lm_bound_fns[0]) == LM_MAX_S && sizeof(lm_merge_fns) / sizeof(lm_merge_fns[0]) == LM_MAX_S,
              "one bound and one merge kernel per slice count");

static int lm_reserve(nafp_index* idx, int64_t nc, int nprobe, int S) {
    LmState* L = idx->ivf->lm;
    const int64_t np = nc * nprobe;
    if (L->cap_q < nc || L->cap_pairs < np || L->cap_cand < np * S) {
        void* old[] = {L->probes, L->gdist, L->qE, L->dkA, L->pairs, L->cand};
        for (void* b : old) if (b) cudaFree(b);
        L->probes = nullptr; L->gdist = nullptr; L->qE = nullptr; L->dkA = nullptr; L->pairs = nullptr; L->cand = nullptr;
        const int64_t cq = std::max(nc, L->cap_q), cp = std::max(np, L->cap_pairs), cc = std::max(np * S, L->cap_cand);
        L->cap_q = 0; L->cap_pairs = 0; L->cap_cand = 0;
        NAFP_CUDA(cudaMalloc(&L->probes, static_cast<size_t>(cp) * sizeof(int32_t)));
        NAFP_CUDA(cudaMalloc(&L->gdist, static_cast<size_t>(cp) * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&L->pairs, static_cast<size_t>(cp) * sizeof(int32_t)));
        NAFP_CUDA(cudaMalloc(&L->cand, static_cast<size_t>(cc) * LM_SLOT * sizeof(uint64_t)));
        NAFP_CUDA(cudaMalloc(&L->qE, static_cast<size_t>(cq) * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&L->dkA, static_cast<size_t>(cq) * sizeof(float)));
        L->cap_q = cq;
        L->cap_pairs = cp;
        L->cap_cand = cc;
    }
    return NAFP_OK;
}

int ivfpq_search_lm(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    IvfPq* s = idx->ivf;
    nafp_ctx* ctx = idx->ctx;
    const int nprobe = idx->nprobe < s->nlist ? idx->nprobe : s->nlist;
    const int nlist = s->nlist;
    const int64_t n_search = (idx->search_rows >= 0 && idx->search_rows < idx->n) ? idx->search_rows : idx->n;
    const int S = lm_slices(k);
    const int64_t chunk_q = LM_CHUNK_Q / S;
    NAFP_TRY(lm_prepare(idx, n_search));
    LmState* L = s->lm;
    NAFP_TRY(ivfpq_reserve_redo(idx, nq));
    int32_t* redo_count = s->redo_rows + s->redo_cap;
    NAFP_CUDA(cudaMemsetAsync(redo_count, 0, sizeof(int32_t), ctx->stream));
    NAFP_CUDA(cudaFuncSetAttribute(ivfpq_lm_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LM_SMEM));
    const LmBoundFn bound_kernel = lm_bound_fns[S - 1];
    const LmMergeFn merge_kernel = lm_merge_fns[S - 1];
    NAFP_CUDA(cudaFuncSetAttribute(bound_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lm_bound_smem(S)));
    int32_t* hist = L->hist;                                        // [LM_WAVES nlist]
    int32_t* cursor = L->hist + LM_WAVES * IVF_MAX_NLIST;           // [LM_WAVES nlist]
    int32_t* counters = L->hist + 2 * LM_WAVES * IVF_MAX_NLIST;     // [LM_WAVES]
    const int nb = LM_WAVES * nlist;
    std::vector<int32_t> h(nb), cur(nb);
    std::vector<LmItem> items;
    for (int64_t q0 = 0; q0 < nq; q0 += chunk_q) {
        const int64_t nc = nq - q0 < chunk_q ? nq - q0 : chunk_q;
        const int64_t np = nc * nprobe;
        const float* qp = q_dev + q0 * D128;
        NAFP_TRY(lm_reserve(idx, nc, nprobe, S));
        NAFP_TRY(coarse_probe(ctx, qp, nc, s->coarse, nlist, nprobe, L->probes, L->gdist, L->qE, L->dmax2));
        NAFP_CUDA(cudaMemsetAsync(hist, 0, nb * sizeof(int32_t), ctx->stream));
        lm_hist_kernel<<<static_cast<unsigned>(std::min<int64_t>((np + 255) / 256, 4 * ctx->sm_count)), 256, 0, ctx->stream>>>(
            L->probes, np, nprobe, nlist, hist);
        NAFP_CUDA(cudaMemcpyAsync(h.data(), hist, nb * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        // work items: (slice of a list, <= 128 of the query rows that probe it in this wave), longest first; slice s of a
        // list of T tiles covers tiles [s T / S, (s + 1) T / S)
        items.clear();
        int n_items[LM_WAVES], first_item[LM_WAVES];
        int32_t run = 0;
        for (int wv = 0; wv < LM_WAVES; ++wv) {
            const size_t first = items.size();
            for (int l = 0; l < nlist; ++l) {
                const int b = wv * nlist + l;
                cur[b] = run;
                const int tiles = (s->h_lend[l] - s->h_loff[l] + LM_ROWS - 1) / LM_ROWS;
                for (int sl = 0; sl < S; ++sl) {
                    const int t0 = static_cast<int>(static_cast<int64_t>(tiles) * sl / S);
                    const int t1 = static_cast<int>(static_cast<int64_t>(tiles) * (sl + 1) / S);
                    if (t1 > t0)
                        for (int o = 0; o < h[b]; o += LM_Q) items.push_back({l, run + o, std::min(LM_Q, h[b] - o), t1 - t0, t0, sl});
                }
                run += h[b];
            }
            std::stable_sort(items.begin() + first, items.end(), [](const LmItem& a, const LmItem& b) { return a.tiles > b.tiles; });
            first_item[wv] = static_cast<int>(first);
            n_items[wv] = static_cast<int>(items.size() - first);
        }
        if (L->items_cap < static_cast<int64_t>(items.size())) {
            if (L->items) cudaFree(L->items);
            L->items = nullptr; L->items_cap = 0;
            const int64_t cap = std::max<int64_t>(static_cast<int64_t>(items.size()) * 2, 1024);
            NAFP_CUDA(cudaMalloc(&L->items, static_cast<size_t>(cap) * sizeof(LmItem)));
            L->items_cap = cap;
        }
        if (!items.empty())
            NAFP_CUDA(cudaMemcpyAsync(L->items, items.data(), items.size() * sizeof(LmItem), cudaMemcpyHostToDevice, ctx->stream));
        NAFP_CUDA(cudaMemcpyAsync(cursor, cur.data(), nb * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
        NAFP_CUDA(cudaMemsetAsync(counters, 0, LM_WAVES * sizeof(int32_t), ctx->stream));
        lm_scatter_kernel<<<static_cast<unsigned>((np + 255) / 256), 256, 0, ctx->stream>>>(L->probes, np, nprobe, nlist, cursor, L->pairs);
        NAFP_CUDA(cudaMemsetAsync(L->cand, 0, static_cast<size_t>(np) * S * LM_SLOT * sizeof(uint64_t), ctx->stream));
        NAFP_CUDA(cudaMemsetAsync(L->dkA, 0x7f, static_cast<size_t>(nc) * sizeof(float), ctx->stream));     // 0x7f7f7f7f = 3.4e38: "no bound"
        ctx->launches += 2;
        for (int wv = 0; wv < LM_WAVES; ++wv) {
            if (n_items[wv] > 0) {
                const int grid = std::min(n_items[wv], ctx->sm_count);
                ivfpq_lm_scan_kernel<<<grid, LM_THREADS, LM_SMEM, ctx->stream>>>(
                    qp, nprobe, S, L->items + first_item[wv], n_items[wv], counters + wv, L->pairs, L->tab, s->lcodes, L->lh, s->loff,
                    L->gdist, wv ? L->dkA : nullptr, L->qE, L->cand);
                ctx->launches++;
                for (int e = 0; e < n_items[wv]; ++e) L->tiles_run += items[first_item[wv] + e].tiles;
                L->items_run += n_items[wv];
            }
            bool later = false;
            for (int x = wv + 1; x < LM_WAVES; ++x) later = later || n_items[x] > 0;
            if (later) {               // the bound the later waves' thresholds are built from
                const int pend = std::min(wv == 0 ? 1 : LM_WAVE1_END, nprobe);
                bound_kernel<<<static_cast<unsigned>((nc + 7) / 8), 256, lm_bound_smem(S), ctx->stream>>>(
                    qp, nc, nprobe, pend, k, L->cand, L->probes, L->gdist, L->qE, s->coarse, s->pq, s->lcodes, L->dkA);
                ctx->launches++;
            }
        }
        merge_kernel<<<static_cast<unsigned>(nc), 128, 0, ctx->stream>>>(qp, q0, nprobe, k, L->cand, L->probes, L->gdist, L->qE, L->dkA,
                                                                                 s->coarse, s->pq, s->lcodes, s->lids, idx->label_offset,
                                                                                 D_dev + q0 * k, I_dev + q0 * k, s->redo_rows, redo_count);
        ctx->launches++;
        NAFP_CUDA(cudaGetLastError());
    }
    int32_t n_redo = 0;
    NAFP_CUDA(cudaMemcpyAsync(&n_redo, redo_count, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n_redo > 0) NAFP_TRY(ivfpq_redo_rows(idx, q_dev, n_redo, k, D_dev, I_dev));      // (counted in IvfPq::lut_rows)
    return NAFP_OK;
}

}  // namespace nafp
