// Exact flat (squared-L2) index on B200: bf16 tensor-core scan with shared-threshold candidate
// filtering, exact fp32 re-rank with a provable error bound, exact fp32 fallback scan.
//
// Replaces faiss.IndexFlatL2 as used by the reference (eval/utils/get_index_faiss.py:58,
// eval/eval_faiss.py:147-148,211).  Ranking score  s(q,x) = q.x - 0.5|x|^2  (argmax s == argmin
// |q-x|^2), distance reported as |q|^2 - 2 s.
//
// One scan pass handles up to 512 query rows against the whole database:
//   flat_prep_kernel    fp32 queries -> bf16 A-operand tile, |q|^2, pass state reset
//   flat_scan_kernel    persistent, one CTA per SM, launched as clusters of two CTAs: the CTA of cluster rank r scores
//                       pass rows [r h, r h + h), h = 128 or 256.  256-row DB tiles are handed out to the pairs by a
//                       global counter; rank 0 loads each tile ONCE and TMA multicast writes it into both CTAs' rings
//                       (half the HBM bytes per score of one CTA per tile).  Per CTA:
//                       TMA (SWIZZLE_128B) -> smem ring of K blocks -> tcgen05.mma (M = 128
//                       queries, N = 256 DB rows, K = 128, bf16, fp32 accumulators double-buffered in
//                       TMEM) -> epilogue threads own one query each: a 3-input max over the tile's
//                       columns and ONE compare against  T + min_tile 0.5|x|^2 ; a 32-column chunk in
//                       which a lane fires gets the exact  q.x - 0.5|x|^2 > T  test in straight-line
//                       code and its hits' row ids join the CTA's pool.
//                       T is a per-query threshold that all CTAs share through L2 (the kg-th largest
//                       of the running maxima per (pair, accumulator column half) -- disjoint row sets, so a
//                       valid lower bound on the kg-th best score -- maintained by one reducer warp per CTA,
//                       lock-free); every pair first scans eight "warm" tiles max-only (re-visited at the end)
//                       so that the thresholds are tight before the first candidate is appended.
//   flat_select_kernel  per query: gather survivors, exact fp32 re-score, sort, and PROVE the
//                       top-k: every dropped row has bf16 score <= T, hence exact score <= T + eps
//                       with eps = (2u+u^2)|q|max|x| (u = 2^-8); if the k-th exact score is not
//                       above that, the query is handed to the fallback.
//   flat_brute_*        exact fp32 CUDA-core scan for flagged queries / tiny databases.
#include <cfloat>
#include <climits>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

#include "index.h"
#include "ptx.cuh"
#include "topk.cuh"

namespace nafp {

// ------------------------------------------------------------------------------------------
// small kernels: row conversion at add(), query preparation
// ------------------------------------------------------------------------------------------
__global__ void flat_convert_rows_kernel(const float* __restrict__ x32, __nv_bfloat16* __restrict__ x16,
                                         float* __restrict__ hn, int32_t* __restrict__ maxn2, int64_t row0,
                                         int64_t n) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
    float mx = 0.f;
    for (int64_t r = row0 + warp; r < row0 + n; r += nwarps) {
        const float4 v = reinterpret_cast<const float4*>(x32 + r * D128)[lane];
        __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
        __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
        uint2 packed;
        packed.x = *reinterpret_cast<uint32_t*>(&a);
        packed.y = *reinterpret_cast<uint32_t*>(&b);
        reinterpret_cast<uint2*>(x16 + r * D128)[lane] = packed;
        float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) hn[r] = 0.5f * ss;
        mx = fmaxf(mx, ss);
    }
    if (lane == 0 && mx > 0.f) atomicMax(maxn2, __float_as_int(mx));
}

__global__ void flat_fill_kernel(float* hn, int64_t from, int64_t to, float v) {
    int64_t i = from + static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < to) hn[i] = v;
}

// one warp per query row of the pass (rows >= nq are zero padding).  The pass takes rows
// p0 .. p0+nq-1 of q_all, or -- for a retry pass -- the rows listed in src_list[src_off ..].
__global__ void flat_prep_kernel(const float* __restrict__ q_all, const int32_t* __restrict__ src_list, int src_off,
                                 int64_t p0, int nq, int nq_pad, int grid_scan,
                                 __nv_bfloat16* __restrict__ qbf, float* __restrict__ q32,
                                 float* __restrict__ qn2, int32_t* __restrict__ Mx, int32_t* __restrict__ Tg,
                                 int32_t* __restrict__ flags, int64_t* __restrict__ gidx, int32_t* __restrict__ tile_counter) {
    const int lane = threadIdx.x & 31;
    const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (blockIdx.x == 0 && threadIdx.x == 0) *tile_counter = 0;      // the scan's dynamic tile scheduler
    if (row >= nq_pad) return;
    int64_t g = -1;
    if (row < nq) g = src_list ? static_cast<int64_t>(src_list[src_off + row]) : p0 + row;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g >= 0) v = reinterpret_cast<const float4*>(q_all + g * D128)[lane];
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y);
    __nv_bfloat162 b = __floats2bfloat162_rn(v.z, v.w);
    uint2 packed;
    packed.x = *reinterpret_cast<uint32_t*>(&a);
    packed.y = *reinterpret_cast<uint32_t*>(&b);
    reinterpret_cast<uint2*>(qbf + row * D128)[lane] = packed;
    reinterpret_cast<float4*>(q32 + row * D128)[lane] = v;
    float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (lane == 0) {
        qn2[row] = ss;
        Tg[row] = INT_MIN;
        flags[row] = 0;
        gidx[row] = g;
    }
    for (int c = lane; c < grid_scan; c += 32) Mx[row * grid_scan + c] = INT_MIN;
}

// ------------------------------------------------------------------------------------------
// the scan
// ------------------------------------------------------------------------------------------
constexpr int RING_SLOTS = 4;                           // K-block slots of the DB ring
constexpr int EPI_WARPS = 16;
constexpr int SCAN_THREADS = (3 + EPI_WARPS) * 32;   // warps 0..15 epilogue, 16 reducer, 17 TMA, 18 MMA (+TMEM alloc)
constexpr int TMA_WARP = EPI_WARPS + 1, MMA_WARP = EPI_WARPS + 2;   // (warp EPI_WARPS is the reducer.)  The SM's warp arbiter
                                                     // favours high warp ids: the MMA issuer must never wait for a slot
constexpr int EPI_PARTS = EPI_WARPS / 4;          // the 4 warps of a TMEM lane quadrant split the tile's 256 DB rows
constexpr int PART_COLS = SCAN_TILE / EPI_PARTS;  // 64 DB rows (accumulator columns) per warp per unit
constexpr int SLOT_BYTES = SCAN_TILE * 128;                // 32 KB: one 64-column K block of a 256-row tile
constexpr int BOX_BYTES = TILE_ROWS * 128;                 // 16 KB per TMA box (128 rows)
constexpr int Q_KB_BYTES = NQ_CTA * 128;                   // 32 KB: one K block of the query operand
constexpr int Q_BYTES_MAX = 2 * Q_KB_BYTES;                // 64 KB
constexpr int H_RING = 4;                               // tiles of 0.5|x|^2 kept in shared memory
constexpr int WARM_TILES = 8;                           // tiles every pair scans max-only before it uses thresholds
constexpr int SCAN_SMEM = Q_BYTES_MAX + RING_SLOTS * SLOT_BYTES + H_RING * SCAN_TILE * 4 + 3 * NQ_CTA * 4 + 256 + 1024;
constexpr uint16_t PAIR_MASK = 0b11, RANK0_MASK = 0b01;       // multicast targets: both CTAs of the pair / rank 0
constexpr int NEG_INF_ORD = static_cast<int>(0x807FFFFFu);  // f2ord(-inf)
static_assert(PART_COLS == 64, "epilogue reads two 32-column chunks per unit");

struct ScanBars {
    uint64_t full[RING_SLOTS];
    uint64_t empty[RING_SLOTS];    // only rank 0's is used: both CTAs' MMA warps release a slot there
    uint64_t tfull[2];
    uint64_t tempty[2];
    uint64_t qfull;
    uint32_t tmem_base;
    int done;          // epilogue warps that finished
    int tile_of[8];    // work item i (mod 8) -> DB tile, -1 = no more work (written by the TMA producer)
};

__device__ __forceinline__ void smem_red_max(int* p, int v) {
    asm volatile("red.shared.max.s32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ int smem_atom_inc(int* p) {
    int old;
    asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(p)) : "memory");
    return old;
}
__device__ __forceinline__ int smem_atom_add(int* p, int v) {
    int old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(p)), "r"(v) : "memory");
    return old;
}
__device__ __forceinline__ int smem_ld_volatile(const int* p) {
    int v;
    asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
// lane 0 arrives; predicated instead of branched so the warp never diverges on the hot path
__device__ __forceinline__ void mbar_arrive_lane0(uint64_t* bar, int lane) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.eq.s32 p, %1, 0;\n\t@p mbarrier.arrive.shared::cta.b64 _, [%0];\n\t}" ::"r"(smem_u32(bar)),
        "r"(lane)
        : "memory");
}
// A chunk (32 accumulator columns = 32 DB rows) in which some lane's maximum passed the prefilter: every lane
// tests its 32 scores exactly -- s = v - 0.5|x|^2 > T -- in straight-line code (bit mask of the hits, exact chunk
// maximum); only then the lanes with hits diverge: one shared-memory add reserves their pool slots, the pool takes
// the row ids (flat_select re-scores every survivor in fp32, the scan's score is not needed again), the running
// maximum of the query takes the chunk maximum.  The first version inlined 32 predicated append bodies (14 KB of
// branchy code); this one is ~150 instructions.  nvalid < 32 only in a tile that holds halo / padding rows.
template <bool EDGE>
__device__ __forceinline__ void scan_chunk_hits(const uint32_t (&v)[32], const float* __restrict__ hc, float t_exact, int nvalid,
                                                uint32_t rbase, int* cnt_q, int* lmax_q, uint64_t* pool_q) {
    uint32_t m = 0;
    float best = -INFINITY;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        if (!EDGE || j < nvalid) {
            const float sj = __uint_as_float(v[j]) - hc[j];
            m |= (sj > t_exact) ? (1u << j) : 0u;
            best = fmaxf(best, sj);
        }
    }
    if (m) {
        smem_red_max(lmax_q, f2ord(best));
        int pos = smem_atom_add(cnt_q, __popc(m));
        while (m) {
            const int j = __ffs(m) - 1;
            m &= m - 1;
            if (pos < POOL_CAP) pool_q[pos] = rbase + j;
            ++pos;
        }
    }
}

// Orientation: the MMA's M side (TMEM lanes) are the QUERIES, its N side (accumulator columns) the
// DB rows of the tile.  An epilogue thread therefore owns one query per 128-query half: its
// threshold is ONE register, and the hot loop is a 3-input max over the columns followed by a single
// compare -- no per-score add, no threshold traffic.  -0.5|x|^2 enters the prefilter through the
// minimum over the warp's 64 rows and is applied exactly only to the few scores that pass it.
__global__ void __launch_bounds__(SCAN_THREADS, 1)
flat_scan_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_db,
                 const float* __restrict__ hn, int32_t* __restrict__ tile_counter, int64_t n_search, int n_tiles, int nq,
                 int n_half, int kg, int32_t* __restrict__ Mx, int32_t* __restrict__ Tg, uint64_t* __restrict__ pool,
                 int32_t* __restrict__ cnt, int32_t* __restrict__ flags) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* q_s = smem;                                   // [kb 2][256 query rows][128 B]
    uint8_t* b_s = smem + Q_BYTES_MAX;                     // [slot][256 DB rows][128 B]
    float* h_s = reinterpret_cast<float*>(b_s + RING_SLOTS * SLOT_BYTES);     // [H_RING][256] 0.5|x|^2 of the tile's rows
    int* lmax_s = reinterpret_cast<int*>(h_s + H_RING * SCAN_TILE);          // [column half 2][NQ_CTA]
    int* cnt_s = lmax_s + 2 * NQ_CTA;                                         // [NQ_CTA]
    ScanBars* bars = reinterpret_cast<ScanBars*>(cnt_s + NQ_CTA);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // Clusters of two CTAs (cluster rank = cta & 1).  Both CTAs of a pair score the same DB tiles, each against its own
    // n_half x 128 query rows: rank 0's producer draws the tiles and multicasts each one into both CTAs' shared
    // memory, so a tile crosses HBM once per pair.  G CTAs, C = G / 2 pairs.  The maxima that build the thresholds
    // come from G sources, one per (pair, accumulator column half): disjoint row sets.
    const int G = gridDim.x;
    const int cta = blockIdx.x;
    const int rank = cta & 1, clu = cta >> 1, C = G >> 1;
    const int qrow0 = rank * n_half * 128;                 // this CTA's first row of the pass
    // Work items of a pair: `warm` tiles clu, clu + C, ... scanned max-only (their exact maxima seed the shared
    // thresholds, which are ready -- no wait -- when the last of them is done; a row scanned at tile t survives
    // with probability ~ kg / (rows seen so far), so the first tiles of a pass would otherwise append, and pay
    // for, half of all survivors), then tiles handed out by a global counter (SMs do not all stream at the same
    // rate: with a static split the slowest CTA finished 35 % after the fastest), then the warm tiles again
    // (with thresholds), then the end marker.  Rank 0's TMA producer draws the tiles and tells the MMA issuers and
    // the epilogues of both CTAs through bars->tile_of.
    const int warm = max(1, min(WARM_TILES, n_tiles / C));

    for (int i = threadIdx.x; i < NQ_CTA; i += blockDim.x) {
        lmax_s[i] = INT_MIN;
        lmax_s[NQ_CTA + i] = INT_MIN;
        cnt_s[i] = 0;
    }
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmap_q);
        tma_prefetch_desc(&tmap_db);
        for (int s = 0; s < RING_SLOTS; ++s) {
            mbar_init(&bars->full[s], 1);
            mbar_init(&bars->empty[s], 2);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bars->tfull[a], 1);
            mbar_init(&bars->tempty[a], EPI_WARPS);
        }
        mbar_init(&bars->qfull, 1);
        bars->done = 0;
        mbar_fence_init();
    }
    if (warp == MMA_WARP) {
        tmem_alloc(&bars->tmem_base, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    cluster_sync();                // the peer's barriers are initialised before the first remote arrive / commit
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, bars->tmem_base, 0);     // provably warp-uniform

    if (warp == TMA_WARP) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            const int q_rows = n_half * 128;
            mbar_arrive_expect_tx(&bars->qfull, 2u * q_rows * 128u);
            for (int kb = 0; kb < 2; ++kb)
                for (int r0 = 0; r0 < q_rows; r0 += 32)
                    tma_load_2d(q_s + kb * Q_KB_BYTES + r0 * 128, &tmap_q, &bars->qfull, kb * 64, qrow0 + r0);
        }
        if (lane == 0 && rank == 0) {
            // Rank 0 delivers every item to both CTAs.  Its empty[s] completes when both MMA warps have released the
            // slot.  It arms the peer's full[s] remotely; the tile id reaches the peer's tile_of by st.async, which
            // completes on the peer's full[s0], so the id becomes visible there together with the slot's data.
            const uint32_t peer_full0 = map_shared_rank(&bars->full[0], 1);       // the peer's full[s]: + 8 s
            const uint32_t peer_tile_of0 = map_shared_rank(&bars->tile_of[0], 1);
            int tile = clu;
            int revisit = -1;                                   // >= 0: index of the warm tile being revisited
            int nxt = warm * C + atomicAdd(tile_counter, 1);    // drawn one item ahead: the round trip hides behind the loads
            int i = 0;
            for (;; ++i) {
                const int kc0 = 2 * i;
                const uint32_t ph = (kc0 / RING_SLOTS) & 1;
                const int s0 = kc0 % RING_SLOTS;
                mbar_wait_parked(&bars->empty[s0], ph ^ 1);
                bars->tile_of[i & 7] = tile;                      // released to this CTA's consumers by the arrive below
                mbar_arrive_expect_tx_remote(peer_full0 + 8 * s0, (tile < 0 ? 0 : SLOT_BYTES + SCAN_TILE * 4) + 4);
                st_async_remote(peer_tile_of0 + 4 * (i & 7), tile, peer_full0 + 8 * s0);
                if (tile < 0) {
                    mbar_arrive(&bars->full[s0]);
                    break;
                }
#pragma unroll
                for (int kb = 0; kb < 2; ++kb) {
                    const int s = s0 + kb;
                    if (kb == 1) {
                        mbar_wait_parked(&bars->empty[s], ph ^ 1);
                        mbar_arrive_expect_tx_remote(peer_full0 + 8 * s, SLOT_BYTES);
                    }
                    mbar_arrive_expect_tx(&bars->full[s], SLOT_BYTES + (kb == 0 ? SCAN_TILE * 4 : 0));
                    // the tile's 0.5|x|^2 travel with its first K block.  Ring of 4: entry i is rewritten for
                    // item i+4, whose load is issued after item i+2's MMAs (in both CTAs), which start after item i's
                    // epilogue
                    if (kb == 0)
                        bulk_load_1d_multicast(h_s + (i % H_RING) * SCAN_TILE, hn + static_cast<int64_t>(tile) * SCAN_TILE,
                                               SCAN_TILE * 4, &bars->full[s], PAIR_MASK);
                    uint8_t* dst = b_s + s * SLOT_BYTES;
                    tma_load_2d_multicast(dst, &tmap_db, &bars->full[s], kb * 64, tile * SCAN_TILE, PAIR_MASK);
                    tma_load_2d_multicast(dst + BOX_BYTES, &tmap_db, &bars->full[s], kb * 64, tile * SCAN_TILE + TILE_ROWS,
                                          PAIR_MASK);
                }
                if (i + 1 < warm) {
                    tile = clu + (i + 1) * C;
                } else if (revisit < 0 && nxt < n_tiles) {
                    tile = nxt;
                    nxt = warm * C + atomicAdd(tile_counter, 1);
                } else {
                    ++revisit;
                    tile = revisit < warm ? clu + revisit * C : -1;
                }
            }
            // The peer's MMA warp commits into this CTA's empty barriers: wait for its last commits (the K blocks
            // 2i-3 .. 2i-1 of the last items) before this CTA may leave.  K block kc of a slot is the (kc / 4)-th use.
            for (int kc = 2 * i + 1; kc < 2 * i + RING_SLOTS; ++kc)
                mbar_wait_parked(&bars->empty[kc % RING_SLOTS], ((kc / RING_SLOTS) & 1) ^ 1);
        }
        __syncwarp();
    } else if (warp == MMA_WARP) {
        // ------------------------------------------------------------ MMA issuer
        // unit = (tile, 128-query half): D[query][db row] in accumulator (unit & 1).  The second K block's
        // slot is released as soon as the last unit's MMAs on it are issued, the first one's four MMAs earlier; a slot is
        // released on rank 0's empty barrier, which counts both CTAs of the pair.
        // The whole warp runs the loop (uniform control flow keeps descriptors and counters in uniform
        // registers); one elected lane issues.
        const bool leader = elect_one();
        const uint32_t idesc = umma_idesc_f16(1u, 128u, static_cast<uint32_t>(SCAN_TILE));
        const uint64_t adesc0 = umma_desc_sw128(smem_u32(q_s));
        const uint64_t bdesc0 = umma_desc_sw128(smem_u32(b_s));
        mbar_wait_parked(&bars->qfull, 0);
        uint32_t uc = 0;
        bool more = true;
        for (int i = 0; more; ++i) {
            const int s0 = (2 * i) % RING_SLOTS, s1 = s0 + 1;
            const uint32_t ph = ((2 * i) / RING_SLOTS) & 1;
            for (int hq = 0; hq < n_half; ++hq, ++uc) {
                const int acc = uc & 1;
                const uint32_t aph = (uc >> 1) & 1;
                const bool last = hq == n_half - 1;
                mbar_wait_parked(&bars->tempty[acc], aph ^ 1);
                if (hq == 0) {
                    mbar_wait_parked_cluster(&bars->full[s0], ph);       // completed from rank 0 (tile id, data)
                    if (smem_ld_volatile(&bars->tile_of[i & 7]) < 0) {      // end marker: wake the epilogue and stop
                        if (leader) tc_commit(&bars->tfull[acc]);
                        __syncwarp();
                        more = false;
                        break;
                    }
                }
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * SCAN_TILE;
                const uint64_t a_kb0 = adesc0 + static_cast<uint64_t>((hq * (128 * 128)) >> 4);
                const uint64_t a_kb1 = a_kb0 + static_cast<uint64_t>(Q_KB_BYTES >> 4);
                const uint64_t b_kb0 = bdesc0 + static_cast<uint64_t>((s0 * SLOT_BYTES) >> 4);
                const uint64_t b_kb1 = b_kb0 + static_cast<uint64_t>(SLOT_BYTES >> 4);
                if (leader) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) tc_mma_f16(d_tmem, a_kb0 + 2 * j, b_kb0 + 2 * j, idesc, j != 0 ? 1u : 0u);
                    if (last) tc_commit_multicast(&bars->empty[s0], RANK0_MASK);
                }
                if (hq == 0) {
                    mbar_wait_parked_cluster(&bars->full[s1], ph);
                    tc_fence_after();
                }
                if (leader) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) tc_mma_f16(d_tmem, a_kb1 + 2 * j, b_kb1 + 2 * j, idesc, 1u);
                    if (last) tc_commit_multicast(&bars->empty[s1], RANK0_MASK);
                    tc_commit(&bars->tfull[acc]);
                }
                __syncwarp();
            }
        }
        __syncwarp();
    } else if (warp < EPI_WARPS) {
        // ------------------------------------------------------------ epilogue (EPI_WARPS warps)
        // Warp e reads TMEM lane quadrant (warp & 3) -- 32 queries per half -- and the 64 accumulator
        // columns (DB rows) [64 part, 64 part + 64) of every unit: column half part >> 1.  Query rows are local
        // (0 .. n_half * 128 - 1, pass row qrow0 + local row).
        const int qd = warp & 3;
        const int e = warp;               // 0..EPI_WARPS-1
        const int part = e >> 2;          // 0..EPI_PARTS-1
        constexpr int QPW = NQ_CTA / EPI_WARPS;      // queries whose maxima (both column halves) this warp publishes
        static_assert(2 * QPW == 32, "one lane per (query, column half) when maxima are published");
        const int q_rows = n_half * 128;
        int* lmax_part = lmax_s + (part >> 1) * NQ_CTA;
        const float NEG_INF = -INFINITY;
        int pub = INT_MIN;
        int thr_ord[2] = {NEG_INF_ORD, NEG_INF_ORD};
        float t_exact[2], t_pre[2];       // exact threshold; same minus a rounding margin (prefilter base)
        bool active[2];
#pragma unroll
        for (int hq = 0; hq < 2; ++hq) {
            active[hq] = hq < n_half && qrow0 + (hq * 128 + qd * 32 + lane) < nq;
            t_exact[hq] = active[hq] ? NEG_INF : INFINITY;      // padding queries never fire
            t_pre[hq] = t_exact[hq];
        }
        uint64_t* my_pool = pool + static_cast<int64_t>(cta) * NQ_CTA * POOL_CAP;
        const uint32_t ns32 = static_cast<uint32_t>(n_search);
        // shared thresholds of this thread's queries -> registers; true when all of the warp's are known
        auto load_thresholds = [&](int (&tg)[2]) {
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) tg[hq] = active[hq] ? ld_relaxed(&Tg[qrow0 + hq * 128 + qd * 32 + lane]) : INT_MIN;
        };
        auto apply_thresholds = [&](const int (&tg)[2]) -> bool {
            bool valid = true;
#pragma unroll
            for (int hq = 0; hq < 2; ++hq) {
                if (active[hq]) {
                    if (tg[hq] > thr_ord[hq]) {
                        thr_ord[hq] = tg[hq];
                        const float t = ord2f(tg[hq]);
                        t_exact[hq] = t;
                        t_pre[hq] = t - fabsf(t) * (1.f / 1048576.f) - 1e-37f;
                    }
                    valid = valid && (thr_ord[hq] > NEG_INF_ORD);
                }
            }
            return __all_sync(0xffffffffu, valid);
        };
        // publish this CTA's running maxima: warp e owns local queries [QPW e, QPW e + QPW), lane / QPW is the column
        // half, and source (pair, column half) is column 2 clu + half of Mx
        auto publish_maxima = [&]() {
            const int ql = e * QPW + (lane % QPW), half = lane / QPW;
            if (ql < q_rows && qrow0 + ql < nq) {
                const int m = smem_ld_volatile(&lmax_s[half * NQ_CTA + ql]);
                if (m > pub) {
                    st_relaxed(&Mx[(qrow0 + ql) * G + 2 * clu + half], m);
                    pub = m;
                }
            }
        };
        const uint32_t tlane = tmem_base + (static_cast<uint32_t>(qd * 32) << 16) + part * PART_COLS;
        uint32_t uc = 0;

        // ---- items 0 .. warm-1 (tiles clu, clu + C, ...) are scanned "max-only": their exact scores feed the
        // running maxima from which the shared thresholds are built; they come back, with thresholds, as the
        // last items.
        for (int w = 0; w < warm; ++w) {
            const uint32_t row0 = static_cast<uint32_t>(clu + w * C) * SCAN_TILE + part * PART_COLS;
            const float* h_part = h_s + (w % H_RING) * SCAN_TILE + part * PART_COLS;
            // rows of (numerically) equal norm, all searchable -- fingerprints are unit vectors --: the best score of a
            // chunk is its maximum minus the common 0.5|x|^2 (FMNMX3 chain).  Otherwise (reconstructions of an
            // IVF-PQ index, raw vectors, halo / padding rows): exact, column by column.
            bool edge = (static_cast<uint32_t>(clu + w * C) + 1u) * SCAN_TILE > ns32;
            float hx = 0.f;
            for (int hq = 0; hq < n_half; ++hq, ++uc) {
                const int acc = uc & 1;
                mbar_wait_parked(&bars->tfull[acc], (uc >> 1) & 1);
                if (hq == 0 && !edge) {
                    const float a = h_part[lane], b = h_part[32 + lane];
                    const float hmax_w = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(a, b))));
                    const float hmin_w = __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(fminf(a, b))));
                    hx = hmax_w * (1.f + 1.f / 1048576.f);
                    edge = !(hmax_w - hmin_w <= hmax_w * (1.f / 262144.f));
                }
                tc_fence_after();
                float munit = NEG_INF;
#pragma unroll 1
                for (int c = 0; c < PART_COLS / 32; ++c) {
                    uint32_t v[32];
                    tmem_ld_32x32(tlane + acc * SCAN_TILE + c * 32, v);
                    tc_wait_ld();
                    if (!edge) {
                        float gm[4];
#pragma unroll
                        for (int g = 0; g < 4; ++g) {
                            float m = fmax3(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1]), __uint_as_float(v[8 * g + 2]));
                            m = fmax3(m, __uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4]));
                            m = fmax3(m, __uint_as_float(v[8 * g + 5]), __uint_as_float(v[8 * g + 6]));
                            gm[g] = fmaxf(m, __uint_as_float(v[8 * g + 7]));
                        }
                        munit = fmaxf(munit, fmaxf(fmax3(gm[0], gm[1], gm[2]), gm[3]) - hx);
                    } else {
                        const float* hc = h_part + c * 32;
                        const int nvalid = static_cast<int>(min(ns32 - min(ns32, row0 + c * 32), 32u));   // rows < n_search
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (j < nvalid) munit = fmaxf(munit, __uint_as_float(v[j]) - hc[j]);
                    }
                }
                if (hq == 0 ? active[0] : active[1]) smem_red_max(&lmax_part[hq * 128 + qd * 32 + lane], f2ord(munit));
                tc_fence_before();
                __syncwarp();
                mbar_arrive_lane0(&bars->tempty[acc], lane);
            }
            publish_maxima();
        }
        // ---- wait (bounded) for the thresholds of this warp's queries
        {
            int tg[2];
            bool ok = false;
            for (int spin = 0; spin < 4096 && !ok; ++spin) {
                publish_maxima();          // the other warps' tile-0 maxima of the queries this warp publishes
                load_thresholds(tg);
                ok = apply_thresholds(tg);
                if (!ok) __nanosleep(100);
            }
            // not ok after ~0.5 ms: scan on with -inf thresholds; the pools overflow and the exact fallback
            // answers those queries
        }
        // ---- the items the producer draws for this CTA, ending with the warm tiles again and the end marker
        for (int i = warm;; ++i) {
            int tg[2] = {INT_MIN, INT_MIN};
            // one refresh every four tiles: a coherent load takes ~2 us under the scan's own traffic -- longer than a
            // tile -- and after the warm tiles the thresholds move slowly (refreshing every tile cost 8 % of a
            // 7 M-row pass).  Loads issued now, consumed after the tile.
            const bool rf = i > warm && (i & 3) == 0;
            if (rf) load_thresholds(tg);
            const float* h_part = h_s + (i % H_RING) * SCAN_TILE + part * PART_COLS;
            uint32_t row0 = 0;
            float hm = 0.f;
            bool end = false, edge = false;
            for (int hq = 0; hq < n_half; ++hq, ++uc) {
                const int acc = uc & 1;
                mbar_wait_parked(&bars->tfull[acc], (uc >> 1) & 1);
                if (hq == 0) {
                    const int tile = smem_ld_volatile(&bars->tile_of[i & 7]);
                    if (tile < 0) {
                        end = true;
                        break;
                    }
                    row0 = static_cast<uint32_t>(tile) * SCAN_TILE + part * PART_COLS;
                    // prefilter offset: s = v - h > T implies v > T + min(h) over this warp's 64 rows (minus a
                    // rounding margin); the rows' 0.5|x|^2 arrived in shared memory with the tile
                    const float hmin_w =
                        __uint_as_float(__reduce_min_sync(0xffffffffu, __float_as_uint(fminf(h_part[lane], h_part[32 + lane]))));
                    hm = hmin_w * (1.f - 1.f / 1048576.f);
                    // the tile holds rows that do not take part in the search (halo, padding)
                    edge = (static_cast<uint32_t>(tile) + 1u) * SCAN_TILE > ns32;
                }
                const float tp = (hq == 0 ? t_pre[0] : t_pre[1]) + hm;
                tc_fence_after();
                const uint32_t taddr = tlane + acc * SCAN_TILE;
#pragma unroll 1
                for (int c = 0; c < PART_COLS / 32; ++c) {
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + c * 32, v);
                    tc_wait_ld();
                    // maxima of the four 8-column groups (FMNMX3), then of the chunk
                    float gm[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {
                        float m = fmax3(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1]), __uint_as_float(v[8 * g + 2]));
                        m = fmax3(m, __uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4]));
                        m = fmax3(m, __uint_as_float(v[8 * g + 5]), __uint_as_float(v[8 * g + 6]));
                        gm[g] = fmaxf(m, __uint_as_float(v[8 * g + 7]));
                    }
                    const float ma = fmaxf(fmax3(gm[0], gm[1], gm[2]), gm[3]);
                    const bool fired = ma > tp;
                    if (__any_sync(0xffffffffu, fired)) {
                        // rare -- except in the first thresholded tiles of a pass, while the thresholds are still
                        // loose (an event per warp per tile): see scan_chunk_hits
                        const int q = hq * 128 + qd * 32 + lane;
                        const float te = hq == 0 ? t_exact[0] : t_exact[1];
                        const uint32_t rbase = row0 + c * 32;
                        if (!edge)
                            scan_chunk_hits<false>(v, h_part + c * 32, te, 32, rbase, &cnt_s[q], &lmax_part[q], my_pool + q * POOL_CAP);
                        else
                            scan_chunk_hits<true>(v, h_part + c * 32, te, static_cast<int>(min(ns32 - min(ns32, rbase), 32u)), rbase,
                                                  &cnt_s[q], &lmax_part[q], my_pool + q * POOL_CAP);
                        __syncwarp();
                    }
                }
                tc_fence_before();
                __syncwarp();
                mbar_arrive_lane0(&bars->tempty[acc], lane);
            }
            if (end) break;
            if (rf) apply_thresholds(tg);
            if (i < warm + 32 || (i & 3) == 0) publish_maxima();
        }
        publish_maxima();
        __syncwarp();
        // all epilogue warps are done appending before counts are published
        asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory");
        {
            const int ql = e * QPW + lane;
            if (lane < QPW && ql < q_rows && qrow0 + ql < nq) {
                const int c = cnt_s[ql];
                cnt[cta * NQ_CTA + ql] = min(c, POOL_CAP);
                if (c > POOL_CAP) flags[qrow0 + ql] = 1;      // pool overflow -> exact fallback answers this query
            }
        }
        if (lane == 0) smem_atom_inc(&bars->done);
    } else {
        // ------------------------------------------------------------ threshold reducer (last warp)
        // For the queries assigned to this CTA: T = kg-th largest of the G maxima (one per pair and accumulator column
        // half, over disjoint row sets).  At least kg distinct rows score >= T, so dropping rows that score <= T can
        // never lose a top-kg row.
        // The thresholds converge within the first few dozen tiles; afterwards the select runs rarely so
        // that this warp stops competing for its sub-partition's issue slots.
        uint32_t round = 0;
        while (smem_ld_volatile(&bars->done) < EPI_WARPS) {
            for (int q = cta; q < nq; q += G) {
                uint32_t u[5];
#pragma unroll
                for (int t = 0; t < 5; ++t) {
                    const int g = lane + 32 * t;
                    const int m = g < G ? ld_relaxed(&Mx[q * G + g]) : INT_MIN;
                    u[t] = static_cast<uint32_t>(m) ^ 0x80000000u;
                }
                uint32_t res = 0;
                for (int bit = 31; bit >= 0; --bit) {
                    const uint32_t cand = res | (1u << bit);
                    int c = 0;
#pragma unroll
                    for (int t = 0; t < 5; ++t) c += (u[t] >= cand) ? 1 : 0;
                    c = __reduce_add_sync(0xffffffffu, c);
                    if (c >= kg) res = cand;
                }
                const int T = static_cast<int>(res ^ 0x80000000u);
                if (lane == 0 && T > NEG_INF_ORD && T > ld_relaxed(&Tg[q])) st_relaxed(&Tg[q], T);
            }
            ++round;
            // the select competes with four epilogue warps for its sub-partition's issue slots: once the first
            // thresholds are out (a few rounds), one refresh every few tiles is as good as a continuous one
            if (round < 6) {
                __nanosleep(100);
            } else {
                for (int nap = 0; nap < 8 && smem_ld_volatile(&bars->done) < EPI_WARPS; ++nap) __nanosleep(500);   // prompt exit
            }
        }
    }

    tc_fence_before();
    cluster_sync();                // no remote arrive, commit or multicast targets a CTA that has left
    if (warp == MMA_WARP) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------
// survivors -> exact fp32 re-rank + proof
// ------------------------------------------------------------------------------------------
struct SelBatch {
    int np[SEL_SLOTS];       // query rows of the pass held in every slot
    int h[SEL_SLOTS];        // query rows per CTA of that pass: row q is local row q % h of the CTAs of rank q / h
    int grid_alloc;          // CTA dimension the pool / cnt arrays were allocated with
};

// grid (NQ_MAX, slots): block (q, slot) answers row q of the scan pass parked in `slot`; its survivors are in the pools
// of the grid_scan / 2 CTAs 2 c + rank that held it
__global__ void __launch_bounds__(256)
flat_select_kernel(SelBatch batch, int k, int grid_scan, int64_t n_rows, const float* __restrict__ q32,
                   const float* __restrict__ qn2, const float* __restrict__ x32, const float* __restrict__ hn,
                   const int32_t* __restrict__ maxn2, const int32_t* __restrict__ Tg,
                   const uint64_t* __restrict__ pool, const int32_t* __restrict__ cnt, int32_t* __restrict__ flags,
                   const int64_t* __restrict__ gidx, int32_t* __restrict__ fail_list, int32_t* __restrict__ fail_count,
                   int64_t label_offset, float* __restrict__ D, int64_t* __restrict__ I,
                   unsigned long long* __restrict__ stats) {
    // D / I are the caller's full output arrays; this pass's row q lands at global row gidx[q].
    // A query whose top-k cannot be proven is appended to fail_list (global row) and answered later.
    __shared__ uint64_t keys[SELECT_CAP];
    __shared__ int total_s;
    const int q = blockIdx.x;
    const int slot = blockIdx.y;
    if (q >= batch.np[slot]) return;
    q32 += static_cast<int64_t>(slot) * NQ_MAX * D128;
    qn2 += slot * NQ_MAX;
    Tg += slot * NQ_MAX;
    pool += static_cast<int64_t>(slot) * batch.grid_alloc * NQ_CTA * POOL_CAP;
    cnt += static_cast<int64_t>(slot) * batch.grid_alloc * NQ_CTA;
    flags += slot * NQ_MAX;
    gidx += slot * NQ_MAX;
    const int64_t g = gidx[q];
    if (flags[q] != 0) {                 // pool overflow seen by the scan
        if (threadIdx.x == 0) {
            fail_list[atomicAdd(fail_count, 1)] = static_cast<int32_t>(g);
            atomicAdd(&stats[5], 1ull);
        }
        return;
    }
    if (threadIdx.x == 0) total_s = 0;
    __syncthreads();
    bool over = false;
    const int rank = q / batch.h[slot], ql = q - rank * batch.h[slot];
    for (int pr = threadIdx.x; pr < grid_scan / 2; pr += blockDim.x) {
        const int cta = 2 * pr + rank;
        const int c = cnt[cta * NQ_CTA + ql];
        if (c > 0) {
            const int base = atomicAdd(&total_s, c);
            if (base + c <= SELECT_CAP) {
                const uint64_t* src = pool + (static_cast<int64_t>(cta) * NQ_CTA + ql) * POOL_CAP;
                for (int i = 0; i < c; ++i) keys[base + i] = src[i];
            } else {
                over = true;
            }
        }
    }
    if (__syncthreads_or(over ? 1 : 0)) {
        if (threadIdx.x == 0) {
            flags[q] = 1;
            fail_list[atomicAdd(fail_count, 1)] = static_cast<int32_t>(g);
            atomicAdd(&stats[5], 1ull);
        }
        return;
    }
    const int total = total_s;
    const int64_t need = n_rows < k ? n_rows : k;
    if (total < need) {
        if (threadIdx.x == 0) {
            flags[q] = 1;
            fail_list[atomicAdd(fail_count, 1)] = static_cast<int32_t>(g);
            atomicAdd(&stats[5], 1ull);
        }
        return;
    }
    // exact fp32 re-score: 8 lanes per survivor (16 dims each), 4 survivors per warp per round,
    // so every lane has 4 independent 16-byte loads in flight
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sub = lane >> 3, l8 = lane & 7;
    float4 qv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) qv[c] = reinterpret_cast<const float4*>(q32 + q * D128 + l8 * 16)[c];
    for (int i0 = warp * 4; i0 < total; i0 += 32) {
        const int i = i0 + sub;
        const bool ok = i < total;
        const uint32_t row = ok ? static_cast<uint32_t>(keys[i]) : 0u;
        const float4* xr = reinterpret_cast<const float4*>(x32 + static_cast<int64_t>(row) * D128 + l8 * 16);
        const float4 a0 = xr[0], a1 = xr[1], a2 = xr[2], a3 = xr[3];
        const float hh = hn[row];
        float s = a0.x * qv[0].x + a0.y * qv[0].y + a0.z * qv[0].z + a0.w * qv[0].w;
        s += a1.x * qv[1].x + a1.y * qv[1].y + a1.z * qv[1].z + a1.w * qv[1].w;
        s += a2.x * qv[2].x + a2.y * qv[2].y + a2.z * qv[2].z + a2.w * qv[2].w;
        s += a3.x * qv[3].x + a3.y * qv[3].y + a3.z * qv[3].z + a3.w * qv[3].w;
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        __syncwarp();
        if (ok && l8 == 0) keys[i] = score_key(s - hh, row);
    }
    int npow = 1;
    while (npow < total) npow <<= 1;
    __syncthreads();
    for (int i = total + threadIdx.x; i < npow; i += blockDim.x) keys[i] = 0;
    __syncthreads();
    block_sort_u64<false>(keys, npow);
    // proof: every row that is not a survivor has bf16 score <= T, hence exact score <= T + eps
    const int tgo = Tg[q];
    if (tgo > NEG_INF_ORD) {
        const float qn = sqrtf(qn2[q]);
        const float xn = sqrtf(__int_as_float(*maxn2));
        const float u = 0.00390625f;
        const float eps = (2.f * u + u * u) * qn * xn * 1.01f + 1e-5f * qn * xn + 1e-30f;
        const float bound = ord2f(tgo) + eps;
        const float sk = key_score(keys[need - 1]);
        if (!(sk > bound)) {
            if (threadIdx.x == 0) {
                flags[q] = 2;
                fail_list[atomicAdd(fail_count, 1)] = static_cast<int32_t>(g);
                atomicAdd(&stats[6], 1ull);
            }
            return;
        }
    }
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        if (j < need) {
            const uint64_t key = keys[j];
            D[g * k + j] = fmaxf(qn2[q] - 2.f * key_score(key), 0.f);
            I[g * k + j] = static_cast<int64_t>(key_row(key)) + label_offset;
        } else {
            D[g * k + j] = INFINITY;
            I[g * k + j] = -1;
        }
    }
    if (threadIdx.x == 0) atomicAdd(&stats[3], static_cast<unsigned long long>(total));
}

// ------------------------------------------------------------------------------------------
// exact fp32 fallback (CUDA cores): queries the bf16 bound could not prove, and tiny databases.
// grid (BRUTE_CHUNKS, n_entries): entry e answers global query row list[list_off + e] (or
// list_off + e when list is NULL).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
flat_brute_scan_kernel(int k, int64_t n_rows, const float* __restrict__ q_all, const float* __restrict__ x32,
                       const float* __restrict__ hn, const int32_t* __restrict__ list, int64_t list_off,
                       uint64_t* __restrict__ part) {
    __shared__ uint64_t lists[8][MAX_K];
    const int e = blockIdx.y;
    const int64_t g = list ? static_cast<int64_t>(list[list_off + e]) : list_off + e;
    const int chunk = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t per = (n_rows + BRUTE_CHUNKS - 1) / BRUTE_CHUNKS;
    const int64_t r0 = chunk * per;
    const int64_t r1 = r0 + per < n_rows ? r0 + per : n_rows;
    uint64_t* lst = lists[warp];
    for (int i = lane; i < k; i += 32) lst[i] = 0;
    __syncwarp();
    const float4 qv = reinterpret_cast<const float4*>(q_all + g * D128)[lane];
    uint64_t kth = 0;     // current k-th best key of this warp (0 = list not full)
    for (int64_t r = r0 + warp; r < r1; r += 8) {
        const float s = warp_dot128(qv, x32 + r * D128, lane) - hn[r];
        const uint64_t key = score_key(s, static_cast<uint32_t>(r));
        if (key > kth) {             // warp-uniform
            if (lane == 0) {
                int p = k - 1;
                while (p > 0 && lst[p - 1] < key) {
                    lst[p] = lst[p - 1];
                    --p;
                }
                lst[p] = key;
            }
            __syncwarp();
            kth = lst[k - 1];
            __syncwarp();            // every lane has read the list before lane 0 inserts again (racecheck: WAR warning;
                                     // the shuffles of the next dot product ordered it in practice)
        }
    }
    __syncthreads();
    // block merge: k rounds of arg-max over the 8 warp lists (each sorted descending)
    if (warp == 0) {
        uint64_t* out = part + (static_cast<int64_t>(e) * BRUTE_CHUNKS + chunk) * MAX_K;
        int head = 0;     // lane w < 8 owns the read cursor of list w
        for (int j = 0; j < k; ++j) {
            const uint64_t cand = (lane < 8 && head < k) ? lists[lane][head] : 0;
            const uint64_t best = warp_max_u64(cand);
            if (lane < 8 && cand == best && best != 0) ++head;   // keys are unique (row id inside)
            if (lane == 0) out[j] = best;
        }
    }
}

__global__ void __launch_bounds__(256)
flat_brute_merge_kernel(int k, const float* __restrict__ q_all, const int32_t* __restrict__ list, int64_t list_off,
                        uint64_t* __restrict__ part, int64_t label_offset, float* __restrict__ D,
                        int64_t* __restrict__ I, unsigned long long* __restrict__ stats) {
    __shared__ uint64_t red[8];
    __shared__ float qn2_s;
    const int e = blockIdx.x;
    const int64_t g = list ? static_cast<int64_t>(list[list_off + e]) : list_off + e;
    uint64_t* p = part + static_cast<int64_t>(e) * BRUTE_CHUNKS * MAX_K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        const float4 v = reinterpret_cast<const float4*>(q_all + g * D128)[lane];
        float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) qn2_s = ss;
    }
    __syncthreads();
    for (int j = 0; j < k; ++j) {
        uint64_t best = 0;
        for (int c = threadIdx.x; c < BRUTE_CHUNKS * k; c += blockDim.x) {
            const uint64_t v = p[(c / k) * MAX_K + (c % k)];
            best = v > best ? v : best;
        }
        const uint64_t w = block_max_u64(best, red);
        if (threadIdx.x == 0) {
            if (w != 0) {
                D[g * k + j] = fmaxf(qn2_s - 2.f * key_score(w), 0.f);
                I[g * k + j] = static_cast<int64_t>(key_row(w)) + label_offset;
            } else {
                D[g * k + j] = INFINITY;
                I[g * k + j] = -1;
            }
        }
        if (w != 0)
            for (int c = threadIdx.x; c < BRUTE_CHUNKS * k; c += blockDim.x) {
                uint64_t* slot = &p[(c / k) * MAX_K + (c % k)];
                if (*slot == w) *slot = 0;
            }
        __syncthreads();
    }
    if (threadIdx.x == 0) atomicAdd(&stats[1], 1ull);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
constexpr int PROF_RING = 8192;
static int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

int index_reserve(nafp_index* idx, int64_t n_total) {
    if (n_total <= idx->cap) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    const int64_t new_cap = round_up(n_total, TILE_ROWS);
    float* x32 = nullptr;
    __nv_bfloat16* x16 = nullptr;
    float* hn = nullptr;
    NAFP_CUDA(cudaMalloc(&x32, static_cast<size_t>(new_cap) * idx->d * sizeof(float)));
    if (idx->scan_copy) {
        NAFP_CUDA(cudaMalloc(&x16, static_cast<size_t>(new_cap) * idx->d * sizeof(__nv_bfloat16)));
        NAFP_CUDA(cudaMalloc(&hn, static_cast<size_t>(new_cap + SCAN_TILE) * sizeof(float)));
        NAFP_CUDA(cudaMemsetAsync(x16, 0, static_cast<size_t>(new_cap) * idx->d * sizeof(__nv_bfloat16), ctx->stream));
    }
    if (idx->n > 0) {
        NAFP_CUDA(cudaMemcpyAsync(x32, idx->x32, static_cast<size_t>(idx->n) * idx->d * sizeof(float),
                                  cudaMemcpyDeviceToDevice, ctx->stream));
        if (idx->scan_copy) {
            NAFP_CUDA(cudaMemcpyAsync(x16, idx->x16, static_cast<size_t>(idx->n) * idx->d * sizeof(__nv_bfloat16),
                                      cudaMemcpyDeviceToDevice, ctx->stream));
            NAFP_CUDA(cudaMemcpyAsync(hn, idx->hn, static_cast<size_t>(idx->n) * sizeof(float),
                                      cudaMemcpyDeviceToDevice, ctx->stream));
        }
    }
    if (idx->scan_copy) {
        const int64_t cnt = new_cap + SCAN_TILE - idx->n;
        const int threads = 256;
        const int64_t blocks = (cnt + threads - 1) / threads;
        flat_fill_kernel<<<static_cast<unsigned>(blocks), threads, 0, ctx->stream>>>(hn, idx->n, new_cap + SCAN_TILE, INFINITY);
        ctx->launches++;
        NAFP_CUDA(cudaGetLastError());
    }
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (idx->x32) cudaFree(idx->x32);
    if (idx->x16) cudaFree(idx->x16);
    if (idx->hn) cudaFree(idx->hn);
    idx->x32 = x32;
    idx->x16 = x16;
    idx->hn = hn;
    idx->cap = new_cap;
    if (!idx->scan_copy) return NAFP_OK;
    // DB tensor map: [cap rows][128 bf16], box 64 columns x 128 rows, 128-byte swizzle
    const uint64_t dims[2] = {static_cast<uint64_t>(idx->d), static_cast<uint64_t>(new_cap)};
    const uint64_t strides[2] = {2, static_cast<uint64_t>(idx->d) * 2};
    const uint32_t box[2] = {64, TILE_ROWS};
    NAFP_TRY(make_tensor_map(&idx->tmap_db, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, x16, dims, strides, box, nullptr,
                             CU_TENSOR_MAP_SWIZZLE_128B));
    idx->tmap_db_valid = true;
    return NAFP_OK;
}

int flat_add_dev(nafp_index* idx, const float* x, int64_t n, bool src_is_host) {
    if (n == 0) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    if (idx->n + n > idx->cap) {
        int64_t want = idx->cap * 2;
        if (want < idx->n + n) want = idx->n + n;
        NAFP_TRY(index_reserve(idx, want));
    }
    NAFP_CUDA(cudaMemcpyAsync(idx->x32 + idx->n * idx->d, x, static_cast<size_t>(n) * idx->d * sizeof(float),
                              src_is_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    if (idx->scan_copy) {
        const int threads = 256;
        int64_t blocks = (n * 32 + threads - 1) / threads;
        if (blocks > ctx->sm_count * 16) blocks = ctx->sm_count * 16;
        flat_convert_rows_kernel<<<static_cast<unsigned>(blocks), threads, 0, ctx->stream>>>(idx->x32, idx->x16, idx->hn,
                                                                                            idx->maxn2, idx->n, n);
        ctx->launches++;
        NAFP_CUDA(cudaGetLastError());
    }
    if (src_is_host) NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    idx->n += n;
    return NAFP_OK;
}

// flat_scan_kernel runs as clusters of two CTAs
static cudaLaunchConfig_t scan_launch_config(int grid, cudaStream_t stream, cudaLaunchAttribute (&attr)[1]) {
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(SCAN_THREADS);
    cfg.dynamicSmemBytes = SCAN_SMEM;
    cfg.stream = stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cfg;
}

static int ensure_scratch(nafp_index* idx) {
    if (idx->scratch_ready) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaFuncSetAttribute(flat_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SCAN_SMEM));
    // one CTA per SM (shared memory); the scan runs as many CTA pairs as can be resident at once
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = scan_launch_config(2 * (ctx->sm_count / 2), ctx->stream, attr);
    int clusters = 0;
    NAFP_CUDA(cudaOccupancyMaxActiveClusters(&clusters, flat_scan_kernel, &cfg));
    NAFP_REQUIRE(clusters >= 1, NAFP_ERR_UNSUPPORTED, "flat scan: no CTA pair of the scan kernel fits on this device");
    idx->grid = 2 * clusters;
    NAFP_REQUIRE(idx->grid <= 160, NAFP_ERR_UNSUPPORTED, "flat scan: %d CTAs (reducer handles <= 160)", idx->grid);
    const int G = idx->grid;
    NAFP_CUDA(cudaMalloc(&idx->qbf, NQ_MAX * D128 * sizeof(__nv_bfloat16)));
    NAFP_CUDA(cudaMalloc(&idx->q32, SEL_SLOTS * NQ_MAX * D128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&idx->qn2, SEL_SLOTS * NQ_MAX * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&idx->Mx, static_cast<size_t>(NQ_MAX) * G * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&idx->Tg, SEL_SLOTS * NQ_MAX * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&idx->pool, SEL_SLOTS * static_cast<size_t>(G) * NQ_CTA * POOL_CAP * sizeof(uint64_t)));
    NAFP_CUDA(cudaMalloc(&idx->cnt, SEL_SLOTS * static_cast<size_t>(G) * NQ_CTA * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&idx->flags, SEL_SLOTS * NQ_MAX * sizeof(int32_t)));
    NAFP_CUDA(cudaMalloc(&idx->gidx, SEL_SLOTS * NQ_MAX * sizeof(int64_t)));
    NAFP_CUDA(cudaMalloc(&idx->brute_part, static_cast<size_t>(BRUTE_SLOTS) * BRUTE_CHUNKS * MAX_K * sizeof(uint64_t)));
    NAFP_CUDA(cudaMalloc(&idx->stats, 8 * sizeof(unsigned long long)));
    NAFP_CUDA(cudaMalloc(&idx->tile_counter, sizeof(int32_t)));
    NAFP_CUDA(cudaMemsetAsync(idx->stats, 0, 8 * sizeof(unsigned long long), ctx->stream));
    const uint64_t dims[2] = {static_cast<uint64_t>(D128), static_cast<uint64_t>(NQ_MAX)};
    const uint64_t strides[2] = {2, static_cast<uint64_t>(D128) * 2};
    const uint32_t box[2] = {64, 32};
    NAFP_TRY(make_tensor_map(&idx->tmap_q, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, idx->qbf, dims, strides, box, nullptr,
                             CU_TENSOR_MAP_SWIZZLE_128B));
    idx->scratch_ready = true;
    return NAFP_OK;
}

static int brute_rounds(nafp_index* idx, const float* q_dev, const int32_t* list, int64_t first, int64_t count, int k,
                        int64_t n_search, float* D_dev, int64_t* I_dev) {
    nafp_ctx* ctx = idx->ctx;
    for (int64_t off = 0; off < count; off += BRUTE_SLOTS) {
        const int n = static_cast<int>(count - off < BRUTE_SLOTS ? count - off : BRUTE_SLOTS);
        flat_brute_scan_kernel<<<dim3(BRUTE_CHUNKS, n), 256, 0, ctx->stream>>>(k, n_search, q_dev, idx->x32, idx->hn, list,
                                                                              first + off, idx->brute_part);
        flat_brute_merge_kernel<<<n, 256, 0, ctx->stream>>>(k, q_dev, list, first + off, idx->brute_part, idx->label_offset,
                                                            D_dev, I_dev, idx->stats);
        ctx->launches += 2;
    }
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

static int scan_pass(nafp_index* idx, const float* q_dev, const int32_t* src_list, int src_off, int64_t p0, int np, int kg,
                     int grid_scan, int n_tiles, int64_t n_search, int slot) {
    nafp_ctx* ctx = idx->ctx;
    const int n_half = np > NQ_MAX / 2 ? 2 : 1;      // 128-row query blocks per CTA; rank r takes rows [r h, r h + h)
    const int nq_pad = 2 * n_half * 128;
    const int64_t G = idx->grid;
    float* q32 = idx->q32 + static_cast<int64_t>(slot) * NQ_MAX * D128;
    float* qn2 = idx->qn2 + slot * NQ_MAX;
    int32_t* Tg = idx->Tg + slot * NQ_MAX;
    uint64_t* pool = idx->pool + static_cast<int64_t>(slot) * G * NQ_CTA * POOL_CAP;
    int32_t* cnt = idx->cnt + static_cast<int64_t>(slot) * G * NQ_CTA;
    int32_t* flags = idx->flags + slot * NQ_MAX;
    int64_t* gidx = idx->gidx + slot * NQ_MAX;
    flat_prep_kernel<<<(nq_pad * 32 + 255) / 256, 256, 0, ctx->stream>>>(q_dev, src_list, src_off, p0, np, nq_pad, grid_scan,
                                                                         idx->qbf, q32, qn2, idx->Mx, Tg, flags, gidx, idx->tile_counter);
    const bool prof = idx->profile && idx->prof_n < PROF_RING;
    if (prof) cudaEventRecord(idx->prof_ev[2 * idx->prof_n], ctx->stream);
    cudaLaunchAttribute attr[1];
    const cudaLaunchConfig_t cfg = scan_launch_config(grid_scan, ctx->stream, attr);
    NAFP_CUDA(cudaLaunchKernelEx(&cfg, flat_scan_kernel, idx->tmap_q, idx->tmap_db, static_cast<const float*>(idx->hn),
                                 idx->tile_counter, n_search, n_tiles, np, n_half, kg, idx->Mx, Tg, pool, cnt, flags));
    if (prof) {
        cudaEventRecord(idx->prof_ev[2 * idx->prof_n + 1], ctx->stream);
        idx->prof_n++;
    }
    ctx->launches += 2;
    idx->last_h = n_half * 128;
    return NAFP_OK;
}

// exact re-rank + proof of every pass parked in slots [0, n_slots): one launch
static int select_batch(nafp_index* idx, const SelBatch& batch, int n_slots, int k, int grid_scan, int64_t n_search,
                        int32_t* fail_list, int32_t* fail_count, float* D_dev, int64_t* I_dev) {
    nafp_ctx* ctx = idx->ctx;
    flat_select_kernel<<<dim3(NQ_MAX, n_slots), 256, 0, ctx->stream>>>(batch, k, grid_scan, n_search, idx->q32, idx->qn2, idx->x32,
                                                                       idx->hn, idx->maxn2, idx->Tg, idx->pool, idx->cnt, idx->flags,
                                                                       idx->gidx, fail_list, fail_count, idx->label_offset, D_dev,
                                                                       I_dev, idx->stats);
    ctx->launches++;
    return NAFP_OK;
}

// Exact top-k of nq query rows.  Asynchronous on the ctx stream except for ONE 8-byte read-back at
// the end (how many rows the bf16 bound could not prove); those rows -- ~0.02 % on the synthetic
// workloads -- get a second scan pass with a much lower shared threshold (kg = all CTAs), and only
// what still cannot be proven (duplicates, pathological ties) goes to the exact CUDA-core scan.
int flat_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    nafp_ctx* ctx = idx->ctx;
    NAFP_REQUIRE(k >= 1 && k <= MAX_K, NAFP_ERR_INVALID, "search: k=%d outside [1,%d]", k, MAX_K);
    NAFP_REQUIRE(idx->d == D128, NAFP_ERR_UNSUPPORTED, "search: d=%d (the tensor-core scan is built for d=128)", idx->d);
    NAFP_REQUIRE(idx->scan_copy, NAFP_ERR_STATE, "search: this index keeps no bf16 scan copy of its rows (IVF-PQ types)");
    NAFP_REQUIRE(nq < (1ll << 31), NAFP_ERR_INVALID, "search: more than 2^31 query rows in one call");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_TRY(ensure_scratch(idx));
    if (nq == 0) return NAFP_OK;
    const int64_t n_search = (idx->search_rows >= 0 && idx->search_rows < idx->n) ? idx->search_rows : idx->n;
    const int n_tiles = static_cast<int>((n_search + SCAN_TILE - 1) / SCAN_TILE);
    const int kg = k + 28;
    // CTA pairs: at most one per tile.  grid_scan is also the number of maxima the thresholds are taken from
    const int grid_scan = 2 * std::max(1, std::min(n_tiles, idx->grid / 2));
    const bool brute = (n_search < 8192) || (kg > grid_scan) || (k > 64);
    idx->host_rows += nq;
    if (brute) return brute_rounds(idx, q_dev, nullptr, 0, nq, k, n_search, D_dev, I_dev);

    if (idx->fail_cap < 2 * nq) {
        if (idx->fail_list) cudaFree(idx->fail_list);
        idx->fail_list = nullptr;
        idx->fail_cap = 0;
        NAFP_CUDA(cudaMalloc(&idx->fail_list, static_cast<size_t>(2 * nq + 2) * sizeof(int32_t)));
        idx->fail_cap = 2 * nq;
    }
    int32_t* list1 = idx->fail_list;                 // rows that failed the first pass
    int32_t* list2 = idx->fail_list + nq;            // rows that failed the retry pass too
    int32_t* counts = idx->fail_list + 2 * nq;       // [2]
    NAFP_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), ctx->stream));
    SelBatch batch;
    batch.grid_alloc = idx->grid;
    int slot = 0;
    for (int64_t p0 = 0; p0 < nq; p0 += NQ_MAX) {
        const int np = static_cast<int>(nq - p0 < NQ_MAX ? nq - p0 : NQ_MAX);
        NAFP_TRY(scan_pass(idx, q_dev, nullptr, 0, p0, np, kg, grid_scan, n_tiles, n_search, slot));
        batch.h[slot] = idx->last_h;
        batch.np[slot++] = np;
        idx->host_passes++;
        if (slot == SEL_SLOTS || p0 + NQ_MAX >= nq) {
            NAFP_TRY(select_batch(idx, batch, slot, k, grid_scan, n_search, list1, counts, D_dev, I_dev));
            slot = 0;
        }
    }
    NAFP_CUDA(cudaGetLastError());
    int32_t h[2] = {0, 0};
    NAFP_CUDA(cudaMemcpyAsync(h, counts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (h[0] > 0) {
        // second chance: a threshold about one spread of the per-source maxima lower (~2x the survivors)
        const int kg_retry = 2 * kg < grid_scan - 2 ? 2 * kg : (grid_scan - 2 > kg ? grid_scan - 2 : kg);
        slot = 0;
        for (int off = 0; off < h[0]; off += NQ_MAX) {
            const int np = h[0] - off < NQ_MAX ? h[0] - off : NQ_MAX;
            NAFP_TRY(scan_pass(idx, q_dev, list1, off, 0, np, kg_retry, grid_scan, n_tiles, n_search, slot));
            batch.h[slot] = idx->last_h;
            batch.np[slot++] = np;
            idx->host_passes++;
            if (slot == SEL_SLOTS || off + NQ_MAX >= h[0]) {
                NAFP_TRY(select_batch(idx, batch, slot, k, grid_scan, n_search, list2, counts + 1, D_dev, I_dev));
                slot = 0;
            }
        }
        NAFP_CUDA(cudaMemcpyAsync(h, counts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        if (h[1] > 0) NAFP_TRY(brute_rounds(idx, q_dev, list2, 0, h[1], k, n_search, D_dev, I_dev));
    }
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

}  // namespace nafp

using namespace nafp;

extern "C" {

int nafp_index_create(nafp_ctx* ctx, int type, int d, int nlist, int pq_m, int pq_nbits, nafp_index** out) {
    NAFP_REQUIRE(ctx && out, NAFP_ERR_INVALID, "nafp_index_create: NULL argument");
    *out = nullptr;
    NAFP_REQUIRE(type == NAFP_INDEX_FLAT_L2 || type == NAFP_INDEX_IVFPQ || type == NAFP_INDEX_IVF_FLAT || type == NAFP_INDEX_IVFPQR,
                 NAFP_ERR_UNSUPPORTED, "nafp_index_create: index type %d is not built (l2, ivfpq, ivf, ivfpq-rr)", type);
    NAFP_REQUIRE(d == D128, NAFP_ERR_UNSUPPORTED, "nafp_index_create: d=%d; only d=128 (MODEL.EMB_SZ) is built", d);
    NAFP_CUDA(cudaSetDevice(ctx->device));
    nafp_index* idx = new nafp_index();
    idx->ctx = ctx;
    idx->type = type;
    idx->d = d;
    idx->scan_copy = type == NAFP_INDEX_FLAT_L2 || type == NAFP_INDEX_IVF_FLAT;
    if (cudaMalloc(&idx->maxn2, sizeof(int32_t)) != cudaSuccess ||
        cudaMemsetAsync(idx->maxn2, 0, sizeof(int32_t), ctx->stream) != cudaSuccess) {
        set_error("nafp_index_create: cudaMalloc failed");
        delete idx;
        return NAFP_ERR_CUDA;
    }
    if (type != NAFP_INDEX_FLAT_L2) {
        int s = type == NAFP_INDEX_IVF_FLAT ? ivfflat_create(idx, nlist) : ivfpq_create(idx, nlist, pq_m, pq_nbits);
        if (s == NAFP_OK && type == NAFP_INDEX_IVFPQR) s = ivfpqr_enable(idx);
        if (s != NAFP_OK) {
            if (idx->ivf) ivfpq_destroy(idx);
            cudaFree(idx->maxn2);
            delete idx;
            return s;
        }
    }
    *out = idx;
    return NAFP_OK;
}

int nafp_index_destroy(nafp_index* idx) {
    if (!idx) return NAFP_OK;
    cudaSetDevice(idx->ctx->device);
    cudaStreamSynchronize(idx->ctx->stream);
    if (idx->ivf) ivfpq_destroy(idx);
    for (auto& e : idx->prof_ev) cudaEventDestroy(e);
    void* bufs[] = {idx->x32, idx->x16, idx->hn, idx->tile_counter, idx->maxn2, idx->qbf, idx->q32, idx->qn2, idx->Mx, idx->Tg,
                    idx->pool, idx->cnt, idx->flags, idx->gidx, idx->fail_list, idx->brute_part, idx->stats, idx->stage_q, idx->stage_D,
                    idx->stage_I};
    for (void* b : bufs)
        if (b) cudaFree(b);
    delete idx;
    return NAFP_OK;
}

int nafp_index_train(nafp_index* idx, const float* x_host, int64_t n, int64_t seed) {
    NAFP_RANGE("nafp_index_train");
    NAFP_REQUIRE(idx, NAFP_ERR_INVALID, "nafp_index_train: idx is NULL");
    if (idx->type == NAFP_INDEX_FLAT_L2) return NAFP_OK;
    NAFP_REQUIRE(x_host && n > 0, NAFP_ERR_INVALID, "nafp_index_train: empty training set");
    return ivfpq_train(idx, x_host, n, seed);
}

int nafp_index_is_trained(nafp_index* idx);

static int add_common(nafp_index* idx, const float* x, int64_t n, bool host) {
    NAFP_REQUIRE(idx && (n == 0 || x) && n >= 0, NAFP_ERR_INVALID, "nafp_index_add: bad arguments");
    NAFP_REQUIRE(idx->n + n < (1ll << 32), NAFP_ERR_UNSUPPORTED, "nafp_index_add: more than 2^32 rows per shard");
    if (idx->type != NAFP_INDEX_FLAT_L2)
        NAFP_REQUIRE(nafp_index_is_trained(idx) == 1, NAFP_ERR_STATE, "nafp_index_add: IVF index is not trained");
    const int64_t row0 = idx->n;
    NAFP_TRY(flat_add_dev(idx, x, n, host));
    if (idx->type != NAFP_INDEX_FLAT_L2) NAFP_TRY(ivfpq_add_rows(idx, row0, n));
    return NAFP_OK;
}
int nafp_index_add(nafp_index* idx, const float* x_host, int64_t n) {
    NAFP_RANGE("nafp_index_add");
    return add_common(idx, x_host, n, true);
}
int nafp_index_add_dev(nafp_index* idx, const float* x_dev, int64_t n) {
    NAFP_RANGE("nafp_index_add_dev");
    return add_common(idx, x_dev, n, false);
}

int nafp_index_reserve(nafp_index* idx, int64_t n_total) {
    NAFP_REQUIRE(idx && n_total >= 0, NAFP_ERR_INVALID, "nafp_index_reserve: bad arguments");
    NAFP_CUDA(cudaSetDevice(idx->ctx->device));
    return index_reserve(idx, n_total);
}

int64_t nafp_index_ntotal(nafp_index* idx) { return idx ? idx->n : 0; }

int nafp_index_set_nprobe(nafp_index* idx, int nprobe) {
    NAFP_REQUIRE(idx && nprobe >= 1, NAFP_ERR_INVALID, "nafp_index_set_nprobe: bad arguments");
    idx->nprobe = nprobe;
    return NAFP_OK;
}
int nafp_index_set_search_rows(nafp_index* idx, int64_t n_rows) {
    NAFP_REQUIRE(idx, NAFP_ERR_INVALID, "nafp_index_set_search_rows: idx is NULL");
    idx->search_rows = n_rows;
    return NAFP_OK;
}
int nafp_index_set_label_offset(nafp_index* idx, int64_t offset) {
    NAFP_REQUIRE(idx, NAFP_ERR_INVALID, "nafp_index_set_label_offset: idx is NULL");
    idx->label_offset = offset;
    return NAFP_OK;
}

int nafp_index_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev) {
    NAFP_RANGE("nafp_index_search_dev");
    NAFP_REQUIRE(idx && nq >= 0 && (nq == 0 || (q_dev && D_dev && I_dev)), NAFP_ERR_INVALID,
                 "nafp_index_search_dev: bad arguments");
    if (idx->type != NAFP_INDEX_FLAT_L2) return ivfpq_search_dev(idx, q_dev, nq, k, D_dev, I_dev);
    return flat_search_dev(idx, q_dev, nq, k, D_dev, I_dev);
}

int nafp_index_search(nafp_index* idx, const float* q_host, int64_t nq, int k, float* D_host, int64_t* I_host) {
    NAFP_RANGE("nafp_index_search");
    NAFP_REQUIRE(idx && nq >= 0 && (nq == 0 || (q_host && D_host && I_host)), NAFP_ERR_INVALID,
                 "nafp_index_search: bad arguments");
    NAFP_REQUIRE(k >= 1 && k <= MAX_K, NAFP_ERR_INVALID, "search: k=%d outside [1,%d]", k, MAX_K);
    if (nq == 0) return NAFP_OK;
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    if (idx->stage_q_rows < nq) {
        if (idx->stage_q) cudaFree(idx->stage_q);
        idx->stage_q = nullptr;
        idx->stage_q_rows = 0;
        NAFP_CUDA(cudaMalloc(&idx->stage_q, static_cast<size_t>(nq) * idx->d * sizeof(float)));
        idx->stage_q_rows = nq;
    }
    if (idx->stage_out_elems < nq * k) {
        if (idx->stage_D) cudaFree(idx->stage_D);
        if (idx->stage_I) cudaFree(idx->stage_I);
        idx->stage_D = nullptr;
        idx->stage_I = nullptr;
        idx->stage_out_elems = 0;
        NAFP_CUDA(cudaMalloc(&idx->stage_D, static_cast<size_t>(nq) * k * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&idx->stage_I, static_cast<size_t>(nq) * k * sizeof(int64_t)));
        idx->stage_out_elems = nq * k;
    }
    NAFP_CUDA(cudaMemcpyAsync(idx->stage_q, q_host, static_cast<size_t>(nq) * idx->d * sizeof(float),
                              cudaMemcpyHostToDevice, ctx->stream));
    NAFP_TRY(nafp_index_search_dev(idx, idx->stage_q, nq, k, idx->stage_D, idx->stage_I));
    NAFP_CUDA(cudaMemcpyAsync(D_host, idx->stage_D, static_cast<size_t>(nq) * k * sizeof(float), cudaMemcpyDeviceToHost,
                              ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(I_host, idx->stage_I, static_cast<size_t>(nq) * k * sizeof(int64_t),
                              cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

int nafp_index_reconstruct_host(nafp_index* idx, int64_t i0, int64_t n, float* out_host) {
    NAFP_RANGE("nafp_index_reconstruct_host");
    NAFP_REQUIRE(idx && out_host && i0 >= 0 && n >= 0 && i0 + n <= idx->n, NAFP_ERR_INVALID,
                 "nafp_index_reconstruct_host: range [%lld, %lld) outside [0, %lld)", (long long)i0,
                 (long long)(i0 + n), (long long)(idx ? idx->n : 0));
    if (n == 0) return NAFP_OK;
    NAFP_CUDA(cudaMemcpyAsync(out_host, idx->x32 + i0 * idx->d, static_cast<size_t>(n) * idx->d * sizeof(float),
                              cudaMemcpyDeviceToHost, idx->ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(idx->ctx->stream));
    return NAFP_OK;
}

int nafp_index_profile_scans(nafp_index* idx, int enable, double* total_ms, int64_t* n_scans) {
    // enable != 0: start timing every scan-kernel launch with CUDA events on the ctx stream;
    // then (any value): report and reset what was collected since the previous call
    NAFP_REQUIRE(idx, NAFP_ERR_INVALID, "nafp_index_profile_scans: idx is NULL");
    nafp_ctx* ctx = idx->ctx;
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    double sum = 0.0;
    for (int64_t i = 0; i < idx->prof_n; ++i) {
        float ms = 0.f;
        NAFP_CUDA(cudaEventElapsedTime(&ms, idx->prof_ev[2 * i], idx->prof_ev[2 * i + 1]));
        sum += ms;
    }
    if (total_ms) *total_ms = sum;
    if (n_scans) *n_scans = idx->prof_n;
    idx->prof_n = 0;
    if (enable && idx->prof_ev.empty()) {
        idx->prof_ev.resize(2 * PROF_RING);
        for (auto& e : idx->prof_ev) NAFP_CUDA(cudaEventCreate(&e));
    }
    idx->profile = enable != 0;
    return NAFP_OK;
}

int nafp_index_last_search_stats(nafp_index* idx, int64_t* out4) {
    NAFP_REQUIRE(idx && out4, NAFP_ERR_INVALID, "nafp_index_last_search_stats: bad arguments");
    for (int i = 0; i < 8; ++i) out4[i] = 0;
    if (idx->ivf && idx->type != NAFP_INDEX_IVF_FLAT) {     // IVF-PQ: rows searched, rows answered by the LUT kernel, list-major work items / tiles
        ivfpq_take_stats(idx, out4);
        return NAFP_OK;
    }
    if (!idx->stats) return NAFP_OK;
    unsigned long long h[8];
    NAFP_CUDA(cudaMemcpyAsync(h, idx->stats, sizeof(h), cudaMemcpyDeviceToHost, idx->ctx->stream));
    NAFP_CUDA(cudaMemsetAsync(idx->stats, 0, sizeof(h), idx->ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(idx->ctx->stream));
    for (int i = 0; i < 8; ++i) out4[i] = static_cast<int64_t>(h[i]);
    out4[0] = idx->host_rows;
    out4[2] = idx->host_passes;
    idx->host_rows = idx->host_passes = 0;
    return NAFP_OK;
}

}  // extern "C"
