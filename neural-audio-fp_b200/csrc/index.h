// nafp_index: device-resident flat store (+ optional IVF-PQ structures) shared by
// flat_search.cu, ivfpq.cu and seq_match.cu.
#pragma once
#include <cuda_bf16.h>

#include "common.h"
#include <vector>

namespace nafp {

constexpr int D128 = 128;            // fingerprint dimension the tensor-core scan is built for
constexpr int NQ_MAX = 512;          // query rows per scan pass: one CTA pair, NQ_CTA rows per CTA
constexpr int NQ_CTA = 256;          // query rows of one scan CTA (two MMA M blocks of 128)
constexpr int TILE_ROWS = 128;       // DB rows per TMA box / allocation granule
constexpr int SCAN_TILE = 256;       // DB rows per scan tile (MMA N)
constexpr int POOL_CAP = 128;        // candidate slots per (CTA, query) per pass
constexpr int MAX_K = 128;
constexpr int BRUTE_CHUNKS = 296;        // CTAs per query of the exact fallback scan (2 per SM)
constexpr int BRUTE_SLOTS = 32;          // queries per fallback launch
constexpr int SELECT_CAP = 4096;     // candidates re-ranked in fp32 per query, at most
constexpr int SEL_SLOTS = 16;        // scan passes whose survivors are re-ranked by ONE flat_select launch

struct IvfPq;                        // ivfpq.cu

}  // namespace nafp

struct nafp_index {
    nafp_ctx* ctx = nullptr;
    int type = 0;
    int d = 0;
    int64_t n = 0;            // rows stored
    int64_t cap = 0;          // rows allocated (multiple of TILE_ROWS)
    float* x32 = nullptr;             // [cap][d] exact rows (re-rank, reconstruct, sequence scoring)
    __nv_bfloat16* x16 = nullptr;     // [cap][d] scan copy
    float* hn = nullptr;              // [cap + SCAN_TILE] 0.5*|x|^2, +inf for unused rows
    int32_t* maxn2 = nullptr;         // device scalar: bits of max |x|^2 (non-negative float)
    bool scan_copy = true;            // x16 / hn exist (flat and IVF-Flat indexes; the IVF-PQ types search their codes)
    int64_t label_offset = 0;
    int64_t search_rows = -1;     // leading rows that take part in search (-1 = all); the rest are halo
    CUtensorMap tmap_db;
    CUtensorMap tmap_q;
    bool tmap_db_valid = false;

    // per-pass scratch (allocated on first search); q32 .. gidx hold SEL_SLOTS passes
    int last_h = 0;                   // query rows per CTA of the last scan pass
    bool scratch_ready = false;
    int grid = 0;                     // scan CTAs: 2 x the CTA pairs that fit on the device at once
    __nv_bfloat16* qbf = nullptr;     // [NQ_MAX][d]
    float* q32 = nullptr;             // [NQ_MAX][d] (pass-local copy, zero padded)
    float* qn2 = nullptr;             // [NQ_MAX]
    int32_t* Mx = nullptr;            // [NQ_MAX][grid] running max per (cluster, accumulator column half) (ordered int)
    int32_t* Tg = nullptr;            // [NQ_MAX] shared threshold (ordered int)
    uint64_t* pool = nullptr;         // [grid][NQ_CTA][POOL_CAP] per (CTA, local query row)
    int32_t* cnt = nullptr;           // [grid][NQ_CTA]
    int32_t* flags = nullptr;         // [NQ_MAX] != 0 -> answered by the exact fallback
    int64_t* gidx = nullptr;          // [NQ_MAX] global query row of every pass row
    int32_t* fail_list = nullptr;     // [2 nq + 2] rows to retry / to scan exactly, + the two counters
    int64_t fail_cap = 0;
    uint64_t* brute_part = nullptr;   // [BRUTE_SLOTS][BRUTE_CHUNKS][MAX_K]
    unsigned long long* stats = nullptr;   // [8] device counters
    int32_t* tile_counter = nullptr;  // device scalar: next DB tile the scan's producers draw
    // staging for the host entry points
    float* stage_q = nullptr;  int64_t stage_q_rows = 0;
    float* stage_D = nullptr;  int64_t* stage_I = nullptr;  int64_t stage_out_elems = 0;

    int64_t host_rows = 0, host_passes = 0;   // since the last nafp_index_last_search_stats

    // optional CUDA-event timing of every scan launch (bench roofline): ring of event pairs
    bool profile = false;
    std::vector<cudaEvent_t> prof_ev;     // [2 * PROF_RING]
    int64_t prof_n = 0;

    int nprobe = 1;
    nafp::IvfPq* ivf = nullptr;
};

namespace nafp {
int flat_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev);
int flat_add_dev(nafp_index* idx, const float* x_dev, int64_t n, bool src_is_host);
int index_reserve(nafp_index* idx, int64_t n_total);
// ivfpq.cu
int ivfpq_create(nafp_index* idx, int nlist, int m, int nbits);
int ivfflat_create(nafp_index* idx, int nlist);
int ivfpqr_enable(nafp_index* idx);       // IVFPQR: adds the refinement quantizer to a freshly created IVF-PQ state
void ivfpq_destroy(nafp_index* idx);
int ivfpq_train(nafp_index* idx, const float* x_host, int64_t n, int64_t seed);
int ivfpq_add_rows(nafp_index* idx, int64_t row0, int64_t n);
int ivfpq_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev);
void ivfpq_take_stats(nafp_index* idx, int64_t* out8);
}  // namespace nafp
