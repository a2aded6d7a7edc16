// IVF-PQ state shared by ivfpq.cu (training, encoding, lists, LUT scan, IVF-Flat scan + filter) and ivfpq_lm.cu
// (the list-major compressed-domain tensor-core scan).
#pragma once
#include "index.h"

namespace nafp {

constexpr int PQ_MAX_M = 64;
constexpr int PQ_KSUB = 256;
constexpr int IVF_MAX_NLIST = 1024;
constexpr int REFINE_M = 4, REFINE_KSUB = 16, REFINE_DSUB = 32, REFINE_KFACTOR = 4;
constexpr int IVF_SCAN_CAP = 512;         // candidate buffer per (query, list) CTA: two 512-key sorts per list instead of two 1024-key ones

struct LmState;                       // ivfpq_lm.cu

struct IvfPq {
    bool lut_only = false;        // NAFP_IVFPQ_PATH=lut when the index was created: every search runs the LUT kernel
    LmState* lm = nullptr;        // list-major scan: per-position row terms, bf16 codebook table, work lists, candidates
    int nlist = 256, m = 64, dsub = 2;
    bool flat_lists = false;      // IVF-Flat: the lists hold the stored rows themselves (no product quantizer)
    bool trained = false;
    float* coarse = nullptr;      // [nlist][128]
    float* pq = nullptr;          // [m][256][dsub]
    int32_t* assign = nullptr;    // [cap] list of every row (row order)
    uint8_t* codes = nullptr;     // [cap][m]
    int64_t cap = 0;
    // list-sorted copy
    bool dirty = true;
    // Every list starts at a multiple of 128 positions (LIST_TILE); its codes are stored tile by tile, transposed for the
    // list-major scan (lcode_off): inside a tile of 128 positions, [K block = sub / 32][position / 4][sub % 32][position % 4]
    // bytes, so that a warp whose lanes are sub-quantizers reads the codes of 4 positions with one coalesced 128-byte
    // load and then indexes the codebook table of ITS sub-quantizer -- one shared-memory bank per lane, no conflicts.
    uint8_t* lcodes = nullptr;    // [padded positions][m], tile-transposed
    int32_t* lids = nullptr;      // [padded positions] row id, -1 = padding
    int32_t* loff = nullptr;      // [nlist + 1] first position of every list (multiples of 128)
    int32_t* lend = nullptr;      // [nlist] one past the last used position
    std::vector<int32_t> h_loff, h_lend;      // host copies (work lists of the list-major scan)
    int64_t lists_version = 0;    // bumped by every rebuild of the list-sorted copy
    int64_t sorted_cap = 0;
    // IVFPQR (index_type 'ivfpq-rr', get_index_faiss.py:75-85): second-level product quantizer of the first level's
    // residual x - xhat, M_refine 4 sub-spaces of 32 dims x 16 centroids (4 bit) = 2 bytes per row; the search asks the
    // IVF-PQ for k * k_factor (faiss default 4) candidates and re-ranks them by |q - (xhat + rhat)|^2
    bool refine = false;
    float* rpq = nullptr;         // [4][16][32]
    uint8_t* rcodes = nullptr;    // [cap][2]: nibbles (sub 0 | sub 1 << 4), (sub 2 | sub 3 << 4)
    float* refD = nullptr;        // [nq_cap][REFINE_K]
    int64_t* refI = nullptr;
    int64_t ref_nq = 0;
    // search scratch
    int32_t* probes = nullptr;    // [nq_cap][nprobe_cap]
    float* partD = nullptr;       // [nprobe][nq_cap][k]
    int64_t* partI = nullptr;
    int64_t scratch_nq = 0;
    int scratch_nprobe = 0, scratch_k = 0;
    // IVF-Flat: the flat scan of the stored rows gives IVFFLAT_K candidates per query row, the filter keeps the ones
    // in probed lists; rows it cannot answer are redone by an exact scan of their probed lists (ivfpq_redo_rows)
    float* candD = nullptr;       // [nq_cap][IVFFLAT_K]
    int64_t* candI = nullptr;
    int64_t cand_nq = 0;
    int32_t* probes_all = nullptr;    // [nq][nprobe] of the whole call
    int64_t probes_all_elems = 0;
    int32_t* redo_rows = nullptr; // query rows the filter or the list-major scan could not answer, + counter at [cap]
    float* redo_q = nullptr;      // gathered copies of those rows, and their results
    float* redo_D = nullptr;
    int64_t* redo_I = nullptr;
    int64_t redo_cap = 0;
    unsigned long long lut_rows = 0;      // rows answered by the LUT kernel since creation (statistics)
};
constexpr int IVFFLAT_K = 64;             // IVF-Flat candidates per query row, fetched from the flat scan



constexpr int LIST_TILE = 128;
// byte offset of the code of sub-quantizer `sub` of list position `pos` (m sub-quantizers per row)
__host__ __device__ __forceinline__ int64_t lcode_off(int64_t pos, int sub, int m) {
    const int mlo = m < 32 ? m : 32;
    const int r = static_cast<int>(pos & (LIST_TILE - 1));
    return (pos >> 7) * (LIST_TILE * m) + (sub / mlo) * (LIST_TILE * mlo) + (r >> 2) * (4 * mlo) + (sub % mlo) * 4 + (r & 3);
}

// ivfpq.cu
// the nprobe nearest coarse centroids of every row of q[nq][128] -> probes[nq][nprobe]; optionally their distances
// gdist[nq][nprobe] and the list-major scan's rounding bound qE[nq] (from dmax2).  One launch on ctx->stream.
int coarse_probe(nafp_ctx* ctx, const float* q, int64_t nq, const float* coarse, int nlist, int nprobe, int32_t* probes,
                 float* gdist = nullptr, float* qE = nullptr, const int32_t* dmax2 = nullptr);
int build_lists(nafp_index* idx);
int ivfpq_search_lut(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev);
int ivfpq_redo_rows(nafp_index* idx, const float* q_dev, int32_t n_redo, int k, float* D_dev, int64_t* I_dev);
int ivfpq_reserve_redo(nafp_index* idx, int64_t nq);
// ivfpq_lm.cu
int ivfpq_lm_supported(const nafp_index* idx, int k);
int ivfpq_search_lm(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev, int64_t* I_dev);
void ivfpq_lm_destroy(IvfPq* s);
void ivfpq_lm_take_stats(IvfPq* s, int64_t* items, int64_t* tiles);

}  // namespace nafp
