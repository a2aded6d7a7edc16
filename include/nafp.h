/*
 * nafp.h -- C ABI of libnafp.so: the B200 (sm_100a) fingerprinting + retrieval hot path of
 * mimbres/neural-audio-fp, as a drop-in for the native work the reference reaches through
 * TensorFlow/kapre (extractor) and faiss (index).  The reference has no FFI of its own (it is
 * pure Python over third-party wheels), so each entry point cites the reference *call site*
 * whose native work it replaces (paths relative to the reference tree).
 *
 * Conventions
 *   - every function returns 0 on success, a negative nafp_status on error;
 *     nafp_last_error() returns a thread-local message for the last failing call.
 *   - plain pointers and sizes only; all counts are int64_t; no exceptions cross the ABI.
 *   - `*_dev` pointers are device memory on the ctx's GPU, `*_host` pointers are host memory.
 *     The library never frees caller memory.  Calls taking device pointers are asynchronous on
 *     the ctx stream (nafp_sync to wait); calls taking host pointers return when the result is
 *     in the host buffer.
 *   - one nafp_ctx per (process, GPU); a ctx is not thread-safe, different ctxs are independent.
 */
#ifndef NAFP_H_
#define NAFP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nafp_ctx nafp_ctx;
typedef struct nafp_index nafp_index;

typedef enum {
    NAFP_OK = 0,
    NAFP_ERR_INVALID = -1,    /* bad argument */
    NAFP_ERR_CUDA = -2,       /* CUDA runtime / driver error (message has the CUDA string) */
    NAFP_ERR_STATE = -3,      /* call out of order (e.g. search before train/add, no weights) */
    NAFP_ERR_UNSUPPORTED = -4 /* valid in the reference but outside the hot path built here */
} nafp_status;

enum { NAFP_INDEX_FLAT_L2 = 0, NAFP_INDEX_IVFPQ = 1, NAFP_INDEX_IVF_FLAT = 2, NAFP_INDEX_IVFPQR = 3 };

/* ------------------------------------------------------------------ library / context */
int nafp_version(void);
const char* nafp_last_error(void);
/* number of CUDA devices visible, or a negative status when the driver is unusable */
int nafp_device_count(void);

int nafp_ctx_create(int device, nafp_ctx** out);
int nafp_ctx_destroy(nafp_ctx* ctx);
int nafp_sync(nafp_ctx* ctx);
/* the ctx's cudaStream_t (so a host can record CUDA events on the launching stream) */
void* nafp_ctx_stream(nafp_ctx* ctx);
/* adopt an external stream (e.g. torch's current stream) for all later work of this ctx;
 * NULL restores the ctx's own stream */
int nafp_ctx_set_stream(nafp_ctx* ctx, void* cuda_stream);
/* kernels launched by this library through this ctx since creation (bench "gpu_launches") */
int64_t nafp_ctx_launch_count(nafp_ctx* ctx);

/* device / pinned-host memory helpers so a host needs nothing but this library */
int nafp_malloc(nafp_ctx* ctx, int64_t bytes, void** out_dev);
int nafp_free(nafp_ctx* ctx, void* dev);
int nafp_malloc_host(nafp_ctx* ctx, int64_t bytes, void** out_host); /* pinned */
int nafp_free_host(nafp_ctx* ctx, void* host);
int nafp_memcpy_h2d(nafp_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes); /* async */
int nafp_memcpy_d2h(nafp_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes); /* async */
/* CUDA-event timing on the ctx stream: ms between the two marks (syncs on the second) */
int nafp_timer_start(nafp_ctx* ctx);
int nafp_timer_stop(nafp_ctx* ctx, float* out_ms);

/* ------------------------------------------------------------------ synthetic inputs
 * Seeded, counter-based generators for the shapes BASELINE.json names (no datasets offline; the
 * full-scale inputs are far too large to stage from the host).  Row / segment i depends only on
 * (seed, i), so any shard regenerates its own slice.  Measurement and test infrastructure. */
/* unit-norm 128-d rows with AR(1) correlation `rho` inside `track_len`-row tracks -> out_dev (n_rows,128) */
int nafp_synth_fp_rows(nafp_ctx* ctx, int64_t seed, int64_t row0, int64_t n_rows, int32_t track_len,
                       float rho, float* out_dev);
/* one-second 8 kHz "music-like" segments -> out_dev (n_seg, 8000) float32 */
int nafp_synth_audio(nafp_ctx* ctx, int64_t seed, int64_t seg0, int64_t n_seg, float* out_dev);

/* ------------------------------------------------------------------ extractor
 * Replaces the native work behind `test_step(X, m_pre, m_fp)` (model/generate.py:83-88):
 * Melspec_layer.call (model/fp/melspec/melspectrogram.py:102-112) and FingerPrinter.call
 * (model/fp/nnfp.py:224-231).
 */

/* Weights of the FingerPrinter (model/fp/nnfp.py:48-71,132-151), host pointers, float32:
 *   conv_w[l]  HWIO kernel of conv l (l = 2*i for the 1x3 conv of ConvLayer i, 2*i+1 for its 3x1)
 *              i.e. 3*Cin*Cout floats laid out [tap][cin][cout]
 *   conv_b[l]  Cout floats
 *   ln_g[l], ln_b[l]  LayerNormalization gamma/beta of that conv's output, F*T*C floats, (F,T,C) order
 *   div_w1 (128,8,32) div_b1 (128,32) div_w2 (128,32,1) div_b2 (128,1)
 * The library converts and keeps its own device copies. */
int nafp_weights_load(nafp_ctx* ctx, const float* const* conv_w, const float* const* conv_b,
                      const float* const* ln_g, const float* const* ln_b, const float* div_w1,
                      const float* div_b1, const float* div_w2, const float* div_b2);

/* MODEL.BN of the weights (model/fp/nnfp.py:20-83: ConvLayer(norm=...)), TF 2.4 Keras semantics, eps 1e-3:
 *   NAFP_NORM_LAYER_NORM2D  LayerNormalization(axis=(1,2,3)): gamma / beta (F,T,C)      = nafp_weights_load
 *   NAFP_NORM_LAYER_NORM1D  LayerNormalization(axis=-1): over the C channels of each position, gamma / beta (C)
 *   NAFP_NORM_BATCH_NORM    BatchNormalization(axis=-1) in inference mode (test_step sets trainable = False):
 *                           gamma, beta, moving mean, moving variance (C) */
enum { NAFP_NORM_LAYER_NORM2D = 0, NAFP_NORM_LAYER_NORM1D = 1, NAFP_NORM_BATCH_NORM = 2 };

/* nafp_weights_load for any MODEL.BN: norm_g[l] / norm_b[l] hold F*T*C floats for NAFP_NORM_LAYER_NORM2D and C floats
 * otherwise; norm_mean / norm_var (C floats per layer) are given for NAFP_NORM_BATCH_NORM and NULL otherwise.  The
 * norm belongs to the loaded weights: the next load replaces it.  A failed load leaves no usable weights. */
int nafp_weights_load_norm(nafp_ctx* ctx, int32_t norm, const float* const* conv_w, const float* const* conv_b,
                           const float* const* norm_g, const float* const* norm_b, const float* const* norm_mean,
                           const float* const* norm_var, const float* div_w1, const float* div_b1,
                           const float* div_w2, const float* div_b2);

/* Log-mel front end.  x_dev: (n_seg, 8000) float32 segments (the (B,1,8000) batches of
 * model/generate.py:178 flattened).  Rows are processed in consecutive groups of `group_size`
 * (= BSZ.TS_BATCH_SZ; the last group may be partial), each group sharing the batch-global max
 * of melspectrogram.py:108.  mel_dev: (n_seg, 256, 32) float32, element [b,f,t] -- the
 * (B,256,32,1) tensor the reference hands to the encoder. */
int nafp_logmel_forward(nafp_ctx* ctx, const float* x_dev, int64_t n_seg, int64_t group_size,
                        float* mel_dev);

/* The same without the finishing pass: raw log10(mel + 0.06) and the per-group maxima (int32 per group: the float
 * maximum in an order-preserving integer encoding; may be NULL) -- what the fused nafp_fingerprint path hands to the
 * encoder's first layer, which applies "- max, clamp -80" itself.  Timed by bench.py for the log-mel roofline. */
int nafp_logmel_forward_raw(nafp_ctx* ctx, const float* x_dev, int64_t n_seg, int64_t group_size,
                            float* mel_dev, int32_t* group_max_dev);

/* MODEL.FEAT (config/default.yaml:38): enable != 0 selects 'melspec_maxnorm' = Melspec_layer(segment_norm=True)
 * (melspectrogram.py:110-111: x = (x - min/2) / |min/2 + 1e-10| over the batch tensor, after the max subtraction and
 * the clamp) for nafp_logmel_forward and the nafp_fingerprint* entry points of this ctx; 0 (default) = 'melspec'. */
int nafp_logmel_set_segment_norm(nafp_ctx* ctx, int32_t enable);

/* FingerPrinter encoder: mel_dev (n_seg,256,32) float32 -> emb_dev (n_seg,128) float32,
 * L2-normalised (model/fp/nnfp.py:224-231).  Requires nafp_weights_load. */
int nafp_encoder_forward(nafp_ctx* ctx, const float* mel_dev, int64_t n_seg, float* emb_dev);

/* test_step: logmel + encoder.  Device buffers, async. */
int nafp_fingerprint(nafp_ctx* ctx, const float* x_dev, int64_t n_seg, int64_t group_size,
                     float* emb_dev);
/* test_step with host buffers (what `emb = test_step(X,...); emb.numpy()` does,
 * model/generate.py:179-180): H2D of x_host, compute, D2H into emb_host, returns when done. */
int nafp_fingerprint_host(nafp_ctx* ctx, const float* x_host, int64_t n_seg, int64_t group_size,
                          float* emb_host);
/* int16 PCM variant: applies the reference's x / 2**15 (model/utils/audio_utils.py:243-244) on
 * the device; pcm_host is (n_seg, 8000) int16. */
int nafp_fingerprint_pcm16_host(nafp_ctx* ctx, const int16_t* pcm_host, int64_t n_seg,
                                int64_t group_size, float* emb_host);
/* The same for whole-track sample runs: pcm_host holds n_samples int16 samples (tracks back to back); segment s is
 * the window [seg_off[s], seg_off[s] + 8000) of it, of which the first seg_valid[s] (<= 8000) samples are real and
 * the rest is zero padding (get_fns_seg_list / load_audio, model/utils/audio_utils.py:140-264, with the 0.5 s hop
 * applied on the device: overlapping segments are uploaded once). */
int nafp_fingerprint_pcm16_tracks_host(nafp_ctx* ctx, const int16_t* pcm_host, int64_t n_samples,
                                       const int64_t* seg_off_host, const int32_t* seg_valid_host,
                                       int64_t n_seg, int64_t group_size, float* emb_host);
/* Debug/parity taps: activation of conv `layer` (0..15) after its normalisation (any MODEL.BN) for the LAST
 * nafp_encoder_forward call, as float32 (n_seg, F, T, C) into out_host. */
int nafp_encoder_activation_host(nafp_ctx* ctx, int layer, int64_t n_seg, float* out_host);

/* ------------------------------------------------------------------ index
 * Replaces the object returned by get_index() (eval/utils/get_index_faiss.py:10-121) for
 * index_type 'l2' (faiss.IndexFlatL2, :58), 'ivfpq' (faiss.IndexIVFPQ(flat,d,256,64,8), :69-74),
 * 'ivf' (faiss.IndexIVFFlat(flat,d,400), :63-66; pq_m / pq_nbits are ignored for it) and 'ivfpq-rr'
 * (faiss.IndexIVFPQR, :75-85: the IVF-PQ search for 4 k candidates, re-ranked with a 4 x 4-bit refinement quantizer).
 */
int nafp_index_create(nafp_ctx* ctx, int type, int d, int nlist, int pq_m, int pq_nbits,
                      nafp_index** out);
int nafp_index_destroy(nafp_index* idx);
/* index.train(x) (get_index_faiss.py:113,116): no-op for FLAT_L2; k-means for IVFPQ / IVF_FLAT. */
int nafp_index_train(nafp_index* idx, const float* x_host, int64_t n, int64_t seed);
/* index.add(x) (eval/eval_faiss.py:147-148): appends n rows; labels are insertion order. */
int nafp_index_add(nafp_index* idx, const float* x_host, int64_t n);
int nafp_index_add_dev(nafp_index* idx, const float* x_dev, int64_t n);
/* IVF-PQ only: export / import the trained quantizers (coarse (nlist,128), pq (M,256,128/M), float32),
 * e.g. to reuse one training across shards; import is only allowed on an empty index. */
int nafp_index_ivfpq_get_params(nafp_index* idx, float* coarse_host, float* pq_host);
int nafp_index_ivfpq_set_params(nafp_index* idx, const float* coarse_host, const float* pq_host);
/* IVFPQR ('ivfpq-rr', faiss.IndexIVFPQR(flat, d, 256, 64, 8, M_refine 4, nbits_refine 4), get_index_faiss.py:75-85):
 * the refinement codebooks ((4, 16, 32) float32) in addition to nafp_index_ivfpq_get/set_params. */
int nafp_index_ivfpqr_get_refine(nafp_index* idx, float* refine_pq_host);
int nafp_index_ivfpqr_set_refine(nafp_index* idx, const float* refine_pq_host);
/* The two levels of an IVFPQR search, for a row-sharded index whose shards must return what one index over all rows
 * returns: (1) every shard's first-level top kc (= 4 k) by ADC distance, all-gathered and merged by
 * nafp_topk_merge_dev into the global top kc; (2) every shard re-ranks the merged candidates whose labels it owns
 * (its searched rows) by |q - (xhat + rhat)|^2 and returns its own sorted top k (+inf / -1 padding); those
 * lists merge into the global top k.  nafp_index_search_dev runs both on one index.  kc <= 128. */
int nafp_index_ivfpqr_first_level_dev(nafp_index* idx, const float* q_dev, int64_t nq, int kc, float* D_dev,
                                      int64_t* I_dev);
int nafp_index_ivfpqr_rerank_dev(nafp_index* idx, const float* q_dev, int64_t nq, const int64_t* candI_dev, int kc,
                                 int k, float* D_dev, int64_t* I_dev);
/* IVF-Flat and IVF-PQ: the coarse quantizer alone ((nlist,128) float32); import only on an empty index
 * (an IVF-Flat index counts as trained afterwards). */
int nafp_index_ivf_get_coarse(nafp_index* idx, float* coarse_host);
int nafp_index_ivf_set_coarse(nafp_index* idx, const float* coarse_host);
/* pre-size the device store (optional; avoids regrowth copies for very large databases) */
int nafp_index_reserve(nafp_index* idx, int64_t n_total);
int64_t nafp_index_ntotal(nafp_index* idx);
int nafp_index_is_trained(nafp_index* idx);
/* index.nprobe = v (get_index_faiss.py:120); ignored by FLAT_L2 */
int nafp_index_set_nprobe(nafp_index* idx, int nprobe);
/* labels returned by search are local_row + label_offset (row-sharded multi-GPU databases) */
int nafp_index_set_label_offset(nafp_index* idx, int64_t offset);
/* only the first n_rows rows take part in search; later rows (the halo copied from the next shard)
 * are only reconstructed / sequence-scored.  -1 = all rows. */
int nafp_index_set_search_rows(nafp_index* idx, int64_t n_rows);

/* D, I = index.search(q, k) (eval/eval_faiss.py:211): squared-L2 distances ascending, int64
 * labels, -1 / +inf padding when fewer than k rows exist.  k <= 128. */
int nafp_index_search(nafp_index* idx, const float* q_host, int64_t nq, int k, float* D_host,
                      int64_t* I_host);
int nafp_index_search_dev(nafp_index* idx, const float* q_dev, int64_t nq, int k, float* D_dev,
                          int64_t* I_dev);
/* index.reconstruct_n(i0, n) -> (n,d) float32 (the reference's fake_recon_index rows,
 * eval/eval_faiss.py:167-171, without touching dummy_db.mm on disk). FLAT_L2 only. */
int nafp_index_reconstruct_host(nafp_index* idx, int64_t i0, int64_t n, float* out_host);
/* counters since the previous call of this function, out8[0..7]: [0] query rows, [1] rows answered
 * by the exact fp32 fallback scan, [2] scan passes, [3] candidates re-ranked in fp32,
 * [5] fallback rows due to candidate-pool overflow / small database, [6] fallback rows because
 * the bf16 error bound could not prove the top-k, [4],[7] reserved. */
int nafp_index_last_search_stats(nafp_index* idx, int64_t* out8);

/* CUDA-event timing of the scan kernel alone, on the launching stream (bench roofline):
 * enable != 0 arms it; every call returns and resets the summed duration / launch count since the
 * previous call (at most 8192 launches are recorded between calls). */
int nafp_index_profile_scans(nafp_index* idx, int enable, double* total_ms, int64_t* n_scans);

/* developer probe of the last flat scan pass (512 entries each, one per query row of a pass): fallback flags,
 * shared thresholds, survivors per query row */
int nafp_index_debug_last_pass(nafp_index* idx, int32_t* flags512, float* thr512, int32_t* total512);
/* developer probe: per-CTA survivor counts [grid][512] (0 where a CTA does not hold the query row) and the tile index
 * at which each CTA first saw a shared threshold per query row [grid][512] (-1 = never; entries 504..511 are in-kernel
 * timestamps when the pass has <= 504 rows); the first call arms the probe */
int nafp_index_debug_enable(nafp_index* idx, int32_t* cnt_out, int32_t* first_out, int32_t* grid_out);

/* ------------------------------------------------------------------ sequence matcher
 * Replaces the body of the hot loop eval/eval_faiss.py:204-232 for a batch of test ids.
 *   q_host      (n_query_rows, d) float32 -- the whole `query` memmap (or a slice)
 *   test_ids    n_test start rows into q
 *   seq_lens    n_len sequence lengths (each <= 32)
 * For every (test id, sl): q = query[id : id+sl] (clamped at n_query_rows, :208); top-k_probe
 * segment search (:211); offset compensation (:215-216); unique candidates >= 0 (:219);
 * score = mean_j q[j].recon[c+j] over the rows that exist (:222-229); the 10 best by score,
 * ties to the lower id (:232).  recon = this index's rows (flat) -- [dummy_db; db].
 * Outputs: pred_ids_host (n_test, n_len, 10) int64 (-1 padded), pred_scores_host same shape
 * float32 (may be NULL). */
int nafp_seq_match(nafp_index* idx, const float* q_host, int64_t n_query_rows,
                   const int64_t* test_ids, int64_t n_test, const int32_t* seq_lens, int32_t n_len,
                   int32_t k_probe, int64_t* pred_ids_host, float* pred_scores_host);

/* Building blocks of nafp_seq_match on device buffers, for a database row-sharded over several
 * GPUs (SURVEY §8 e): each rank searches its shard, the host all-gathers the per-rank top-k
 * (NCCL), nafp_topk_merge_dev merges them, every rank scores the candidates it owns
 * (-inf for the others), the host max-reduces the score tables, nafp_seq_top_dev picks the 10 best.
 *   rowmap_dev       (n_test*max_len) int32: row of the search-result table for (test id, offset), -1 past the end
 *   uniq_rows_dev    the distinct query rows some (test id, offset) needs, ascending (capacity n_test*max_len)
 *   I_dev            (n_uniq, k_probe) merged global labels of those rows
 *   cand_ids_dev     (n_test, 1024) int64 sorted unique candidate start ids, -1 padded
 *   cand_scores_dev  (n_test, n_len, 1024) float32, -inf where not a member / not owned
 *   n_cand_dev       (n_test) int32 */
/* plan: overlapping query sequences share rows; each needed row is searched once.  scratch_dev holds
 * 2*n_query_rows+1 int32.  Synchronises once to return the number of unique rows. */
int nafp_seq_plan_dev(nafp_ctx* ctx, const int64_t* test_ids_dev, int64_t n_test, int32_t max_len,
                      int64_t n_query_rows, int32_t* scratch_dev, int32_t* rowmap_dev,
                      int32_t* uniq_rows_dev, int64_t* n_uniq_out);
int nafp_seq_gather_rows_dev(nafp_ctx* ctx, const float* q_dev, const int32_t* rows_dev, int64_t n_rows,
                             float* out_dev);
int nafp_seq_cand_dev(nafp_index* idx, const float* q_dev, int64_t n_query_rows,
                      const int64_t* test_ids_dev, int64_t n_test, const int32_t* seq_lens_dev,
                      int32_t n_len, int32_t max_len, int32_t k_probe, const int64_t* I_dev,
                      const int32_t* rowmap_dev, int64_t n_rows_global, int64_t owned_lo, int64_t owned_hi,
                      int64_t* cand_ids_dev, float* cand_scores_dev, int32_t* n_cand_dev);
int nafp_seq_top_dev(nafp_ctx* ctx, int64_t n_test, int32_t n_len, const int64_t* cand_ids_dev,
                     const float* cand_scores_dev, const int32_t* n_cand_dev,
                     int64_t* pred_ids_dev, float* pred_scores_dev);
/* merge n_shards top-k lists: D_all/I_all (n_shards, nq, k) -> (nq, k), ordered by (distance, label) */
int nafp_topk_merge_dev(nafp_ctx* ctx, const float* D_all_dev, const int64_t* I_all_dev,
                        int32_t n_shards, int64_t nq, int32_t k, float* D_out_dev, int64_t* I_out_dev);

/* ------------------------------------------------------------------ in-training mini search (SURVEY §8 f3)
 * Replaces the TensorFlow / numpy work of model/utils/mini_search_subroutines.py, called from
 * mini_search_validation (model/trainer.py:80-108).
 *   q_host   (n_q, n_aug, d) float32 query embeddings, db_host (n_db, d) float32 (d is 128 for g(f), 1024 for f). */
/* pairwise_distances_for_eval (:29-90): out_host (n_aug, n_q, n_db) float32 -- dot products when return_dotprod != 0,
 * else max(|a|^2 + |b|^2 - 2 a.b, 0), its square root (zeros kept) when squared == 0. */
int nafp_pairwise_dists_host(nafp_ctx* ctx, const float* q_host, const float* db_host, int64_t n_q, int64_t n_aug,
                             int64_t n_db, int64_t d, int32_t return_dotprod, int32_t squared, float* out_host);
/* conv_eye_func (:93-120): x_host (n_aug, n_q, n_db) -> out_host (n_aug, n_q-s+1, n_db-s+1),
 * out[a,i,j] = sum_{t<s} x[a,i+t,j+t] (Conv2D with an s x s identity kernel, 'valid'). */
int nafp_conv_eye_host(nafp_ctx* ctx, const float* x_host, int64_t n_aug, int64_t n_q, int64_t n_db, int32_t s,
                       float* out_host);
/* mini_search_eval (:123-236): for every scope s, target i < n_q-s+1 and augmentation a the rank of item
 * gt = i + gt_id_offset in argsort(conv[a,i,:]) (descending for argmax != 0, which works on dot products);
 * outputs per scope: top-1/3/10 accuracy in percent and the mean rank (doubles, n_scopes each). */
int nafp_mini_search_host(nafp_ctx* ctx, const float* q_host, const float* db_host, int64_t n_q, int64_t n_aug,
                          int64_t n_db, int64_t d, const int32_t* scopes, int32_t n_scopes, int32_t argmax,
                          int64_t gt_id_offset, double* top1, double* top3, double* top10, double* mean_rank);

#ifdef __cplusplus
}
#endif
#endif /* NAFP_H_ */
