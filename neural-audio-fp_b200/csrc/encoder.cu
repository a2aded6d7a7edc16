// FingerPrinter encoder (SURVEY §8 a2-a4): the reference's model/fp/nnfp.py on B200.
//
// LayerNormalization over (F,T,C) with per-element gamma/beta sits between every two convolutions
// (nnfp.py:66-79).  A convolution is linear, so the normalisation of layer l is FOLDED THROUGH conv l+1:
//
//     LN_l(y)[p,ci]        = a (gamma[p,ci] y[p,ci]) + c gamma[p,ci] + beta[p,ci],   a = rstd, c = -rstd mean  (per segment)
//     conv_{l+1}(LN_l(y))  = a * conv(z) + c * Cg + Cb,      z = gamma (.) y,   Cg = conv(gamma),   Cb = bias + conv(beta)
//
// Every layer stores z = gamma (.) ELU(...) ONCE in fp16 (no pre-LN scratch, no normalise pass: the
// pre-LN -> LN round trip was 41 % of the encoder's HBM traffic), its epilogue accumulates the statistics of
// ELU(...), and the NEXT layer's epilogue applies (a, c) to its own accumulator.  Cg / Cb / gamma are
// per-(output position, channel) constants: tiles are handed out POSITION-STATIONARY (a CTA keeps one
// (position tile, channel tile) for all the segments it processes), so gamma and Cb live in the 256 TMEM columns
// the two 128-column accumulators leave free and Cg in 16 registers -- they are read from L2 once per launch.
//
//   conv0_kernel       1x3 conv with C_in = 1 (K = 3): CUDA cores, fused with the log-mel max subtraction /
//                      clamp, bias, ELU, statistics and the gamma scaling; one pass, one store.
//   ln_stats_kernel    partial sums -> (a, c) per segment (fixed order: fingerprints are bit-reproducible)
//   conv_gemm_kernel   the other 15 separable convolutions as implicit GEMMs on tcgen05:
//                      M = 128 output positions (NHWC rows), N = 128 channels, K = 3 taps x C_in.
//                      The A operand of each (tap, 64-channel block) is ONE TMA box of the previous
//                      layer's fp16 activation: stride-2 axes are split into (parity, half) dimensions of
//                      the tensor map, TF 'SAME' zero padding is TMA out-of-bounds fill.  Persistent CTAs,
//                      6-stage smem ring, fp32 accumulators double-buffered in TMEM, 16 epilogue warps;
//                      layers with K <= 384 keep their weights resident in shared memory.
//   fold_kernel        (weights load) Cg / Cb of every layer in fp64
//   ln1d_kernel        MODEL.BN 'layer_norm1d': per-position LayerNorm over C, in place (L1a: fused into conv0_kernel)
//   (MODEL.BN 'batch_norm' is the fold with constant factors, all layers split precision: nafp_weights_load_norm)
//   divenc_kernel      last LayerNorm + divide-and-encode head (128 x [8->32 ELU, 32->1]); l2norm_kernel.
// fp16 operands / fp32 accumulation; the six small layers from L6a on run split precision (hi + lo operands).
// Measured against the fp64 oracle the fingerprints agree to a few 1e-4 (gate: cosine >= 0.9999, max abs <= 1e-3).
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "common.h"
#include "ptx.cuh"

namespace nafp {

int logmel_run(nafp_ctx* ctx, const void* x_dev, bool pcm16, int64_t n_seg, int64_t group_size, float* mel_dev,
               bool finish, const int32_t** gmax_out, const int64_t* seg_off, const int32_t* seg_valid);
bool logmel_segment_norm(nafp_ctx* ctx);

constexpr int ENC_LAYERS = 16;
#ifndef NAFP_ENC_CHUNK_MAX
#define NAFP_ENC_CHUNK_MAX 4000
#endif
constexpr int ENC_CHUNK_MAX = NAFP_ENC_CHUNK_MAX;    // most segments of one encoder pass (2.3 MB of activations each): at 1,000 the
                                       // six last layers have fewer tiles than the chip has SMs
constexpr int ENC_CHUNK_MIN = 1000;    // the activation arena starts here and grows on demand (encoder_reserve)
constexpr int EMB = 128;
constexpr float LN_EPS = 1e-3f;        // Keras LayerNormalization default
constexpr float L2_EPS = 1e-12f;       // tf.math.l2_normalize default

struct ConvGeom {
    int axis, stride, pad_lo;          // axis 0 = time (1x3), 1 = frequency (3x1)
    int f_in, t_in, c_in, f_out, t_out, c_out;
    int ms;                            // output positions per segment
    int mode;                          // TMA addressing mode, see conv_gemm_kernel
    int tap_lo, tap_hi;                // taps that touch real data (others are all padding)
    int bt, bf, bb;                    // box extents in output positions: time, freq, segments
    int nt;                            // N tile: 128 (position-stationary, >= 128 positions per segment) or 256
    int ksplit;                        // 3 = this layer's input is stored [hi | hi | lo] per position and its
                                       // weights [hi | lo | hi] per tap (hi + lo = the fp32 value to 2^-22):
                                       // the same implicit GEMM then computes hi.hi + hi.lo + lo.hi
    int osplit;                        // split factor of this layer's stored output (= ksplit of its consumer)
};
constexpr int ENC_SPLIT_FROM = 10;     // layers >= L6a run split precision.  Measured on B200 (120 segments x 3 weight sets, fp64 oracle;
                                       // seg/s of a 4,000-segment pass): from L4a (round 1's choice) 636 k, rms 8.0e-5, max 3.9e-4;
                                       // from L6a 760 k, rms 1.0e-4, max 4.9e-4; no split 821 k, rms 1.3e-4, max 6.1e-4 (gate 1e-3).
                                       // One fp16 rounding per layer instead of round 1's two (LayerNorm folding) is what made
                                       // room: round 1 measured 1.0e-3 without the split.

struct ConvParams {
    int m_total, ms, n_seg, c_in, c_out, n_ntiles;
    int mode, pad_lo, tap_lo, tap_hi, kb_per_tap, bf, bb;
    int groups;      // 32-row groups per segment (>= 1): slots of the LayerNorm partial sums
    int osplit;      // 1 = z stored as fp16, 3 = [hi | hi | lo]
    int combos;      // (position tiles per segment) x (channel tiles): what a CTA stays on
    int n_streams;   // CTAs per combo; CTA c works on combo c % combos, unit c / combos, + n_streams, ...
    int n_units;     // units per combo: segments (ms >= 128) or 128-row groups of whole segments (ms < 128)
    int tma_store;   // 1 = z leaves through a swizzled shared-memory tile and TMA stores (full-tile layers, fp16 output)
};

struct EncoderState {
    ConvGeom g[ENC_LAYERS];
    float* w0 = nullptr;                       // conv0_a kernel [3][128]
    float* bias0 = nullptr;
    __half* wt[ENC_LAYERS] = {};               // [c_out][3*c_in] fp16, K-major
    float* ln_g[ENC_LAYERS] = {};              // gamma, (F,T,C)
    float* ln_b15 = nullptr;                   // beta of the last layer (the head applies the last LayerNorm itself)
    float* cbeta[ENC_LAYERS] = {};             // Cb = bias + conv(beta of the previous layer), fp32 (F,T,C) of this layer
    __half* cgam[ENC_LAYERS] = {};             // Cg = conv(gamma of the previous layer), fp16
    std::vector<float> h_g[ENC_LAYERS], h_b[ENC_LAYERS];     // host copies for the activation probe
    float *dw1 = nullptr, *db1 = nullptr, *dw2 = nullptr, *db2 = nullptr;
    __half* x[ENC_LAYERS] = {};                // z = gamma (.) ELU(pre-activation), fp16 (split layers: [hi | hi | lo])
    int cap = 0;                               // segments the arena below holds (ENC_CHUNK_MIN .. ENC_CHUNK_MAX)
    float2* stat = nullptr;                    // [ENC_LAYERS][cap] (a, c) = (rstd, -rstd mean)
    float* part = nullptr;                     // [cap][PART_SLOTS][2] partial LayerNorm sums of the running layer
    float* mel = nullptr;                      // (cap, 256, 32) for the fused entry points
    void* xin[2] = {nullptr, nullptr};         // (cap, 8000) staging for the *_host entry points, double-buffered:
    cudaStream_t copy_stream = nullptr;        // the upload of pass i+1 runs on copy_stream under the kernels of pass i
    cudaEvent_t ev_up[2] = {nullptr, nullptr}; // xin[b] has landed
    cudaEvent_t ev_free[2] = {nullptr, nullptr};   // the last pass that read xin[b] has finished
    float* emb = nullptr;                      // (cap, 128)
    float* raw = nullptr;                      // (cap, 128) head outputs before the L2 normalisation
    CUtensorMap tmA[ENC_LAYERS], tmB[ENC_LAYERS], tmO[ENC_LAYERS];     // activation in, weights, activation out (TMA store)
    bool weights = false;
    int64_t last_n = 0;                        // segments of the last pass (activation probe)
    int norm = NAFP_NORM_LAYER_NORM2D;         // MODEL.BN of the loaded weights (nafp_weights_load_norm)
    int split_from = 0;                        // first split-precision layer of g (split_point(norm))
    float* ln_c = nullptr;                     // [16][gamma 1024 | beta 1024] per-channel LayerNorm of 'layer_norm1d'
    float2* unit = nullptr;                    // [cap] (1, 0): the stat buffer of layers whose output is stored normalised
};
constexpr int PART_SLOTS = 256;                // most partial-sum slots per segment of any layer (L1b: 64 groups x <= 4 parts)

static const int kHidden[8] = {128, 128, 256, 256, 512, 512, 1024, 1024};      // nnfp.py:193
static const int kStrideT[8] = {2, 2, 2, 2, 1, 2, 1, 2};                        // nnfp.py:194-197 (1x3 conv)

static void same_pad(int n_in, int k, int s, int* n_out, int* lo) {
    *n_out = (n_in + s - 1) / s;
    int total = (*n_out - 1) * s + k - n_in;
    if (total < 0) total = 0;
    *lo = total / 2;
}

// split_from: first layer whose operands are split (hi + lo), split_point(norm)
static void build_geometry(ConvGeom* g, int split_from) {
    int f = 256, t = 32, c = 1;
    for (int i = 0; i < 8; ++i) {
        for (int half = 0; half < 2; ++half) {
            ConvGeom& L = g[2 * i + half];
            L.axis = half;
            L.stride = half == 0 ? kStrideT[i] : 2;
            L.f_in = f; L.t_in = t; L.c_in = c; L.c_out = kHidden[i];
            if (half == 0) { same_pad(t, 3, L.stride, &L.t_out, &L.pad_lo); L.f_out = f; }
            else           { same_pad(f, 3, L.stride, &L.f_out, &L.pad_lo); L.t_out = t; }
            L.ms = L.f_out * L.t_out;
            const int n_in = half == 0 ? L.t_in : L.f_in, n_out = half == 0 ? L.t_out : L.f_out;
            L.tap_lo = 3; L.tap_hi = -1;
            for (int tap = 0; tap < 3; ++tap) {
                bool any = false;
                for (int o = 0; o < n_out; ++o) {
                    const int src = o * L.stride + tap - L.pad_lo;
                    if (src >= 0 && src < n_in) any = true;
                }
                if (any) { if (tap < L.tap_lo) L.tap_lo = tap; if (tap > L.tap_hi) L.tap_hi = tap; }
            }
            if (n_out == 1 || L.stride == 1) L.mode = half == 0 ? 0 : 3;
            else L.mode = half == 0 ? 1 : 2;
            L.bt = L.t_out;
            L.bb = L.ms >= 128 ? 1 : 128 / L.ms;
            L.bf = L.ms >= 128 ? 128 / L.t_out : L.f_out;
            L.nt = 128;
            f = L.f_out; t = L.t_out; c = L.c_out;
        }
    }
    // N = 256 where measured faster (4,000-segment pass, round 2): L5b, L6b, L7b, L8a, L8b -- the layers whose A
    // operand is tiny and whose time is the re-streaming of the weights
    constexpr unsigned nt256 = (1u << 9) | (1u << 11) | (1u << 13) | (1u << 14) | (1u << 15);
    for (int l = 1; l < 16; ++l)
        if (((nt256 >> l) & 1u) && g[l].c_out >= 256 && g[l].ms < 128) g[l].nt = 256;
    for (int l = 0; l < 16; ++l) g[l].ksplit = l >= split_from ? 3 : 1;
    for (int l = 0; l < 16; ++l) g[l].osplit = l + 1 < 16 ? g[l + 1].ksplit : 3;     // the head reads hi + lo too
}

// ELU(v) = v > 0 ? v : e^v - 1.  Only the v <= 0 side reaches the exponential, where e^v is in (0, 1]: the bare
// MUFU ex2 (flush-to-zero) is exact enough (2 ulp, absolute error 2^-22 after the -1) and saves the
// denormal-range fix-up of __expf -- 5 of the ~15 instructions per output element of the conv epilogues.
__device__ __forceinline__ float elu(float v) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(v * 1.4426950408889634f));
    return v > 0.f ? v : e - 1.f;
}

// ------------------------------------------------------------------------------------------
// conv0 (L1a): (B,256,32) fp32 log-mel -> z = gamma (.) ELU(conv + bias), (B,256,16,128) fp16, stride 2 in
// time, pad (0,1).  K = 3: CUDA cores; fused with the log-mel max subtraction / clamp and the LayerNorm sums.
// ------------------------------------------------------------------------------------------
// Lane owns 4 channels = 2 packed fp32 pairs: FFMA2 / FMUL2 / FADD2 do two channels per issue slot (the kernel was
// issue-bound: ~12.7 instructions per output element, now ~9).
struct Conv0Lane {
    uint64_t w[3][2], bia[2];
};
__device__ __forceinline__ void conv0_load_lane(const float* __restrict__ w0, const float* __restrict__ b0, int lane,
                                                Conv0Lane& L) {
#pragma unroll
    for (int tap = 0; tap < 3; ++tap) {
        const float4 v = reinterpret_cast<const float4*>(w0 + tap * 128)[lane];
        L.w[tap][0] = pk2(v.x, v.y);
        L.w[tap][1] = pk2(v.z, v.w);
    }
    const float4 v = reinterpret_cast<const float4*>(b0)[lane];
    L.bia[0] = pk2(v.x, v.y);
    L.bia[1] = pk2(v.z, v.w);
}
// ELU of a packed pair; same arithmetic as elu(): v > 0 ? v : ex2(v log2 e) - 1
__device__ __forceinline__ uint64_t elu2(uint64_t v) {
    float a, b, ua, ub, ea, eb;
    upk2(mul2(v, pk2(1.4426950408889634f, 1.4426950408889634f)), ua, ub);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(ea) : "f"(ua));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(eb) : "f"(ub));
    float wa, wb;
    upk2(add2(pk2(ea, eb), pk2(-1.f, -1.f)), wa, wb);
    upk2(v, a, b);
    return pk2(a > 0.f ? a : wa, b > 0.f ? b : wb);
}
// a warp per frequency row; the row's 32 log-mel values are one coalesced load, the three taps of every output
// position come from warp shuffles, the 16 positions of the row are unrolled
__device__ __forceinline__ void conv0_row(float v, const Conv0Lane& L, int tp, uint64_t (&o)[2]) {
    const float x0 = __shfl_sync(0xffffffffu, v, 2 * tp);
    const float x1 = __shfl_sync(0xffffffffu, v, 2 * tp + 1);
    const float x2 = tp < 15 ? __shfl_sync(0xffffffffu, v, (2 * tp + 2) & 31) : 0.f;      // SAME padding (0, 1)
    const uint64_t p0 = pk2(x0, x0), p1 = pk2(x1, x1), p2 = pk2(x2, x2);
#pragma unroll
    for (int c = 0; c < 2; ++c) o[c] = elu2(fma2(p2, L.w[2][c], fma2(p1, L.w[1][c], fma2(p0, L.w[0][c], L.bia[c]))));
}

// grid (256 / CONV0_ROWS, ceil(n_seg / CONV0_SEGS)): block (bx, by) covers CONV0_ROWS frequency rows of CONV0_SEGS
// segments, so that the block's gamma rows (128 KB, 4 B per element, shared by all segments) come from L1 after
// the first segment.  One slot of partial sums per (segment, block, warp): CONV0_SLOTS per segment.
constexpr int CONV0_ROWS = 16, CONV0_SEGS = 16;
constexpr int CONV0_SLOTS = (256 / CONV0_ROWS) * 8;
// LN1D ('layer_norm1d'): every output position is normalised over its 128 channels before the store -- a lane holds
// 4 channels of the position, so its statistics are a warp reduction (two passes, fp32, fixed order); ln_c holds
// gamma [0, 128) and beta [1024, 1152) of the layer, and no partial sums are written.
// SPLIT: the output is stored [hi | hi | lo] per position (L1b runs split precision: 'batch_norm', see build_geometry).
template <bool LN1D, bool SPLIT = false>
__global__ void __launch_bounds__(256)
conv0_kernel(const float* __restrict__ mel, const int32_t* __restrict__ gmax, int64_t group_size, int n_seg,
             const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ gamma,
             __half* __restrict__ x, float* __restrict__ part, const float* __restrict__ ln_c) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int seg0 = blockIdx.y * CONV0_SEGS;
    constexpr int PER_SEG = 256 * 16 * 128;
    Conv0Lane L;
    conv0_load_lane(w0, b0, lane, L);
    float4 lg, lb;
    if constexpr (LN1D) {
        lg = reinterpret_cast<const float4*>(ln_c)[lane];
        lb = reinterpret_cast<const float4*>(ln_c + 1024)[lane];
    }
    const bool raw = gmax != nullptr;
#pragma unroll 1
    for (int k = 0; k < CONV0_SEGS; ++k) {
        const int seg = seg0 + k;
        if (seg >= n_seg) break;
        const float sub = raw ? ord2f(gmax[seg / group_size]) : 0.f;
        uint64_t s1 = pk2(0.f, 0.f), s2 = pk2(0.f, 0.f);
#pragma unroll 1
        for (int r = 0; r < CONV0_ROWS / 8; ++r) {
            const int f = blockIdx.x * CONV0_ROWS + warp * (CONV0_ROWS / 8) + r;
            float v = __ldg(mel + static_cast<int64_t>(seg) * 8192 + f * 32 + lane);
            if (raw) v = fmaxf(v - sub, -80.f);                 // "- batch max, clamp -80" (melspectrogram.py:108-109)
            const ulonglong2* g_row = reinterpret_cast<const ulonglong2*>(gamma + static_cast<int64_t>(f) * (16 * 128)) + lane;
            uint2* orow = reinterpret_cast<uint2*>(x + static_cast<int64_t>(seg) * PER_SEG + static_cast<int64_t>(f) * (16 * 128)) + lane;
#pragma unroll
            for (int tp = 0; tp < 16; ++tp) {
                uint64_t o[2];
                conv0_row(v, L, tp, o);
                float z0, z1, z2, z3;
                if constexpr (LN1D) {
                    float y0, y1, y2, y3;
                    upk2(o[0], y0, y1);
                    upk2(o[1], y2, y3);
                    float m = (y0 + y1) + (y2 + y3);
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) m += __shfl_xor_sync(0xffffffffu, m, off);
                    m *= 1.f / 128.f;
                    y0 -= m; y1 -= m; y2 -= m; y3 -= m;
                    float q = (y0 * y0 + y1 * y1) + (y2 * y2 + y3 * y3);
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) q += __shfl_xor_sync(0xffffffffu, q, off);
                    const float rstd = rsqrtf(q * (1.f / 128.f) + LN_EPS);
                    z0 = fmaf(lg.x, y0 * rstd, lb.x);
                    z1 = fmaf(lg.y, y1 * rstd, lb.y);
                    z2 = fmaf(lg.z, y2 * rstd, lb.z);
                    z3 = fmaf(lg.w, y3 * rstd, lb.w);
                } else {
                    const ulonglong2 g = __ldg(g_row + tp * 32);
                    s1 = add2(s1, add2(o[0], o[1]));
                    s2 = fma2(o[0], o[0], fma2(o[1], o[1], s2));
                    upk2(mul2(o[0], g.x), z0, z1);
                    upk2(mul2(o[1], g.y), z2, z3);
                }
                __half2 h0 = __floats2half2_rn(z0, z1), h1 = __floats2half2_rn(z2, z3);
                uint2 pk;
                pk.x = *reinterpret_cast<uint32_t*>(&h0);
                pk.y = *reinterpret_cast<uint32_t*>(&h1);
                if constexpr (SPLIT) {
                    const float2 b0 = __half22float2(h0), b1 = __half22float2(h1);
                    __half2 l0 = __floats2half2_rn(z0 - b0.x, z1 - b0.y), l1 = __floats2half2_rn(z2 - b1.x, z3 - b1.y);
                    uint2 lo;
                    lo.x = *reinterpret_cast<uint32_t*>(&l0);
                    lo.y = *reinterpret_cast<uint32_t*>(&l1);
                    uint2* srow = reinterpret_cast<uint2*>(x + (static_cast<int64_t>(seg) * PER_SEG + static_cast<int64_t>(f) * (16 * 128)) * 3) + lane;
                    srow[tp * 96] = pk;                 // 384 halves per position: hi (32 uint2), hi, lo
                    srow[tp * 96 + 32] = pk;
                    srow[tp * 96 + 64] = lo;
                } else {
                    orow[tp * 32] = pk;
                }
            }
        }
        if constexpr (LN1D) continue;
        float a1, b1, a2, b2;
        upk2(s1, a1, b1);
        upk2(s2, a2, b2);
        float t1 = a1 + b1, t2 = a2 + b2;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            t1 += __shfl_xor_sync(0xffffffffu, t1, o);
            t2 += __shfl_xor_sync(0xffffffffu, t2, o);
        }
        if (lane == 0)
            reinterpret_cast<float2*>(part)[static_cast<int64_t>(seg) * CONV0_SLOTS + blockIdx.x * 8 + warp] = make_float2(t1, t2);
    }
}

// partial (sum, sum of squares) slots of one layer -> (a, c) = (rstd, -rstd * mean) per segment: one warp per
// segment, fixed order, double accumulation (bit-reproducible)
__global__ void __launch_bounds__(256)
ln_stats_kernel(const float* __restrict__ part, int slots, int per_seg, int n_seg, float2* __restrict__ stat) {
    const int lane = threadIdx.x & 31;
    const int seg = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (seg >= n_seg) return;
    const float2* p = reinterpret_cast<const float2*>(part) + static_cast<int64_t>(seg) * slots;
    double a = 0.0, b = 0.0;
    for (int i = lane; i < slots; i += 32) {
        const float2 v = p[i];
        a += v.x;
        b += v.y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == 0) {
        const float inv_n = 1.f / static_cast<float>(per_seg);
        const float mean = static_cast<float>(a) * inv_n;
        const float var = fmaxf(static_cast<float>(b) * inv_n - mean * mean, 0.f);
        const float rstd = rsqrtf(var + LN_EPS);
        stat[seg] = make_float2(rstd, -rstd * mean);
    }
}

// 'layer_norm1d' after conv layers 1 .. 14: one warp per output position normalises its C = 32 PER channels in
// place, gamma (.) (y - mean) rstd + beta, in the stored format (fp16, or [hi | hi | lo] re-split).  Two passes in
// fp32 over the lane's registers, then a fixed shuffle tree: bit-reproducible, independent of the pass size.
template <int PER>
__global__ void __launch_bounds__(256)
ln1d_kernel(__half* __restrict__ x, int64_t n_pos, int split, const float* __restrict__ gamma, const float* __restrict__ beta) {
    constexpr int C = PER * 32;
    constexpr int VEC = PER < 8 ? PER : 8;            // halves per load: 8 or 16 bytes, consecutive lanes adjacent
    constexpr int NV = PER / VEC;
    const int lane = threadIdx.x & 31;
    const int64_t pos = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (pos >= n_pos) return;
    __half* row = x + pos * C * (split ? 3 : 1);
    float v[PER];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int c0 = (j * 32 + lane) * VEC;
        __half2 h[VEC / 2], l[VEC / 2];
        if constexpr (VEC == 8) *reinterpret_cast<uint4*>(h) = *reinterpret_cast<const uint4*>(row + c0);
        else                    *reinterpret_cast<uint2*>(h) = *reinterpret_cast<const uint2*>(row + c0);
        if (split) {
            if constexpr (VEC == 8) *reinterpret_cast<uint4*>(l) = *reinterpret_cast<const uint4*>(row + 2 * C + c0);
            else                    *reinterpret_cast<uint2*>(l) = *reinterpret_cast<const uint2*>(row + 2 * C + c0);
        }
#pragma unroll
        for (int k = 0; k < VEC / 2; ++k) {
            float2 f = __half22float2(h[k]);
            if (split) {
                const float2 g = __half22float2(l[k]);
                f.x += g.x;
                f.y += g.y;
            }
            v[j * VEC + 2 * k] = f.x;
            v[j * VEC + 2 * k + 1] = f.y;
        }
    }
    float m = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) m += v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
    m *= 1.f / C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        v[i] -= m;
        q = fmaf(v[i], v[i], q);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q * (1.f / C) + LN_EPS);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int c0 = (j * 32 + lane) * VEC;
        __half2 h[VEC / 2], l[VEC / 2];
#pragma unroll
        for (int k = 0; k < VEC / 2; ++k) {
            const int c = c0 + 2 * k;
            const float z0 = fmaf(__ldg(gamma + c), v[j * VEC + 2 * k] * rstd, __ldg(beta + c));
            const float z1 = fmaf(__ldg(gamma + c + 1), v[j * VEC + 2 * k + 1] * rstd, __ldg(beta + c + 1));
            h[k] = __floats2half2_rn(z0, z1);
            if (split) {
                const float2 back = __half22float2(h[k]);
                l[k] = __floats2half2_rn(z0 - back.x, z1 - back.y);
            }
        }
        if constexpr (VEC == 8) {
            *reinterpret_cast<uint4*>(row + c0) = *reinterpret_cast<const uint4*>(h);
            if (split) {
                *reinterpret_cast<uint4*>(row + C + c0) = *reinterpret_cast<const uint4*>(h);
                *reinterpret_cast<uint4*>(row + 2 * C + c0) = *reinterpret_cast<const uint4*>(l);
            }
        } else {
            *reinterpret_cast<uint2*>(row + c0) = *reinterpret_cast<const uint2*>(h);
            if (split) {
                *reinterpret_cast<uint2*>(row + C + c0) = *reinterpret_cast<const uint2*>(h);
                *reinterpret_cast<uint2*>(row + 2 * C + c0) = *reinterpret_cast<const uint2*>(l);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// implicit-GEMM separable convolution on tcgen05
// ------------------------------------------------------------------------------------------
// Two tile shapes:
//   NTILE = 128 (layers with >= 128 positions per segment, L1b .. L3b): 6-stage ring, two 128-column accumulators,
//                gamma / Cb STATIONARY in the other 256 TMEM columns, Cg in registers (position-stationary CTAs);
//   NTILE = 256 (the ten small layers, several whole segments per 128-row tile): 4-stage ring, two 256-column
//                accumulators (TMEM full); these layers are bound by the L2 -> SM operand fetch (weights are
//                re-streamed for every M tile), which the wider tile cuts by 25 %; their parameters repeat every
//                `ms` rows and are read per tile through L1 (<= 9 % of the operand bytes).
constexpr int CONV_MAX_STAGES = 6;
#ifndef NAFP_CONV_EPI_WARPS
#define NAFP_CONV_EPI_WARPS 8      // measured: 5.65 ms per 4,000 segments with 8 warps (152 registers, two chunks of TMEM loads
#endif                             // in flight per warp) against 5.99 ms with 16 (96 registers, spills)
constexpr int CONV_EPI_WARPS = NAFP_CONV_EPI_WARPS;      // 4 (or 2) per TMEM lane quadrant: each takes a share of the tile's columns
constexpr int CONV_EPI_PARTS = CONV_EPI_WARPS / 4;
constexpr int CONV_THREADS = (2 + CONV_EPI_WARPS) * 32;   // warp 0 TMA, warp 1 MMA (+TMEM alloc), warps 2.. epilogue
constexpr int CONV_A_BYTES = 128 * 128;    // 128 rows x 64 fp16
constexpr int CONV_RING_BYTES = 192 * 1024;
constexpr int CONV_STAGE_BYTES = 128 * 256;          // output staging: 128 rows x 128 fp16 channels, two SWIZZLE_128B halves
constexpr int CONV_SMEM = CONV_RING_BYTES + CONV_STAGE_BYTES + 256 + 1024;
constexpr int TMEM_GAMMA = 256, TMEM_CBETA = 384;          // NTILE = 128: column offsets of the parameter planes

struct ConvBars {
    uint64_t full[CONV_MAX_STAGES];
    uint64_t empty[CONV_MAX_STAGES];
    uint64_t tfull[2];
    uint64_t tempty[2];
    uint64_t bfull;            // resident-weights mode: all K blocks of the CTA's N tile have landed
    uint32_t tmem_base;
};

// one 16-column chunk of the epilogue: v = a acc + c Cg + Cb; y = ELU(v); statistics of y; z = gamma y -> hi (and lo).
// Packed fp32 pairs (FFMA2 / FMUL2 / FADD2): two columns per issue slot.
__device__ __forceinline__ void conv_epi_chunk(const uint32_t (&va)[16], const uint32_t (&vg)[16], const uint32_t (&vb)[16],
                                               const uint32_t* cg, uint64_t sta, uint64_t stc, bool split, uint64_t& s1,
                                               uint64_t& s2, uint32_t (&hi)[8], uint32_t (&lo)[8]) {
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
        const float2 cgv = __half22float2(*reinterpret_cast<const __half2*>(&cg[j >> 1]));
        // conv(LN(y_prev)) = a * conv(z) + c * Cg + Cb  (bias is inside Cb)
#ifdef NAFP_EPI_PACKED      // measured slower here (register pairs under the 96-register cap): 6.28 vs 5.99 ms per 4,000 segments
        const uint64_t acc = pk2(__uint_as_float(va[j]), __uint_as_float(va[j + 1]));
        const uint64_t cb = pk2(__uint_as_float(vb[j]), __uint_as_float(vb[j + 1]));
        const uint64_t y = elu2(fma2(sta, acc, fma2(stc, pk2(cgv.x, cgv.y), cb)));
        s1 = add2(s1, y);
        s2 = fma2(y, y, s2);
        float z0, z1;
        upk2(mul2(y, pk2(__uint_as_float(vg[j]), __uint_as_float(vg[j + 1]))), z0, z1);
#else
        float sa, sc, t1a, t1b, t2a, t2b;
        upk2(sta, sa, sc); upk2(stc, sc, sc);
        const float y0 = elu(fmaf(sa, __uint_as_float(va[j]), fmaf(sc, cgv.x, __uint_as_float(vb[j]))));
        const float y1 = elu(fmaf(sa, __uint_as_float(va[j + 1]), fmaf(sc, cgv.y, __uint_as_float(vb[j + 1]))));
        upk2(s1, t1a, t1b); upk2(s2, t2a, t2b);
        s1 = pk2(t1a + y0, t1b + y1);
        s2 = pk2(fmaf(y0, y0, t2a), fmaf(y1, y1, t2b));
        const float z0 = y0 * __uint_as_float(vg[j]), z1 = y1 * __uint_as_float(vg[j + 1]);
#endif
        __half2 hh = __floats2half2_rn(z0, z1);
        hi[j >> 1] = *reinterpret_cast<uint32_t*>(&hh);
        if (split) {
            const float2 back = __half22float2(hh);
            __half2 ll = __floats2half2_rn(z0 - back.x, z1 - back.y);
            lo[j >> 1] = *reinterpret_cast<uint32_t*>(&ll);
        }
    }
}

template <int NTILE>
// 18 warps: five share a sub-partition's 16 K registers -> at most 96 per thread (112 does not launch)
__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const ConvParams p, const float2* __restrict__ stat_in, const float* __restrict__ gamma,
                 const float* __restrict__ cbeta, const __half* __restrict__ cgam, __half* __restrict__ x_out,
                 float* __restrict__ part) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    constexpr int CONV_B_BYTES = NTILE * 128;                   // NTILE channels x 64 fp16
    constexpr int CONV_STAGES = CONV_RING_BYTES / (CONV_A_BYTES + CONV_B_BYTES);      // 6 / 4
    constexpr int CPW = NTILE / CONV_EPI_PARTS;                 // columns per epilogue warp: 32 / 64
    constexpr bool STATIONARY = NTILE == 128;
    uint8_t* a_s = smem;                                        // [stage][128][128 B]
    uint8_t* b_s = smem + CONV_STAGES * CONV_A_BYTES;           // [stage][NTILE][128 B]  (or the resident weights)
    uint8_t* o_s = smem + CONV_RING_BYTES;                      // [half 2][128 rows][128 B] output staging (tma_store)
    ConvBars* bars = reinterpret_cast<ConvBars*>(o_s + CONV_STAGE_BYTES);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_taps = p.tap_hi - p.tap_lo + 1;
    const int k_iters = n_taps * p.kb_per_tap;
    // this CTA's fixed (position tile, channel tile) and its stream of units
    const int combo = blockIdx.x % p.combos, stream = blockIdx.x / p.combos;
    const int ptile = combo / p.n_ntiles, ntile = combo % p.n_ntiles;
    const int n0 = ntile * NTILE;
    // Weights resident: when all K blocks of the N tile fit into the B ring's space (K <= 384: L1b .. L3a), B is
    // loaded ONCE and only A streams -- half the TMA / L2 traffic of those layers.
    const bool b_resident = k_iters <= CONV_STAGES;

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if (p.tma_store) tma_prefetch_desc(&tmO);
        for (int s = 0; s < CONV_STAGES; ++s) {
            mbar_init(&bars->full[s], 1);
            mbar_init(&bars->empty[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&bars->tfull[a], 1);
            mbar_init(&bars->tempty[a], CONV_EPI_WARPS);
        }
        mbar_init(&bars->bfull, 1);
        mbar_fence_init();
    }
    if (warp == 1) {
        tmem_alloc(&bars->tmem_base, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, bars->tmem_base, 0);     // provably warp-uniform

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer
        if (lane == 0) {
            int it = 0;
            if (b_resident) {
                mbar_arrive_expect_tx(&bars->bfull, static_cast<uint32_t>(k_iters * CONV_B_BYTES));
                int k = 0;
                for (int tap = p.tap_lo; tap <= p.tap_hi; ++tap)
                    for (int kb = 0; kb < p.kb_per_tap; ++kb, ++k)
                        tma_load_2d(b_s + k * CONV_B_BYTES, &tmB, &bars->bfull, tap * p.c_in + kb * 64, n0);
            }
            // A box (tap, channels c0 ..) of unit u into ring slot dst
            // (an L2 prefetch of the next unit's A boxes was measured slower: 7.5 vs 6.9 ms per 4,000 segments -- the
            // prefetch requests compete with the loads for the same TMA / L2 request slots)
            auto a_box = [&](uint8_t* dst, uint64_t* bar, int u, int tap, int c0) {
                int b0, f0;
                if (p.ms >= 128) { b0 = u;        f0 = ptile * p.bf; }
                else             { b0 = u * p.bb; f0 = 0; }
                // mode 0: (c,t,f,b)        time conv, unit stride in the box: t = tap - pad
                // mode 1: (c,tp,th,f,b)    time conv stride 2: t = 2 t' + tap -> parity tap&1, half t' + (tap>>1)
                // mode 2: (c,t,fp,fh,b)    freq conv stride 2: f = 2 f' + tap
                // mode 3: (c,t,f,b)        freq conv with a single output row: f = tap - pad
                if (p.mode == 0)      tma_load_4d(dst, &tmA, bar, c0, tap - p.pad_lo, f0, b0);
                else if (p.mode == 1) tma_load_5d(dst, &tmA, bar, c0, tap & 1, tap >> 1, f0, b0);
                else if (p.mode == 2) tma_load_5d(dst, &tmA, bar, c0, 0, tap & 1, f0 + (tap >> 1), b0);
                else                  tma_load_4d(dst, &tmA, bar, c0, 0, f0 + tap - p.pad_lo, b0);
            };
            for (int u = stream; u < p.n_units; u += p.n_streams) {
                for (int tap = p.tap_lo; tap <= p.tap_hi; ++tap) {
                    for (int kb = 0; kb < p.kb_per_tap; ++kb, ++it) {
                        const int s = it % CONV_STAGES;
                        const uint32_t ph = (it / CONV_STAGES) & 1;
                        mbar_wait(&bars->empty[s], ph ^ 1);
                        mbar_arrive_expect_tx(&bars->full[s], CONV_A_BYTES + (b_resident ? 0 : CONV_B_BYTES));
                        const int c0 = kb * 64;
                        a_box(a_s + s * CONV_A_BYTES, &bars->full[s], u, tap, c0);
                        if (!b_resident) tma_load_2d(b_s + s * CONV_B_BYTES, &tmB, &bars->full[s], tap * p.c_in + c0, n0);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer
        // The whole warp runs the loop (uniform control flow: descriptors and counters stay in uniform
        // registers, no ELECT / R2UR waterfall around every MMA); one elected lane issues.
        const bool leader = elect_one();
        const uint32_t idesc = umma_idesc_f16(0u, 128, NTILE);
        const uint64_t adesc0 = umma_desc_sw128(smem_u32(a_s));
        const uint64_t bdesc0 = umma_desc_sw128(smem_u32(b_s));
        if (b_resident) mbar_wait(&bars->bfull, 0);
        int it = 0, lt = 0;
        for (int u = stream; u < p.n_units; u += p.n_streams, ++lt) {
            const int acc = lt & 1;
            const uint32_t aph = (lt >> 1) & 1;
            mbar_wait(&bars->tempty[acc], aph ^ 1);
            const uint32_t d_tmem = tmem_base + acc * NTILE;
            for (int k = 0; k < k_iters; ++k, ++it) {
                const int s = it % CONV_STAGES;
                const uint32_t ph = (it / CONV_STAGES) & 1;
                mbar_wait(&bars->full[s], ph);
                tc_fence_after();
                if (leader) {
                    const uint64_t adesc = adesc0 + static_cast<uint64_t>((s * CONV_A_BYTES) >> 4);
                    const uint64_t bdesc = bdesc0 + static_cast<uint64_t>(((b_resident ? k : s) * CONV_B_BYTES) >> 4);
#pragma unroll
                    for (int j = 0; j < 4; ++j) tc_mma_f16(d_tmem, adesc + 2 * j, bdesc + 2 * j, idesc, (k | j) != 0 ? 1u : 0u);
                    tc_commit(&bars->empty[s]);
                    if (k == k_iters - 1) tc_commit(&bars->tfull[acc]);
                }
                __syncwarp();
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------ epilogue (CONV_EPI_WARPS warps)
        const int qd = warp & 3;               // TMEM lane quadrant = rows 32 qd .. 32 qd + 31 of the tile
        const int cpart = (warp - 2) >> 2;     // which quarter of the tile's columns
        const int r = qd * 32 + lane;          // row of the tile
        const int n_base = n0 + cpart * CPW;
        const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(qd * 32) << 16);
        // this thread's (position, CPW channels) of the per-element constants
        const int pos = p.ms >= 128 ? ptile * 128 + r : r % p.ms;
        const int64_t poff = static_cast<int64_t>(pos) * p.c_out + n_base;
        uint32_t cg[STATIONARY ? CPW / 2 : 1];      // half2 pairs
        if constexpr (STATIONARY) {
            // ---- stationary: gamma and Cb into the free TMEM columns, Cg into registers, once per launch
            const uint4* gs = reinterpret_cast<const uint4*>(gamma + poff);
            const uint4* bs = reinterpret_cast<const uint4*>(cbeta + poff);
            const uint4* cs = reinterpret_cast<const uint4*>(cgam + poff);
#pragma unroll
            for (int h = 0; h < CPW / 16; ++h) {
                uint32_t v[16];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint4 q = __ldg(gs + h * 4 + j);
                    v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
                }
                tmem_st_32x16(lane_base + TMEM_GAMMA + cpart * CPW + h * 16, v);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint4 q = __ldg(bs + h * 4 + j);
                    v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w;
                }
                tmem_st_32x16(lane_base + TMEM_CBETA + cpart * CPW + h * 16, v);
            }
#pragma unroll
            for (int j = 0; j < CPW / 8; ++j) {            // 8 fp16 values per 16-byte load
                const uint4 q = __ldg(cs + j);
                cg[4 * j] = q.x; cg[4 * j + 1] = q.y; cg[4 * j + 2] = q.z; cg[4 * j + 3] = q.w;
            }
            tc_wait_st();
        }
        const int seg_len = p.ms < 32 ? p.ms : 32;     // rows of one segment inside this warp (power of two)
        const int row_halves = p.c_out * p.osplit;     // halves per stored row
        const bool split = p.osplit != 1;
        // no integer division in the tile loop: a row's segment and its 32-row group follow from per-thread constants
        const bool big = p.ms >= 128;
        const int seg_in_unit = big ? 0 : r / p.ms;    // ms < 128: the unit holds bb = 128 / ms whole segments
        const int grp = p.ms >= 32 ? pos >> 5 : 0;
        const int64_t slot_lane = (static_cast<int64_t>(grp) * p.n_ntiles + ntile) * CONV_EPI_PARTS + cpart;
        const int slots_per_seg = p.groups * p.n_ntiles * CONV_EPI_PARTS;
        int lt = 0;
        float2 st_next = make_float2(0.f, 0.f);
        {
            const int b0 = big ? stream : stream * p.bb + seg_in_unit;
            if (stream < p.n_units && b0 < p.n_seg) st_next = __ldg(stat_in + b0);
        }
        for (int u = stream; u < p.n_units; u += p.n_streams, ++lt) {
            const int acc = lt & 1;
            const uint32_t aph = (lt >> 1) & 1;
            const int m = (big ? u * p.ms + ptile * 128 : u * 128) + r;      // output row (NHWC position index)
            const int b = big ? u : u * p.bb + seg_in_unit;
            const bool row_ok = b < p.n_seg;
            const float2 st = st_next;
            {           // the next unit's (a, c) while this one is processed
                const int un = u + p.n_streams;
                const int bn = big ? un : un * p.bb + seg_in_unit;
                if (un < p.n_units && bn < p.n_seg) st_next = __ldg(stat_in + bn);
            }
            __half* xrow = x_out + static_cast<int64_t>(m) * row_halves + n_base;
            // TMA-store layers: the previous unit's tile must have left the staging buffer before it is rewritten
            const bool use_tma = STATIONARY && CPW == 64 && p.tma_store;
            if (use_tma) {
                if (warp == 2 && lane == 0 && lt > 0) tma_store_wait_read();
                asm volatile("bar.sync 1, %0;" ::"n"(CONV_EPI_WARPS * 32) : "memory");
            }
            mbar_wait(&bars->tfull[acc], aph);
            tc_fence_after();
            uint64_t ps1 = pk2(0.f, 0.f), ps2 = pk2(0.f, 0.f);
            const uint64_t sta = pk2(st.x, st.x), stc = pk2(st.y, st.y);
#pragma unroll
            for (int h = 0; h < CPW / 16; ++h) {
                uint32_t va[16], vg[16], vb[16], cgl[8];
                tmem_ld_32x16(lane_base + acc * NTILE + cpart * CPW + h * 16, va);
                if constexpr (STATIONARY) {
                    tmem_ld_32x16(lane_base + TMEM_GAMMA + cpart * CPW + h * 16, vg);
                    tmem_ld_32x16(lane_base + TMEM_CBETA + cpart * CPW + h * 16, vb);
                } else {
                    // per tile through L1: the tile's rows repeat every ms positions and the next tile reads the same lines
                    const uint4* gs = reinterpret_cast<const uint4*>(gamma + poff + h * 16);
                    const uint4* bs = reinterpret_cast<const uint4*>(cbeta + poff + h * 16);
                    const uint4* cs = reinterpret_cast<const uint4*>(cgam + poff + h * 16);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint4 q = __ldg(gs + j), w = __ldg(bs + j);
                        vg[4 * j] = q.x; vg[4 * j + 1] = q.y; vg[4 * j + 2] = q.z; vg[4 * j + 3] = q.w;
                        vb[4 * j] = w.x; vb[4 * j + 1] = w.y; vb[4 * j + 2] = w.z; vb[4 * j + 3] = w.w;
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const uint4 q = __ldg(cs + j);
                        cgl[4 * j] = q.x; cgl[4 * j + 1] = q.y; cgl[4 * j + 2] = q.z; cgl[4 * j + 3] = q.w;
                    }
                }
                tc_wait_ld();
                if (h == CPW / 16 - 1) {           // the accumulator is in registers: hand it back to the MMA warp
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&bars->tempty[acc]);
                }
                uint32_t hi[8], lo[8];
                // (loading chunk h + 1 while chunk h is computed was measured slower: 7.07 vs 6.26 ms per 4,000 segments)
                conv_epi_chunk(va, vg, vb, STATIONARY ? &cg[(STATIONARY ? h : 0) * 8] : cgl, sta, stc, split, ps1, ps2, hi, lo);
                if (use_tma) {
                    // row r of half `cpart`: 16-byte chunk c of the 128-byte row sits at chunk (c ^ (r & 7)) (SWIZZLE_128B);
                    // 8 consecutive rows cover all 32 banks: a warp's store is conflict-free
                    uint8_t* srow = o_s + cpart * (CONV_STAGE_BYTES / 2) + r * 128;
                    *reinterpret_cast<uint4*>(srow + (((2 * h) ^ (r & 7)) << 4)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(srow + (((2 * h + 1) ^ (r & 7)) << 4)) = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                } else if (row_ok) {
                    uint4* dst = reinterpret_cast<uint4*>(xrow + h * 16);
                    dst[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    dst[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                    if (split) {        // [hi | hi | lo] per position
                        uint4* d1 = reinterpret_cast<uint4*>(xrow + p.c_out + h * 16);
                        uint4* d2 = reinterpret_cast<uint4*>(xrow + 2 * p.c_out + h * 16);
                        d1[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                        d1[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
                        d2[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        d2[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
                    }
                }
            }
            if (use_tma) {
                // generic-proxy writes -> visible to the async proxy, all 8 warps done, then ONE thread stores the tile:
                // two boxes of 64 channels x 128 rows = 32 KB contiguous in global memory (was 64 scattered 32-byte
                // stores per warp: 32 L1 wavefronts per instruction)
                fence_proxy_async_smem();
                asm volatile("bar.sync 1, %0;" ::"n"(CONV_EPI_WARPS * 32) : "memory");
                if (warp == 2 && lane == 0) {
                    const int m0 = u * p.ms + ptile * 128;
                    tma_store_2d(&tmO, o_s, n0, m0);
                    tma_store_2d(&tmO, o_s + CONV_STAGE_BYTES / 2, n0 + 64, m0);
                    tma_store_commit();
                }
            }
            // LayerNorm statistics of ELU(...): reduce over the rows of the same segment inside the warp, then one
            // slot per (segment, 32-row group, N tile, column part) -- no atomics, so the sums (and with
            // them every fingerprint) are bit-reproducible
            float s1, s2;
            {
                float a, b;
                upk2(ps1, a, b);
                s1 = a + b;
                upk2(ps2, a, b);
                s2 = a + b;
            }
            if (!row_ok) { s1 = 0.f; s2 = 0.f; }
            if (seg_len == 32) {
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                }
            } else {
                for (int o = 1; o < seg_len; o <<= 1) {
                    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                }
            }
            if (row_ok && (lane & (seg_len - 1)) == 0)
                reinterpret_cast<float2*>(part)[static_cast<int64_t>(b) * slots_per_seg + slot_lane] = make_float2(s1, s2);
        }
    }

    if (warp == 2 && lane == 0 && p.tma_store) tma_store_wait_all();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------
// weights load: Cg = conv(gamma_prev) (fp16, with the weights as the MMA sees them), Cb = bias + conv(beta_prev) (fp32),
// one thread per (output position, output channel), fp64 accumulation
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
fold_kernel(const float* __restrict__ w /* [3][c_in][c_out] */, const float* __restrict__ bias, const float* __restrict__ g_in,
            const float* __restrict__ b_in, ConvGeom L, int round_w, __half* __restrict__ cgam, float* __restrict__ cbeta) {
    const int co = blockIdx.x * blockDim.x + threadIdx.x;
    const int po = blockIdx.y;
    if (co >= L.c_out) return;
    const int fo = po / L.t_out, to = po % L.t_out;
    double ag = 0.0, ab = bias[co];
    for (int tap = 0; tap < 3; ++tap) {
        int f = fo, t = to;
        if (L.axis == 0) t = to * L.stride + tap - L.pad_lo;
        else             f = fo * L.stride + tap - L.pad_lo;
        if (f < 0 || f >= L.f_in || t < 0 || t >= L.t_in) continue;        // SAME zero padding
        const float* gp = g_in + (static_cast<int64_t>(f) * L.t_in + t) * L.c_in;
        const float* bp = b_in + (static_cast<int64_t>(f) * L.t_in + t) * L.c_in;
        const float* wp = w + static_cast<int64_t>(tap) * L.c_in * L.c_out + co;
        for (int ci = 0; ci < L.c_in; ++ci) {
            const float wv = wp[static_cast<int64_t>(ci) * L.c_out];
            const float wg = round_w ? __half2float(__float2half_rn(wv)) : wv;
            ag += static_cast<double>(wg) * gp[ci];
            ab += static_cast<double>(wv) * bp[ci];
        }
    }
    const int64_t o = static_cast<int64_t>(po) * L.c_out + co;
    cgam[o] = __float2half_rn(static_cast<float>(ag));
    cbeta[o] = static_cast<float>(ab);
}

// ------------------------------------------------------------------------------------------
// divide-and-encode head (nnfp.py:132-156): block (q, 128 segments) -- the 8x32 + 32 weights of slice q
// sit in shared memory and are broadcast to the 128 segments; then one warp per segment L2-normalises.
// x: (B, 3 x 1024) z of the last conv, [hi | hi | lo]; the last LayerNorm is applied here:
// LN(y)[c] = a z[c] + c gamma[c] + beta[c]; slice q = features 8q .. 8q+7 (nnfp.py:155)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
divenc_kernel(const __half* __restrict__ x, const float2* __restrict__ stat, const float* __restrict__ gamma,
              const float* __restrict__ beta, int n_seg, const float* __restrict__ w1, const float* __restrict__ b1,
              const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ raw) {
    __shared__ float W1[8 * 32], B1[32], W2[32], G[8], Bt[8];
    const int q = blockIdx.x;
    for (int i = threadIdx.x; i < 256; i += 128) W1[i] = w1[q * 256 + i];
    if (threadIdx.x < 32) {
        B1[threadIdx.x] = b1[q * 32 + threadIdx.x];
        W2[threadIdx.x] = w2[q * 32 + threadIdx.x];
    }
    if (threadIdx.x < 8) {
        G[threadIdx.x] = gamma[q * 8 + threadIdx.x];
        Bt[threadIdx.x] = beta[q * 8 + threadIdx.x];
    }
    __syncthreads();
    const int seg = blockIdx.y * 128 + threadIdx.x;
    if (seg >= n_seg) return;
    const float2 st = stat[seg];
    const uint4 rv = *reinterpret_cast<const uint4*>(x + static_cast<int64_t>(seg) * 3072 + q * 8);
    const uint4 rl = *reinterpret_cast<const uint4*>(x + static_cast<int64_t>(seg) * 3072 + 2048 + q * 8);
    const __half2* hv = reinterpret_cast<const __half2*>(&rv);
    const __half2* hl = reinterpret_cast<const __half2*>(&rl);
    float in[8];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(hv[j]), g = __half22float2(hl[j]);
        in[2 * j] = fmaf(st.x, f.x + g.x, fmaf(st.y, G[2 * j], Bt[2 * j]));
        in[2 * j + 1] = fmaf(st.x, f.y + g.y, fmaf(st.y, G[2 * j + 1], Bt[2 * j + 1]));
    }
    float acc = b2[q];
#pragma unroll 8
    for (int u = 0; u < 32; ++u) {
        float hsum = B1[u];
#pragma unroll
        for (int sdim = 0; sdim < 8; ++sdim) hsum += in[sdim] * W1[sdim * 32 + u];
        hsum = hsum > 0.f ? hsum : expm1f(hsum);
        acc += hsum * W2[u];
    }
    raw[static_cast<int64_t>(seg) * EMB + q] = acc;
}

__global__ void __launch_bounds__(256)
l2norm_kernel(const float* __restrict__ raw, int n_seg, float* __restrict__ emb) {
    const int lane = threadIdx.x & 31;
    const int seg = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (seg >= n_seg) return;
    const float4 v = reinterpret_cast<const float4*>(raw + static_cast<int64_t>(seg) * EMB)[lane];
    float ss = v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const float inv = rsqrtf(fmaxf(ss, L2_EPS));
    reinterpret_cast<float4*>(emb + static_cast<int64_t>(seg) * EMB)[lane] = make_float4(v.x * inv, v.y * inv, v.z * inv, v.w * inv);
}

// ------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------
static_assert(ENC_SPLIT_FROM >= 2, "conv0_kernel writes split output only without the fused layer_norm1d");
// First split-precision layer for a MODEL.BN.  'batch_norm' needs every layer split: its per-channel scale
// gamma / sqrt(var + eps) reaches ~30 on channels ELU saturates (variance near 0), and any fp16 rounding of an
// activation before that scale -- even L1a's output, or the normalised value -- carries the fingerprints past 1e-3
// (measured on B200 with the default split point: max-abs 1.6-4.6e-3; an fp16-storage model of the network on the
// host gives 0.9-3e-3 for every split point from L1b's output on and rounding-level error with L1a's output split).
static int split_point(int norm) { return norm == NAFP_NORM_BATCH_NORM ? 1 : ENC_SPLIT_FROM; }

// the weight operands and their tensor maps: sized by the split point of the geometry
static int encoder_weight_buffers(EncoderState* s) {
    for (int l = 1; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        if (s->wt[l]) cudaFree(s->wt[l]);
        s->wt[l] = nullptr;
        NAFP_CUDA(cudaMalloc(&s->wt[l], static_cast<size_t>(L.c_out) * 3 * L.c_in * L.ksplit * sizeof(__half)));
        const uint64_t C = static_cast<uint64_t>(L.c_in) * L.ksplit;
        const uint64_t wd[2] = {3 * C, static_cast<uint64_t>(L.c_out)};
        const uint64_t ws[2] = {2, 3 * C * 2};
        const uint32_t wb[2] = {64, static_cast<uint32_t>(L.nt)};
        NAFP_TRY(make_tensor_map(&s->tmB[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, s->wt[l], wd, ws, wb, nullptr,
                                 CU_TENSOR_MAP_SWIZZLE_128B));
    }
    return NAFP_OK;
}

static int encoder_init(nafp_ctx* ctx) {
    if (ctx->encoder) return NAFP_OK;
    EncoderState* s = new EncoderState();
    ctx->encoder = s;              // before the first fallible call: nafp_ctx_destroy releases it
    s->split_from = split_point(NAFP_NORM_LAYER_NORM2D);
    build_geometry(s->g, s->split_from);
    NAFP_CUDA(cudaMalloc(&s->w0, 3 * 128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->bias0, 128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->ln_b15, 1024 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->ln_c, ENC_LAYERS * 2048 * sizeof(float)));
    for (int l = 0; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        const size_t per = static_cast<size_t>(L.ms) * L.c_out;
        NAFP_CUDA(cudaMalloc(&s->ln_g[l], per * sizeof(float)));
        if (l == 0) continue;
        NAFP_CUDA(cudaMalloc(&s->cbeta[l], per * sizeof(float)));
        NAFP_CUDA(cudaMalloc(&s->cgam[l], per * sizeof(__half)));
    }
    NAFP_CUDA(cudaMalloc(&s->dw1, 128 * 8 * 32 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->db1, 128 * 32 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->dw2, 128 * 32 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->db2, 128 * sizeof(float)));
    NAFP_TRY(encoder_weight_buffers(s));
    NAFP_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM));
    NAFP_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, CONV_SMEM));
    NAFP_CUDA(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
        NAFP_CUDA(cudaEventCreateWithFlags(&s->ev_up[b], cudaEventDisableTiming));
        NAFP_CUDA(cudaEventCreateWithFlags(&s->ev_free[b], cudaEventDisableTiming));
    }
    return NAFP_OK;
}

static void encoder_release_arena(EncoderState* s) {
    for (int l = 0; l < ENC_LAYERS; ++l) {
        if (s->x[l]) cudaFree(s->x[l]);
        s->x[l] = nullptr;
    }
    void** bufs[] = {reinterpret_cast<void**>(&s->stat), reinterpret_cast<void**>(&s->unit), reinterpret_cast<void**>(&s->part),
                     reinterpret_cast<void**>(&s->raw), reinterpret_cast<void**>(&s->mel), &s->xin[0], &s->xin[1],
                     reinterpret_cast<void**>(&s->emb)};
    for (void** b : bufs) {
        if (*b) cudaFree(*b);
        *b = nullptr;
    }
    s->cap = 0;
    s->last_n = 0;
}

// The activation arena (2.3 MB per segment) and the activation tensor maps are sized for `cap` segments; a pass of
// more segments than that re-allocates them (ENC_CHUNK_MIN, then the request rounded up to 1,000, <= ENC_CHUNK_MAX).
static int encoder_reserve(nafp_ctx* ctx, int64_t n) {
    EncoderState* s = ctx->encoder;
    if (n <= s->cap) return NAFP_OK;
    int64_t cap = (n + 999) / 1000 * 1000;
    if (cap < ENC_CHUNK_MIN) cap = ENC_CHUNK_MIN;
    if (cap > ENC_CHUNK_MAX) cap = ENC_CHUNK_MAX;
    NAFP_REQUIRE(n <= cap, NAFP_ERR_INVALID, "encoder: %lld segments in one pass (at most %d)", (long long)n, ENC_CHUNK_MAX);
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    encoder_release_arena(s);
    for (int l = 0; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        const size_t per = static_cast<size_t>(L.ms) * L.c_out;
        // +128 rows of slack: the GEMM epilogue never writes past m_total, TMA boxes may read past it
        const size_t x_elems = (static_cast<size_t>(cap) * per + 128 * L.c_out) * L.osplit;
        NAFP_CUDA(cudaMalloc(&s->x[l], x_elems * sizeof(__half)));
        NAFP_CUDA(cudaMemset(s->x[l], 0, x_elems * sizeof(__half)));
    }
    NAFP_CUDA(cudaMalloc(&s->stat, static_cast<size_t>(ENC_LAYERS) * cap * sizeof(float2)));
    {
        const std::vector<float2> unit(static_cast<size_t>(cap), make_float2(1.f, 0.f));
        NAFP_CUDA(cudaMalloc(&s->unit, unit.size() * sizeof(float2)));
        NAFP_CUDA(cudaMemcpy(s->unit, unit.data(), unit.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    NAFP_CUDA(cudaMalloc(&s->part, static_cast<size_t>(cap) * PART_SLOTS * 2 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->mel, static_cast<size_t>(cap) * 8192 * sizeof(float)));
    for (int b = 0; b < 2; ++b) NAFP_CUDA(cudaMalloc(&s->xin[b], static_cast<size_t>(cap) * 8000 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->emb, static_cast<size_t>(cap) * EMB * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&s->raw, static_cast<size_t>(cap) * EMB * sizeof(float)));
    // activation tensor maps (rows past the live batch are masked by the epilogue)
    for (int l = 1; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        const uint64_t C = static_cast<uint64_t>(L.c_in) * L.ksplit, T = L.t_in, F = L.f_in, B = cap;
        uint64_t dims[5], str[5];
        uint32_t box[5];
        int rank;
        if (L.mode == 0 || L.mode == 3) {
            rank = 4;
            dims[0] = C; dims[1] = T; dims[2] = F; dims[3] = B;
            str[0] = 2; str[1] = C * 2; str[2] = T * C * 2; str[3] = F * T * C * 2;
            box[0] = 64; box[1] = L.bt; box[2] = L.bf; box[3] = L.bb;
        } else if (L.mode == 1) {
            rank = 5;
            dims[0] = C; dims[1] = 2; dims[2] = T / 2; dims[3] = F; dims[4] = B;
            str[0] = 2; str[1] = C * 2; str[2] = 2 * C * 2; str[3] = T * C * 2; str[4] = F * T * C * 2;
            box[0] = 64; box[1] = 1; box[2] = L.bt; box[3] = L.bf; box[4] = L.bb;
        } else {
            rank = 5;
            dims[0] = C; dims[1] = T; dims[2] = 2; dims[3] = F / 2; dims[4] = B;
            str[0] = 2; str[1] = C * 2; str[2] = T * C * 2; str[3] = 2 * T * C * 2; str[4] = F * T * C * 2;
            box[0] = 64; box[1] = L.bt; box[2] = 1; box[3] = L.bf; box[4] = L.bb;
        }
        NAFP_TRY(make_tensor_map(&s->tmA[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, s->x[l - 1], dims, str, box, nullptr,
                                 CU_TENSOR_MAP_SWIZZLE_128B));
        // output map for the TMA-store layers: rows = NHWC positions of all segments, box = 128 rows x 64 channels
        const uint64_t od[2] = {static_cast<uint64_t>(L.c_out) * L.osplit, static_cast<uint64_t>(cap) * L.ms + 128};
        const uint64_t os[2] = {2, static_cast<uint64_t>(L.c_out) * L.osplit * 2};
        const uint32_t ob[2] = {64, 128};
        NAFP_TRY(make_tensor_map(&s->tmO[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, s->x[l], od, os, ob, nullptr,
                                 CU_TENSOR_MAP_SWIZZLE_128B));
    }
    s->cap = static_cast<int>(cap);
    return NAFP_OK;
}

void encoder_destroy(nafp_ctx* ctx) {
    EncoderState* s = ctx->encoder;
    if (!s) return;
    encoder_release_arena(s);
    for (int l = 0; l < ENC_LAYERS; ++l) {
        void* bufs[] = {s->ln_g[l], s->cbeta[l], s->cgam[l], s->wt[l]};
        for (void* b : bufs) if (b) cudaFree(b);
    }
    void* bufs[] = {s->w0, s->bias0, s->ln_b15, s->ln_c, s->dw1, s->db1, s->dw2, s->db2};
    for (void* b : bufs) if (b) cudaFree(b);
    for (int b = 0; b < 2; ++b) {
        if (s->ev_up[b]) cudaEventDestroy(s->ev_up[b]);
        if (s->ev_free[b]) cudaEventDestroy(s->ev_free[b]);
    }
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    delete s;
    ctx->encoder = nullptr;
}

// (a, c) of layer l's stored activation: per-segment LayerNorm statistics, or (1, 0) where the stored values need no
// per-segment factor -- layers 0 .. 14 of 'layer_norm1d' (stored normalised by conv0 / ln1d_kernel; the last layer's
// output is one position, where the per-channel LayerNorm is the per-segment one) and every layer of 'batch_norm'
// (its affine map is in the planes)
static bool layer_has_stats(const EncoderState* s, int l) {
    return s->norm == NAFP_NORM_LAYER_NORM2D || (s->norm == NAFP_NORM_LAYER_NORM1D && l == ENC_LAYERS - 1);
}
static float2* layer_stat(const EncoderState* s, int l) {
    return layer_has_stats(s, l) ? s->stat + static_cast<size_t>(l) * s->cap : s->unit;
}

// one pass over n <= cap segments (encoder_reserve); mel is either final (gmax == nullptr) or raw log-mel + group maxima
static int encoder_pass(nafp_ctx* ctx, const float* mel, const int32_t* gmax, int64_t group_size, int n, float* emb_dev) {
    EncoderState* s = ctx->encoder;
    cudaStream_t st = ctx->stream;
    const bool ln1d = s->norm == NAFP_NORM_LAYER_NORM1D;
    for (int l = 0; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        float2* stat = s->stat + static_cast<size_t>(l) * s->cap;
        const int per = L.ms * L.c_out;
        int slots;
        if (l == 0) {
            auto kern = ln1d ? conv0_kernel<true> : L.osplit != 1 ? conv0_kernel<false, true> : conv0_kernel<false>;
            kern<<<dim3(256 / CONV0_ROWS, (n + CONV0_SEGS - 1) / CONV0_SEGS), 256, 0, st>>>(
                mel, gmax, group_size, n, s->w0, s->bias0, s->ln_g[0], s->x[0], s->part, ln1d ? s->ln_c : nullptr);
            slots = CONV0_SLOTS;
        } else {
            ConvParams p;
            p.m_total = n * L.ms; p.ms = L.ms; p.n_seg = n; p.c_in = L.c_in * L.ksplit; p.c_out = L.c_out;
            p.n_ntiles = L.c_out / L.nt;
            p.mode = L.mode; p.pad_lo = L.pad_lo; p.tap_lo = L.tap_lo; p.tap_hi = L.tap_hi;
            p.kb_per_tap = L.c_in * L.ksplit / 64; p.bf = L.bf; p.bb = L.bb;
            p.groups = L.ms >= 32 ? L.ms / 32 : 1;
            p.osplit = L.osplit;
            p.combos = (L.ms >= 128 ? L.ms / 128 : 1) * p.n_ntiles;
            p.n_units = L.ms >= 128 ? n : (p.m_total + 127) / 128;
            p.n_streams = ctx->sm_count / p.combos;
            if (p.n_streams > p.n_units) p.n_streams = p.n_units;
            if (p.n_streams < 1) p.n_streams = 1;
            p.tma_store = (L.nt == 128 && L.ms >= 128 && L.osplit == 1 && CONV_EPI_PARTS == 2) ? 1 : 0;
            slots = p.groups * p.n_ntiles * CONV_EPI_PARTS;
            auto kern = L.nt == 128 ? conv_gemm_kernel<128> : conv_gemm_kernel<256>;
            kern<<<p.combos * p.n_streams, CONV_THREADS, CONV_SMEM, st>>>(
                s->tmA[l], s->tmB[l], s->tmO[l], p, layer_stat(s, l - 1), s->ln_g[l], s->cbeta[l], s->cgam[l],
                s->x[l], s->part);
            if (ln1d && l < ENC_LAYERS - 1) {
                const int64_t n_pos = static_cast<int64_t>(n) * L.ms;
                const unsigned blocks = static_cast<unsigned>((n_pos + 7) / 8);
                const float* g1 = s->ln_c + static_cast<size_t>(l) * 2048;
                const int sp = L.osplit != 1;
                auto kern1 = L.c_out == 128 ? ln1d_kernel<4> : L.c_out == 256 ? ln1d_kernel<8>
                           : L.c_out == 512 ? ln1d_kernel<16> : ln1d_kernel<32>;
                kern1<<<blocks, 256, 0, st>>>(s->x[l], n_pos, sp, g1, g1 + 1024);
                ctx->launches += 1;
            }
        }
        ctx->launches += 1;
        if (layer_has_stats(s, l)) {
            ln_stats_kernel<<<(n + 7) / 8, 256, 0, st>>>(s->part, slots, per, n, stat);
            ctx->launches += 1;
        }
    }
    divenc_kernel<<<dim3(EMB, (n + 127) / 128), 128, 0, st>>>(s->x[ENC_LAYERS - 1], layer_stat(s, ENC_LAYERS - 1),
                                                              s->ln_g[ENC_LAYERS - 1], s->ln_b15, n, s->dw1, s->db1, s->dw2,
                                                              s->db2, s->raw);
    l2norm_kernel<<<(n * 32 + 255) / 256, 256, 0, st>>>(s->raw, n, emb_dev);
    ctx->launches += 2;
    NAFP_CUDA(cudaGetLastError());
    s->last_n = n;
    return NAFP_OK;
}

static int fingerprint_dev(nafp_ctx* ctx, const void* x_dev, bool pcm16, int64_t n_seg, int64_t group_size,
                           float* emb_dev, const int64_t* seg_off = nullptr, const int32_t* seg_valid = nullptr) {
    EncoderState* s = ctx->encoder;
    // chunks are whole groups so that every group's batch-global max is complete (melspectrogram.py:108)
    int64_t chunk = group_size <= ENC_CHUNK_MAX ? (ENC_CHUNK_MAX / group_size) * group_size : 0;
    NAFP_REQUIRE(chunk > 0, NAFP_ERR_UNSUPPORTED, "fingerprint: group_size %lld exceeds the %d-segment encoder pass",
                 (long long)group_size, ENC_CHUNK_MAX);
    NAFP_TRY(encoder_reserve(ctx, n_seg < chunk ? n_seg : chunk));
    const size_t elt = pcm16 ? sizeof(int16_t) : sizeof(float);
    // 'melspec_maxnorm' needs the group minimum as well: the log-mel is finished by its own elementwise pass
    // instead of being folded into conv0
    const bool finish = logmel_segment_norm(ctx);
    for (int64_t s0 = 0; s0 < n_seg; s0 += chunk) {
        const int n = static_cast<int>(n_seg - s0 < chunk ? n_seg - s0 : chunk);
        const int32_t* gmax = nullptr;
        // (n_seg, 8000) rows, or windows of track sample runs addressed through seg_off (absolute sample offsets)
        const void* xin = seg_off ? x_dev : static_cast<const uint8_t*>(x_dev) + static_cast<size_t>(s0) * 8000 * elt;
        NAFP_TRY(logmel_run(ctx, xin, pcm16, n, group_size, s->mel, finish, &gmax, seg_off ? seg_off + s0 : nullptr,
                            seg_valid ? seg_valid + s0 : nullptr));
        NAFP_TRY(encoder_pass(ctx, s->mel, finish ? nullptr : gmax, group_size, n, emb_dev + s0 * EMB));
    }
    return NAFP_OK;
}

}  // namespace nafp

using namespace nafp;

extern "C" {

int nafp_weights_load(nafp_ctx* ctx, const float* const* conv_w, const float* const* conv_b, const float* const* ln_g,
                      const float* const* ln_b, const float* div_w1, const float* div_b1, const float* div_w2,
                      const float* div_b2) {
    return nafp_weights_load_norm(ctx, NAFP_NORM_LAYER_NORM2D, conv_w, conv_b, ln_g, ln_b, nullptr, nullptr, div_w1, div_b1,
                                  div_w2, div_b2);
}

// The other MODEL.BN values run through the same GEMM kernels with other per-element planes and per-segment factors:
//   'layer_norm1d': layers 0 .. 14 store their output normalised (conv0_kernel<true> / ln1d_kernel, per-channel
//                gamma / beta in ln_c), so their planes are 1 / 0 and their consumers read (a, c) = (1, 0); the last
//                layer's output is one position, where the per-channel LayerNorm is the per-segment one with (1, 1, C)
//                parameters: the layer_norm2d path;
//   'batch_norm' (inference): y -> s y + t per channel, s = gamma / sqrt(var + eps), t = beta - mean s (fp64 here),
//                is the fold with (a, c) = (1, 0) and the planes s / t broadcast over (F,T): the layers store
//                z = s (.) y, fold_kernel gives Cb = bias + conv(t), the head adds t.  No statistics, no extra pass;
//                every layer runs split precision (split_point), so z keeps what t cancels later.
// The split point belongs to the norm: a load that changes it rebuilds the geometry, the weight operands and the
// activation arena.  Every pointer is checked before the first device write.
int nafp_weights_load_norm(nafp_ctx* ctx, int32_t norm, const float* const* conv_w, const float* const* conv_b,
                           const float* const* norm_g, const float* const* norm_b, const float* const* norm_mean,
                           const float* const* norm_var, const float* div_w1, const float* div_b1, const float* div_w2,
                           const float* div_b2) {
    NAFP_RANGE("nafp_weights_load");
    NAFP_REQUIRE(ctx && conv_w && conv_b && norm_g && norm_b && div_w1 && div_b1 && div_w2 && div_b2, NAFP_ERR_INVALID,
                 "nafp_weights_load: NULL argument");
    NAFP_REQUIRE(norm == NAFP_NORM_LAYER_NORM2D || norm == NAFP_NORM_LAYER_NORM1D || norm == NAFP_NORM_BATCH_NORM,
                 NAFP_ERR_INVALID, "nafp_weights_load_norm: norm %d (0 layer_norm2d, 1 layer_norm1d, 2 batch_norm)", (int)norm);
    const bool bn = norm == NAFP_NORM_BATCH_NORM;
    NAFP_REQUIRE(bn ? (norm_mean && norm_var) : (!norm_mean && !norm_var), NAFP_ERR_INVALID,
                 "nafp_weights_load_norm: norm_mean / norm_var are given exactly for batch_norm");
    for (int l = 0; l < ENC_LAYERS; ++l)
        NAFP_REQUIRE(conv_w[l] && conv_b[l] && norm_g[l] && norm_b[l] && (!bn || (norm_mean[l] && norm_var[l])),
                     NAFP_ERR_INVALID, "nafp_weights_load: layer %d NULL", l);
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_TRY(encoder_init(ctx));
    EncoderState* s = ctx->encoder;
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    s->weights = false;                // until this load completes
    const int split_from = split_point(norm);
    if (split_from != s->split_from) {
        encoder_release_arena(s);      // activation sizes and maps follow the split point (encoder_reserve)
        build_geometry(s->g, split_from);
        s->split_from = split_from;
        NAFP_TRY(encoder_weight_buffers(s));
    }
    // per-layer planes: the caller's (F,T,C) arrays for layer_norm2d, built here otherwise
    std::vector<float> plane_g[ENC_LAYERS], plane_b[ENC_LAYERS];
    const float* ln_g[ENC_LAYERS];
    const float* ln_b[ENC_LAYERS];
    std::vector<float> lnc;
    if (norm == NAFP_NORM_LAYER_NORM1D) lnc.assign(static_cast<size_t>(ENC_LAYERS) * 2048, 0.f);
    for (int l = 0; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        if (norm == NAFP_NORM_LAYER_NORM2D) {
            ln_g[l] = norm_g[l];
            ln_b[l] = norm_b[l];
            continue;
        }
        const int C = L.c_out;
        std::vector<float> sc(C), sh(C);
        for (int c = 0; c < C; ++c) {
            const float g = norm_g[l][c], b = norm_b[l][c];
            if (bn) {
                const double k = static_cast<double>(g) / std::sqrt(static_cast<double>(norm_var[l][c]) + LN_EPS);
                sc[c] = static_cast<float>(k);
                sh[c] = static_cast<float>(static_cast<double>(b) - static_cast<double>(norm_mean[l][c]) * k);
            } else if (l == ENC_LAYERS - 1) {
                sc[c] = g;
                sh[c] = b;
            } else {
                sc[c] = 1.f;
                sh[c] = 0.f;
                lnc[static_cast<size_t>(l) * 2048 + c] = g;
                lnc[static_cast<size_t>(l) * 2048 + 1024 + c] = b;
            }
        }
        plane_g[l].resize(static_cast<size_t>(L.ms) * C);
        plane_b[l].resize(static_cast<size_t>(L.ms) * C);
        for (int pos = 0; pos < L.ms; ++pos) {
            std::copy(sc.begin(), sc.end(), plane_g[l].begin() + static_cast<size_t>(pos) * C);
            std::copy(sh.begin(), sh.end(), plane_b[l].begin() + static_cast<size_t>(pos) * C);
        }
        ln_g[l] = plane_g[l].data();
        ln_b[l] = plane_b[l].data();
    }
    if (!lnc.empty())
        NAFP_CUDA(cudaMemcpy(s->ln_c, lnc.data(), lnc.size() * sizeof(float), cudaMemcpyHostToDevice));
    struct Tmp {                       // fp32 weights / beta of the running layer, only needed by fold_kernel
        float *w = nullptr, *bias = nullptr, *beta_prev = nullptr, *beta_cur = nullptr;
        ~Tmp() { cudaFree(w); cudaFree(bias); cudaFree(beta_prev); cudaFree(beta_cur); }
    } tmp;
    NAFP_CUDA(cudaMalloc(&tmp.w, static_cast<size_t>(3) * 1024 * 1024 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&tmp.bias, 1024 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&tmp.beta_prev, static_cast<size_t>(256) * 16 * 128 * sizeof(float)));
    NAFP_CUDA(cudaMalloc(&tmp.beta_cur, static_cast<size_t>(256) * 16 * 128 * sizeof(float)));
    for (int l = 0; l < ENC_LAYERS; ++l) {
        const ConvGeom& L = s->g[l];
        NAFP_REQUIRE(conv_w[l] && conv_b[l] && ln_g[l] && ln_b[l], NAFP_ERR_INVALID, "nafp_weights_load: layer %d NULL", l);
        const size_t per = static_cast<size_t>(L.ms) * L.c_out;
        s->h_g[l].assign(ln_g[l], ln_g[l] + per);
        s->h_b[l].assign(ln_b[l], ln_b[l] + per);
        NAFP_CUDA(cudaMemcpy(s->ln_g[l], ln_g[l], per * sizeof(float), cudaMemcpyHostToDevice));
        NAFP_CUDA(cudaMemcpy(tmp.beta_cur, ln_b[l], per * sizeof(float), cudaMemcpyHostToDevice));
        if (l == 0) {
            NAFP_CUDA(cudaMemcpy(s->w0, conv_w[0], 3 * 128 * sizeof(float), cudaMemcpyHostToDevice));
            NAFP_CUDA(cudaMemcpy(s->bias0, conv_b[0], 128 * sizeof(float), cudaMemcpyHostToDevice));
        } else {
            // HWIO [tap][cin][cout] -> K-major B operand [cout][tap*cin + cin] in fp16
            // split layers: per tap [hi | lo | hi], matching the [hi | hi | lo] activations
            const int ce = L.c_in * L.ksplit, K = 3 * ce;
            std::vector<__half> wt(static_cast<size_t>(L.c_out) * K);
            for (int tap = 0; tap < 3; ++tap)
                for (int ci = 0; ci < L.c_in; ++ci) {
                    const float* src = conv_w[l] + (static_cast<size_t>(tap) * L.c_in + ci) * L.c_out;
                    for (int co = 0; co < L.c_out; ++co) {
                        const __half hi = __float2half_rn(src[co]);
                        __half* row = &wt[static_cast<size_t>(co) * K + tap * ce];
                        row[ci] = hi;
                        if (L.ksplit == 3) {
                            row[L.c_in + ci] = __float2half_rn(src[co] - __half2float(hi));
                            row[2 * L.c_in + ci] = hi;
                        }
                    }
                }
            NAFP_CUDA(cudaMemcpy(s->wt[l], wt.data(), wt.size() * sizeof(__half), cudaMemcpyHostToDevice));
            // the previous layer's LayerNorm folded through this convolution: Cg = conv(gamma_prev), Cb = bias + conv(beta_prev)
            NAFP_CUDA(cudaMemcpy(tmp.w, conv_w[l], static_cast<size_t>(3) * L.c_in * L.c_out * sizeof(float), cudaMemcpyHostToDevice));
            NAFP_CUDA(cudaMemcpy(tmp.bias, conv_b[l], L.c_out * sizeof(float), cudaMemcpyHostToDevice));
            fold_kernel<<<dim3((L.c_out + 127) / 128, L.ms), 128, 0, ctx->stream>>>(tmp.w, tmp.bias, s->ln_g[l - 1], tmp.beta_prev, L,
                                                                                   L.ksplit == 1 ? 1 : 0, s->cgam[l], s->cbeta[l]);
            ctx->launches += 1;
            NAFP_CUDA(cudaGetLastError());
            NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
        }
        std::swap(tmp.beta_prev, tmp.beta_cur);
    }
    NAFP_CUDA(cudaMemcpy(s->ln_b15, ln_b[ENC_LAYERS - 1], 1024 * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->dw1, div_w1, 128 * 8 * 32 * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->db1, div_b1, 128 * 32 * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->dw2, div_w2, 128 * 32 * sizeof(float), cudaMemcpyHostToDevice));
    NAFP_CUDA(cudaMemcpy(s->db2, div_b2, 128 * sizeof(float), cudaMemcpyHostToDevice));
    s->norm = norm;
    s->weights = true;
    return NAFP_OK;
}

int nafp_encoder_forward(nafp_ctx* ctx, const float* mel_dev, int64_t n_seg, float* emb_dev) {
    NAFP_RANGE("nafp_encoder_forward");
    NAFP_REQUIRE(ctx && n_seg >= 0 && (n_seg == 0 || (mel_dev && emb_dev)), NAFP_ERR_INVALID,
                 "nafp_encoder_forward: bad arguments");
    NAFP_REQUIRE(ctx->encoder && ctx->encoder->weights, NAFP_ERR_STATE, "nafp_encoder_forward: call nafp_weights_load first");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_TRY(encoder_reserve(ctx, n_seg < ENC_CHUNK_MAX ? n_seg : ENC_CHUNK_MAX));
    for (int64_t s0 = 0; s0 < n_seg; s0 += ENC_CHUNK_MAX) {
        const int n = static_cast<int>(n_seg - s0 < ENC_CHUNK_MAX ? n_seg - s0 : ENC_CHUNK_MAX);
        NAFP_TRY(encoder_pass(ctx, mel_dev + s0 * 8192, nullptr, 1, n, emb_dev + s0 * EMB));
    }
    return NAFP_OK;
}

int nafp_fingerprint(nafp_ctx* ctx, const float* x_dev, int64_t n_seg, int64_t group_size, float* emb_dev) {
    NAFP_RANGE("nafp_fingerprint");
    NAFP_REQUIRE(ctx && n_seg >= 0 && group_size >= 1 && (n_seg == 0 || (x_dev && emb_dev)), NAFP_ERR_INVALID,
                 "nafp_fingerprint: bad arguments");
    NAFP_REQUIRE(ctx->encoder && ctx->encoder->weights, NAFP_ERR_STATE, "nafp_fingerprint: call nafp_weights_load first");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    return fingerprint_dev(ctx, x_dev, false, n_seg, group_size, emb_dev);
}

static int fingerprint_host(nafp_ctx* ctx, const void* x_host, bool pcm16, int64_t n_seg, int64_t group_size,
                            float* emb_host) {
    NAFP_REQUIRE(ctx && n_seg >= 0 && group_size >= 1 && (n_seg == 0 || (x_host && emb_host)), NAFP_ERR_INVALID,
                 "nafp_fingerprint_host: bad arguments");
    NAFP_REQUIRE(ctx->encoder && ctx->encoder->weights, NAFP_ERR_STATE, "nafp_fingerprint_host: call nafp_weights_load first");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    EncoderState* s = ctx->encoder;
    const int64_t chunk = group_size <= ENC_CHUNK_MAX ? (ENC_CHUNK_MAX / group_size) * group_size : 0;
    NAFP_REQUIRE(chunk > 0, NAFP_ERR_UNSUPPORTED, "fingerprint: group_size %lld exceeds the %d-segment encoder pass",
                 (long long)group_size, ENC_CHUNK_MAX);
    NAFP_TRY(encoder_reserve(ctx, n_seg < chunk ? n_seg : chunk));      // before s->xin / s->emb are read below
    const size_t elt = pcm16 ? sizeof(int16_t) : sizeof(float);
    const uint8_t* src = static_cast<const uint8_t*>(x_host);
    // Pieces of whole groups: a short first piece (its upload is the only one no kernel hides: 16 MB instead of 64 MB
    // of int16 PCM), then full encoder passes; the upload of piece i + 1 runs on the copy stream under the kernels of
    // piece i.
    std::vector<int64_t> piece_at;           // start segment of every piece, + n_seg
    {
        int64_t first = (1000 / group_size) * group_size;
        if (first < group_size) first = group_size;
        if (first > chunk || n_seg < 2 * first) first = chunk;
        for (int64_t s0 = 0; s0 < n_seg; s0 += (s0 == 0 ? first : chunk)) piece_at.push_back(s0);
        piece_at.push_back(n_seg);
    }
    const int n_pieces = static_cast<int>(piece_at.size()) - 1;
    auto upload = [&](int i, int b) -> cudaError_t {      // piece i -> xin[b], on the copy stream
        const int64_t s0 = piece_at[i], n = piece_at[i + 1] - s0;
        cudaError_t e = cudaStreamWaitEvent(s->copy_stream, s->ev_free[b], 0);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s->xin[b], src + static_cast<size_t>(s0) * 8000 * elt, static_cast<size_t>(n) * 8000 * elt,
                                cudaMemcpyHostToDevice, s->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(s->ev_up[b], s->copy_stream);
        return e;
    };
    // the copy stream starts behind everything already queued on the compute stream (it may still read xin[0/1])
    for (int b = 0; b < 2; ++b) NAFP_CUDA(cudaEventRecord(s->ev_free[b], ctx->stream));
    if (n_pieces > 0) NAFP_CUDA(upload(0, 0));
    for (int i = 0, b = 0; i < n_pieces; ++i, b ^= 1) {
        const int64_t s0 = piece_at[i], n = piece_at[i + 1] - s0;
        if (i + 1 < n_pieces) NAFP_CUDA(upload(i + 1, b ^ 1));     // under this piece's kernels
        NAFP_CUDA(cudaStreamWaitEvent(ctx->stream, s->ev_up[b], 0));
        NAFP_TRY(fingerprint_dev(ctx, s->xin[b], pcm16, n, group_size, s->emb));
        NAFP_CUDA(cudaEventRecord(s->ev_free[b], ctx->stream));
        NAFP_CUDA(cudaMemcpyAsync(emb_host + s0 * EMB, s->emb, static_cast<size_t>(n) * EMB * sizeof(float),
                                  cudaMemcpyDeviceToHost, ctx->stream));
    }
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

int nafp_fingerprint_host(nafp_ctx* ctx, const float* x_host, int64_t n_seg, int64_t group_size, float* emb_host) {
    NAFP_RANGE("nafp_fingerprint_host");
    return fingerprint_host(ctx, x_host, false, n_seg, group_size, emb_host);
}
int nafp_fingerprint_pcm16_host(nafp_ctx* ctx, const int16_t* pcm_host, int64_t n_seg, int64_t group_size,
                                float* emb_host) {
    NAFP_RANGE("nafp_fingerprint_pcm16_host");
    return fingerprint_host(ctx, pcm_host, true, n_seg, group_size, emb_host);
}

// generate.py's path: whole-track int16 sample runs + one (offset, valid length) pair per segment; the overlapping
// 1 s segments (0.5 s hop) are cut by the log-mel kernel, so every sample is uploaded once instead of twice and the
// host never materialises the (n_seg, 8000) array.
int nafp_fingerprint_pcm16_tracks_host(nafp_ctx* ctx, const int16_t* pcm_host, int64_t n_samples, const int64_t* seg_off_host,
                                       const int32_t* seg_valid_host, int64_t n_seg, int64_t group_size, float* emb_host) {
    NAFP_RANGE("nafp_fingerprint_pcm16_tracks_host");
    NAFP_REQUIRE(ctx && n_seg >= 0 && n_samples >= 0 && group_size >= 1 &&
                     (n_seg == 0 || (pcm_host && seg_off_host && seg_valid_host && emb_host)),
                 NAFP_ERR_INVALID, "nafp_fingerprint_pcm16_tracks_host: bad arguments");
    NAFP_REQUIRE(ctx->encoder && ctx->encoder->weights, NAFP_ERR_STATE,
                 "nafp_fingerprint_pcm16_tracks_host: call nafp_weights_load first");
    if (n_seg == 0) return NAFP_OK;
    for (int64_t i = 0; i < n_seg; ++i)
        NAFP_REQUIRE(seg_off_host[i] >= 0 && seg_valid_host[i] >= 0 && seg_valid_host[i] <= 8000 &&
                         seg_off_host[i] + seg_valid_host[i] <= n_samples,
                     NAFP_ERR_INVALID, "nafp_fingerprint_pcm16_tracks_host: segment %lld reads [%lld, +%d) of %lld samples",
                     (long long)i, (long long)seg_off_host[i], (int)seg_valid_host[i], (long long)n_samples);
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));      // the staging buffer may be re-allocated below
    // one staging buffer, every part 256-byte aligned: samples (+1 so that it is never empty), offsets, valid
    // lengths, fingerprints
    const int64_t pcm_bytes = (n_samples + 1) * 2, pcm_pad = (pcm_bytes + 255) / 256 * 256;
    const int64_t off_bytes = (n_seg * 8 + 255) / 256 * 256, val_bytes = (n_seg * 4 + 255) / 256 * 256;
    const int64_t emb_bytes = n_seg * EMB * static_cast<int64_t>(sizeof(float));
    NAFP_TRY(ensure_dev(ctx, &ctx->stage_dev, &ctx->stage_dev_bytes, pcm_pad + off_bytes + val_bytes + emb_bytes));
    uint8_t* base = static_cast<uint8_t*>(ctx->stage_dev);
    int16_t* pcm_dev = reinterpret_cast<int16_t*>(base);
    int64_t* off_dev = reinterpret_cast<int64_t*>(base + pcm_pad);
    int32_t* val_dev = reinterpret_cast<int32_t*>(base + pcm_pad + off_bytes);
    float* emb_dev = reinterpret_cast<float*>(base + pcm_pad + off_bytes + val_bytes);
    NAFP_CUDA(cudaMemcpyAsync(pcm_dev, pcm_host, static_cast<size_t>(n_samples) * 2, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(off_dev, seg_off_host, static_cast<size_t>(n_seg) * 8, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(val_dev, seg_valid_host, static_cast<size_t>(n_seg) * 4, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_TRY(fingerprint_dev(ctx, pcm_dev, true, n_seg, group_size, emb_dev, off_dev, val_dev));
    NAFP_CUDA(cudaMemcpyAsync(emb_host, emb_dev, static_cast<size_t>(emb_bytes), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

// The same for source files at any rate: the runs are resampled to one 8 kHz track buffer by one launch, which the
// segments then index as above.
int nafp_fingerprint_pcm16_sources_host(nafp_ctx* ctx, const int16_t* pcm_host, int64_t n_pcm, const int64_t* runs_host,
                                        int64_t n_runs, const int64_t* seg_off_host, const int32_t* seg_valid_host,
                                        int64_t n_seg, int64_t group_size, float* emb_host) {
    NAFP_RANGE("nafp_fingerprint_pcm16_sources_host");
    const char* fn = "nafp_fingerprint_pcm16_sources_host";
    NAFP_REQUIRE(ctx && n_seg >= 0 && n_pcm >= 0 && n_runs >= 0 && group_size >= 1 &&
                     (n_seg == 0 || (seg_off_host && seg_valid_host && emb_host)) && (n_runs == 0 || runs_host) &&
                     (n_pcm == 0 || pcm_host),
                 NAFP_ERR_INVALID, "%s: bad arguments", fn);
    NAFP_REQUIRE(ctx->encoder && ctx->encoder->weights, NAFP_ERR_STATE, "%s: call nafp_weights_load first", fn);
    std::vector<SourceRun> runs(static_cast<size_t>(n_runs));
    int64_t n_samples = 0;
    for (int64_t r = 0; r < n_runs; ++r) {
        const int64_t* u = runs_host + r * 7;
        NAFP_REQUIRE(u[3] >= 1 && u[3] <= 0x7fffffff && u[4] >= 1 && u[4] <= 0x7fffffff, u[3] < 1 || u[4] < 1 ? NAFP_ERR_INVALID : NAFP_ERR_UNSUPPORTED,
                     "%s: run %lld has %lld channels at %lld Hz", fn, (long long)r, (long long)u[3], (long long)u[4]);
        NAFP_TRY(resample_check_run(fn, u[1], u[2], static_cast<int32_t>(u[3]), static_cast<int32_t>(u[4]), 8000, u[5], u[6]));
        NAFP_REQUIRE(u[0] >= 0 && u[0] <= n_pcm && u[2] * u[3] <= n_pcm - u[0], NAFP_ERR_INVALID,
                     "%s: run %lld reads [%lld, +%lld) of %lld samples", fn, (long long)r, (long long)u[0],
                     (long long)(u[2] * u[3]), (long long)n_pcm);
        runs[r] = SourceRun{u[0], u[1], u[2], u[5], u[6], n_samples, static_cast<int32_t>(u[3]), static_cast<int32_t>(u[4])};
        n_samples += u[6];
    }
    for (int64_t i = 0; i < n_seg; ++i)
        NAFP_REQUIRE(seg_off_host[i] >= 0 && seg_valid_host[i] >= 0 && seg_valid_host[i] <= 8000 &&
                         seg_off_host[i] + seg_valid_host[i] <= n_samples,
                     NAFP_ERR_INVALID, "%s: segment %lld reads [%lld, +%d) of %lld resampled samples", fn, (long long)i,
                     (long long)seg_off_host[i], (int)seg_valid_host[i], (long long)n_samples);
    if (n_seg == 0) return NAFP_OK;
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));      // the staging buffer may be re-allocated below
    // one staging buffer, every part 256-byte aligned: source samples, 8 kHz samples (+1 so that neither is empty),
    // offsets, valid lengths, fingerprints
    const int64_t src_pad = ((n_pcm + 1) * 2 + 255) / 256 * 256, pcm_pad = ((n_samples + 1) * 2 + 255) / 256 * 256;
    const int64_t off_bytes = (n_seg * 8 + 255) / 256 * 256, val_bytes = (n_seg * 4 + 255) / 256 * 256;
    const int64_t emb_bytes = n_seg * EMB * static_cast<int64_t>(sizeof(float));
    NAFP_TRY(ensure_dev(ctx, &ctx->stage_dev, &ctx->stage_dev_bytes, src_pad + pcm_pad + off_bytes + val_bytes + emb_bytes));
    uint8_t* base = static_cast<uint8_t*>(ctx->stage_dev);
    int16_t* src_dev = reinterpret_cast<int16_t*>(base);
    int16_t* pcm_dev = reinterpret_cast<int16_t*>(base + src_pad);
    int64_t* off_dev = reinterpret_cast<int64_t*>(base + src_pad + pcm_pad);
    int32_t* val_dev = reinterpret_cast<int32_t*>(base + src_pad + pcm_pad + off_bytes);
    float* emb_dev = reinterpret_cast<float*>(base + src_pad + pcm_pad + off_bytes + val_bytes);
    NAFP_CUDA(cudaMemcpyAsync(src_dev, pcm_host, static_cast<size_t>(n_pcm) * 2, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(off_dev, seg_off_host, static_cast<size_t>(n_seg) * 8, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(val_dev, seg_valid_host, static_cast<size_t>(n_seg) * 4, cudaMemcpyHostToDevice, ctx->stream));
    NAFP_TRY(resample_launch(ctx, src_dev, runs.data(), n_runs, 8000, pcm_dev));
    NAFP_TRY(fingerprint_dev(ctx, pcm_dev, true, n_seg, group_size, emb_dev, off_dev, val_dev));
    NAFP_CUDA(cudaMemcpyAsync(emb_host, emb_dev, static_cast<size_t>(emb_bytes), cudaMemcpyDeviceToHost, ctx->stream));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

int nafp_encoder_activation_host(nafp_ctx* ctx, int layer, int64_t n_seg, float* out_host) {
    NAFP_RANGE("nafp_encoder_activation_host");
    NAFP_REQUIRE(ctx && ctx->encoder && out_host && layer >= 0 && layer < ENC_LAYERS, NAFP_ERR_INVALID,
                 "nafp_encoder_activation_host: bad arguments");
    EncoderState* s = ctx->encoder;
    NAFP_REQUIRE(n_seg >= 0 && n_seg <= s->last_n, NAFP_ERR_INVALID,
                 "nafp_encoder_activation_host: %lld segments requested, last pass had %lld", (long long)n_seg,
                 (long long)s->last_n);
    const ConvGeom& L = s->g[layer];
    const size_t per = static_cast<size_t>(L.ms) * L.c_out, n = static_cast<size_t>(n_seg) * per;
    std::vector<__half> tmp(n * L.osplit);
    std::vector<float2> st(static_cast<size_t>(n_seg));
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    NAFP_CUDA(cudaMemcpy(tmp.data(), s->x[layer], tmp.size() * sizeof(__half), cudaMemcpyDeviceToHost));
    NAFP_CUDA(cudaMemcpy(st.data(), layer_stat(s, layer), st.size() * sizeof(float2), cudaMemcpyDeviceToHost));
    // the device keeps z = gamma (.) ELU(...); LN(y) = a z + c gamma + beta with (a, c) = (rstd, -rstd mean) of the segment
    // ('layer_norm1d' before the last layer: z is the normalised value, (a, c) = (1, 0), gamma = 1, beta = 0;
    // 'batch_norm': (a, c) = (1, 0) and the planes are the folded scale / shift)
    const size_t C = L.c_out;
    for (size_t i = 0; i < n; ++i) {
        const size_t b = i / per, e = i % per;
        float z;
        if (L.osplit == 1) {
            z = __half2float(tmp[i]);
        } else {                // [hi | hi | lo] per position
            const size_t pos = i / C, c = i % C;
            z = __half2float(tmp[pos * 3 * C + c]) + __half2float(tmp[pos * 3 * C + 2 * C + c]);
        }
        out_host[i] = st[b].x * z + st[b].y * s->h_g[layer][e] + s->h_b[layer][e];
    }
    return NAFP_OK;
}

}  // extern "C"
