// Polyphase resampling of 16-bit PCM to the model rate, on the device: any rate with max(up, down) <= 1024, 1..8
// interleaved channels, int16 out.  The filter is resample_poly's default (firwin(2 hl + 1, 1 / max(up, down),
// window=('kaiser', 5.0)) * up, hl = 10 max(up, down)), built here in fp64; every output is one fp64 sum over
// ascending input frames, rounded half to even and saturated:
//   y[m] = rint_sat( sum_n s[n] h[hl + m down - n up] / C ),   s[n] = sum of the C channels of frame n (exact int)
// Equal rates need no filter: hl = 0 and h = {1}, so a mono run is a copy and a multi-channel run is round(mean).
#include <algorithm>
#include <cmath>
#include <map>
#include <numeric>
#include <utility>
#include <vector>

#include "common.h"

namespace nafp {

constexpr int RS_THREADS = 256;                       // one output per thread per sub-tile
constexpr int RS_SUBTILES = 16;                       // a CTA writes RS_THREADS * RS_SUBTILES outputs of one run
constexpr int64_t RS_TILE = int64_t(RS_THREADS) * RS_SUBTILES;
constexpr int RS_STAGE_MAX = 8192;                    // staged frames per chunk (fp64 channel sums)

struct RsFilter {                                      // polyphase table [phase p < up][tap k < K] = h[p + k up], 0-padded
    int32_t up, down, hl, K;
    const double* tab;
};
struct RsRun {
    int64_t pcm_off, frame0, n_frames, m0, n_out, out_off, tile0;
    int32_t channels, filt;
};

struct ResampleState {
    std::map<std::pair<int32_t, int32_t>, RsFilter> filters;     // (fs_in, fs_out) -> device table
    void* desc = nullptr;                                        // this call's filters + runs
    int64_t desc_bytes = 0;
    int smem_optin = 0;
};

__device__ __forceinline__ int64_t floor_div(int64_t a, int64_t b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// One CTA: RS_TILE consecutive outputs of one run, RS_THREADS at a time.  Per sub-tile the input frames it reads
// are staged in chunks of `stage` channel sums (ascending), so each thread's sum runs over ascending frames.
__global__ void __launch_bounds__(RS_THREADS) resample_kernel(const int16_t* __restrict__ pcm,
                                                              const RsRun* __restrict__ runs, int n_runs,
                                                              const RsFilter* __restrict__ filts, int tab_doubles,
                                                              int stage, int16_t* __restrict__ out) {
    extern __shared__ double rs_smem[];
    double* tab = rs_smem;
    double* xs = rs_smem + tab_doubles;
    const int64_t b = blockIdx.x;
    int lo = 0, hi = n_runs - 1;                      // the run whose tiles hold this CTA
    while (lo < hi) {
        const int mid = (lo + hi + 1) / 2;
        if (runs[mid].tile0 <= b) lo = mid; else hi = mid - 1;
    }
    const RsRun R = runs[lo];
    const RsFilter F = filts[R.filt];
    for (int i = threadIdx.x; i < F.up * F.K; i += RS_THREADS) tab[i] = F.tab[i];
    const int16_t* in = pcm + R.pcm_off;
    const int C = R.channels;
    const int64_t t0 = (b - R.tile0) * RS_TILE;                   // first output of the tile, relative to m0
    for (int st = 0; st < RS_SUBTILES; ++st) {
        const int64_t ra = t0 + int64_t(st) * RS_THREADS;
        if (ra >= R.n_out) break;                                  // uniform over the CTA
        const int64_t ma = R.m0 + ra;
        const int64_t mb = R.m0 + min(ra + RS_THREADS, R.n_out) - 1;
        const int64_t n_lo = floor_div(F.hl + ma * F.down, F.up) - (F.K - 1);
        const int64_t n_end = floor_div(F.hl + mb * F.down, F.up) + 1;
        const int64_t m = ma + threadIdx.x;
        const bool active = m <= mb;
        const int64_t nh = floor_div(F.hl + m * F.down, F.up);    // frame of tap 0
        const double* tp = tab + (F.hl + m * F.down - nh * F.up) * F.K;
        double acc = 0.0;
        for (int64_t c0 = n_lo; c0 < n_end; c0 += stage) {
            const int64_t c1 = min(c0 + stage, n_end);
            __syncthreads();                                       // the previous chunk is consumed
            for (int64_t n = c0 + threadIdx.x; n < c1; n += RS_THREADS) {
                const int64_t f = n - R.frame0;                     // frames outside the window read as zero
                int s = 0;
                if (f >= 0 && f < R.n_frames) {
                    const int16_t* q = in + f * C;
                    for (int c = 0; c < C; ++c) s += q[c];
                }
                xs[n - c0] = static_cast<double>(s);
            }
            __syncthreads();
            if (active) {
                // taps k with frame nh - k in [c0, c1), k descending = frames ascending
                const int k_hi = static_cast<int>(min(int64_t(F.K - 1), nh - c0));
                const int k_lo = static_cast<int>(max(int64_t(0), nh - c1 + 1));
                const double* xp = xs + (nh - c0);
#pragma unroll 4
                for (int k = k_hi; k >= k_lo; --k) acc = fma(xp[-k], tp[k], acc);
            }
        }
        if (active) {
            const double y = fmin(fmax(rint(acc / C), -32768.0), 32767.0);
            out[R.out_off + (m - R.m0)] = static_cast<int16_t>(y);
        }
    }
}

// I0 by its power series (converges fast for the Kaiser beta of 5)
static double bessel_i0(double x) {
    double sum = 1.0, term = 1.0;
    const double q = x * x / 4.0;
    for (int k = 1; k < 200; ++k) {
        term *= q / (static_cast<double>(k) * k);
        sum += term;
        if (term < 1e-17 * sum) break;
    }
    return sum;
}

int resample_ratio(int32_t fs_in, int32_t fs_out, int32_t* up, int32_t* down, int32_t* hl) {
    NAFP_REQUIRE(fs_in > 0 && fs_out > 0, NAFP_ERR_INVALID, "resample: sample rates %d -> %d must be positive",
                 (int)fs_in, (int)fs_out);
    const int32_t g = std::gcd(fs_in, fs_out);
    *up = fs_out / g;
    *down = fs_in / g;
    NAFP_REQUIRE(std::max(*up, *down) <= NAFP_RESAMPLE_MAX_RATIO, NAFP_ERR_UNSUPPORTED,
                 "resample: %d Hz -> %d Hz needs up %d / down %d; max(up, down) <= %d is supported", (int)fs_in,
                 (int)fs_out, (int)*up, (int)*down, NAFP_RESAMPLE_MAX_RATIO);
    *hl = *up == *down ? 0 : 10 * std::max(*up, *down);
    return NAFP_OK;
}

int resample_check_run(const char* fn, int64_t frame0, int64_t n_frames, int32_t channels, int32_t fs_in,
                       int32_t fs_out, int64_t m0, int64_t n_out) {
    NAFP_REQUIRE(channels >= 1, NAFP_ERR_INVALID, "%s: %d channels", fn, (int)channels);
    NAFP_REQUIRE(channels <= NAFP_RESAMPLE_MAX_CHANNELS, NAFP_ERR_UNSUPPORTED, "%s: %d channels; at most %d are supported",
                 fn, (int)channels, NAFP_RESAMPLE_MAX_CHANNELS);
    NAFP_REQUIRE(frame0 >= 0 && n_frames >= 0 && m0 >= 0 && n_out >= 0, NAFP_ERR_INVALID,
                 "%s: negative frame0 %lld / n_frames %lld / m0 %lld / n_out %lld", fn, (long long)frame0,
                 (long long)n_frames, (long long)m0, (long long)n_out);
    NAFP_REQUIRE(m0 <= (int64_t(1) << 40) && n_out <= (int64_t(1) << 40) && frame0 <= (int64_t(1) << 40) &&
                     n_frames <= (int64_t(1) << 40),
                 NAFP_ERR_INVALID, "%s: counts beyond 2^40", fn);
    int32_t up, down, hl;
    return resample_ratio(fs_in, fs_out, &up, &down, &hl);
}

static int resample_filter(nafp_ctx* ctx, int32_t fs_in, int32_t fs_out, RsFilter* out) {
    if (!ctx->resample) ctx->resample = new ResampleState();
    ResampleState* s = ctx->resample;
    auto it = s->filters.find({fs_in, fs_out});
    if (it != s->filters.end()) {
        *out = it->second;
        return NAFP_OK;
    }
    int32_t up, down, hl;
    NAFP_TRY(resample_ratio(fs_in, fs_out, &up, &down, &hl));
    const int L = 2 * hl + 1;
    std::vector<double> h(L, 1.0);
    if (hl > 0) {
        // scipy.signal.firwin(L, 1 / max(up, down), window=('kaiser', 5.0)), scaled to unit DC gain, then * up
        const double pi = 3.14159265358979323846, cut = 1.0 / std::max(up, down), beta = 5.0, alpha = 0.5 * (L - 1);
        const double i0b = bessel_i0(beta);
        double sum = 0.0;
        for (int i = 0; i < L; ++i) {
            const double t = i - alpha, x = cut * t;
            const double sinc = x == 0.0 ? 1.0 : std::sin(pi * x) / (pi * x);
            const double r = t / alpha;
            h[i] = cut * sinc * bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
        }
        for (int i = 0; i < L; ++i) sum += h[i];
        for (int i = 0; i < L; ++i) h[i] = h[i] / sum * up;
    }
    const int K = 2 * hl / up + 1;
    std::vector<double> tab(static_cast<size_t>(up) * K, 0.0);
    for (int p = 0; p < up; ++p)
        for (int k = 0; k < K && p + k * up < L; ++k) tab[static_cast<size_t>(p) * K + k] = h[p + k * up];
    double* dev = nullptr;
    NAFP_CUDA(cudaMalloc(&dev, tab.size() * sizeof(double)));
    NAFP_CUDA(cudaMemcpy(dev, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    RsFilter f{up, down, hl, K, dev};
    s->filters[{fs_in, fs_out}] = f;
    *out = f;
    return NAFP_OK;
}

// One launch for every run of the call.  runs[r] (host) holds pcm_off / frame0 / n_frames / channels / m0 / n_out /
// out_off, already checked; fs_in[r] picks its filter.
int resample_launch(nafp_ctx* ctx, const int16_t* pcm_dev, const SourceRun* runs, int64_t n_runs, int32_t fs_out,
                    int16_t* out_dev) {
    NAFP_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->resample) ctx->resample = new ResampleState();
    ResampleState* s = ctx->resample;
    if (!s->smem_optin) {
        NAFP_CUDA(cudaDeviceGetAttribute(&s->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
        NAFP_CUDA(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s->smem_optin));
    }
    std::vector<RsFilter> filts;
    std::map<int32_t, int32_t> slot;
    std::vector<RsRun> rr;
    int64_t tiles = 0;
    int tab_doubles = 0, need_stage = 1;
    for (int64_t r = 0; r < n_runs; ++r) {
        const SourceRun& u = runs[r];
        if (u.n_out == 0) continue;
        auto it = slot.find(u.fs_in);
        if (it == slot.end()) {
            RsFilter f;
            NAFP_TRY(resample_filter(ctx, u.fs_in, fs_out, &f));
            it = slot.emplace(u.fs_in, static_cast<int32_t>(filts.size())).first;
            filts.push_back(f);
            tab_doubles = std::max(tab_doubles, f.up * f.K);
            // frames one sub-tile reads: ((RS_THREADS - 1) down + 2 hl) / up + 2 at most
            const int64_t fr = ((RS_THREADS - 1) * int64_t(f.down) + 2 * int64_t(f.hl)) / f.up + 2;
            need_stage = static_cast<int>(std::max<int64_t>(need_stage, std::min<int64_t>(fr, RS_STAGE_MAX)));
        }
        rr.push_back(RsRun{u.pcm_off, u.frame0, u.n_frames, u.m0, u.n_out, u.out_off, tiles, u.channels, it->second});
        tiles += (u.n_out + RS_TILE - 1) / RS_TILE;
    }
    if (rr.empty()) return NAFP_OK;
    tab_doubles = (tab_doubles + 1) / 2 * 2;
    const int room = (s->smem_optin - tab_doubles * 8) / 8;
    const int stage = std::max(1, std::min(need_stage, room));
    const int64_t smem = (int64_t(tab_doubles) + stage) * 8;
    NAFP_REQUIRE(smem <= s->smem_optin && tiles <= 0x7fffffff, NAFP_ERR_UNSUPPORTED,
                 "resample: %lld bytes of shared memory / %lld tiles", (long long)smem, (long long)tiles);
    const int64_t fbytes = static_cast<int64_t>(filts.size() * sizeof(RsFilter) + 255) / 256 * 256;
    const int64_t bytes = fbytes + static_cast<int64_t>(rr.size() * sizeof(RsRun));
    if (s->desc_bytes < bytes) {
        NAFP_CUDA(cudaStreamSynchronize(ctx->stream));          // an earlier launch may still read the old table
        NAFP_TRY(ensure_dev(ctx, &s->desc, &s->desc_bytes, bytes));
    }
    uint8_t* d = static_cast<uint8_t*>(s->desc);
    NAFP_CUDA(cudaMemcpyAsync(d, filts.data(), filts.size() * sizeof(RsFilter), cudaMemcpyHostToDevice, ctx->stream));
    NAFP_CUDA(cudaMemcpyAsync(d + fbytes, rr.data(), rr.size() * sizeof(RsRun), cudaMemcpyHostToDevice, ctx->stream));
    resample_kernel<<<static_cast<unsigned>(tiles), RS_THREADS, static_cast<size_t>(smem), ctx->stream>>>(
        pcm_dev, reinterpret_cast<const RsRun*>(d + fbytes), static_cast<int>(rr.size()),
        reinterpret_cast<const RsFilter*>(d), tab_doubles, stage, out_dev);
    ctx->launches++;
    NAFP_CUDA(cudaGetLastError());
    return NAFP_OK;
}

void resample_destroy(nafp_ctx* ctx) {
    if (!ctx->resample) return;
    for (auto& kv : ctx->resample->filters) cudaFree(const_cast<double*>(kv.second.tab));
    if (ctx->resample->desc) cudaFree(ctx->resample->desc);
    delete ctx->resample;
    ctx->resample = nullptr;
}

}  // namespace nafp

using namespace nafp;

// Device-to-device resampling of one track's window (audio_utils.py:140-264 reads 8 kHz mono only).
extern "C" int nafp_resample_pcm16_dev(nafp_ctx* ctx, const int16_t* in_dev, int64_t frame0, int64_t n_frames,
                                       int32_t channels, int32_t fs_in, int32_t fs_out, int64_t m0, int64_t n_out,
                                       int16_t* out_dev) {
    NAFP_RANGE("nafp_resample_pcm16_dev");
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_resample_pcm16_dev: ctx is NULL");
    NAFP_TRY(resample_check_run("nafp_resample_pcm16_dev", frame0, n_frames, channels, fs_in, fs_out, m0, n_out));
    NAFP_REQUIRE((n_out == 0 || out_dev) && (n_frames == 0 || in_dev), NAFP_ERR_INVALID,
                 "nafp_resample_pcm16_dev: NULL buffer");
    if (n_out == 0) return NAFP_OK;
    const SourceRun run{0, frame0, n_frames, m0, n_out, 0, channels, fs_in};
    return resample_launch(ctx, in_dev, &run, 1, fs_out, out_dev);
}
