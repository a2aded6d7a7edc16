// Shared host-side plumbing of libnafp: context, error reporting, launch accounting,
// TMA tensor-map encoding through the driver entry point (libcuda is NOT a link-time dependency,
// so the library still loads -- and reports "no device" -- on a machine without a driver).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>      // header-only NVTX v3: ranges cost nothing unless a profiler injects itself

#include "../../include/nafp.h"

namespace nafp {

void set_error(const char* fmt, ...);
const char* get_error();

#define NAFP_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            nafp::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return NAFP_ERR_CUDA;                                                               \
        }                                                                                       \
    } while (0)

#define NAFP_REQUIRE(cond, status, ...)  \
    do {                                 \
        if (!(cond)) {                   \
            nafp::set_error(__VA_ARGS__); \
            return (status);             \
        }                                \
    } while (0)

#define NAFP_TRY(expr)             \
    do {                           \
        int _s = (expr);           \
        if (_s != NAFP_OK) return _s; \
    } while (0)

// NVTX range around every compute entry point of the C ABI (SURVEY §5: the tracing hook of this path;
// `nsys` / `ncu --nvtx` show them, e.g. `ncu --nvtx --nvtx-include "nafp_fingerprint/"`)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};
#define NAFP_RANGE(name) nafp::NvtxRange _nvtx_range_(name)

struct LogmelState;
struct EncoderState;
struct ResampleState;

}  // namespace nafp

struct nafp_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;       // stream all work is issued on
    cudaStream_t own_stream = nullptr;   // the one this ctx created
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    int64_t launches = 0;
    nafp::LogmelState* logmel = nullptr;
    nafp::EncoderState* encoder = nullptr;
    nafp::ResampleState* resample = nullptr;
    // reusable staging buffers for the *_host entry points
    void* stage_dev = nullptr;
    int64_t stage_dev_bytes = 0;
    void* stage_pinned = nullptr;
    int64_t stage_pinned_bytes = 0;
    // workspace of the clip matcher (search results, candidate sorts, scores)
    void* clip_ws = nullptr;
    int64_t clip_ws_bytes = 0;
};

namespace nafp {

inline int ensure_dev(nafp_ctx* ctx, void** buf, int64_t* cap, int64_t bytes) {
    if (*cap >= bytes) return NAFP_OK;
    if (*buf) NAFP_CUDA(cudaFree(*buf));
    *buf = nullptr;
    *cap = 0;
    NAFP_CUDA(cudaMalloc(buf, static_cast<size_t>(bytes)));
    *cap = bytes;
    return NAFP_OK;
}
inline int ensure_pinned(void** buf, int64_t* cap, int64_t bytes) {
    if (*cap >= bytes) return NAFP_OK;
    if (*buf) NAFP_CUDA(cudaFreeHost(*buf));
    *buf = nullptr;
    *cap = 0;
    NAFP_CUDA(cudaMallocHost(buf, static_cast<size_t>(bytes)));
    *cap = bytes;
    return NAFP_OK;
}

// 2-D..4-D tiled tensor map; dims/strides innermost first (strides in bytes, strides[0] implied).
int make_tensor_map(CUtensorMap* out, CUtensorMapDataType dtype, int rank, void* base,
                    const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                    const uint32_t* elem_strides, CUtensorMapSwizzle swizzle);

// module destructors (called from nafp_ctx_destroy)
void logmel_destroy(nafp_ctx* ctx);
void encoder_destroy(nafp_ctx* ctx);
void resample_destroy(nafp_ctx* ctx);

// resampler (resample.cu): one run is a window of one track's source frames and the outputs m0 .. m0 + n_out - 1 it
// yields, written at out_off of the output buffer
struct SourceRun {
    int64_t pcm_off, frame0, n_frames, m0, n_out, out_off;
    int32_t channels, fs_in;
};
int resample_ratio(int32_t fs_in, int32_t fs_out, int32_t* up, int32_t* down, int32_t* hl);
int resample_check_run(const char* fn, int64_t frame0, int64_t n_frames, int32_t channels, int32_t fs_in,
                       int32_t fs_out, int64_t m0, int64_t n_out);
int resample_launch(nafp_ctx* ctx, const int16_t* pcm_dev, const SourceRun* runs, int64_t n_runs, int32_t fs_out,
                    int16_t* out_dev);

}  // namespace nafp
