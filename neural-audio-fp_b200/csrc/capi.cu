// Context, error reporting, memory helpers and the TMA tensor-map encoder of libnafp.
#include <cstring>

#include "common.h"

namespace nafp {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_err; }

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(p);
    return fn;
}

int make_tensor_map(CUtensorMap* out, CUtensorMapDataType dtype, int rank, void* base,
                    const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                    const uint32_t* elem_strides, CUtensorMapSwizzle swizzle) {
    PFN_encodeTiled fn = get_encode_fn();
    NAFP_REQUIRE(fn != nullptr, NAFP_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
    cuuint64_t gdim[5], gstr[5];
    cuuint32_t bx[5], es[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bx[i] = box[i];
        es[i] = elem_strides ? elem_strides[i] : 1;
    }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i + 1];
    CUresult r = fn(out, dtype, static_cast<cuuint32_t>(rank), base, gdim, gstr, bx, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    NAFP_REQUIRE(r == CUDA_SUCCESS, NAFP_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return NAFP_OK;
}

}  // namespace nafp

using namespace nafp;

extern "C" {

int nafp_version(void) { return 100; }

const char* nafp_last_error(void) { return get_error(); }

int nafp_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return NAFP_ERR_CUDA;
    }
    return n;
}

int nafp_ctx_create(int device, nafp_ctx** out) {
    NAFP_REQUIRE(out != nullptr, NAFP_ERR_INVALID, "nafp_ctx_create: out is NULL");
    *out = nullptr;
    int n = nafp_device_count();
    if (n < 0) return n;
    NAFP_REQUIRE(device >= 0 && device < n, NAFP_ERR_INVALID, "nafp_ctx_create: device %d of %d", device, n);
    NAFP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    NAFP_CUDA(cudaGetDeviceProperties(&prop, device));
    NAFP_REQUIRE(prop.major == 10, NAFP_ERR_UNSUPPORTED,
                 "nafp: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device,
                 prop.major, prop.minor);
    nafp_ctx* ctx = new nafp_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    NAFP_CUDA(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    NAFP_CUDA(cudaEventCreate(&ctx->ev0));
    NAFP_CUDA(cudaEventCreate(&ctx->ev1));
    *out = ctx;
    return NAFP_OK;
}

int nafp_ctx_destroy(nafp_ctx* ctx) {
    if (!ctx) return NAFP_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    logmel_destroy(ctx);
    encoder_destroy(ctx);
    resample_destroy(ctx);
    if (ctx->stage_dev) cudaFree(ctx->stage_dev);
    if (ctx->stage_pinned) cudaFreeHost(ctx->stage_pinned);
    if (ctx->clip_ws) cudaFree(ctx->clip_ws);
    cudaEventDestroy(ctx->ev0);
    cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return NAFP_OK;
}

int nafp_sync(nafp_ctx* ctx) {
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_sync: ctx is NULL");
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    return NAFP_OK;
}

int nafp_ctx_set_stream(nafp_ctx* ctx, void* cuda_stream) {
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_ctx_set_stream: ctx is NULL");
    NAFP_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return NAFP_OK;
}

void* nafp_ctx_stream(nafp_ctx* ctx) { return ctx ? static_cast<void*>(ctx->stream) : nullptr; }

int64_t nafp_ctx_launch_count(nafp_ctx* ctx) { return ctx ? ctx->launches : 0; }

int nafp_malloc(nafp_ctx* ctx, int64_t bytes, void** out_dev) {
    NAFP_REQUIRE(ctx && out_dev && bytes >= 0, NAFP_ERR_INVALID, "nafp_malloc: bad arguments");
    NAFP_CUDA(cudaSetDevice(ctx->device));
    NAFP_CUDA(cudaMalloc(out_dev, static_cast<size_t>(bytes > 0 ? bytes : 1)));
    return NAFP_OK;
}
int nafp_free(nafp_ctx* ctx, void* dev) {
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_free: ctx is NULL");
    if (dev) NAFP_CUDA(cudaFree(dev));
    return NAFP_OK;
}
int nafp_malloc_host(nafp_ctx* ctx, int64_t bytes, void** out_host) {
    NAFP_REQUIRE(ctx && out_host && bytes >= 0, NAFP_ERR_INVALID, "nafp_malloc_host: bad arguments");
    NAFP_CUDA(cudaMallocHost(out_host, static_cast<size_t>(bytes > 0 ? bytes : 1)));
    return NAFP_OK;
}
int nafp_free_host(nafp_ctx* ctx, void* host) {
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_free_host: ctx is NULL");
    if (host) NAFP_CUDA(cudaFreeHost(host));
    return NAFP_OK;
}
int nafp_memcpy_h2d(nafp_ctx* ctx, void* dst_dev, const void* src_host, int64_t bytes) {
    NAFP_REQUIRE(ctx && (bytes == 0 || (dst_dev && src_host)), NAFP_ERR_INVALID, "nafp_memcpy_h2d: bad arguments");
    if (bytes) NAFP_CUDA(cudaMemcpyAsync(dst_dev, src_host, (size_t)bytes, cudaMemcpyHostToDevice, ctx->stream));
    return NAFP_OK;
}
int nafp_memcpy_d2h(nafp_ctx* ctx, void* dst_host, const void* src_dev, int64_t bytes) {
    NAFP_REQUIRE(ctx && (bytes == 0 || (dst_host && src_dev)), NAFP_ERR_INVALID, "nafp_memcpy_d2h: bad arguments");
    if (bytes) NAFP_CUDA(cudaMemcpyAsync(dst_host, src_dev, (size_t)bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return NAFP_OK;
}
int nafp_timer_start(nafp_ctx* ctx) {
    NAFP_REQUIRE(ctx, NAFP_ERR_INVALID, "nafp_timer_start: ctx is NULL");
    NAFP_CUDA(cudaEventRecord(ctx->ev0, ctx->stream));
    return NAFP_OK;
}
int nafp_timer_stop(nafp_ctx* ctx, float* out_ms) {
    NAFP_REQUIRE(ctx && out_ms, NAFP_ERR_INVALID, "nafp_timer_stop: bad arguments");
    NAFP_CUDA(cudaEventRecord(ctx->ev1, ctx->stream));
    NAFP_CUDA(cudaEventSynchronize(ctx->ev1));
    NAFP_CUDA(cudaEventElapsedTime(out_ms, ctx->ev0, ctx->ev1));
    return NAFP_OK;
}

}  // extern "C"
