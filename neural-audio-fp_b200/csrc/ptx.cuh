// Thin inline-PTX wrappers for the sm_100a features the kernels use:
// mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc / mma / commit / ld / fences), and the cluster
// forms the flat scan's CTA pairs use (multicast loads, remote arrives, st.async, cluster barrier).
// Every MMA is cta_group::1: a pair shares its B operand through multicast, not through cta_group::2.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace nafp {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch error (trap), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 26)) __trap();
    }
}
// Same, for the single-thread producer / MMA roles: let the hardware park the thread (suspend-time
// hint) instead of burning issue slots of the sub-partition it shares with the epilogue warps.
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred P;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, P;\n\t}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(2000u)
            : "memory");
        if (ok) return;
        if (++spins > (1u << 24)) __trap();
    }
}
// Same, with cluster-scope acquire: for a barrier that a peer CTA completes (remote arrive, st.async), so that
// what the peer wrote before it is visible here and to whatever this thread signals next.
__device__ __forceinline__ void mbar_wait_parked_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n\t.reg .pred P;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, P;\n\t}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(2000u)
            : "memory");
        if (ok) return;
        if (++spins > (1u << 24)) __trap();
    }
}

// ---------------------------------------------------------------- clusters
// all threads of all CTAs of the cluster; release / acquire order shared-memory accesses across it
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same object in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_shared_rank(const void* p, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
    return r;
}
// arrive (+ expect bytes) on a peer CTA's mbarrier.  .relaxed: the data it announces carries its own completion,
// and .release would cost a GPU-wide memory barrier per call
__device__ __forceinline__ void mbar_arrive_expect_tx_remote(uint32_t bar_cluster, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.relaxed.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_cluster), "r"(bytes)
                 : "memory");
}
// 4-byte store into a peer CTA's shared memory that completes 4 bytes of transaction on the peer's mbarrier
__device__ __forceinline__ void st_async_remote(uint32_t dst_cluster, int32_t v, uint32_t bar_cluster) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(dst_cluster), "r"(v),
                 "r"(bar_cluster)
                 : "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
// same box delivered to the same shared-memory offset, and completed on the same mbarrier offset, in every CTA of
// `cta_mask` (bit i = cluster rank i); one read from L2 / HBM
__device__ __forceinline__ void tma_load_2d_multicast(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1,
                                                      uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* smem_dst, const void* tmap, uint64_t* bar, int32_t c0, int32_t c1, int32_t c2, int32_t c3, int32_t c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
// TMA store: shared memory tile -> global tensor box (bulk async-group completion)
__device__ __forceinline__ void tma_store_2d(const void* tmap, const void* smem_src, int32_t c0, int32_t c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the source shared memory of all committed stores has been read (it may be overwritten)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all committed stores are complete
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// packed fp32 pairs (FFMA2 / FADD2 / FMUL2: two fp32 operations per issue slot)
__device__ __forceinline__ uint64_t pk2(float a, float b) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void upk2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}

// make generic-proxy smem writes visible to the async proxy (TMA / tcgen05 operand reads)
// plain (non-tensor) bulk copy global -> shared, completion counted on an mbarrier; 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_load_1d_multicast(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar,
                                                       uint16_t cta_mask) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (fp16/bf16 operands, fp32 accumulate)
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// same, arriving on the mbarrier at this offset in every CTA of `cta_mask` (bit i = cluster rank i)
__device__ __forceinline__ void tc_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp gets lane (base_lane + i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
// 32 lanes x 64 consecutive fp32 columns (one round trip instead of two)
__device__ __forceinline__ void tmem_ld_32x64(uint32_t taddr, uint32_t (&v)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, %48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31]), "=r"(v[32]), "=r"(v[33]), "=r"(v[34]), "=r"(v[35]), "=r"(v[36]), "=r"(v[37]), "=r"(v[38]), "=r"(v[39]), "=r"(v[40]), "=r"(v[41]), "=r"(v[42]), "=r"(v[43]), "=r"(v[44]), "=r"(v[45]), "=r"(v[46]), "=r"(v[47]), "=r"(v[48]), "=r"(v[49]), "=r"(v[50]), "=r"(v[51]), "=r"(v[52]), "=r"(v[53]), "=r"(v[54]), "=r"(v[55]), "=r"(v[56]), "=r"(v[57]), "=r"(v[58]), "=r"(v[59]), "=r"(v[60]), "=r"(v[61]), "=r"(v[62]), "=r"(v[63])
        : "r"(taddr)
        : "memory");
}
// one column: lane l gets TMEM lane (base + l) of column taddr
__device__ __forceinline__ uint32_t tmem_ld_32x1(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}

// registers -> TMEM, 32 lanes x 16 consecutive 32-bit columns (thread i writes lane base_lane + i)
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand, SWIZZLE_128B, rows of 128 bytes:
// 8-row x 128 B swizzle atoms stacked every 1024 B (SBO).  Field layout per
// cute/arch/mma_sm100_desc.hpp (SmemDescriptor): addr>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type [61,64) (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
    d |= static_cast<uint64_t>(1) << 16;            // LBO (ignored for swizzled K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;    // SBO = 1024 B
    d |= static_cast<uint64_t>(1) << 46;            // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;            // SWIZZLE_128B
    return d;
}
// Instruction descriptor for kind::f16: fp32 accumulate, A/B both K-major.
// fmt: 0 = fp16, 1 = bf16.  (InstrDescriptor in mma_sm100_desc.hpp)
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t fmt, uint32_t M, uint32_t N) {
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ---------------------------------------------------------------- misc
// order-preserving map float -> int32 (signed compare of the result == float compare)
__device__ __forceinline__ int32_t f2ord(float f) {
    int32_t b = __float_as_int(f);
    return b >= 0 ? b : (b ^ 0x7FFFFFFF);
}
__device__ __forceinline__ float ord2f(int32_t o) {
    return __int_as_float(o >= 0 ? o : (o ^ 0x7FFFFFFF));
}
__device__ __forceinline__ int32_t ld_relaxed(const int32_t* p) {
    int32_t v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(int32_t* p, int32_t v) {
    asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// 128-d fp32 dot product by one warp: lane holds 4 consecutive elements of `a`; every lane returns
// the same bits (xor butterfly adds commute pairwise).
__device__ __forceinline__ float warp_dot128(const float4 a, const float* __restrict__ xrow, int lane) {
    const float4 b = reinterpret_cast<const float4*>(xrow)[lane];
    float s = a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

}  // namespace nafp
