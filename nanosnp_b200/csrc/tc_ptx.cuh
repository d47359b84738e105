// Raw PTX for the tcgen05 kernels (model_tc.cu, haplotype_tc.cu): mbarriers, cluster barriers, TMEM allocation, tcgen05.mma /
// commit / ld, UMMA descriptors, fp16 hi/lo splitting and bulk copies.  Internal linkage: every including file gets its own copy.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

namespace nsnp {
namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// cluster-scope wait for the hand-off between the two CTAs of a pair
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_LOOP_C:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE_C;\n\t"
        "bra WAIT_LOOP_C;\n\t"
        "DONE_C:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// Relaxed remote arrive: execution ordering only.  The operand rows were already made visible to the async proxy by
// fence.proxy.async and the TMEM reads retired (tcgen05.fence); a .release at cluster scope would additionally drain this
// thread's outstanding GLOBAL stores (the layer-0 output rows) on every step.
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint64_t* bar, uint32_t target_cta) {
    uint32_t raddr;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(smem_u32(bar)), "r"(target_cta));
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(raddr) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Per-step hand-off inside a CTA pair.  Every thread has already made its shared-memory operand writes visible to
// the async proxy (fence.proxy.async) and retired its TMEM loads, so only execution ordering is needed here; a
// .release arrive would additionally drain this thread's outstanding GLOBAL stores (the layer-0 output rows) to L2
// at cluster scope on every step, which ncu showed as 37% of all stall samples (membar).
__device__ __forceinline__ void cluster_sync_exec() {
    asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }

template <int CG> __device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    if (CG == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    } else {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
}
template <int CG> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
template <int CG> __device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    if (CG == 1)
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
    else
        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                     ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// kind::tf32 (fp32 operand words, K = 8 per instruction), one CTA: same descriptors and accumulator as umma_f16<1>
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
template <int CG> __device__ __forceinline__ void umma_commit(uint64_t* bar) {
    if (CG == 1)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n\t"
        "tcgen05.wait::ld.sync.aligned;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// 16 consecutive fp32 columns, no wait: pair with tmem_wait_ld() before the registers are read
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ int2 ldg_nc_volatile(const int2* p) {      // stays where it is written: issued before the MMA wait
    int2 v;
    asm volatile("ld.global.nc.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor, mma_sm100_desc.hpp):
//   bits [0,14) start>>4, [16,30) leading-dim byte offset>>4 (between the two 16-byte K chunks of one MMA),
//   [32,46) stride byte offset>>4 (between 8-row groups), [46,48) version = 1, [61,64) layout = 0.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (bit 4), A=B=f16 (0), K-major both, N>>3 at 17, M>>4 at 24
__host__ __device__ constexpr uint32_t make_idesc(int m, int n) { return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24); }

struct HiLo8 { uint4 hi, lo; };
__device__ __forceinline__ uint32_t h2_bits(__half2 h) { return *reinterpret_cast<uint32_t*>(&h); }
// 8 floats -> 8 fp16 "hi" + 8 fp16 "lo" (v - float(hi)), two values per cvt.rn.f16x2.f32
__device__ __forceinline__ HiLo8 split8(const float (&v)[8]) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        const float2 f = __half22float2(hh);
        h[i] = h2_bits(hh);
        l[i] = h2_bits(__floats2half2_rn(v[2 * i] - f.x, v[2 * i + 1] - f.y));
    }
    HiLo8 o;
    o.hi = make_uint4(h[0], h[1], h[2], h[3]);
    o.lo = make_uint4(l[0], l[1], l[2], l[3]);
    return o;
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared (UBLKCP): one instruction moves a contiguous block, completion is counted on an mbarrier,
// and the data lands through the async proxy (no generic->async proxy fence needed before the MMAs read it)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* gsrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}

}  // namespace
}  // namespace nsnp
