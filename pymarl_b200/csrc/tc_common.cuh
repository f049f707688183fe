// Blackwell (sm_100a) primitives used by the tensor-core kernels: mbarrier, bulk async copy,
// TMEM allocation, tcgen05.mma / commit / ld, UMMA shared-memory and instruction descriptors.
// Everything is inline PTX; no CUTLASS dependency.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace pmb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
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
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---- packed fp32 pairs (sm_100: FFMA2 - two IEEE fp32 operations per instruction, same rounding as the scalar form) ----
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_make(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_split(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
// the two halves of a bf16x2 word as an fp32 pair (element 0 = low half)
__device__ __forceinline__ f32x2 f2_from_bf16x2(uint32_t w) { return f2_make(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// generic-proxy smem writes -> visible to the async proxy (tensor core / bulk copy engine)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 1-D bulk copy global -> shared, completion counted in bytes on an mbarrier (TMA engine, no tensor map)
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 1-D bulk copy shared -> global (TMA engine), tracked by the per-thread bulk async-group
__device__ __forceinline__ void bulk_copy_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all but the newest N groups have finished READING shared memory (the source may be overwritten)
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// ... have completed (the global writes are done)
template <int N>
__device__ __forceinline__ void bulk_wait_group() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }

// ---- TMEM ----------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot_smem, uint32_t ncols) {   // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {       // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// ---- programmatic dependent launch ----------------------------------------------------------
// launch_dependents: this CTA no longer holds back the next kernel of the stream (if that one was launched with
// programmatic stream serialization); wait: everything the previous kernel of the stream did is complete and visible
// (a no-op when this kernel was launched the ordinary way)
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base_lane + i)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns from registers: thread i of the warp writes lane (base_lane + i)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        :
        : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
          "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
          "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
// this thread's tcgen05.st have completed (before a fence / barrier hands the columns to the tensor core)
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- UMMA descriptors ------------------------------------------------------------------------
// Shared-memory matrix descriptor, 128-byte swizzle (cute::UMMA::SmemDescriptor): start address
// [0,14) >>4, leading byte offset [16,30) >>4, stride byte offset [32,46) >>4, version [46,48) = 1,
// layout type [61,64) = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor for kind::f16 with BF16 A/B and FP32 accumulation
// (cute::UMMA::InstrDescriptor): c_format [4,6) = 1 (F32), a_format [7,10) = 1 (BF16),
// b_format [10,13) = 1, a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major),
// n_dim [17,23) = N >> 3, m_dim [24,29) = M >> 4.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] . B[smem], issued by ONE thread on behalf of the CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem]: A (M x K, K-major) is read from tensor memory - lane = row of A, two bf16 per 32-bit
// column (lower k in the low half), so one K = 16 step is 8 columns
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        :
        : "r"(tmem_d), "r"(tmem_a), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// byte offset of element (row r, 16-byte chunk j) inside a [rows][128 B] tile with the 128-byte
// swizzle (Swizzle<3,4,3>): chunk index XOR (row mod 8).  The tile base must be 1024-byte aligned.
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t r, uint32_t j) {
    return r * 128u + ((j ^ (r & 7u)) << 4);
}

}  // namespace tc
}  // namespace pmb
