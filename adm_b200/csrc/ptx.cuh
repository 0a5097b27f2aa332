// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM).
// Everything here is device-side and header-only.  No CUTLASS dependency.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace adm {

// Error flag written by device code when a bounded wait expires (deadlock guard).  Read by adm_last_error().
static __device__ int g_device_error = 0;  // one copy per translation unit (no -rdc)

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
}
__device__ __forceinline__ uint32_t mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {  // acquire at cluster scope
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok;
}
// Bounded wait: a pipeline bug must never hang the GPU box.  ~4 s at 2 GHz, then flag + trap.  `code` names the wait
// site in g_device_error.
template <typename TryWait>
__device__ __forceinline__ void bounded_wait(TryWait try_wait, int code) {
    if (try_wait()) return;
    const long long t0 = clock64();
    while (!try_wait()) {
        if (clock64() - t0 > 8000000000LL) {
            g_device_error = code;
            __threadfence_system();
            asm volatile("trap;");
        }
    }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int code) {
    bounded_wait([=] { return mbar_try_wait(bar, parity); }, code);
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity, int code) {
    bounded_wait([=] { return mbar_try_wait_cluster(bar, parity); }, code);
}
// Distributed shared memory: the address of this CTA's shared variable `saddr` in the cluster CTA `rank`.
__device__ __forceinline__ uint32_t mapa_shared(uint32_t saddr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
    return r;
}
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t caddr) {
    float4 v;
    asm volatile("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(caddr));
    return v;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t caddr) {  // release at cluster scope
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(caddr) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32.  Issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 16 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 consecutive fp32 columns of this warp's 32 lanes.
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
// registers -> TMEM: this warp's 32 lanes x 8 / 16 consecutive 32-bit columns.
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
                 "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15, %16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem desc]: the A operand is read from tensor memory (lane = row m, 32-bit column k / 2 holds
// the bf16 pair (k, k + 1), K-major by construction; a 16-deep k-step advances the A address by 8 columns).  Verified
// bit-exact on B200 by tools/exp/umma_tmem_a.cu (profiles/r03_umma_tmem_a_operand_experiment.txt).
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// ---------------------------------------------------------------- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor (sm_100 "version 1"), SWIZZLE_128B.
//  K-major : rows of 128 B (64 bf16 of K), 8-row groups 1024 B apart  -> LBO unused (1), SBO = 1024.
//  MN-major: chunks of [K rows][128 B = 64 bf16 of MN]; 8-row K groups 1024 B apart (SBO), 64-wide MN chunks
//            chunk_bytes apart (LBO).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;  // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;  // SWIZZLE_128B
    return d;
}
// Instruction descriptor for kind::f16 with bf16 inputs, fp32 accumulate.
__device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
    uint32_t d = 0;
    d |= 1u << 4;   // D format fp32
    d |= 1u << 7;   // A format bf16
    d |= 1u << 10;  // B format bf16
    d |= (a_mn_major ? 1u : 0u) << 15;
    d |= (b_mn_major ? 1u : 0u) << 16;
    d |= static_cast<uint32_t>(N >> 3) << 17;
    d |= static_cast<uint32_t>(M >> 4) << 24;
    return d;
}

}  // namespace adm
