// PTX wrappers shared by the tcgen05 kernels: mbarrier, TMA (cp.async.bulk.tensor), UMMA descriptors,
// tcgen05.mma / commit / ld.  Hand-written inline PTX for sm_100a; encodings follow the sm_100
// SmemDescriptor / InstrDescriptor bit layouts.
#pragma once
#include "kernels.cuh"

namespace kzb {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2,
                                            int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::
            "r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}

// 1-D bulk copy global -> shared (16-byte aligned, size a multiple of 16), completion on an mbarrier
__device__ __forceinline__ void bulk_load_1d(uint64_t* bar, void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// multicast variant: the box lands at the same CTA-relative offset in every CTA of `cta_mask`, and each destination
// CTA's barrier (same offset) receives the complete_tx for the bytes written there
__device__ __forceinline__ void tma_load_2d_multicast(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1,
                                                      uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
        "[%2], %5;" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster (release at cluster scope)
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// wait that also acquires what CTAs of the cluster released before arriving
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_CLUSTER:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_CLUSTER;\n\t"
        "bra WAIT_CLUSTER;\n\t"
        "DONE_CLUSTER:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// Programmatic dependent launch (kernels launched with cudaLaunchAttributeProgrammaticStreamSerialization): the next kernel of
// the stream may start once every CTA of this one has called launch_dependents (or exited); it must call grid_dep_wait before
// it touches anything the previous kernel wrote.
__device__ __forceinline__ void grid_dep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 "SmemDescriptor"):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major) | [32,46) SBO >> 4
//   [46,48) version = 1 | [49,52) base offset = 0 | [61,64) layout type: 2 = SWIZZLE_128B
// 8-row groups are 1024 B apart (SBO), rows inside a group 128 B apart.
// The descriptor is built as its address-independent upper part OR the 14-bit start-address field, so the MMA
// issue loop only does one integer add per operand (the issue thread is otherwise the bottleneck: measured
// ~100 cycles per tcgen05.mma when the full descriptor is rebuilt each time vs 64 cycles of tensor work).
__device__ __forceinline__ uint64_t umma_desc_sw128_hi() {
    return (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t smem_addr) { return (smem_addr >> 4) & 0x3FFF; }

// Instruction descriptor, kind::f16: c=f32 [4,6)=1, a=bf16 [7,10)=1, b=bf16 [10,13)=1, both K-major,
// N>>3 at [17,23), M>>4 at [24,29).
__device__ __forceinline__ uint32_t umma_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
// Instruction descriptor, kind::tf32: c=f32 [4,6)=1, a=tf32 [7,10)=2, b=tf32 [10,13)=2, both K-major; N, M as above.
__device__ __forceinline__ uint32_t umma_idesc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
// the instruction descriptor of one 128-byte-per-row operand type: bf16 (kind::f16) or f32 rounded to TF32 (kind::tf32)
template <typename T>
__device__ __forceinline__ uint32_t umma_idesc(int m, int n) {
    if constexpr (sizeof(T) == 4)
        return umma_idesc_tf32(m, n);
    else
        return umma_idesc_bf16(m, n);
}

__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// commit that arrives on the barrier at the same offset in every CTA of `cta_mask` (releases a multicast-filled slot)
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(cta_mask)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
        "[%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
// TMA store (shared -> global) of one box, bulk-group completion
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}

}  // namespace tc
}  // namespace kzb
