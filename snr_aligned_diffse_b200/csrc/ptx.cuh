// Inline-PTX wrappers for the Blackwell (sm_100a) async machinery used by the implicit-GEMM kernel:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and UMMA descriptors.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done;
}
// Non-blocking probe (try_wait may suspend the warp for an implementation-defined time; a loop that polls two barriers
// in turn must not)
__device__ __forceinline__ uint32_t mbar_test_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    return done;
}
// Bounded wait: a protocol bug must fault the launch (trap -> cudaErrorLaunchFailure), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
        if (spins > (1u << 22)) {
            asm volatile("trap;");
        }
    }
}

// One lane of the (fully converged) warp is elected; every other lane gets false.  Keeping the MMA / TMA issue loops
// warp-uniform and predicating only the issue instruction lets the compiler hold descriptors in uniform registers
// (a loop under `if (lane == 0)` is divergent code: every tcgen05.mma then needs five R2UR moves in a waterfall loop).
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- TMA loads (tile mode, mbarrier completion)
__device__ __forceinline__ void tma_load_4d(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                            int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                            int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// TMA store of a shared-memory tile (bulk-group completion); out-of-bounds elements are not written
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t smem_src, int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
        ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still have to READ their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {  // whole warp
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> f32, issued by ONE thread.
__device__ __forceinline__ void mma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// 32 lanes x 32 consecutive fp32 columns: thread i of the warp receives lane (base_lane + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t* v) {  // whole warp
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
// 32 lanes x 4 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x32_x4(uint32_t taddr, uint32_t* v) {  // whole warp
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- 2-CTA (cta_group::2) variants
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in the cluster's rank-0 (leader) CTA
__device__ __forceinline__ uint32_t mapa_rank0(uint32_t smem_addr) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(smem_addr));
    return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// arrive + expect-tx on a barrier addressed in cluster space (may live in the peer CTA)
__device__ __forceinline__ void mbar_arrive_expect_tx_remote(uint32_t cluster_bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.release.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t smem_dst, const CUtensorMap* map, uint32_t cluster_bar, int c0,
                                                int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t smem_dst, const CUtensorMap* map, uint32_t cluster_bar, int c0,
                                                int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(cluster_bar), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t smem_result, uint32_t ncols) {  // whole warp, both CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish2() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A (128 rows per CTA) * B^T (N/2 rows per CTA); issued by ONE thread of the leader CTA
__device__ __forceinline__ void mma_bf16_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive (once) on the barrier at this shared-memory offset in BOTH CTAs when the issued MMAs retire
__device__ __forceinline__ void mma_commit_2sm(uint32_t bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(bar), "h"((uint16_t)3)
        : "memory");
}

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor for a K-major operand tile stored as rows of 128 bytes
// (64 bf16) with the 128-byte swizzle TMA writes: 8-row atoms of 1024 B, atoms stacked along M/N.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4 (unused for swizzled K-major: 1)
//   bits [32,46) stride byte offset >> 4   bits [46,48) version = 1 (sm_100)
//   bits [61,64) layout type: 2 = SWIZZLE_128B
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// Instruction descriptor, kind::f16: D=f32 (bit 4), A=B=bf16 (bits 7,10), both K-major, N>>3 at 17, M>>4 at 24.
__host__ __device__ __forceinline__ uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

}  // namespace ptx
