// umma.cuh -- thin PTX wrappers for the sm_100a tensor-core path (tcgen05.mma / tensor memory / mbarrier / cp.async).
// Only what the sparse conv needs; layouts and encodings are spelled out where they are used.
#pragma once
#include "common.cuh"

// all tcgen05.mma issued so far by this thread -> one arrival on the mbarrier when they have completed
__device__ __forceinline__ void umma_commit(u32 bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// One lane of a converged warp.  Issue tcgen05.mma from `if (elect_one())` inside warp-uniform control flow: the descriptors
// then live in uniform registers; from `if (lane == 0)` ptxas wraps every UTCHMMA in an election loop (~140 clk per MMA,
// tools/micro/umma_rate.cu).
__device__ __forceinline__ bool elect_one() {
    u32 pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tmem_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld16(u32 taddr, u32 (&d)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7]), "=r"(d[8]),
                   "=r"(d[9]), "=r"(d[10]), "=r"(d[11]), "=r"(d[12]), "=r"(d[13]), "=r"(d[14]), "=r"(d[15])
                 : "r"(taddr) : "memory");
}

__device__ __forceinline__ void tmem_ld8(u32 taddr, u32 (&d)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]), "=r"(d[4]), "=r"(d[5]), "=r"(d[6]), "=r"(d[7]) : "r"(taddr) : "memory");
}

// ---- mbarrier
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(u32 bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait with an explicit suspend-time hint: the warp sleeps in hardware until the phase completes or the hint (ns) runs out.
// Bounded: a mis-programmed pipeline must fault the launch (trap), never hang the GPU.
__device__ __forceinline__ void mbar_wait_hint(u32 bar, u32 parity) {
#pragma unroll 1
    for (u32 spins = 0; spins < (1u << 20); ++spins) {
        u32 done;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(done) : "r"(bar), "r"(parity), "r"(100000u) : "memory");
        if (done) return;
    }
    __trap();
}

// ---- cp.async (no "memory" clobber: ordering against commit / wait / barrier statements is kept by their volatile-ness, and a
// clobber here would chain every table load in front of a copy behind the previous copy)
__device__ __forceinline__ void cp_async16(u32 dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
