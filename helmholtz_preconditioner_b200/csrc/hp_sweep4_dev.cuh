// Device helpers shared by the cluster sweep kernels (csrc/hp_sweep4.cu: one right-hand side per launch,
// csrc/hp_sweep4m.cu: several): thread roles, named barriers, distributed-shared-memory stores, bounded mbarrier waits.
#pragma once
#include "hp_sweep_common.cuh"
#include "hp_sweep4.h"

#define HP4_CRIT 96          // critical group: warps 0-2
#define HP4_PROD 32          // warp 3: issues every TMA copy (its lane 0), driven by the empty barriers of the rings
#define HP4_OFF 256          // off-path group: warps 4-11
#define HP4_POLL 32          // warp 12: fetches the gf partials of the right neighbour from L2 ahead of the critical group
#define HP4_THREADS (HP4_CRIT + HP4_PROD + HP4_OFF + HP4_POLL)
#define HP4_CW (HP4_CRIT / 32)

__device__ __forceinline__ void bar_crit4() { asm volatile("bar.sync 1, 96;" ::: "memory"); }
__device__ __forceinline__ void bar_off4() { asm volatile("bar.sync 2, 256;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ unsigned int mapa_u32(unsigned int local_addr, unsigned int rank) {
    unsigned int r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
// one complex number into the shared memory of a CTA of the cluster; the 16 bytes are counted on that CTA's mbarrier
__device__ __forceinline__ void st_async_cplx(unsigned int remote_addr, cplx v, unsigned int remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b64 [%0], {%1, %2}, [%3];"
                 ::"r"(remote_addr), "l"(__double_as_longlong(v.x)), "l"(__double_as_longlong(v.y)), "r"(remote_bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_cluster(unsigned long long* bar, unsigned int parity) {
    unsigned int ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// bounded wait: a runaway wait (a bug) marks the CTA dead, all later waits fall through and the kernel terminates.
// The spin loop is kept out of line: ~20 wait sites would otherwise carry a 4x unrolled copy each (a third of the
// kernel's instructions), and the hot path of a wait is a single try_wait.
static __device__ __noinline__ void mbar_wait4_slow(unsigned long long* bar, unsigned int parity, unsigned int* abort_flag,
                                             volatile unsigned int* dead) {
    unsigned int spins = 0;
#pragma unroll 1
    while (!mbar_try_cluster(bar, parity)) {
        if (*dead) break;
        if (++spins > (1u << 20)) { hp_raise_abort(abort_flag); *dead = 1u; break; }
        if ((spins & 0x3FF) == 0 && *((volatile unsigned int*)abort_flag)) { *dead = 1u; break; }
    }
}
__device__ __forceinline__ void mbar_wait4(unsigned long long* bar, unsigned int parity, unsigned int* abort_flag,
                                           volatile unsigned int* dead) {
    if (!mbar_try_cluster(bar, parity)) mbar_wait4_slow(bar, parity, abort_flag, dead);
}
// hand-over of plain shared-memory stores between warps of the CTA: release on the arrive, acquire on the wait
__device__ __forceinline__ void mbar_arrive_rel4(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait_acq4(unsigned long long* bar, unsigned int parity, unsigned int* abort_flag,
                                               volatile unsigned int* dead) {
    mbar_wait4(bar, parity, abort_flag, dead);      // try_wait has acquire semantics by default
    __syncwarp();
}
__device__ __forceinline__ void mbar_arrive_local(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// field accesses of the multi-vector kernels: a right-hand-side slot whose field pointer is null is inactive (masked),
// every load of it reads 0 and every store is dropped.  A per-lane predicate, nothing else: the zero column runs through
// the products like any other input, so active slots compute exactly what they compute in a full launch.
__device__ __forceinline__ cplx ldcg_slot(const cplx* u, size_t i) { return u ? ldcg(u + i) : cmake(0.0, 0.0); }
__device__ __forceinline__ void st_slot(cplx* u, size_t i, cplx v) {
    if (u) u[i] = v;
}
__device__ __forceinline__ void ring_fill4(unsigned char* dst, const cplx* src, unsigned int bytes, unsigned long long* bar) {
    mbar_expect_tx(bar, bytes);
    for (unsigned int o = 0; o < bytes; o += HP_BULK_CHUNK)
        bulk_g2s(dst + o, (const char*)src + o, min(HP_BULK_CHUNK, bytes - o), bar);
}

