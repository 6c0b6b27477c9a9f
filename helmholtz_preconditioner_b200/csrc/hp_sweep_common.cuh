// Pieces shared by the sweep kernels: arguments, self-validating exchange words, TMA/mbarrier wrappers.
#pragma once
#include "hp_internal.cuh"

#define HP_RING 4
#define HP_RMAX 8           // right-hand sides one launch of the multi-vector cluster kernel carries at most
#define HP_SPIN_LIMIT (1u << 21)

struct HpSweepArgs {
    int n, b;
    HpLayout lay;
    const int *leaf_start, *leaf_q, *sep;
    const cplx* packets;
    const cplx* mleaf;        // transfer matrices [strip][dir][leaf][2b][2b] (pipelined kernel)
    const cplx* rsep;         // separator recurrence rows [strip][dir][P-1][b][3b] (cluster kernel)
    int m_lo;
    int mode, m_from, m_to, diag_mode;
    cplx* u;
    cplx* um[HP_RMAX];        // multi-vector cluster kernel (csrc/hp_sweep4m.cu): the fields of the right-hand sides
    const cplx* vin;
    cplx* yout;
    cplx* xch;                // exchange ring: HP_RING slots of slot_stride complex numbers
    size_t oGP, oGR, oXS, oVS, slot_stride;      // (cluster kernel: oXS = partial x [P-1][K*NRQ], oGP = gf partials [P][K][b])
    unsigned int* bar;        // [1] abort flag of the running launch (a spin ran into HP_SPIN_LIMIT), cleared before every launch;
                              // [2] sticky copy, cleared by the setup only (hp_sweep_status, checked on the product path)
    const cplx *s2t, *is1t;
    double ih2;
    long long* dbg;           // optional [G][8] per-phase cycle sums (thread 0 of every CTA), NULL = off
};

__device__ __forceinline__ cplx ldcg(const cplx* p) {
    double2 v = __ldcg(reinterpret_cast<const double2*>(p));
    return v;
}
// the same load pinned where it is written: the compiler may sink a plain load down to its first use, i.e. behind the
// mbarrier waits of the strip (the point of an early load is that its DRAM latency passes during those waits)
__device__ __forceinline__ cplx ldcg_now(const cplx* p) {
    cplx v;
    asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}

// ---- self-validating exchange words -----------------------------------------------------------------
#define HP_SENTINEL 0xFFFFFFFFFFFFFFFFull
__device__ __forceinline__ void xput(cplx* p, cplx v) {
    asm volatile("st.relaxed.gpu.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void xarm(cplx* p) {
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %1};" ::"l"(p), "l"(HP_SENTINEL) : "memory");
}
__device__ __forceinline__ bool xtry(const cplx* p, cplx& v) {
    unsigned long long lo, hi;
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(p) : "memory");
    v.x = __longlong_as_double((long long)lo);
    v.y = __longlong_as_double((long long)hi);
    return lo != HP_SENTINEL && hi != HP_SENTINEL;
}
// the load alone (issue several back to back, then test with xvalid)
__device__ __forceinline__ void xload(const cplx* p, unsigned long long& lo, unsigned long long& hi) {
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "l"(p) : "memory");
}
__device__ __forceinline__ bool xvalid(unsigned long long lo, unsigned long long hi) { return lo != HP_SENTINEL && hi != HP_SENTINEL; }
// a runaway wait: stop this launch (flag [0]) and leave a mark that survives it (flag [1], read by hp_sweep_status)
__device__ __forceinline__ void hp_raise_abort(unsigned int* abort_flag) {
    atomicExch(abort_flag, 1u);
    atomicExch(abort_flag + 1, 1u);
}
// spin until the word is valid; on a runaway spin raise the abort flag (the kernel then terminates)
__device__ __forceinline__ cplx xget(const cplx* p, unsigned int* abort_flag) {
    cplx v;
    unsigned int spins = 0;
    while (!xtry(p, v)) {
        if (++spins > HP_SPIN_LIMIT) { hp_raise_abort(abort_flag); break; }
        if ((spins & 0xFFF) == 0 && *((volatile unsigned int*)abort_flag)) break;
    }
    return v;
}

__device__ __forceinline__ unsigned int smem_u32(const void* p) { return (unsigned int)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned int bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned int bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, unsigned int bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned int parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

__device__ __forceinline__ cplx hp_warp_sum2(cplx v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
        v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
    }
    return v;
}
// coupling A_{j+1,j}[c] = c3 of grid row j+1 = s2((j+.5)h)/(h^2 s1(ih)) = A_{j,j+1}[c] (c4 of row j); rowfac is
// the x2 part for the pair (j, j+1), 1-based j
__device__ __forceinline__ cplx hp_rowfac(const HpSweepArgs& a, int j) { return cscale(a.ih2, a.s2t[2 * j + 1]); }

#define HP_BULK_CHUNK 32768u
