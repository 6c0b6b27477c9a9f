// Cluster sweep kernel for EIGHT right-hand sides on the FP64 tensor cores (DMMA.8x8x4, mma.sync m8n8k4 f64).
//
// Same skeleton as csrc/hp_sweep4m.cu (clusters, distributed shared memory, one hand-over of the separator solution
// through L2 per strip, warp-specialised groups, TMA rings).  With eight vectors every phase of a strip is a small
// complex matrix product with N = 8 columns:
//     leaf product      Y0 = W(t) V          [CW x q] [q x 8]        all 8 off-path warps (4 row tiles x 2 halves of q)
//     interface data    Gb = Gc(t) Vb        [2b x CW] [CW x 8]      off-path warps 4-7
//     correction        C  = Gc(t-1)^T X3    [CW x 2b] [2b x 8]      off-path warps 0-3 (these own the per-column state)
//     separator rhs     P  = R(t) X3         [b x 3b] [3b x 8]       critical warps, 3b split three ways
//     separator rows    X  = N(t) Rho        [NRQ x b] [b x 8]       critical warps
// In the scalar kernel each complex multiply-add costs about one 16-byte shared-memory load per lane, and the
// shared-memory pipe (71 % busy in ncu, FP64 pipe 18 %) bounds the strip.  An 8x8x4 tile needs one operand load per lane
// for 8 multiply-adds per lane and no cross-lane reduction.  A complex tile product is three real DMMAs (see CFrag).
// Fragment layout (PTX mma.m8n8k4.f64): with g = lane/4, t = lane%4 a lane holds A[g][t], B[t][g], C[g][2t], C[g][2t+1].
// Operand strides in shared memory are chosen so that the 8 lanes of a quarter warp hit 32 different banks: rows that
// follow each other in a tile are 4 matrix rows apart (tile row g <-> matrix row 4 g + tile index), vector arrays have
// strides = 4 mod 8 complex numbers.
#include "hp_sweep4_dev.cuh"

#include <stdlib.h>
#include <string.h>

#define RT 8
#define HP4D_THREADS (HP4_CRIT + HP4_PROD + HP4_OFF)   // 12 warps: three per scheduler, up to 168 registers per thread
#define HP4D_NPOLL 3        // off-path warps 4..6 fetch the gf partials of the right neighbour after their interface products
#define HP4D_PW 4          // words per lane and round of the poll warp
#define HP4D_EW 3          // gathered entries per warp and batch

struct Hp4dPlan {
    int RC, NCH, S;                     // rows per W chunk, chunks per strip (all resident at once), slots of the W ring
    int QPV, CWV, BV, B3V, NRQV;        // padded strides (complex numbers)
    size_t w_st, g_st, n_st, r_st;      // stage strides in bytes
    size_t total;
};

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// Complex accumulator fragment.  The FP64 pipe is what every phase of a strip waits for once the operands come from
// registers (DMMA and DFMA share one datapath: 64 multiply-adds per clock and SM, tools/micro/dmma_mix.cu), so a complex
// tile product is formed with THREE real DMMAs instead of four (Karatsuba / "3M"):
//     p1 = ar br,  p2 = ai bi,  p3 = (ar + ai)(br + bi);     re = p1 - p2,   im = p3 - p1 - p2
// The three accumulators are independent chains.  The imaginary part is formed with one more rounding of size
// eps (|p1| + |p2| + |p3|): norm-wise as accurate as the four-product form (tests: 1e-13 against the scalar kernels).
struct CFrag {
    double p1[2], p2[2], p3[2];
    __device__ __forceinline__ cplx get(int i) const { return cmake(p1[i] - p2[i], p3[i] - p1[i] - p2[i]); }
    __device__ __forceinline__ void add(int i, cplx v) { p1[i] += v.x; p3[i] += v.x + v.y; }
};
__device__ __forceinline__ void cfrag_zero(CFrag& c) { c.p1[0] = c.p1[1] = c.p2[0] = c.p2[1] = c.p3[0] = c.p3[1] = 0.0; }
// C += A B for complex fragments
__device__ __forceinline__ void cmma(CFrag& c, cplx a, cplx b) {
    dmma884(c.p1[0], c.p1[1], a.x, b.x);
    dmma884(c.p2[0], c.p2[1], a.y, b.y);
    dmma884(c.p3[0], c.p3[1], a.x + a.y, b.x + b.y);
}
// A dependent DMMA waits ~200 cycles for its accumulator (tools/micro/dmma.cu: one warp with 8 independent chains issues
// one DMMA per 25 cycles), 12 times the 16 cycles it occupies the pipe: every product below runs its k-steps on
// NST interleaved accumulator sets (3 NST independent chains) that are summed at the end.
#define NST 4
__device__ __forceinline__ void cfrag_zero4(CFrag (&c)[NST]) {
#pragma unroll
    for (int i = 0; i < NST; ++i) cfrag_zero(c[i]);
}
__device__ __forceinline__ cplx cfrag_get4(const CFrag (&c)[NST], int i) {
    CFrag t;
    t.p1[i] = (c[0].p1[i] + c[1].p1[i]) + (c[2].p1[i] + c[3].p1[i]);
    t.p2[i] = (c[0].p2[i] + c[1].p2[i]) + (c[2].p2[i] + c[3].p2[i]);
    t.p3[i] = (c[0].p3[i] + c[1].p3[i]) + (c[2].p3[i] + c[3].p3[i]);
    return t.get(i);
}
__device__ __forceinline__ cplx cz() { return cmake(0.0, 0.0); }

// State of the separator column b-1 carried from strip to strip for two right-hand sides, one per lane that owns it
// (4 lanes of critical warp 0).  It lives in shared memory: held in registers, it pushed the critical warps past the
// 168-register cap and the whole per-strip loop spilled to local memory.
struct HpSepState { cplx usbase[2], vsb[2], o_usep[2], o_usbase[2], o_c, cis1, ys[2], usep[2]; };
// u[i] -> shared memory without a register (cp.async, waited for with cp_async_wait_all); a masked slot (u = NULL) or
// take = false gives 0 and reads nothing (src-size 0; `any` is only a valid address)
__device__ __forceinline__ void cp_async_slot(cplx* dst, const cplx* u, size_t i, bool take, const void* any) {
    const bool rd = take && u;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(rd ? (const void*)(u + i) : any),
                 "r"(rd ? 16 : 0) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// MODE: 0 forward, 1 backward (reference diagonal), 2 backward (paper diagonal)
template <int MODE, bool DBG, int BT, int KT>
__global__ void __launch_bounds__(HP4D_THREADS, 1) hp_sweep4d_kernel(HpSweepArgs a, Hp4dPlan pl) {
    constexpr int a_mode = MODE == 0 ? 0 : 1;
    constexpr int a_diag = MODE == 2 ? 1 : 0;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = BT ? BT : a.b, b2 = 2 * b, b3 = 3 * b, n = a.n, K = KT ? KT : a.lay.K, P = a.lay.P, QP = a.lay.QP, CW = a.lay.CW;
    const int NS = a.lay.NS, NRQ = a.lay.NRQ, NXG = a.lay.NXG;
    const int QPV = pl.QPV, CWV = pl.CWV, BV = pl.BV, B3V = pl.B3V, NRQV = pl.NRQV;
    const int PP = P | 1;
    const int g_ = blockIdx.x, l = g_ / K, k = g_ - l * K;
    const int tid = threadIdx.x, lane = tid & 31;
    const int fg = lane >> 2, ft = lane & 3;       // fragment coordinates
    const int q = a.leaf_q[l], ls = a.leaf_start[l];
    const int lc0 = (q * k) / K, lc1 = (q * (k + 1)) / K, ncols = lc1 - lc0, c0 = ls + lc0;
    unsigned int* abort_flag = a.bar + 1;
    const int step = a_mode == 1 ? -1 : 1;
    const int nsteps = a_mode == 0 ? a.m_to - a.m_from + 1 : a.m_from - a.m_to + 1;
    const int dir = a_mode == 1 ? 1 : 0;
    const double sg = a_diag == 0 ? 1.0 : -1.0;
    const bool any_sep = NS > 0;
    const bool has_sep = l < P - 1;
    const int nrq_own = has_sep ? max(0, min(NRQ, NS - NRQ * k)) : 0;
    const int nxg_own = any_sep ? max(0, min(NXG, b3 - NXG * k)) : 0;
    const int S = pl.S, RC = pl.RC, NCH = pl.NCH;

    // ---- shared memory carve-up (hp_sweep4d_plan)
    unsigned char* ringW = smem_raw;
    unsigned char* ringG = ringW + (size_t)S * pl.w_st;
    unsigned char* ringN = ringG + 3 * pl.g_st;
    unsigned char* ringR = ringN + 2 * pl.n_st;
    cplx* vb = reinterpret_cast<cplx*>(ringR + 2 * pl.r_st);     // [RT][CWV]
    cplx* v_leaf = vb + (size_t)RT * CWV;                        // [2][RT][QPV]       (DSMEM target)
    cplx* y0p = v_leaf + 2 * (size_t)RT * QPV;                   // [2][RT][CWV]       leaf product, two halves of q
    cplx* x3 = y0p + 2 * (size_t)RT * CWV;                       // [2][RT][B3V]       (DSMEM target)
    cplx* glp = x3 + 2 * (size_t)RT * B3V;                       // [2][K][b][RT]      (DSMEM target)
    cplx* rho_p = glp + 2 * (size_t)K * b * RT;                  // [3][RT][BV]        partial sums of -rho (one per critical warp)
    cplx* gfp = rho_p + 3 * (size_t)RT * BV;                     // [2][b][RT]         gf partials of leaf l+1, summed over its K parts
    HpSepState* sep_st = reinterpret_cast<HpSepState*>(gfp + 2 * (size_t)b * RT);   // [4]   one per lane ft of the separator column
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(sep_st + 4);
    unsigned long long* barW = mbar;                 // [S]
    unsigned long long* barG = barW + S;             // [3]
    unsigned long long* barN = barG + 3;             // [2]
    unsigned long long* barR = barN + 2;             // [2]
    unsigned long long* barX = barR + 2;             // [2]
    unsigned long long* barGL = barX + 2;            // [2]
    unsigned long long* barV = barGL + 2;            // [2]
    unsigned long long* eW = barV + 2;               // [S]
    unsigned long long* eG = eW + S;                 // [3]
    unsigned long long* eN = eG + 3;                 // [2]
    unsigned long long* eR = eN + 2;                 // [2]
    unsigned long long* barGF = eR + 2;              // [2]
    unsigned long long* eGF = barGF + 2;             // [2]
    volatile unsigned int* dead = reinterpret_cast<volatile unsigned int*>(eGF + 2);

    const cplx* pk_base = a.packets + (size_t)g_ * a.lay.PK;
    const size_t strip_stride = (size_t)a.lay.G * a.lay.PK;
    const int m0 = a.m_from;
    const unsigned int x_bytes = (unsigned int)(b3 * RT * sizeof(cplx)), gl_bytes = (unsigned int)((size_t)K * b * RT * sizeof(cplx)),
                       v_bytes = (unsigned int)(q * RT * sizeof(cplx));

    if (tid == 0) {
        for (int i = 0; i < S + 13; ++i) mbar_init(&mbar[i], 1);
        for (int i = 0; i < S + 3; ++i) mbar_init(&eW[i], HP4_OFF / 32);
        for (int i = 0; i < 4; ++i) mbar_init(&eN[i], HP4_CW);
        for (int i = 0; i < 2; ++i) { mbar_init(&barGF[i], HP4D_NPOLL); mbar_init(&eGF[i], HP4_CW); }
        *dead = 0u;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async;" ::: "memory");
        for (int p = 0; p < 2; ++p) {
            if (any_sep) mbar_expect_tx(&barX[p], x_bytes);
            if (has_sep) mbar_expect_tx(&barGL[p], gl_bytes);
            mbar_expect_tx(&barV[p], v_bytes);
        }
    }
    // the padding of the vector arrays is read by the tile loads (multiplied by zero rows/columns): keep it finite
    for (int i = tid; i < (int)(((unsigned char*)mbar - (unsigned char*)vb) / sizeof(cplx)); i += HP4D_THREADS) vb[i] = cz();
    __syncthreads();
    cluster_sync_all();

    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = 0;
#define HPD_TICK(i) do { if (DBG && lane == 0 && (tid == 0 || tid == HP4_CRIT + HP4_PROD)) { long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } } while (0)

    if (tid < HP4_CRIT) {
        // =====================================================================================================
        // critical group (3 warps).  A lane's accumulator fragment covers entry / row "fg" of a tile and the
        // right-hand sides 2 ft, 2 ft + 1.
        // =====================================================================================================
        const int ctid = tid, cw = ctid >> 5;
        // separator column: the lanes of warp 0 whose fragment holds entry b-1 (tile (b-1)/8, row (b-1)%8) keep its state for
        // their two right-hand sides
        const int sep_tile = (b - 1) >> 3;
        const bool is_sep = has_sep && cw == 0 && fg == ((b - 1) & 7);
        const int sep_col = has_sep ? a.sep[l] : 0;
        HpSepState& ss = sep_st[ft];                  // zero from the fill above; touched by the is_sep lanes only
        if (is_sep) {
            const cplx cis1s = a.is1t[2 * (sep_col + 1)];
            ss.cis1 = cis1s;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                cplx* u = a.um[2 * ft + i];
                if (a_mode == 0) ss.vsb[i] = ldcg_slot(u, (size_t)(m0 - 1) * n + sep_col);
                else {
                    const cplx ub = ldcg_slot(u, (size_t)(m0 - 1) * n + sep_col);
                    ss.usbase[i] = ub;
                    ss.vsb[i] = m0 < n ? cfma(cscale(sg, cmul(hp_rowfac(a, m0), cis1s)), ldcg_slot(u, (size_t)m0 * n + sep_col), ub) : ub;
                }
            }
        }
        auto sep_output = [&](int m_prev, int i, cplx ys) {   // y_s = x_l[b-1] of strip m_prev, right-hand side 2 ft + i
            if (k != 0) return;
            cplx* u = a.um[2 * ft + i];
            if (a_mode == 0) st_slot(u, (size_t)m_prev * n + sep_col, cfms(ss.o_c, ys, ss.o_usep[i]));
            else st_slot(u, (size_t)(m_prev - 1) * n + sep_col, a_diag == 0 ? csub(ss.o_usbase[i], ys) : ys);
        };
        const int nks_b = (b3 + 3) >> 2, ks_per = (nks_b + HP4_CW - 1) / HP4_CW;       // k-steps of P = R X3, split over the warps
        const int ntile_e = (b + 7) >> 3;                                              // entry tiles (2 for b = 12)
        const int ntile_r = 4 * ((NRQ + 31) >> 5), nks_c = (b + 3) >> 2;                // row tiles (blocks of 32 rows) / k-steps of X = N Rho

        for (int it = 0; it < nsteps; ++it) {
            const int m = m0 + it * step, mn = m + step;
            const bool more = it + 1 < nsteps;
            const int par = it & 1, ph = (it >> 1) & 1;
            cplx* slot = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride;
            cplx* slot_next = a.xch + (size_t)((it + 1) & (HP_RING - 1)) * a.slot_stride;
            const cplx* x3p = x3 + (size_t)(par ^ 1) * RT * B3V;                                // x3(it-1), [RT][B3V]
            if (DBG && tid == 0) tprev = clock64();
            if (is_sep) {                                   // the field entries of the separator column, used at the end of the strip
#pragma unroll
                for (int i = 0; i < 2; ++i)
                    cp_async_slot(&ss.usep[i], a.um[2 * ft + i], a_mode == 0 ? (size_t)m * n + sep_col : (size_t)(mn - 1) * n + sep_col,
                                  a_mode == 0 || more, a.is1t);
            }
            // ---- x-independent part: the K partial sums of gl (DSMEM) and gf (L2, poll warp), split over the warps
            CFrag acc[2][2];                                // entry tiles 0, 1 (b <= 16: see the host check), two k-streams each
            cfrag_zero(acc[0][0]); cfrag_zero(acc[0][1]); cfrag_zero(acc[1][0]); cfrag_zero(acc[1][1]);
            if (has_sep) {
                mbar_wait4(&barGL[par], ph, abort_flag, dead);
                mbar_wait_acq4(&barGF[par], ph, abort_flag, dead);
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int e = fg + 8 * t;
                    if (t < ntile_e && e < b) {
                        for (int kk = cw; kk < K; kk += HP4_CW) {
                            const size_t o = (((size_t)par * K + kk) * b + e) * RT + 2 * ft;
                            acc[t][0].add(0, glp[o]); acc[t][0].add(1, glp[o + 1]);
                        }
                        if (cw == HP4_CW - 1) {
                            const size_t o = ((size_t)par * b + e) * RT + 2 * ft;
                            acc[t][0].add(0, gfp[o]); acc[t][0].add(1, gfp[o + 1]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_rel4(&eGF[par]);
                mbar_wait4(&barR[par], ph, abort_flag, dead);
            }
            HPD_TICK(0);
            // ---- A: x3(it-1)
            if (it > 0 && any_sep) {
                mbar_wait4(&barX[par ^ 1], ((it - 1) >> 1) & 1, abort_flag, dead);
                if (ctid == 0 && it + 1 < nsteps) mbar_expect_tx(&barX[par ^ 1], x_bytes);
            }
            HPD_TICK(1);
            if (has_sep) {
                // ---- B: P = R(it) X3(it-1): this warp's share of the 3b columns, both entry tiles
                const cplx* R = reinterpret_cast<const cplx*>(ringR + par * pl.r_st);
                if (it > 0) {
                    const int ks_end = min(nks_b, (cw + 1) * ks_per);
                    for (int ks0 = cw * ks_per; ks0 < ks_end; ks0 += 2) {
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const int c = 4 * (ks0 + j) + ft;
                            const bool on = ks0 + j < ks_end && c < b3;
                            const cplx bv = on ? x3p[(size_t)fg * B3V + c] : cz();
                            const cplx a0 = (on && fg < b) ? R[(size_t)fg * b3 + c] : cz();
                            const cplx a1 = (on && ntile_e > 1 && fg + 8 < b) ? R[(size_t)(fg + 8) * b3 + c] : cz();
                            cmma(acc[0][j], a0, bv);
                            cmma(acc[1][j], a1, bv);
                        }
                    }
                }
                // -rho = pre + R x3 - [e = b-1] vsb ; the three warps' shares are summed by the readers
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int e = fg + 8 * t;
                    if (t < ntile_e && e < b) {
                        cplx r0 = cadd(acc[t][0].get(0), acc[t][1].get(0)), r1 = cadd(acc[t][0].get(1), acc[t][1].get(1));
                        if (is_sep && t == sep_tile) { r0 = csub(r0, ss.vsb[0]); r1 = csub(r1, ss.vsb[1]); }
                        rho_p[((size_t)cw * RT + 2 * ft) * BV + e] = r0;
                        rho_p[((size_t)cw * RT + 2 * ft + 1) * BV + e] = r1;
                    }
                }
            }
            if (is_sep && it > 0) {
                ss.ys[0] = x3p[(size_t)(2 * ft) * B3V + b2 - 1];     // x3(it-1) is overwritten from strip it+1 on
                ss.ys[1] = x3p[(size_t)(2 * ft + 1) * B3V + b2 - 1];
            }
            if (has_sep) {
                bar_crit4();
                HPD_TICK(2);
                // ---- C: own rows of X(it) = N[:, sep l] Rho: row tiles round robin over the warps
                if (nrq_own > 0) mbar_wait4(&barN[par], ph, abort_flag, dead);
                const cplx* Np = reinterpret_cast<const cplx*>(ringN + par * pl.n_st);          // [b][NRQV]
                cplx bq[NST];                                // B fragments of the k-steps (b <= 16)
#pragma unroll
                for (int ks = 0; ks < NST; ++ks) {
                    const int c = 4 * ks + ft;
                    cplx s = cz();
                    if (ks < nks_c && c < b) {
                        const size_t o = (size_t)fg * BV + c;
                        s = cneg(cadd(cadd(rho_p[o], rho_p[(size_t)RT * BV + o]), rho_p[(size_t)2 * RT * BV + o]));
                    }
                    bq[ks] = s;
                }
                for (int tr0 = cw; tr0 < ntile_r; tr0 += 2 * HP4_CW) {          // two row tiles at a time: 8 independent DMMA chains
                    // tile row fg <-> row 32 (tr / 4) + 4 fg + tr % 4: consecutive tile rows are 4 rows apart (banks)
                    const int tr1 = tr0 + HP4_CW;
                    const int row0 = 32 * (tr0 >> 2) + 4 * fg + (tr0 & 3);
                    const int row1 = tr1 < ntile_r ? 32 * (tr1 >> 2) + 4 * fg + (tr1 & 3) : nrq_own;
                    CFrag xa[NST], xb[NST];                      // one accumulator set per k-step (b <= 16: at most 4)
                    cfrag_zero4(xa); cfrag_zero4(xb);
#pragma unroll
                    for (int ks = 0; ks < NST; ++ks) {
                        const int c = 4 * ks + ft;
                        if (ks < nks_c) {                      // warp-uniform
                            const cplx a0 = (row0 < nrq_own && c < b) ? Np[(size_t)c * NRQV + row0] : cz();
                            const cplx a1 = (row1 < nrq_own && c < b) ? Np[(size_t)c * NRQV + row1] : cz();
                            cmma(xa[ks], a0, bq[ks]);
                            cmma(xb[ks], a1, bq[ks]);
                        }
                    }
                    if (row0 < nrq_own) {
                        const size_t o = a.oXS + ((size_t)(NRQ * k + row0) * PP + l) * RT + 2 * ft;
                        xput(slot + o, cfrag_get4(xa, 0)); xput(slot + o + 1, cfrag_get4(xa, 1));
                        xarm(slot_next + o); xarm(slot_next + o + 1);
                    }
                    if (row1 < nrq_own) {
                        const size_t o = a.oXS + ((size_t)(NRQ * k + row1) * PP + l) * RT + 2 * ft;
                        xput(slot + o, cfrag_get4(xb, 0)); xput(slot + o + 1, cfrag_get4(xb, 1));
                        xarm(slot_next + o); xarm(slot_next + o + 1);
                    }
                }
                HPD_TICK(3);
                __syncwarp();
                if (lane == 0) { mbar_arrive_local(&eN[par]); mbar_arrive_local(&eR[par]); }
                if (ctid == 0 && it + 2 < nsteps) mbar_expect_tx(&barGL[par], gl_bytes);
            }
            // ---- D: gather x3(it): a warp load covers 4 separators x 8 right-hand sides of one entry.  The separator column's
            //      field reads of this strip complete before it: x3(it) lets the CTA k = 0 of the leaf overwrite that entry.
            if (is_sep) cp_async_wait_all();
            if (any_sep) {
                const int lr = lane % RT, lsub = lane / RT;
                constexpr int SPL = 32 / RT;
                for (int tb = 0; tb < nxg_own; tb += HP4_CW * HP4D_EW) {
                    int ent[HP4D_EW];
                    cplx val[HP4D_EW];
#pragma unroll
                    for (int o = 0; o < HP4D_EW; ++o) {
                        const int tt = tb + cw + HP4_CW * o;
                        const int e = tt < nxg_own ? (l - 1) * b + NXG * k + tt : -1;
                        ent[o] = (e >= 0 && e < NS) ? e : -1;
                        val[o] = cz();
                    }
                    unsigned int spins = 0;
                    for (;;) {
                        unsigned long long lo[HP4D_EW][RT], hi[HP4D_EW][RT];
#pragma unroll
                        for (int o = 0; o < HP4D_EW; ++o)
#pragma unroll
                            for (int i = 0; i < RT; ++i) {
                                lo[o][i] = hi[o][i] = 0ull;
                                const int sp = lsub + SPL * i;
                                if (ent[o] >= 0 && sp < P - 1) xload(slot + a.oXS + ((size_t)ent[o] * PP + sp) * RT + lr, lo[o][i], hi[o][i]);
                            }
                        bool ok = true;
#pragma unroll
                        for (int o = 0; o < HP4D_EW; ++o) {
                            cplx sacc = cz();
#pragma unroll
                            for (int i = 0; i < RT; ++i) {
                                ok = ok && xvalid(lo[o][i], hi[o][i]);
                                sacc = cadd(sacc, cmake(__longlong_as_double((long long)lo[o][i]), __longlong_as_double((long long)hi[o][i])));
                            }
                            val[o] = sacc;
                        }
                        if (__all_sync(0xffffffffu, ok || *dead)) break;
                        if (++spins > HP_SPIN_LIMIT) { hp_raise_abort(abort_flag); *dead = 1u; }
                        if ((spins & 0xFFF) == 0 && *((volatile unsigned int*)abort_flag)) *dead = 1u;
                    }
                    HPD_TICK(4);
#pragma unroll
                    for (int o = 0; o < HP4D_EW; ++o) {
#pragma unroll
                        for (int of = RT; of < 32; of <<= 1) {
                            val[o].x += __shfl_xor_sync(0xffffffffu, val[o].x, of);
                            val[o].y += __shfl_xor_sync(0xffffffffu, val[o].y, of);
                        }
                    }
#pragma unroll
                    for (int o = 0; o < HP4D_EW; ++o) {
                        const int tt = tb + cw + HP4_CW * o;
                        if (tt < nxg_own)
                            for (int d = lsub; d < K; d += SPL)
                                st_async_cplx(mapa_u32(smem_u32(x3 + ((size_t)par * RT + lr) * B3V + NXG * k + tt), d), val[o],
                                              mapa_u32(smem_u32(&barX[par]), d));
                    }
                }
                HPD_TICK(5);
            }
            // ---- the separator column: output of strip it-1 and the state of strip it+1, after this strip's hand-over so that
            //      neither the field load nor the store holds up the critical warps
            if (is_sep) {
                const cplx cs = cmul(hp_rowfac(a, a_mode == 1 ? mn : m), ss.cis1);
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    if (it > 0) sep_output(m - step, i, ss.ys[i]);
                    const cplx ub = ss.usbase[i], usep = ss.usep[i];
                    ss.o_usep[i] = usep; ss.o_usbase[i] = ub;
                    if (a_mode == 0) ss.vsb[i] = usep;
                    else { ss.vsb[i] = a_diag == 0 ? cfma(cs, ub, usep) : usep; ss.usbase[i] = usep; }
                }
                ss.o_c = cs;
            }
        }
        if (any_sep && nsteps > 0 && is_sep) {
            const int itl = nsteps - 1;
            mbar_wait4(&barX[itl & 1], (itl >> 1) & 1, abort_flag, dead);
#pragma unroll
            for (int i = 0; i < 2; ++i) sep_output(m0 + itl * step, i, x3[((size_t)(itl & 1) * RT + 2 * ft + i) * B3V + b2 - 1]);
        }
        if (DBG && tid == 0)
            for (int i = 0; i < 6; ++i) a.dbg[(size_t)g_ * 16 + i] = tacc[i];
    } else if (tid < HP4_CRIT + HP4_PROD) {
        // =====================================================================================================
        // producer warp: every TMA copy of the sweep.  The columns of N go to rows of NRQV (padded) complex numbers.
        // =====================================================================================================
        if (lane == 0) {
            const unsigned int ncol_bytes = (unsigned int)((size_t)NRQ * sizeof(cplx)), r_bytes = (unsigned int)((size_t)b * b3 * sizeof(cplx));
            const unsigned int g_bytes = (unsigned int)((size_t)b2 * CW * sizeof(cplx)), pk_bytes = (unsigned int)(a.lay.PK * sizeof(cplx));
            const cplx* n_base = pk_base + a.lay.offN;
            const cplx* g_base = pk_base + a.lay.offG;
            const size_t r_stride = (size_t)2 * (P - 1) * b * b3;
            const cplx* r_base = has_sep ? a.rsep + ((size_t)dir * (P - 1) + l) * b * b3 : nullptr;
            for (int it = 0; it < nsteps; ++it) {
                const size_t so = (size_t)(m0 + it * step - a.m_lo);
                if (it + 2 < nsteps) {
                    const char* src = (const char*)(pk_base + (size_t)(m0 + (it + 2) * step - a.m_lo) * strip_stride);
                    for (unsigned int o = 0; o < pk_bytes; o += HP_BULK_CHUNK) bulk_prefetch_l2(src + o, min(HP_BULK_CHUNK, pk_bytes - o));
                }
                if (it >= 3) mbar_wait4(&eG[it % 3], ((it / 3) - 1) & 1, abort_flag, dead);
                ring_fill4(ringG + (size_t)(it % 3) * pl.g_st, g_base + so * strip_stride, g_bytes, &barG[it % 3]);
                if (has_sep) {
                    if (it >= 2) { mbar_wait4(&eN[it & 1], ((it >> 1) - 1) & 1, abort_flag, dead); mbar_wait4(&eR[it & 1], ((it >> 1) - 1) & 1, abort_flag, dead); }
                    if (nrq_own > 0) {
                        mbar_expect_tx(&barN[it & 1], ncol_bytes * b);
                        for (int c = 0; c < b; ++c)
                            bulk_g2s(ringN + (size_t)(it & 1) * pl.n_st + (size_t)c * NRQV * sizeof(cplx), n_base + so * strip_stride + (size_t)c * NRQ,
                                     ncol_bytes, &barN[it & 1]);
                    }
                    ring_fill4(ringR + (size_t)(it & 1) * pl.r_st, r_base + so * r_stride, r_bytes, &barR[it & 1]);
                }
                for (int ch = 0; ch < NCH; ++ch) {
                    const int cidx = it * NCH + ch, sl = cidx % S, r0 = ch * RC;
                    if (cidx >= S) mbar_wait4(&eW[sl], ((cidx / S) - 1) & 1, abort_flag, dead);
                    ring_fill4(ringW + (size_t)sl * pl.w_st, pk_base + so * strip_stride + (size_t)r0 * QP,
                               (unsigned int)((size_t)min(RC, CW - r0) * QP * sizeof(cplx)), &barW[sl]);
                }
            }
        }
    } else {
        // =====================================================================================================
        // off-path group (8 warps).  Warps 0-3 own the per-column state: lane -> column oc = 4 fg + ow, right-hand sides
        // 2 ft and 2 ft + 1 (exactly the accumulator fragment of the correction product).  Warps 4-7 form the interface
        // data of the strip meanwhile.  All 8 warps share the leaf product.
        // =====================================================================================================
        const int ot = tid - HP4_CRIT - HP4_PROD, ow = ot >> 5;
        const bool owner = ow < 4;
        const int oc = 4 * fg + (ow & 3);
        const bool col = owner && oc < ncols;
        const int c = c0 + oc;
        cplx* const u0 = a.um[2 * ft];
        cplx* const u1 = a.um[2 * ft + 1];
        const cplx cis1 = col ? a.is1t[2 * (c + 1)] : cz();
        cplx vbr[2] = {cz(), cz()}, y0prev[2] = {cz(), cz()}, ubase[2] = {cz(), cz()}, ubase_prev[2] = {cz(), cz()};
        cplx coefc = cz();
        if (col) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                cplx* u = i ? u1 : u0;
                if (a_mode == 0) vbr[i] = ldcg_slot(u, (size_t)(m0 - 1) * n + c);
                else {
                    ubase[i] = ldcg_slot(u, (size_t)(m0 - 1) * n + c);
                    vbr[i] = ubase[i];
                    if (m0 < n) vbr[i] = cfma(cscale(sg, cmul(hp_rowfac(a, m0), cis1)), ldcg_slot(u, (size_t)m0 * n + c), vbr[i]);
                }
                vb[(size_t)(2 * ft + i) * CWV + oc] = vbr[i];
            }
        }
        bar_off4();
        // leaf product: warp -> (row tile ow & 3, half ow >> 2 of the k-steps); tile row fg <-> row 4 fg + tile
        const int wrow = 4 * fg + (ow & 3);
        const int nks_w = (q + 3) >> 2, ks_half = (nks_w + 1) >> 1;
        const int ks_lo = (ow >> 2) * ks_half, ks_hi = min(nks_w, ks_lo + ks_half);
        const cplx* wrow_ptr_off = nullptr;                 // set per strip (ring slot of the row's chunk)
        (void)wrow_ptr_off;
        const int nks_g = (ncols + 3) >> 2;                 // k-steps of Gb = Gc Vb
        const int nks_x = (b2 + 3) >> 2;                    // k-steps of C = Gc^T X3

        for (int it = 0; it <= nsteps; ++it) {
            const int m = m0 + it * step, mn = m + step, mp = m - step;
            const bool live = it < nsteps, more = it + 1 < nsteps;
            const int par = it & 1, ph = (it >> 1) & 1;
            cplx* slot = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride;
            cplx* slot_arm = a.xch + (size_t)((it + 2) & (HP_RING - 1)) * a.slot_stride;
            const cplx* Gp = reinterpret_cast<const cplx*>(ringG + (size_t)(it % 3) * pl.g_st);
            const cplx* Gprev = reinterpret_cast<const cplx*>(ringG + (size_t)((it + 2) % 3) * pl.g_st);
            const cplx rf_it = hp_rowfac(a, a_mode == 1 ? mn : m);
            cplx unx[2] = {cz(), cz()};
            if (col && live) {
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    cplx* u = i ? u1 : u0;
                    if (a_mode == 0) unx[i] = ldcg_slot(u, (size_t)m * n + c);
                    else if (more) unx[i] = ldcg_slot(u, (size_t)(mn - 1) * n + c);
                }
            }
            if (DBG && (ot == 0 || ot == 128)) tprev = clock64();
#define HPD_TICK4(i) do { if (DBG && ot == 128) { long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } } while (0)
            if (!owner) {
                // ---- a (warps 4-7): Gb(t) = Gc(t) Vb(t): row tile ow - 4 of the 2b interface components (4 tiles cover b <= 16;
                //      larger b: a second pass), gf -> cluster l-1 (L2), gl -> every CTA of the cluster (DSMEM)
                if (live) {
                    mbar_wait4(&barG[it % 3], (it / 3) & 1, abort_flag, dead);
                    HPD_TICK4(0);
                    if (any_sep) {
                        for (int kap0 = 0; kap0 < b2; kap0 += 32) {
                            const int kap = kap0 + 4 * fg + (ow & 3);
                            CFrag gb[NST];
                            cfrag_zero4(gb);
                            for (int ks0 = 0; ks0 < nks_g; ks0 += NST) {
                                cplx av[NST], bv[NST];
#pragma unroll
                                for (int j = 0; j < NST; ++j) {
                                    const int cc = 4 * (ks0 + j) + ft;
                                    av[j] = (kap < b2 && cc < ncols) ? Gp[(size_t)kap * CW + cc] : cz();
                                    bv[j] = cc < ncols ? vb[(size_t)fg * CWV + cc] : cz();
                                }
#pragma unroll
                                for (int j = 0; j < NST; ++j) cmma(gb[j], av[j], bv[j]);
                            }
                            const cplx r0 = cfrag_get4(gb, 0), r1 = cfrag_get4(gb, 1);
                            if (kap < b) {
                                if (l > 0) {
                                    const size_t o = a.oGP + (((size_t)l * K + k) * b + kap) * RT + 2 * ft;
                                    xput(slot + o, r0); xput(slot + o + 1, r1);
                                    xarm(slot_arm + o); xarm(slot_arm + o + 1);
                                }
                            } else if (kap < b2 && has_sep) {
                                for (int d = 0; d < K; ++d) {
                                    const unsigned int dst = mapa_u32(smem_u32(glp + (((size_t)par * K + k) * b + (kap - b)) * RT + 2 * ft), d);
                                    const unsigned int bar = mapa_u32(smem_u32(&barGL[par]), d);
                                    st_async_cplx(dst, r0, bar);
                                    st_async_cplx(dst + (unsigned int)sizeof(cplx), r1, bar);
                                }
                            }
                        }
                    }
                }
                if (it > 0) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&eG[(it + 2) % 3]);
                }
                if (!live) break;
                HPD_TICK4(1);
                // ---- the gf partials of leaf l+1 for this strip ([K][b][RT] self-validating words in L2, written by the same
                //      phase of the clusters on the right): warps 4..6 sum the K parts of 32 outputs each and hand them to the
                //      critical group in shared memory
                if (has_sep && ow - 4 < HP4D_NPOLL) {
                    const int no = b * RT, nw = K * no;
                    const cplx* src = slot + a.oGP + (size_t)(l + 1) * nw;
                    if (it >= 2) mbar_wait4(&eGF[par], ((it >> 1) - 1) & 1, abort_flag, dead);
                    for (int i0 = 32 * (ow - 4); i0 < no; i0 += 32 * HP4D_NPOLL) {
                        const int idx = i0 + lane;
                        cplx sum = cz();
                        unsigned int spins = 0;
                        for (;;) {
                            unsigned long long lo[8], hi[8];
                            bool ok = true;
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) {
                                lo[kk] = hi[kk] = 0ull;
                                if (kk < K && idx < no) xload(src + (size_t)kk * no + idx, lo[kk], hi[kk]);
                            }
                            sum = cz();
#pragma unroll
                            for (int kk = 0; kk < 8; ++kk) {
                                ok = ok && xvalid(lo[kk], hi[kk]);
                                sum = cadd(sum, cmake(__longlong_as_double((long long)lo[kk]), __longlong_as_double((long long)hi[kk])));
                            }
                            if (__all_sync(0xffffffffu, ok || *dead)) break;
                            if (++spins > HP_SPIN_LIMIT) { hp_raise_abort(abort_flag); *dead = 1u; }
                            if ((spins & 0xFFF) == 0 && *((volatile unsigned int*)abort_flag)) *dead = 1u;
                        }
                        if (idx < no) gfp[(size_t)par * no + idx] = sum;
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive_rel4(&barGF[par]);
                }
                HPD_TICK4(2);
            } else {
                // ---- b (warps 0-3): x3(t-1) arrives: correction C = Gc(t-1)^T [x_{l-1}; x_l], finish strip t-1 on the own
                //      columns, input of strip t to every CTA of the leaf
                cplx v[2] = {vbr[0], vbr[1]};
                if (it > 0) {
                    CFrag cr[NST];
                    cfrag_zero4(cr);
                    if (any_sep) {
                        mbar_wait4(&barX[par ^ 1], ((it - 1) >> 1) & 1, abort_flag, dead);
                        HPD_TICK(2);
                        const cplx* xa = x3 + (size_t)(par ^ 1) * RT * B3V;
                        for (int ks0 = 0; ks0 < nks_x; ks0 += NST) {
                            cplx av[NST], bv[NST];
#pragma unroll
                            for (int j = 0; j < NST; ++j) {
                                const int kap = 4 * (ks0 + j) + ft;
                                av[j] = (oc < ncols && kap < b2) ? Gprev[(size_t)kap * CW + oc] : cz();
                                bv[j] = kap < b2 ? xa[(size_t)fg * B3V + kap] : cz();
                            }
#pragma unroll
                            for (int j = 0; j < NST; ++j) cmma(cr[j], av[j], bv[j]);
                        }
                    }
                    const cplx corr[2] = {cfrag_get4(cr, 0), cfrag_get4(cr, 1)};
                    if (col) {
#pragma unroll
                        for (int i = 0; i < 2; ++i) {
                            cplx* u = i ? u1 : u0;
                            v[i] = cfma(coefc, corr[i], vbr[i]);
                            if (a_mode == 0) st_slot(u, (size_t)mp * n + c, v[i]);
                            else st_slot(u, (size_t)(mp - 1) * n + c, a_diag == 0 ? cadd(csub(ubase_prev[i], y0prev[i]), corr[i]) : csub(y0prev[i], corr[i]));
                        }
                    }
                }
                if (col && live) {
                    for (int d = 0; d < K; ++d) {
                        const unsigned int bar = mapa_u32(smem_u32(&barV[par]), d);
#pragma unroll
                        for (int i = 0; i < 2; ++i)
                            st_async_cplx(mapa_u32(smem_u32(v_leaf + ((size_t)par * RT + 2 * ft + i) * QPV + lc0 + oc), d), v[i], bar);
                    }
                }
                if (it > 0) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive_local(&eG[(it + 2) % 3]);
                }
                if (!live) break;
                HPD_TICK(3);
            }
            // ---- c: leaf product Y0(t) = W(t) V_leaf(t) on the tensor cores: all chunks of the strip are resident
            mbar_wait4(&barV[par], ph, abort_flag, dead);
            HPD_TICK(4);
            HPD_TICK4(3);
            for (int ch = 0; ch < NCH; ++ch) mbar_wait4(&barW[(it * NCH + ch) % S], ((it * NCH + ch) / S) & 1, abort_flag, dead);
            HPD_TICK(7);
            {
                const cplx* vl = v_leaf + (size_t)par * RT * QPV;
                const int wch = wrow / RC;
                const cplx* wr = reinterpret_cast<const cplx*>(ringW + (size_t)((it * NCH + wch) % S) * pl.w_st) + (size_t)(wrow - wch * RC) * QP;
                const bool rowok = wrow < ncols;
                CFrag y[NST];
                cfrag_zero4(y);
                for (int ks0 = ks_lo; ks0 < ks_hi; ks0 += NST) {
                    cplx av[NST], bv[NST];
#pragma unroll
                    for (int j = 0; j < NST; ++j) {
                        const int cq = 4 * (ks0 + j) + ft;
                        const bool on = ks0 + j < ks_hi && cq < q;
                        av[j] = (on && rowok) ? wr[cq] : cz();
                        bv[j] = on ? vl[(size_t)fg * QPV + cq] : cz();
                    }
#pragma unroll
                    for (int j = 0; j < NST; ++j) cmma(y[j], av[j], bv[j]);
                }
                if (rowok) {
                    y0p[((size_t)(ow >> 2) * RT + 2 * ft) * CWV + wrow] = cfrag_get4(y, 0);
                    y0p[((size_t)(ow >> 2) * RT + 2 * ft + 1) * CWV + wrow] = cfrag_get4(y, 1);
                }
            }
            HPD_TICK(0);
            __syncwarp();
            if (lane == 0)
                for (int ch = 0; ch < NCH; ++ch) mbar_arrive_local(&eW[(it * NCH + ch) % S]);
            bar_off4();                                      // y0p complete
            HPD_TICK(5);
            if (ot == 0 && it + 2 < nsteps) mbar_expect_tx(&barV[par], v_bytes);
            if (col) {
                coefc = cmul(rf_it, cis1);
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const size_t o = (size_t)(2 * ft + i) * CWV + oc;
                    const cplx y0 = cadd(y0p[o], y0p[(size_t)RT * CWV + o]);
                    y0prev[i] = y0;
                    if (a_mode == 0) vbr[i] = cfms(coefc, y0, unx[i]);
                    else {
                        vbr[i] = a_diag == 0 ? cfma(coefc, csub(ubase[i], y0), unx[i]) : cfms(coefc, y0, unx[i]);
                        ubase_prev[i] = ubase[i];
                        ubase[i] = unx[i];
                    }
                    vb[o] = vbr[i];
                }
            }
            bar_off4();                                      // vb ready, y0p free for the next strip
            HPD_TICK(6);
            HPD_TICK4(4);
        }
        if (DBG && ot == 0) {
            for (int i = 2; i < 8; ++i) a.dbg[(size_t)g_ * 16 + 8 + i] = tacc[i];
            a.dbg[(size_t)g_ * 16 + 6] = tacc[0];            // leaf product proper (loads + DMMA + store)
        }
        if (DBG && ot == 128) {              // warp 4: G wait, interface product, gf poll, wait V, leaf product + tail barriers
            a.dbg[(size_t)g_ * 16 + 7] = tacc[0] + tacc[1] + tacc[2];
            a.dbg[(size_t)g_ * 16 + 8 + 0] = tacc[3];
            a.dbg[(size_t)g_ * 16 + 8 + 1] = tacc[4];
        }
    }
    __syncthreads();
    cluster_sync_all();
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
static inline size_t al128d(size_t x) { return (x + 127) & ~(size_t)127; }
static inline int pad4mod8(int x) { while ((x & 7) != 4) ++x; return x; }

static int hp_sweep4d_plan(const HpLayout& L, int b, size_t max_smem, Hp4dPlan& pl) {
    if (!L.colN || L.K < 1 || L.K > 8 || L.P - 1 > 32 || L.CW > 32 || b > 16) return 1;     // two entry tiles, one pass of 2b <= 32 interface rows
    pl.QPV = pad4mod8(L.QP); pl.CWV = pad4mod8(L.CW); pl.BV = pad4mod8(b); pl.B3V = pad4mod8(3 * b);
    pl.NRQV = L.NRQ; while ((pl.NRQV & 7) != 1) ++pl.NRQV;
    pl.g_st = al128d((size_t)2 * b * L.CW * sizeof(cplx));
    pl.n_st = al128d(std::max<size_t>(1, (size_t)b * pl.NRQV) * sizeof(cplx));
    pl.r_st = al128d((size_t)b * 3 * b * sizeof(cplx));
    size_t small = sizeof(cplx) * ((size_t)RT * pl.CWV + 2 * (size_t)RT * pl.QPV + 2 * (size_t)RT * pl.CWV + 2 * (size_t)RT * pl.B3V +
                                   2 * (size_t)L.K * b * RT + 2 * (size_t)b * RT + 3 * (size_t)RT * pl.BV) + 4 * sizeof(HpSepState) +
                  8 * (2 * 8 + 13 + 7 + 4) + 16;
    size_t fixed = 3 * pl.g_st + 2 * pl.n_st + 2 * pl.r_st + al128d(small);
    if (fixed + 1024 >= max_smem) return 1;
    size_t avail = max_smem - 1024 - fixed;
    size_t row = (size_t)L.QP * sizeof(cplx);
    for (int RC = 32; RC >= 8; RC >>= 1) {
        size_t w_st = al128d((size_t)RC * row);
        int NCH = (L.CW + RC - 1) / RC;
        int S = (int)std::min<size_t>(8, avail / w_st);
        if (S < NCH) continue;                                  // every chunk of a strip must be resident
        S = NCH == 1 ? std::min(S, 2) : (S / NCH) * NCH;        // a whole number of strips
        pl.RC = RC; pl.NCH = NCH; pl.S = S; pl.w_st = w_st;
        pl.total = (size_t)S * w_st + fixed;
        return 0;
    }
    return 1;
}

template <int MODE, int BT, int KT>
static const void* hp4d_fn(bool dbg) {
    return dbg ? (const void*)hp_sweep4d_kernel<MODE, true, BT, KT> : (const void*)hp_sweep4d_kernel<MODE, false, BT, KT>;
}
static const void* hp4d_select(int mode, bool dbg, int b, int K) {
    if (b == 12 && K == 4) return mode == 0 ? hp4d_fn<0, 12, 4>(dbg) : (mode == 1 ? hp4d_fn<1, 12, 4>(dbg) : hp4d_fn<2, 12, 4>(dbg));
    return mode == 0 ? hp4d_fn<0, 0, 0>(dbg) : (mode == 1 ? hp4d_fn<1, 0, 0>(dbg) : hp4d_fn<2, 0, 0>(dbg));
}

// 0 = the layout of this solver can run the tensor-core kernel (8 right-hand sides per launch)
int hp_sweep4d_supported(hp_solver* s) {
    const HpLayout& L = s->lay;
    if (getenv("HP_NO_DMMA")) return 1;
    if (s->dmma_ok != 0) return s->dmma_ok > 0 ? 0 : 1;
    s->dmma_ok = -1;
    int dev = 0, max_smem = 0, ncl = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    if (cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 1;
    Hp4dPlan pl;
    if (hp_sweep4d_plan(L, s->b, (size_t)max_smem, pl)) return 1;
    const void* fn = hp4d_select(0, false, s->b, L.K);
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total) != cudaSuccess) { cudaGetLastError(); return 1; }
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) cudaGetLastError();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.K * 64); cfg.blockDim = dim3(HP4D_THREADS); cfg.dynamicSmemBytes = pl.total;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = L.K; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&ncl, fn, &cfg) != cudaSuccess) { cudaGetLastError(); return 1; }
    if (ncl < L.P) return 1;
    s->dmma_ok = 1;
    return 0;
}

int hp_sweep4d_launch(hp_solver* s, HpSweepArgs& a, cudaStream_t st) {
    const HpLayout& L = s->lay;
    int dev = 0, max_smem = 0;
    HP_CUDA(cudaGetDevice(&dev));
    HP_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    Hp4dPlan pl;
    if (hp_sweep4d_plan(L, s->b, (size_t)max_smem, pl)) { hp_set_error("sweep: the tensor-core cluster kernel does not fit this partition"); return 1; }
    const int mode = a.mode == 0 ? 0 : (a.diag_mode == 0 ? 1 : 2);
    const void* fn = hp4d_select(mode, a.dbg != nullptr, s->b, L.K);
    HP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.G); cfg.blockDim = dim3(HP4D_THREADS); cfg.dynamicSmemBytes = pl.total; cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = L.K; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeCooperative;
    at[1].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 2;
    void* args[] = {&a, &pl};
    if (hp_profiler_attached() || getenv("HP_NO_COOP") || !s->coop) cfg.numAttrs = 1;      // see hp_sweep4_launch
    cudaError_t e = cudaLaunchKernelExC(&cfg, fn, args);
    if (e != cudaSuccess) {
        cudaGetLastError();
        hp_set_error("sweep: %s cluster launch of %d CTAs (tensor-core kernel, 8 right-hand sides) failed: %s",
                     cfg.numAttrs == 2 ? "cooperative" : "plain", L.G, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}
