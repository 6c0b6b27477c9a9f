// Cluster sweep kernel for several right-hand sides: the strip chain of algo2_4 (/root/reference/code.py:366-380) applied
// to RT vectors in ONE pass over the strip generators.
//
// Same structure as csrc/hp_sweep4.cu (a leaf = a thread-block cluster, distributed shared memory inside the leaf, one
// hand-over of the separator solution through L2 per strip, warp-specialised groups, TMA-fed generator rings); every
// phase carries the RT right-hand sides together:
//   * a generator element is loaded from shared memory once and multiplied into RT accumulators (the leaf product
//     W(t) V, Gc(t) Vb, N rho): the sweep of one vector is a chain of latencies that leaves the FP64 pipe ~10 % busy, so
//     RT vectors cost little more than one, and the 12.6 MB of generators per strip are streamed once for all of them;
//   * the 8 lanes that split a dot product for one vector (hp_sweep4.cu) each own one right-hand side here when RT = 8
//     (RT < 8: 8/RT lanes split the sum of a right-hand side); where 8 lanes hold RT partial sums each, a
//     reduce-scatter over the lanes (7 exchanges instead of 3 RT) leaves lane r with the sum of right-hand side r;
//   * the partial separator solutions cross L2 as [entry][separator][RT] (a producer stores RT consecutive words, a
//     consumer warp reads 32/RT separators x RT right-hand sides per coalesced load).
// Requires the widest leaf part CW <= 32 (8 lanes per column), P - 1 <= 32 separators and RT in {1, 2, 4, 8}; the host
// falls back to one launch per vector otherwise.  RT = 1 runs the same arithmetic as hp_sweep4.cu.
#include "hp_sweep4_dev.cuh"

#include <stdlib.h>
#include <string.h>

#define HP4M_PW 4          // words per lane and round of the poll warp
#define HP4M_EW 3          // gathered entries per warp and batch

// the 8 lanes of a group (lane index j = lane & 7) hold RT partial sums each; on return every lane holds the total of
// right-hand side j % RT (lanes with the same j % RT hold the same number)
template <int RT>
__device__ __forceinline__ cplx group8_reduce_scatter(cplx (&a)[RT], int j) {
    // plain reductions over the lane bits that do not select a right-hand side
#pragma unroll
    for (int o = 4; o >= RT; o >>= 1) {
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            a[i].x += __shfl_xor_sync(0xffffffffu, a[i].x, o);
            a[i].y += __shfl_xor_sync(0xffffffffu, a[i].y, o);
        }
    }
    // scatter stages: keep the half the lane is responsible for, hand the other half to the partner
#pragma unroll
    for (int half = RT / 2; half >= 1; half >>= 1) {
        const bool up = (j & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const cplx keep = up ? a[i + half] : a[i];
            const cplx send = up ? a[i] : a[i + half];
            a[i] = cmake(keep.x + __shfl_xor_sync(0xffffffffu, send.x, half), keep.y + __shfl_xor_sync(0xffffffffu, send.y, half));
        }
    }
    return a[0];
}

// MODE: 0 forward, 1 backward (reference diagonal), 2 backward (paper diagonal)
// BT, KT: PML width and cluster size as compile-time constants (0 = run-time values); RT right-hand sides
template <int MODE, bool DBG, int BT, int KT, int RT>
__global__ void __launch_bounds__(HP4_THREADS, 1) hp_sweep4m_kernel(HpSweepArgs a, Hp4Plan pl) {
    constexpr int a_mode = MODE == 0 ? 0 : 1;
    constexpr int a_diag = MODE == 2 ? 1 : 0;
    constexpr int KS = 8 / RT;                     // lanes that split the sum of one right-hand side
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = BT ? BT : a.b, b2 = 2 * b, b3 = 3 * b, n = a.n, K = KT ? KT : a.lay.K, P = a.lay.P, QP = a.lay.QP, CW = a.lay.CW;
    const int NS = a.lay.NS, NRQ = a.lay.NRQ, NXG = a.lay.NXG;
    const int PP = P | 1;
    const int g = blockIdx.x, l = g / K, k = g - l * K;
    const int tid = threadIdx.x, lane = tid & 31;
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

    // ---- shared memory carve-up (must match hp_sweep4_plan with the same RT; identical in every CTA)
    unsigned char* ringW = smem_raw;
    unsigned char* ringG = ringW + (size_t)S * pl.w_st;
    unsigned char* ringN = ringG + 3 * pl.g_st;
    unsigned char* ringR = ringN + 2 * pl.n_st;
    cplx* vb = reinterpret_cast<cplx*>(ringR + 2 * pl.r_st);     // [RT][CW]
    cplx* v_leaf = vb + (size_t)RT * CW;                         // [2][RT][QP]      (DSMEM target)
    cplx* y0s = v_leaf + 2 * (size_t)RT * QP;                    // [RT][CW]
    cplx* x3 = y0s + (size_t)RT * CW;                            // [2][RT][3b]      (DSMEM target)
    cplx* glp = x3 + 2 * (size_t)RT * b3;                        // [2][K][b][RT]    (DSMEM target)
    cplx* rho_s = glp + 2 * (size_t)K * b * RT;                  // [RT][b]
    cplx* gfp = rho_s + (size_t)RT * b;                          // [2][K][b][RT]
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(gfp + 2 * (size_t)K * b * RT);
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

    const cplx* pk_base = a.packets + (size_t)g * a.lay.PK;
    const size_t strip_stride = (size_t)a.lay.G * a.lay.PK;
    const int m0 = a.m_from;
    const unsigned int x_bytes = (unsigned int)(b3 * RT * sizeof(cplx)), gl_bytes = (unsigned int)((size_t)K * b * RT * sizeof(cplx)),
                       v_bytes = (unsigned int)(q * RT * sizeof(cplx));

    if (tid == 0) {
        for (int i = 0; i < S + 13; ++i) mbar_init(&mbar[i], 1);
        for (int i = 0; i < S + 3; ++i) mbar_init(&eW[i], HP4_OFF / 32);
        for (int i = 0; i < 4; ++i) mbar_init(&eN[i], HP4_CW);
        for (int i = 0; i < 2; ++i) { mbar_init(&barGF[i], 1); mbar_init(&eGF[i], HP4_CW); }
        *dead = 0u;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async;" ::: "memory");
        for (int p = 0; p < 2; ++p) {
            if (any_sep) mbar_expect_tx(&barX[p], x_bytes);
            if (has_sep) mbar_expect_tx(&barGL[p], gl_bytes);
            mbar_expect_tx(&barV[p], v_bytes);
        }
    }
    __syncthreads();
    cluster_sync_all();

    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = 0;
#define HPM_TICK(i) do { if (DBG && lane == 0 && (tid == 0 || tid == HP4_CRIT + HP4_PROD)) { long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } } while (0)

    if (tid < HP4_CRIT) {
        // =====================================================================================================
        // critical group: thread -> (entry e = ctid/8 + 12*pass, right-hand side rr = part % RT, split ks = part / RT)
        // =====================================================================================================
        const int ctid = tid, cw = ctid >> 5, part = ctid & 7, e_lo = ctid >> 3;
        const int rr = part % RT, ks = part / RT;
        constexpr int EPP = HP4_CRIT / 8;
        constexpr int NPASS = (HP_BMAX + EPP - 1) / EPP;
        cplx* const u = a.um[rr];
        const bool is_sep = has_sep && ks == 0 && e_lo == (b - 1) % EPP;
        const bool sep_io = is_sep && u != nullptr;          // field accesses of an empty slot are skipped (reads give 0)
        const int sep_pass = (b - 1) / EPP;
        const int sep_col = has_sep ? a.sep[l] : 0;
        const cplx cis1s = is_sep ? a.is1t[2 * (sep_col + 1)] : cmake(0.0, 0.0);
        cplx usbase = cmake(0.0, 0.0), vsb = cmake(0.0, 0.0);
        cplx o_usep = cmake(0.0, 0.0), o_c = cmake(0.0, 0.0), o_usbase = cmake(0.0, 0.0);
        if (sep_io) {
            if (a_mode == 0) vsb = ldcg(u + (size_t)(m0 - 1) * n + sep_col);
            else {
                usbase = ldcg(u + (size_t)(m0 - 1) * n + sep_col);
                vsb = usbase;
                if (m0 < n) vsb = cfma(cscale(sg, cmul(hp_rowfac(a, m0), cis1s)), ldcg(u + (size_t)m0 * n + sep_col), vsb);
            }
        }
        auto sep_output = [&](int m_prev, cplx ys) {          // y_s = x_l[b-1] of strip m_prev
            if (k != 0 || !sep_io) return;
            if (a_mode == 0) u[(size_t)m_prev * n + sep_col] = cfms(o_c, ys, o_usep);
            else u[(size_t)(m_prev - 1) * n + sep_col] = a_diag == 0 ? csub(o_usbase, ys) : ys;
        };

        for (int it = 0; it < nsteps; ++it) {
            const int m = m0 + it * step, mn = m + step;
            const bool more = it + 1 < nsteps;
            const int par = it & 1, ph = (it >> 1) & 1;
            cplx* slot = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride;
            cplx* slot_next = a.xch + (size_t)((it + 1) & (HP_RING - 1)) * a.slot_stride;
            const cplx* x3p = x3 + ((size_t)(par ^ 1) * RT + rr) * b3;                          // x3(it-1) of the own right-hand side
            if (DBG && tid == 0) tprev = clock64();
            cplx usep = cmake(0.0, 0.0), cs = cmake(0.0, 0.0);
            if (is_sep) {
                cs = cmul(hp_rowfac(a, a_mode == 1 ? mn : m), cis1s);
                if (a_mode == 0) { if (sep_io) usep = ldcg(u + (size_t)m * n + sep_col); }
                else if (more && sep_io) usep = ldcg(u + (size_t)(mn - 1) * n + sep_col);
            }
            // ---- x-independent part of rho_l(it): own-cluster gl partials (DSMEM) + gf partials of leaf l+1 (L2)
            cplx pre[NPASS];
#pragma unroll
            for (int ps = 0; ps < NPASS; ++ps) pre[ps] = cmake(0.0, 0.0);
            if (has_sep) {
                mbar_wait4(&barGL[par], ph, abort_flag, dead);
                mbar_wait_acq4(&barGF[par], ph, abort_flag, dead);
#pragma unroll
                for (int ps = 0; ps < NPASS; ++ps) {
                    const int e = e_lo + EPP * ps;
                    if (e < b) {
                        cplx acc = cmake(0.0, 0.0);
                        for (int kk = ks; kk < K; kk += KS) {
                            const size_t o = (((size_t)par * K + kk) * b + e) * RT + rr;
                            acc = cadd(acc, cadd(glp[o], gfp[o]));
                        }
                        pre[ps] = acc;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_rel4(&eGF[par]);
                mbar_wait4(&barR[par], ph, abort_flag, dead);
            }
            HPM_TICK(0);
            // ---- A: x3(it-1)
            if (it > 0 && any_sep) {
                mbar_wait4(&barX[par ^ 1], ((it - 1) >> 1) & 1, abort_flag, dead);
                if (ctid == 0 && it + 1 < nsteps) mbar_expect_tx(&barX[par ^ 1], x_bytes);
            }
            HPM_TICK(1);
            if (has_sep) {
                // ---- B: rho_l(it) = rho_b - R x3(it-1), every right-hand side on its own lane(s)
                const cplx* R = reinterpret_cast<const cplx*>(ringR + par * pl.r_st);
#pragma unroll
                for (int ps = 0; ps < NPASS; ++ps) {
                    const int e = e_lo + EPP * ps;
                    cplx tot = pre[ps];
                    if (e < b && it > 0) {
                        const cplx* Rr = R + (size_t)e * b3;
                        cplx a0 = cmake(0.0, 0.0), a1 = cmake(0.0, 0.0), a2 = cmake(0.0, 0.0), a3 = cmake(0.0, 0.0);
                        int c = ks;
                        for (; c + 3 * KS < b3; c += 4 * KS) {
                            a0 = cfma(Rr[c], x3p[c], a0);
                            a1 = cfma(Rr[c + KS], x3p[c + KS], a1);
                            a2 = cfma(Rr[c + 2 * KS], x3p[c + 2 * KS], a2);
                            a3 = cfma(Rr[c + 3 * KS], x3p[c + 3 * KS], a3);
                        }
                        for (; c < b3; c += KS) a0 = cfma(Rr[c], x3p[c], a0);
                        tot = cadd(tot, cadd(cadd(a0, a1), cadd(a2, a3)));
                    }
                    if (EPP * ps < b) {                         // warp-uniform
#pragma unroll
                        for (int o = RT; o < 8; o <<= 1) {
                            tot.x += __shfl_xor_sync(0xffffffffu, tot.x, o);
                            tot.y += __shfl_xor_sync(0xffffffffu, tot.y, o);
                        }
                        if (e < b && ks == 0) {
                            cplx rho = cneg(tot);
                            if (is_sep && ps == sep_pass) rho = cadd(rho, vsb);
                            rho_s[(size_t)rr * b + e] = rho;
                        }
                    }
                }
            }
            if (is_sep) {
                if (it > 0) sep_output(m - step, x3p[b2 - 1]);
                o_usep = usep; o_c = cs; o_usbase = usbase;
                if (a_mode == 0) vsb = usep;
                else { vsb = a_diag == 0 ? cfma(cs, usbase, usep) : usep; usbase = usep; }
            }
            if (has_sep) {
                bar_crit4();
                HPM_TICK(2);
                // ---- C: own rows of x(it) restricted to the columns of separator l, all right-hand sides per row
                if (nrq_own > 0) mbar_wait4(&barN[par], ph, abort_flag, dead);
                const cplx* Np = reinterpret_cast<const cplx*>(ringN + par * pl.n_st);
                for (int r = ctid; r < nrq_own; r += HP4_CRIT) {
                    cplx acc[RT];
#pragma unroll
                    for (int i = 0; i < RT; ++i) acc[i] = cmake(0.0, 0.0);
                    for (int c = 0; c < b; ++c) {
                        const cplx np_ = Np[(size_t)c * NRQ + r];
#pragma unroll
                        for (int i = 0; i < RT; ++i) acc[i] = cfma(np_, rho_s[(size_t)i * b + c], acc[i]);
                    }
                    const size_t o = a.oXS + ((size_t)(NRQ * k + r) * PP + l) * RT;
#pragma unroll
                    for (int i = 0; i < RT; ++i) { xput(slot + o + i, acc[i]); xarm(slot_next + o + i); }
                }
                HPM_TICK(3);
                __syncwarp();
                if (lane == 0) { mbar_arrive_local(&eN[par]); mbar_arrive_local(&eR[par]); }
                if (ctid == 0 && it + 2 < nsteps) mbar_expect_tx(&barGL[par], gl_bytes);
            }
            // ---- D: gather x3(it): a warp load covers 32/RT separators x RT right-hand sides of one entry
            if (any_sep) {
                const int lr = lane % RT, lsub = lane / RT;
                constexpr int SPL = 32 / RT;                                // separators per load
                for (int tb = 0; tb < nxg_own; tb += HP4_CW * HP4M_EW) {
                    int ent[HP4M_EW];
                    cplx val[HP4M_EW];
#pragma unroll
                    for (int o = 0; o < HP4M_EW; ++o) {
                        const int tt = tb + cw + HP4_CW * o;
                        const int e = tt < nxg_own ? (l - 1) * b + NXG * k + tt : -1;
                        ent[o] = (e >= 0 && e < NS) ? e : -1;
                        val[o] = cmake(0.0, 0.0);
                    }
                    unsigned int spins = 0;
                    for (;;) {
                        unsigned long long lo[HP4M_EW][RT], hi[HP4M_EW][RT];
#pragma unroll
                        for (int o = 0; o < HP4M_EW; ++o)
#pragma unroll
                            for (int i = 0; i < RT; ++i) {
                                lo[o][i] = hi[o][i] = 0ull;
                                const int sp = lsub + SPL * i;
                                if (ent[o] >= 0 && sp < P - 1) xload(slot + a.oXS + ((size_t)ent[o] * PP + sp) * RT + lr, lo[o][i], hi[o][i]);
                            }
                        bool ok = true;
#pragma unroll
                        for (int o = 0; o < HP4M_EW; ++o) {
                            cplx sacc = cmake(0.0, 0.0);
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
                    HPM_TICK(4);
#pragma unroll
                    for (int o = 0; o < HP4M_EW; ++o) {
#pragma unroll
                        for (int of = RT; of < 32; of <<= 1) {
                            val[o].x += __shfl_xor_sync(0xffffffffu, val[o].x, of);
                            val[o].y += __shfl_xor_sync(0xffffffffu, val[o].y, of);
                        }
                    }
#pragma unroll
                    for (int o = 0; o < HP4M_EW; ++o) {
                        const int tt = tb + cw + HP4_CW * o;
                        if (tt < nxg_own)
                            for (int d = lsub; d < K; d += SPL)
                                st_async_cplx(mapa_u32(smem_u32(x3 + ((size_t)par * RT + lr) * b3 + NXG * k + tt), d), val[o],
                                              mapa_u32(smem_u32(&barX[par]), d));
                    }
                }
                HPM_TICK(5);
            }
        }
        if (any_sep && nsteps > 0 && is_sep) {
            const int itl = nsteps - 1;
            mbar_wait4(&barX[itl & 1], (itl >> 1) & 1, abort_flag, dead);
            sep_output(m0 + itl * step, x3[((size_t)(itl & 1) * RT + rr) * b3 + b2 - 1]);
        }
        if (DBG && tid == 0)
            for (int i = 0; i < 8; ++i) a.dbg[(size_t)g * 16 + i] = tacc[i];
    } else if (tid < HP4_CRIT + HP4_PROD) {
        // =====================================================================================================
        // producer warp: every TMA copy of the sweep (identical to hp_sweep4.cu)
        // =====================================================================================================
        if (lane == 0) {
            const unsigned int n_bytes = (unsigned int)((size_t)b * NRQ * sizeof(cplx)), r_bytes = (unsigned int)((size_t)b * b3 * sizeof(cplx));
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
                    if (nrq_own > 0) ring_fill4(ringN + (size_t)(it & 1) * pl.n_st, n_base + so * strip_stride, n_bytes, &barN[it & 1]);
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
    } else if (tid >= HP4_CRIT + HP4_PROD + HP4_OFF) {
        // =====================================================================================================
        // poll warp: the gf partials of leaf l+1 for strip it ([K][b][RT] self-validating words in L2)
        // =====================================================================================================
        if (has_sep) {
            const int nw = K * b * RT;
            for (int it = 0; it < nsteps; ++it) {
                const int par = it & 1;
                const cplx* src = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride + a.oGP + (size_t)(l + 1) * nw;
                if (it >= 2) mbar_wait4(&eGF[par], ((it >> 1) - 1) & 1, abort_flag, dead);
                for (int w0 = 0; w0 < nw; w0 += 32 * HP4M_PW) {
                    unsigned long long lo[HP4M_PW], hi[HP4M_PW];
                    unsigned int spins = 0;
                    for (;;) {
                        bool ok = true;
#pragma unroll
                        for (int uu = 0; uu < HP4M_PW; ++uu) {
                            const int wd = w0 + lane + 32 * uu;
                            lo[uu] = hi[uu] = 0ull;
                            if (wd < nw) xload(src + wd, lo[uu], hi[uu]);
                        }
#pragma unroll
                        for (int uu = 0; uu < HP4M_PW; ++uu) ok = ok && xvalid(lo[uu], hi[uu]);
                        if (__all_sync(0xffffffffu, ok || *dead)) break;
                        if (++spins > HP_SPIN_LIMIT) { hp_raise_abort(abort_flag); *dead = 1u; }
                        if ((spins & 0xFFF) == 0 && *((volatile unsigned int*)abort_flag)) *dead = 1u;
                    }
#pragma unroll
                    for (int uu = 0; uu < HP4M_PW; ++uu) {
                        const int wd = w0 + lane + 32 * uu;
                        if (wd < nw)
                            gfp[(size_t)par * nw + wd] = cmake(__longlong_as_double((long long)lo[uu]), __longlong_as_double((long long)hi[uu]));
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive_rel4(&barGF[par]);
            }
        }
    } else {
        // =====================================================================================================
        // off-path group: thread -> (column oc = ot/8, right-hand side rr = (ot%8) % RT, split ks = (ot%8) / RT)
        // =====================================================================================================
        const int ot = tid - HP4_CRIT - HP4_PROD, ow = ot >> 5;
        const int cpart = ot & 7, oc = ot >> 3;
        const int rr = cpart % RT, ks = cpart / RT;
        const bool col = oc < ncols, colw = col && ks == 0;
        const bool col_io = col && a.um[rr] != nullptr;      // field accesses of an empty slot are skipped (reads give 0)
        const int c = c0 + oc;
        cplx* const u = a.um[rr];
        const cplx cis1 = col ? a.is1t[2 * (c + 1)] : cmake(0.0, 0.0);
        cplx vbr = cmake(0.0, 0.0), y0prev = cmake(0.0, 0.0), coefc = cmake(0.0, 0.0), ubase = cmake(0.0, 0.0),
             ubase_prev = cmake(0.0, 0.0);
        if (col) {
            if (!col_io) {
            } else if (a_mode == 0) vbr = ldcg(u + (size_t)(m0 - 1) * n + c);
            else {
                ubase = ldcg(u + (size_t)(m0 - 1) * n + c);
                vbr = ubase;
                if (m0 < n) vbr = cfma(cscale(sg, cmul(hp_rowfac(a, m0), cis1)), ldcg(u + (size_t)m0 * n + c), vbr);
            }
            if (colw) vb[(size_t)rr * CW + oc] = vbr;
        }
        bar_off4();
        // leaf product: RC/8 rows per warp, LPR >= 8 lanes per row
        const int RW = RC >> 3, LPR = 32 / RW;
        const int wr_r = ow * RW + lane / LPR, wr_cp = lane % LPR;
        const int gpart = ot & 7, gkap_lo = ot >> 3;

        for (int it = 0; it <= nsteps; ++it) {
            const int m = m0 + it * step, mn = m + step, mp = m - step;
            const bool live = it < nsteps, more = it + 1 < nsteps;
            const int par = it & 1, ph = (it >> 1) & 1;
            cplx* slot = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride;
            cplx* slot_arm = a.xch + (size_t)((it + 2) & (HP_RING - 1)) * a.slot_stride;
            const cplx* Gp = reinterpret_cast<const cplx*>(ringG + (size_t)(it % 3) * pl.g_st);
            const cplx* Gprev = reinterpret_cast<const cplx*>(ringG + (size_t)((it + 2) % 3) * pl.g_st);
            const cplx rf_it = hp_rowfac(a, a_mode == 1 ? mn : m);
            cplx unx = cmake(0.0, 0.0);
            if (col_io && live) {
                if (a_mode == 0) unx = ldcg(u + (size_t)m * n + c);
                else if (more) unx = ldcg(u + (size_t)(mn - 1) * n + c);
            }
            if (DBG && ot == 0) tprev = clock64();
            // ---- a: gb(t) = Gc(t) vb(t) for all right-hand sides: gf -> cluster l-1 (L2), gl -> every CTA of the cluster
            if (live) {
                mbar_wait4(&barG[it % 3], (it / 3) & 1, abort_flag, dead);
                HPM_TICK(0);
                if (any_sep) {
                    for (int kap0 = 0; kap0 < b2; kap0 += HP4_OFF / 8) {
                        const int kap = kap0 + gkap_lo;
                        cplx acc[RT];
#pragma unroll
                        for (int i = 0; i < RT; ++i) acc[i] = cmake(0.0, 0.0);
                        if (kap < b2) {
                            const cplx* gr = Gp + (size_t)kap * CW;
                            for (int cc = gpart; cc < ncols; cc += 8) {
                                const cplx gv = gr[cc];
#pragma unroll
                                for (int i = 0; i < RT; ++i) acc[i] = cfma(gv, vb[(size_t)i * CW + cc], acc[i]);
                            }
                        }
                        const cplx tot = group8_reduce_scatter<RT>(acc, gpart);     // right-hand side gpart % RT
                        if (kap < b) {
                            if (l > 0 && gpart < RT) {
                                const size_t o = a.oGP + (((size_t)l * K + k) * b + kap) * RT + gpart;
                                xput(slot + o, tot);
                                xarm(slot_arm + o);
                            }
                        } else if (kap < b2 && has_sep) {
                            for (int d = gpart / RT; d < K; d += KS)
                                st_async_cplx(mapa_u32(smem_u32(glp + (((size_t)par * K + k) * b + (kap - b)) * RT + (gpart % RT)), d), tot,
                                              mapa_u32(smem_u32(&barGL[par]), d));
                        }
                    }
                }
            }
            HPM_TICK(1);
            // ---- b: x3(t-1) arrives: finish strip t-1 on the own columns, input of strip t
            cplx v = vbr;
            if (it > 0) {
                cplx corr = cmake(0.0, 0.0);
                if (any_sep) {
                    mbar_wait4(&barX[par ^ 1], ((it - 1) >> 1) & 1, abort_flag, dead);
                    HPM_TICK(2);
                    const cplx* xa = x3 + ((size_t)(par ^ 1) * RT + rr) * b3;
                    cplx c1 = cmake(0.0, 0.0);
                    if (col) {
                        int kap = ks;
                        for (; kap + KS < b2; kap += 2 * KS) {
                            corr = cfma(Gprev[(size_t)kap * CW + oc], xa[kap], corr);
                            c1 = cfma(Gprev[(size_t)(kap + KS) * CW + oc], xa[kap + KS], c1);
                        }
                        if (kap < b2) corr = cfma(Gprev[(size_t)kap * CW + oc], xa[kap], corr);
                        corr = cadd(corr, c1);
                    }
#pragma unroll
                    for (int o = RT; o < 8; o <<= 1) {
                        corr.x += __shfl_xor_sync(0xffffffffu, corr.x, o);
                        corr.y += __shfl_xor_sync(0xffffffffu, corr.y, o);
                    }
                }
                if (col) v = cfma(coefc, corr, vbr);
                if (col && live)
                    for (int d = ks; d < K; d += KS)
                        st_async_cplx(mapa_u32(smem_u32(v_leaf + ((size_t)par * RT + rr) * QP + lc0 + oc), d), v, mapa_u32(smem_u32(&barV[par]), d));
                if (colw && col_io) {
                    if (a_mode == 0) u[(size_t)mp * n + c] = v;
                    else {
                        cplx un = a_diag == 0 ? cadd(csub(ubase_prev, y0prev), corr) : csub(y0prev, corr);
                        u[(size_t)(mp - 1) * n + c] = un;
                    }
                }
            } else if (col && live) {
                for (int d = ks; d < K; d += KS)
                    st_async_cplx(mapa_u32(smem_u32(v_leaf + ((size_t)par * RT + rr) * QP + lc0 + oc), d), v, mapa_u32(smem_u32(&barV[par]), d));
            }
            if (it > 0) {
                __syncwarp();
                if (lane == 0) mbar_arrive_local(&eG[(it + 2) % 3]);
            }
            if (!live) break;
            HPM_TICK(3);
            // ---- c: leaf product Y0(t) = W(t) V_leaf(t): a W element is loaded once and feeds RT accumulators
            mbar_wait4(&barV[par], ph, abort_flag, dead);
            HPM_TICK(4);
            const cplx* vl = v_leaf + (size_t)par * RT * QP;
            for (int ch = 0; ch < NCH; ++ch) {
                const int cidx = it * NCH + ch, sl = cidx % S, r0 = ch * RC;
                long long tw0 = 0;
                if (DBG && ot == 0) tw0 = clock64();
                mbar_wait4(&barW[sl], (cidx / S) & 1, abort_flag, dead);
                if (DBG && ot == 0) tacc[7] += clock64() - tw0;
                const cplx* Wc = reinterpret_cast<const cplx*>(ringW + (size_t)sl * pl.w_st);
                cplx acc[RT];
#pragma unroll
                for (int i = 0; i < RT; ++i) acc[i] = cmake(0.0, 0.0);
                if (r0 + wr_r < ncols) {
                    const cplx* wr = Wc + (size_t)wr_r * QP;
                    if (RT == 1) {
                        cplx a1 = cmake(0.0, 0.0), a2 = cmake(0.0, 0.0), a3 = cmake(0.0, 0.0);
                        int cq = wr_cp;
                        for (; cq + 3 * LPR < q; cq += 4 * LPR) {
                            acc[0] = cfma(wr[cq], vl[cq], acc[0]);
                            a1 = cfma(wr[cq + LPR], vl[cq + LPR], a1);
                            a2 = cfma(wr[cq + 2 * LPR], vl[cq + 2 * LPR], a2);
                            a3 = cfma(wr[cq + 3 * LPR], vl[cq + 3 * LPR], a3);
                        }
                        for (; cq < q; cq += LPR) acc[0] = cfma(wr[cq], vl[cq], acc[0]);
                        acc[0] = cadd(cadd(acc[0], a1), cadd(a2, a3));
                    } else {
                        for (int cq = wr_cp; cq < q; cq += LPR) {
                            const cplx wv = wr[cq];
#pragma unroll
                            for (int i = 0; i < RT; ++i) acc[i] = cfma(wv, vl[(size_t)i * QP + cq], acc[i]);
                        }
                    }
                }
                for (int o = LPR >> 1; o >= 8; o >>= 1) {
#pragma unroll
                    for (int i = 0; i < RT; ++i) {
                        acc[i].x += __shfl_xor_sync(0xffffffffu, acc[i].x, o);
                        acc[i].y += __shfl_xor_sync(0xffffffffu, acc[i].y, o);
                    }
                }
                const cplx tot = group8_reduce_scatter<RT>(acc, wr_cp & 7);
                if (wr_cp < RT && r0 + wr_r < ncols) y0s[(size_t)wr_cp * CW + r0 + wr_r] = tot;
                __syncwarp();
                if (lane == 0) mbar_arrive_local(&eW[sl]);
            }
            bar_off4();                                      // y0s complete
            HPM_TICK(5);
            if (ot == 0 && it + 2 < nsteps) mbar_expect_tx(&barV[par], v_bytes);
            if (col) {
                cplx y0 = y0s[(size_t)rr * CW + oc];
                y0prev = y0;
                if (a_mode == 0) {
                    coefc = cmul(rf_it, cis1);
                    vbr = cfms(coefc, y0, unx);
                } else {
                    coefc = cmul(rf_it, cis1);
                    vbr = a_diag == 0 ? cfma(coefc, csub(ubase, y0), unx) : cfms(coefc, y0, unx);
                    ubase_prev = ubase;
                    ubase = unx;
                }
                if (colw) vb[(size_t)rr * CW + oc] = vbr;
            }
            bar_off4();                                      // vb ready, y0s free for the next strip
            HPM_TICK(6);
        }
        if (DBG && ot == 0)
            for (int i = 0; i < 8; ++i) a.dbg[(size_t)g * 16 + 8 + i] = tacc[i];
    }
    __syncthreads();
    cluster_sync_all();
}

// ------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------
template <int MODE, int BT, int KT, int RT>
static const void* hp4m_fn(bool dbg) {
    return dbg ? (const void*)hp_sweep4m_kernel<MODE, true, BT, KT, RT> : (const void*)hp_sweep4m_kernel<MODE, false, BT, KT, RT>;
}
template <int BT, int KT, int RT>
static const void* hp4m_mode(int mode, bool dbg) {
    return mode == 0 ? hp4m_fn<0, BT, KT, RT>(dbg) : (mode == 1 ? hp4m_fn<1, BT, KT, RT>(dbg) : hp4m_fn<2, BT, KT, RT>(dbg));
}
template <int BT, int KT>
static const void* hp4m_rt(int RT, int mode, bool dbg) {
    switch (RT) {
        case 1: return hp4m_mode<BT, KT, 1>(mode, dbg);
        case 2: return hp4m_mode<BT, KT, 2>(mode, dbg);
        case 4: return hp4m_mode<BT, KT, 4>(mode, dbg);
        case 8: return hp4m_mode<BT, KT, 8>(mode, dbg);
    }
    return nullptr;
}
static const void* hp4m_select(int RT, int mode, bool dbg, int b, int K) {
    return (b == 12 && K == 4) ? hp4m_rt<12, 4>(RT, mode, dbg) : hp4m_rt<0, 0>(RT, mode, dbg);
}

// can the layout of this solver run RT right-hand sides per launch?  (0 = yes)
int hp_sweep4m_supported(hp_solver* s, int RT) {
    const HpLayout& L = s->lay;
    if (!L.colN || (RT != 1 && RT != 2 && RT != 4 && RT != 8) || RT > HP_RMAX) return 1;
    if (L.CW > HP4_OFF / 8 || L.P - 1 > 32 || L.K < 1 || L.K > 8 || s->b > HP_BMAX) return 1;
    if (s->multi_ok[RT] != 0) return s->multi_ok[RT] > 0 ? 0 : 1;
    int dev = 0, max_smem = 0, ncl = 0;
    s->multi_ok[RT] = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return 1;
    if (cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 1;
    Hp4Plan pl;
    if (hp_sweep4_plan(L, s->b, (size_t)max_smem, pl, RT)) return 1;
    if (32 / (pl.RC >> 3) < 8) return 1;                      // the leaf product needs at least 8 lanes per row
    const void* fn = hp4m_select(RT, 0, false, s->b, L.K);
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total) != cudaSuccess) { cudaGetLastError(); return 1; }
    if (cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) cudaGetLastError();
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.K * 64); cfg.blockDim = dim3(HP4_THREADS); cfg.dynamicSmemBytes = pl.total;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = L.K; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaOccupancyMaxActiveClusters(&ncl, fn, &cfg) != cudaSuccess) { cudaGetLastError(); return 1; }
    if (ncl < L.P) return 1;
    s->multi_ok[RT] = 1;
    return 0;
}

int hp_sweep4m_launch(hp_solver* s, HpSweepArgs& a, int RT, cudaStream_t st) {
    const HpLayout& L = s->lay;
    int dev = 0, max_smem = 0;
    HP_CUDA(cudaGetDevice(&dev));
    HP_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    Hp4Plan pl;
    if (hp_sweep4_plan(L, s->b, (size_t)max_smem, pl, RT)) { hp_set_error("sweep: the multi-vector cluster kernel does not fit this partition"); return 1; }
    const int mode = a.mode == 0 ? 0 : (a.diag_mode == 0 ? 1 : 2);
    const void* fn = hp4m_select(RT, mode, a.dbg != nullptr, s->b, L.K);
    if (!fn) { hp_set_error("sweep: %d right-hand sides per launch are not supported", RT); return 1; }
    HP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.total));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(L.G); cfg.blockDim = dim3(HP4_THREADS); cfg.dynamicSmemBytes = pl.total; cfg.stream = st;
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
        hp_set_error("sweep: %s cluster launch of %d CTAs (%d right-hand sides) failed: %s", cfg.numAttrs == 2 ? "cooperative" : "plain", L.G, RT,
                     cudaGetErrorString(e));
        return 2;
    }
    return 0;
}
