// The sweeps of algo2_4 (/root/reference/code.py:366-380): a chain of strip solves y = T_m v, each of which
// depends on the previous one.  One persistent cooperative kernel walks the whole chain; per strip every
// CTA streams its packet (csrc/hp_internal.cuh) once.
//
//   S1  g   = Gp v_own                      (2b numbers per CTA)         -> exchange: V (own columns), GP
//       the first CTA of a leaf sums the K partial g in fixed order       -> exchange: GR   (deterministic)
//   S2  y0  = Wp v_leaf                     (own rows of the leaf product; v_leaf <- exchange V)
//       rho = e_b v_s - GR                  (separator right-hand sides;   <- exchange GR, VS)
//       x_S(own rows) = Np rho              (dense separator inverse)     -> exchange: XS
//   S3  y   = y0 - Gf^T x_left - Gl^T x_right  (<- exchange XS), separator columns y_s = x_s[b-1]
//       epilogue: forward   u_{m+1} -= A_{m+1,m} y                           (code.py:370)
//                 backward  u_m <- u_m - y   (reference, :372-380 fused by linearity)  or  u_m <- y (paper)
//       and the input of the next strip is formed in place (S3 runs straight into the next S1).
//
// There is no grid barrier.  CTAs exchange the few numbers that cross them through a ring of four L2-resident
// slots (slot = strip counter mod 4) in which every 8-byte word validates itself: the ring is filled with
// 0xFF bytes (a NaN no arithmetic produces), producers overwrite it with data, consumers spin on the data word
// itself until it differs from the sentinel - one L2 round trip per hand-over, no fences, no atomics.  A
// producer re-arms its words two strips after writing them; by then every consumer has moved on, because a
// CTA cannot finish strip t+1 before all CTAs have finished strip t (S2 needs GR from every leaf).
//
// Packets are independent of the data, so they are fetched ahead of the dependency chain: the TMA variant
// double-buffers whole packets in shared memory with cp.async.bulk + mbarrier (issued one strip ahead, with an
// L2 prefetch two strips ahead); the direct variant (packets too large for two shared-memory stages) reads
// them from global memory behind an L2 prefetch.
#include "hp_sweep_common.cuh"
#include "hp_sweep4.h"

#include <algorithm>

#ifndef HP_SWEEP_THREADS
#define HP_SWEEP_THREADS 256
#endif

template <bool TMA>
__global__ void __launch_bounds__(HP_SWEEP_THREADS) hp_sweep_kernel(HpSweepArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int b = a.b, n = a.n, K = a.lay.K, P = a.lay.P, G = a.lay.G, QP = a.lay.QP, CW = a.lay.CW;
    const int NS = a.lay.NS, NSP = a.lay.NSP, NR = a.lay.NR;
    const int g = blockIdx.x, l = g / K, k = g % K;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = HP_SWEEP_THREADS / 32;
    const int q = a.leaf_q[l], ls = a.leaf_start[l];
    const int lc0 = (q * k) / K, lc1 = (q * (k + 1)) / K, ncols = lc1 - lc0, c0 = ls + lc0;
    const int row0 = g * NR, nrows = max(0, min(NR, NS - row0));
    const unsigned int pk_bytes = (unsigned int)(a.lay.PK * sizeof(cplx));
    const size_t stage_bytes = ((size_t)pk_bytes + 127) & ~(size_t)127;
    unsigned int* abort_flag = a.bar + 1;

    cplx* small = reinterpret_cast<cplx*>(smem_raw + (TMA ? 2 * stage_bytes : 0));
    cplx* v_own = small;                // [CW]
    cplx* v_leaf = v_own + CW;          // [QP]
    cplx* rho = v_leaf + QP;            // [NSP]
    cplx* xlr = rho + NSP;              // [2b]  x_left, x_right
    cplx* xrow = xlr + 2 * b;           // [NR+1] own rows of x_S
    cplx* gpw = xrow + NR + 1;          // [8][2b]  per-warp partial g
    cplx* nred = gpw + (size_t)nwarps * 2 * b;      // [8][4]   per-warp partial separator rows
    cplx* y0w = nred + nwarps * 4;      // [8][CW]  per-warp partial leaf products
    cplx* ypart = y0w + (size_t)nwarps * CW;         // [8][CW]  per-warp partial corrections
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(ypart + (size_t)nwarps * CW);   // [2]

    __shared__ unsigned int s_abort;
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = 0;
#define HP_TICK(i) do { if (a.dbg && tid == 0) { long long t_ = clock64(); tacc[i] += t_ - tprev; tprev = t_; } } while (0)
    const int step = a.mode == 1 ? -1 : 1;
    const int nsteps = a.mode == 2 ? 1 : (a.mode == 0 ? a.m_to - a.m_from + 1 : a.m_from - a.m_to + 1);
    const cplx sgn = cmake(a.diag_mode == 0 ? 1.0 : -1.0, 0.0);
    int m = a.m_from;
    const cplx* pk_base = a.packets + (size_t)g * a.lay.PK;
    const size_t strip_stride = (size_t)G * a.lay.PK;

    if (TMA) {
        if (tid == 0) {
            mbar_init(&mbar[0], 1);
            mbar_init(&mbar[1], 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            asm volatile("fence.proxy.async;" ::: "memory");
        }
        __syncthreads();
        if (tid == 0) {
            // strip 0 -> stage 0, strip 1 -> stage 1, strip 2 -> L2
            for (int sidx = 0; sidx < 2 && sidx < nsteps; ++sidx) {
                const char* src = (const char*)(pk_base + (size_t)(m + sidx * step - a.m_lo) * strip_stride);
                char* dst = (char*)smem_raw + sidx * stage_bytes;
                mbar_expect_tx(&mbar[sidx], pk_bytes);
                for (unsigned int o = 0; o < pk_bytes; o += HP_BULK_CHUNK)
                    bulk_g2s(dst + o, src + o, min(HP_BULK_CHUNK, pk_bytes - o), &mbar[sidx]);
            }
            if (nsteps > 2) {
                const char* src = (const char*)(pk_base + (size_t)(m + 2 * step - a.m_lo) * strip_stride);
                for (unsigned int o = 0; o < pk_bytes; o += HP_BULK_CHUNK) bulk_prefetch_l2(src + o, min(HP_BULK_CHUNK, pk_bytes - o));
            }
        }
    }

    // the separator column this thread owns (the CTA that computes row (j, b-1) of x_S updates column sep[j])
    int sep_j = -1, sep_col = -1;
    if (tid < nrows) {
        int row = row0 + tid;
        int j = row / b;
        if (row - j * b == b - 1) { sep_j = j; sep_col = a.sep[j]; }
    }
    const cplx cis1 = tid < ncols ? a.is1t[2 * (c0 + tid + 1)] : cmake(0.0, 0.0);       // 1/s1 of the own column
    const cplx cis1s = sep_col >= 0 ? a.is1t[2 * (sep_col + 1)] : cmake(0.0, 0.0);      // ... of the own separator column
    // rho entry of this thread (entries beyond the first HP_SWEEP_THREADS are indexed in the loop)
    const int rho_j = tid < NS ? tid / b : 0, rho_kap = tid < NS ? tid - (tid / b) * b : 0;
    // input of the first strip; ubase = the u value the epilogue of this strip combines with y
    cplx ubase = cmake(0.0, 0.0), usbase = cmake(0.0, 0.0);
    if (tid < ncols) {
        int c = c0 + tid;
        cplx v;
        if (a.mode == 2) v = a.vin[c];
        else if (a.mode == 0) { v = ldcg(a.u + (size_t)(m - 1) * n + c); }
        else {
            ubase = ldcg(a.u + (size_t)(m - 1) * n + c);
            v = ubase;
            if (m < n) {
                cplx cp = cmul(cmul(hp_rowfac(a, m), cis1), sgn);
                v = cfma(cp, ldcg(a.u + (size_t)m * n + c), v);
            }
        }
        v_own[tid] = v;
    }
    if (sep_col >= 0) {
        cplx v;
        if (a.mode == 2) v = a.vin[sep_col];
        else if (a.mode == 0) v = ldcg(a.u + (size_t)(m - 1) * n + sep_col);
        else {
            usbase = ldcg(a.u + (size_t)(m - 1) * n + sep_col);
            v = usbase;
            if (m < n) {
                cplx cp = cmul(cmul(hp_rowfac(a, m), cis1s), sgn);
                v = cfma(cp, ldcg(a.u + (size_t)m * n + sep_col), v);
            }
        }
        xput(a.xch + a.oVS + sep_j, v);                 // slot 0
    }
    __syncthreads();

    for (int it = 0; it < nsteps; ++it, m += step) {
        const int mn = m + step;               // next strip
        const bool more = it + 1 < nsteps;
        cplx* slot = a.xch + (size_t)(it & (HP_RING - 1)) * a.slot_stride;
        cplx* slot_next = a.xch + (size_t)((it + 1) & (HP_RING - 1)) * a.slot_stride;
        cplx* slot_arm = a.xch + (size_t)((it + 2) & (HP_RING - 1)) * a.slot_stride;
        const cplx* pk;
        if (TMA) {
            pk = reinterpret_cast<const cplx*>(smem_raw + (it & 1) * stage_bytes);
        } else {
            pk = pk_base + (size_t)(m - a.m_lo) * strip_stride;
            if (more) {   // pull the next strip's packet towards L2 while this one is processed
                const char* nx = (const char*)(pk_base + (size_t)(mn - a.m_lo) * strip_stride);
                for (size_t o = (size_t)tid * 128; o < pk_bytes; o += (size_t)HP_SWEEP_THREADS * 128)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + o));
            }
        }
        const cplx* Wp = pk;
        const cplx* Gp = pk + a.lay.offG;
        const cplx* Np = pk + a.lay.offN;
        // coupling between grid rows for this strip's epilogue (forward: rows m, m+1; backward: next strip's pair)
        const cplx rfac = hp_rowfac(a, a.mode == 1 ? mn : m);
        // early loads of the u values the epilogue needs (written by no other CTA)
        cplx upre = cmake(0.0, 0.0), usep = cmake(0.0, 0.0);
        if (tid < ncols) {
            int c = c0 + tid;
            if (a.mode == 0) upre = ldcg(a.u + (size_t)m * n + c);
            else if (a.mode == 1 && more) upre = ldcg(a.u + (size_t)(mn - 1) * n + c);
        }
        if (sep_col >= 0) {
            if (a.mode == 0) usep = ldcg(a.u + (size_t)m * n + sep_col);
            else if (a.mode == 1 && more) usep = ldcg(a.u + (size_t)(mn - 1) * n + sep_col);
        }
        if (a.dbg && tid == 0) tprev = clock64();
        if (TMA) mbar_wait(&mbar[it & 1], (it >> 1) & 1);
        HP_TICK(0);
        // ---- S1: publish own columns; g = Gp v_own with lanes over the 2b interface components (rows of Gp,
        //      odd row stride -> conflict-free) and warps over column subsets (v_own is a broadcast read)
        if (K > 1 && tid < ncols) xput(slot + c0 + tid, v_own[tid]);
        for (int kap = lane; kap < 2 * b; kap += 32) {
            cplx acc = cmake(0.0, 0.0);
            const cplx* gr = Gp + (size_t)kap * CW;
            for (int cc = warp; cc < ncols; cc += nwarps) acc = cfma(gr[cc], v_own[cc], acc);
            gpw[warp * 2 * b + kap] = acc;
        }
        __syncthreads();
        if (tid < 2 * b) {
            cplx acc = gpw[tid];
#pragma unroll
            for (int w = 1; w < HP_SWEEP_THREADS / 32; ++w) acc = cadd(acc, gpw[w * 2 * b + tid]);
            if (K == 1) xput(slot + a.oGR + (size_t)l * 2 * b + tid, acc);
            else if (k > 0) xput(slot + a.oGP + (size_t)g * 2 * b + tid, acc);
            else gpw[tid] = acc;          // the leaf's first CTA adds the other parts below (same thread)
        }
        // re-arm what this CTA wrote two strips ago (slot it+2 = it-2 mod 4)
        if (K > 1 && tid < ncols) xarm(slot_arm + c0 + tid);
        if (tid < 2 * b) {
            if (K > 1 && k > 0) xarm(slot_arm + a.oGP + (size_t)g * 2 * b + tid);
            if (k == 0) xarm(slot_arm + a.oGR + (size_t)l * 2 * b + tid);
        }
        if (tid < nrows) xarm(slot_arm + a.oXS + row0 + tid);
        if (sep_col >= 0) xarm(slot_arm + a.oVS + sep_j);
        HP_TICK(1);
        if (K > 1 && k == 0 && tid < 2 * b) {
            cplx acc = gpw[tid];
            for (int kk = 1; kk < K; ++kk) acc = cadd(acc, xget(slot + a.oGP + (size_t)(g + kk) * 2 * b + tid, abort_flag));
            xput(slot + a.oGR + (size_t)l * 2 * b + tid, acc);
        }
        HP_TICK(2);
        // ---- S2
        for (int c = tid; c < q; c += HP_SWEEP_THREADS)
            v_leaf[c] = (c >= lc0 && c < lc1) ? v_own[c - lc0] : xget(slot + ls + c, abort_flag);
        if (nrows > 0) {
            for (int e = tid; e < NS; e += HP_SWEEP_THREADS) {
                int j = rho_j, kap = rho_kap;
                if (e != tid) { j = e / b; kap = e - j * b; }
                const cplx* pa = slot + a.oGR + ((size_t)j * 2 + 1) * b + kap;          // Gl of leaf j
                const cplx* pc = slot + a.oGR + ((size_t)(j + 1) * 2) * b + kap;        // Gf of leaf j+1
                const cplx* pv = slot + a.oVS + j;
                const bool need_v = kap == b - 1;
                cplx va, vc, vs = cmake(0.0, 0.0);
                unsigned int spins = 0;
                for (;;) {
                    bool ok = xtry(pa, va);
                    ok = xtry(pc, vc) && ok;
                    if (need_v) ok = xtry(pv, vs) && ok;
                    if (ok) break;
                    if (++spins > HP_SPIN_LIMIT) { hp_raise_abort(abort_flag); break; }
                    if ((spins & 0xFFF) == 0 && *((volatile unsigned int*)abort_flag)) break;
                }
                rho[e] = csub(vs, cadd(va, vc));
            }
        }
        __syncthreads();
        HP_TICK(3);
        // separator rows first (they are on the critical path): threads over the columns of N, 4 rows at a time
        for (int r0 = 0; r0 < nrows; r0 += 4) {
            cplx acc[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = cmake(0.0, 0.0);
            for (int e = tid; e < NS; e += HP_SWEEP_THREADS) {
                cplx r = rho[e];
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (r0 + i < nrows) acc[i] = cfma(Np[(size_t)(r0 + i) * NSP + e], r, acc[i]);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = hp_warp_sum2(acc[i]);
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < 4; ++i) nred[warp * 4 + i] = acc[i];
            }
            __syncthreads();
            if (tid < 4 && r0 + tid < nrows) {
                cplx t = nred[tid];
#pragma unroll
                for (int w = 1; w < HP_SWEEP_THREADS / 32; ++w) t = cadd(t, nred[w * 4 + tid]);
                xput(slot + a.oXS + row0 + r0 + tid, t);
                xrow[r0 + tid] = t;
            }
            if (r0 + 4 < nrows) __syncthreads();
        }
        // leaf product: lanes over the rows of Wp (odd row stride -> conflict-free), warps over column subsets
        for (int cc = lane; cc < ncols; cc += 32) {
            cplx acc = cmake(0.0, 0.0), acc2 = cmake(0.0, 0.0);
            const cplx* wr = Wp + (size_t)cc * QP;
            int c = warp;
            for (; c + nwarps < q; c += 2 * nwarps) { acc = cfma(wr[c], v_leaf[c], acc); acc2 = cfma(wr[c + nwarps], v_leaf[c + nwarps], acc2); }
            if (c < q) acc = cfma(wr[c], v_leaf[c], acc);
            y0w[(size_t)warp * CW + cc] = cadd(acc, acc2);
        }
        HP_TICK(4);
        // ---- S3
        if (tid < 2 * b) {
            int side = tid / b, kap = tid - side * b;
            int j = l - 1 + side;
            xlr[tid] = (j >= 0 && j < P - 1) ? xget(slot + a.oXS + (size_t)j * b + kap, abort_flag) : cmake(0.0, 0.0);
        }
        __syncthreads();
        HP_TICK(5);
        // correction: warp w takes the interface components kap = w, w+8, ...; lanes run over the columns
        for (int cc = lane; cc < ncols; cc += 32) {
            cplx acc = cmake(0.0, 0.0);
            for (int kap = warp; kap < 2 * b; kap += nwarps) acc = cfma(Gp[(size_t)kap * CW + cc], xlr[kap], acc);
            ypart[(size_t)warp * CW + cc] = acc;
        }
        __syncthreads();
        if (tid < ncols) {
            int c = c0 + tid;
            cplx y = cmake(0.0, 0.0);
#pragma unroll
            for (int w = 0; w < HP_SWEEP_THREADS / 32; ++w) y = cadd(y, csub(y0w[(size_t)w * CW + tid], ypart[(size_t)w * CW + tid]));
            if (a.mode == 2) {
                a.yout[c] = y;
            } else if (a.mode == 0) {
                // u_{m+1} -= c3(row m+1) y ; the result is the input of strip m+1
                cplx cp = cmul(rfac, cis1);
                cplx un = cfms(cp, y, upre);
                a.u[(size_t)m * n + c] = un;
                v_own[tid] = un;
            } else {
                cplx un = a.diag_mode == 0 ? csub(ubase, y) : y;
                a.u[(size_t)(m - 1) * n + c] = un;
                if (more) {
                    // input of strip m-1: u_{m-1} (+/-) c4(row m-1) u_m
                    cplx cp = cmul(cmul(rfac, cis1), sgn);
                    ubase = upre;
                    v_own[tid] = cfma(cp, un, upre);
                }
            }
        }
        // separator columns: y_s = x_s[b-1]; the input value of the next strip goes to the next slot
        if (sep_col >= 0) {
            cplx y = xrow[tid];
            if (a.mode == 2) a.yout[sep_col] = y;
            else if (a.mode == 0) {
                cplx cp = cmul(rfac, cis1s);
                cplx un = cfms(cp, y, usep);
                a.u[(size_t)m * n + sep_col] = un;
                if (more) xput(slot_next + a.oVS + sep_j, un);
            } else {
                cplx un = a.diag_mode == 0 ? csub(usbase, y) : y;
                a.u[(size_t)(m - 1) * n + sep_col] = un;
                if (more) {
                    cplx cp = cmul(cmul(rfac, cis1s), sgn);
                    usbase = usep;
                    xput(slot_next + a.oVS + sep_j, cfma(cp, un, usep));
                }
            }
        }
        __syncthreads();
        HP_TICK(6);
        if (TMA && tid == 0) {
            // every thread is done with this stage: refill it with the packet two strips ahead
            if (it + 2 < nsteps) {
                const char* src = (const char*)(pk_base + (size_t)(m + 2 * step - a.m_lo) * strip_stride);
                char* dst = (char*)smem_raw + (it & 1) * stage_bytes;
                mbar_expect_tx(&mbar[it & 1], pk_bytes);
                for (unsigned int o = 0; o < pk_bytes; o += HP_BULK_CHUNK)
                    bulk_g2s(dst + o, src + o, min(HP_BULK_CHUNK, pk_bytes - o), &mbar[it & 1]);
            }
            if (it + 3 < nsteps) {
                const char* src = (const char*)(pk_base + (size_t)(m + 3 * step - a.m_lo) * strip_stride);
                for (unsigned int o = 0; o < pk_bytes; o += HP_BULK_CHUNK) bulk_prefetch_l2(src + o, min(HP_BULK_CHUNK, pk_bytes - o));
            }
        }
        if ((it & 63) == 63) {                 // a runaway spin somewhere: every CTA leaves within 64 strips
            if (tid == 0) s_abort = *((volatile unsigned int*)abort_flag);
            __syncthreads();
            if (s_abort) break;
        }
    }
    if (a.dbg && tid == 0)
        for (int i = 0; i < 8; ++i) a.dbg[(size_t)g * 8 + i] = tacc[i];
}

#define HP2_OFF_COLS 256
size_t hp_sweep2_smem(const HpLayout& L, int b);
int hp_sweep2_launch(hp_solver* s, HpSweepArgs& a, cudaStream_t st);

int hp_sweep_launch(hp_solver* s, int mode, cplx* u, const cplx* vin, cplx* yout, int m_from, int m_to,
                    int diag_mode, cudaStream_t st) {
    if (!s->packets) { hp_set_error("sweep: preconditioner not set up"); return 1; }
    int lo = mode == 1 ? m_to : m_from, hi = mode == 1 ? m_from : m_to;
    if (mode == 2) lo = hi = m_from;
    if (lo > hi) return 0;
    if (lo < s->m_lo || hi > s->m_hi) {
        hp_set_error("sweep: strips %d..%d requested, solver holds %d..%d", lo, hi, s->m_lo, s->m_hi);
        return 1;
    }
    const HpLayout& L = s->lay;
    HpSweepArgs a;
    a.n = s->n; a.b = s->b; a.lay = s->lay;
    a.leaf_start = s->leaf_start; a.leaf_q = s->leaf_q; a.sep = s->sep;
    a.packets = s->packets; a.mleaf = s->mleaf; a.rsep = s->rsep; a.m_lo = s->m_lo;
    a.mode = mode; a.m_from = m_from; a.m_to = m_to; a.diag_mode = diag_mode;
    a.u = u; a.vin = vin; a.yout = yout;
    a.xch = s->xch; a.bar = s->bar;
    a.oGP = (size_t)s->n; a.oGR = a.oGP + (size_t)L.G * 2 * s->b; a.oXS = a.oGR + (size_t)L.P * 2 * s->b;
    a.oVS = a.oXS + L.NSP; a.slot_stride = a.oVS + L.P;
    a.s2t = s->s2t; a.is1t = s->is1t;
    a.ih2 = 1.0 / (s->pml.h * s->pml.h);
    a.dbg = s->dbg;
    const int nw = HP_SWEEP_THREADS / 32;
    size_t small = sizeof(cplx) * ((size_t)(1 + 2 * nw) * L.CW + L.QP + L.NSP + 2 * s->b + L.NR + 1 + (size_t)nw * 2 * s->b + nw * 4) +
                   2 * sizeof(unsigned long long);
    size_t stage = (L.PK * sizeof(cplx) + 127) & ~(size_t)127;
    int max_smem = 0, dev = 0;
    HP_CUDA(cudaGetDevice(&dev));
    HP_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    // variants: classic layout: 1 direct (global loads); 2 staged, block-synchronous phases; 3 pipelined, two hand-overs
    // per strip (csrc/hp_sweep2.cu).  cluster layout: 4 (csrc/hp_sweep4.cu).  0 = automatic.
    int variant = s->sweep_variant;
    if (L.colN) {
        if (variant != 0 && variant != 4) { hp_set_error("sweep: variant %d needs the classic layout (hp_set_layout_mode before setup)", variant); return 1; }
        variant = 4;
        a.oGP = 0; a.oXS = (size_t)L.G * s->b; a.oGR = a.oVS = 0;
        a.slot_stride = a.oXS + (size_t)std::max(L.NS, 1) * (L.P | 1);
    } else {
        if (variant == 4) { hp_set_error("sweep: variant 4 needs the cluster layout (hp_set_layout_mode before setup)"); return 1; }
        bool pipe_ok = L.K <= 16 && L.CW <= HP2_OFF_COLS && 2 * s->b <= 64 && L.NR <= 128 && s->mleaf && hp_sweep2_smem(L, s->b) + 1024 <= (size_t)max_smem;
        bool tma_ok = 2 * stage + small + 1024 <= (size_t)max_smem;
        if (variant == 0) variant = pipe_ok ? 3 : (tma_ok ? 2 : 1);   // measured at 4096^2: 3 (5.9 us/strip) < 2 (7.2)
        if (variant == 3 && !pipe_ok) variant = tma_ok ? 2 : 1;
        if (variant == 2 && !tma_ok) variant = 1;
    }
    // the exchange ring starts all-sentinel (0xFF bytes); bar[1] = abort flag of this launch (a timed-out launch must not
    // stop the next one; its sticky copy bar[2] stays until the next setup)
    HP_CUDA(cudaMemsetAsync(s->xch, 0xFF, sizeof(cplx) * HP_RING * a.slot_stride, st));
    HP_CUDA(cudaMemsetAsync(s->bar + 1, 0, sizeof(unsigned int), st));
    hp_count_launch();
    hp_profile_begin(s, st);
    if (variant == 4) {
        if (hp_sweep4_launch(s, a, st)) return 2;
    } else if (variant == 3) {
        if (hp_sweep2_launch(s, a, st)) return 2;
    } else {
        bool tma = variant == 2;
        size_t smem = small + (tma ? 2 * stage : 0);
        if (smem + 1024 > (size_t)max_smem) { hp_set_error("sweep: %zu bytes of shared memory needed, %d available", smem, max_smem); return 1; }
        const void* fn = tma ? (const void*)hp_sweep_kernel<true> : (const void*)hp_sweep_kernel<false>;
        if (smem > 48 * 1024) HP_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        void* args[] = {&a};
        if (s->coop) HP_CUDA(cudaLaunchCooperativeKernel(fn, dim3(L.G), dim3(HP_SWEEP_THREADS), args, smem, st));
        else HP_CUDA(cudaLaunchKernel(fn, dim3(L.G), dim3(HP_SWEEP_THREADS), args, smem, st));   // contexts: see hp_context_clone
    }
    hp_profile_end(s, st, (int64_t)(hi - lo + 1) * ((int64_t)L.G * L.PK + 3 * (int64_t)s->n + (L.colN ? (int64_t)(L.P - 1) * 3 * s->b * s->b : 0)) *
                              (int64_t)sizeof(cplx));
    return 0;
}

// kernel that one launch carrying R right-hand sides runs with the layout of this solver: 2 = hp_sweep4d (tensor cores,
// R = 8), 1 = hp_sweep4m, 0 = none (the right-hand sides go through the single-vector kernel one by one)
extern "C" int hp_multi_kernel(hp_solver* s, int R) {
    if (!s || !s->packets || R < 1 || R > HP_RMAX) return 0;
    if (R == 8 && !hp_sweep4d_supported(s)) return 2;
    return hp_sweep4m_supported(s, R) ? 0 : 1;
}

int hp_sweep_launch_multi(hp_solver* s, int mode, int R, cplx* const* um, int m_from, int m_to, int diag_mode, cudaStream_t st) {
    if (!s->packets) { hp_set_error("sweep: preconditioner not set up"); return 1; }
    const int kernel = hp_multi_kernel(s, R);
    if (!kernel) { hp_set_error("sweep: %d right-hand sides per launch not supported by this layout", R); return 1; }
    const bool tensor = kernel == 2;
    int first = 0;                                       // null entries are inactive slots (hp_sweep4_dev.cuh: ldcg_slot)
    while (first < R && !um[first]) ++first;
    if (first == R) { hp_set_error("sweep: all %d right-hand-side slots of the launch are empty", R); return 1; }
    int lo = mode == 1 ? m_to : m_from, hi = mode == 1 ? m_from : m_to;
    if (lo > hi) return 0;
    if (lo < s->m_lo || hi > s->m_hi) {
        hp_set_error("sweep: strips %d..%d requested, solver holds %d..%d", lo, hi, s->m_lo, s->m_hi);
        return 1;
    }
    const HpLayout& L = s->lay;
    HpSweepArgs a;
    a.n = s->n; a.b = s->b; a.lay = s->lay;
    a.leaf_start = s->leaf_start; a.leaf_q = s->leaf_q; a.sep = s->sep;
    a.packets = s->packets; a.mleaf = s->mleaf; a.rsep = s->rsep; a.m_lo = s->m_lo;
    a.mode = mode; a.m_from = m_from; a.m_to = m_to; a.diag_mode = diag_mode;
    a.u = um[first]; a.vin = nullptr; a.yout = nullptr;     // not read by hp_sweep4d / hp_sweep4m
    for (int r = 0; r < HP_RMAX; ++r) a.um[r] = r < R ? um[r] : nullptr;
    a.xch = s->xch; a.bar = s->bar;
    a.oGP = 0; a.oXS = (size_t)L.G * s->b * R; a.oGR = a.oVS = 0;
    a.slot_stride = a.oXS + (size_t)std::max(L.NS, 1) * (L.P | 1) * R;
    a.s2t = s->s2t; a.is1t = s->is1t;
    a.ih2 = 1.0 / (s->pml.h * s->pml.h);
    a.dbg = s->dbg;
    HP_CUDA(cudaMemsetAsync(s->xch, 0xFF, sizeof(cplx) * HP_RING * a.slot_stride, st));
    HP_CUDA(cudaMemsetAsync(s->bar + 1, 0, sizeof(unsigned int), st));
    hp_count_launch();
    hp_profile_begin(s, st);
    if (tensor ? hp_sweep4d_launch(s, a, st) : hp_sweep4m_launch(s, a, R, st)) return 2;
    hp_profile_end(s, st, (int64_t)(hi - lo + 1) * ((int64_t)L.G * L.PK + 3 * (int64_t)s->n * R + (int64_t)(L.P - 1) * 3 * s->b * s->b) *
                              (int64_t)sizeof(cplx));
    return 0;
}

// 0 = fine; 1 = a CTA of a sweep kernel gave up waiting for exchange data (synchronises the device)
extern "C" int hp_sweep_status(hp_solver* s) {
    if (!s || !s->bar) return 0;
    unsigned int v[3] = {0, 0, 0};
    if (cudaDeviceSynchronize() != cudaSuccess) return 2;
    if (cudaMemcpy(v, s->bar, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return 2;
    return (v[1] | v[2]) ? 1 : 0;
}

extern "C" int hp_sweep_forward(hp_solver* s, double* u_dev, int m_from, int m_to, void* stream) {
    if (!s) { hp_set_error("hp_sweep_forward: null solver"); return 1; }
    return hp_sweep_launch(s, 0, (cplx*)u_dev, nullptr, nullptr, m_from, m_to, 0, (cudaStream_t)stream);
}

extern "C" int hp_sweep_backward(hp_solver* s, double* u_dev, int m_from, int m_to, int diag_mode, void* stream) {
    if (!s) { hp_set_error("hp_sweep_backward: null solver"); return 1; }
    return hp_sweep_launch(s, 1, (cplx*)u_dev, nullptr, nullptr, m_from, m_to, diag_mode, (cudaStream_t)stream);
}

// largest number of right-hand sides one sweep launch can carry with the layout of this solver (1, 2, 4 or 8)
extern "C" int hp_multi_max(hp_solver* s) {
    if (!s || !s->packets) return 1;
    if (!hp_sweep4d_supported(s)) return 8;
    for (int R = HP_RMAX; R > 1; R >>= 1)
        if (!hp_sweep4m_supported(s, R)) return R;
    return 1;
}
extern "C" int hp_sweep_forward_multi(hp_solver* s, int R, double* const* u_devs, int m_from, int m_to, void* stream) {
    if (!s || !u_devs) { hp_set_error("hp_sweep_forward_multi: null argument"); return 1; }
    return hp_sweep_launch_multi(s, 0, R, (cplx* const*)u_devs, m_from, m_to, 0, (cudaStream_t)stream);
}
extern "C" int hp_sweep_backward_multi(hp_solver* s, int R, double* const* u_devs, int m_from, int m_to, int diag_mode, void* stream) {
    if (!s || !u_devs) { hp_set_error("hp_sweep_backward_multi: null argument"); return 1; }
    return hp_sweep_launch_multi(s, 1, R, (cplx* const*)u_devs, m_from, m_to, diag_mode, (cudaStream_t)stream);
}

extern "C" int hp_strip_apply(hp_solver* s, int m, const double* v_dev, double* y_dev, void* stream) {
    if (!s) { hp_set_error("hp_strip_apply: null solver"); return 1; }
    return hp_sweep_launch(s, 2, nullptr, (const cplx*)v_dev, (cplx*)y_dev, m, m, 0, (cudaStream_t)stream);
}
