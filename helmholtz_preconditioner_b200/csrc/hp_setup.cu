// Setup of the strip solves: algo2_3 of the reference (/root/reference/code.py:345-353) for the strips
// H_m, m = m_lo..m_hi.  Where the reference calls SuperLU on each bn x bn strip operator, every strip is
// reduced here to the generators the sweep kernel streams (csrc/hp_setup_core.h, tools/strip_model.py):
//   leaf samples W, Gf, Gl and the dense separator inverse N, written straight into the per-CTA packets.
// Strips are independent; they are processed in batches of LB strips so that the scratch (the Schur
// chains of every block row) stays bounded.
#include "hp_internal.cuh"
#include "hp_sweep4.h"

#include <algorithm>
#include <chrono>
#include <stdio.h>
#include <stdlib.h>

struct HpSetupArgs {
    HpStripCtx c;
    HpLayout lay;
    const int *leaf_start, *leaf_q, *sep;
    int m0;            // first strip of this batch
    int nb;            // strips in this batch
    int m_lo;          // first strip of the solver (packet index origin)
    int leaf_piped;    // leaf kernel: propagators prefetched through registers (developer switch HP_LEAF_NOPIPE)
    cplx *Finv, *Binv, *gcol;             // [nb][n][bb], [nb][n][bb], [nb][n][b]
    cplx* tp;                             // [nb][P][bb]
    cplx *Sd, *So, *FX, *FXi, *PF, *BX, *BXi, *PB, *Njj;   // [nb][max(ns,1)][bb]
    cplx* packets;
    int* status;
};

__device__ __forceinline__ cplx* hp_packet(const HpSetupArgs& a, int layer_in_batch, int g) {
    return a.packets + ((size_t)(a.m0 - a.m_lo + layer_in_batch) * a.lay.G + g) * a.lay.PK;
}

// thread -> (strip, leaf, direction)
template <int BB>
__global__ void __launch_bounds__(64) hp_chain_kernel(HpSetupArgs a) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int total = a.nb * a.lay.P * 2;
    if (t >= total) return;
    int dir = t & 1, l = (t >> 1) % a.lay.P, lb = (t >> 1) / a.lay.P;
    int m = a.m0 + lb, n = a.c.n, bb = a.c.b * a.c.b;
    int i0 = a.leaf_start[l] + 1, i1 = a.leaf_start[l] + a.leaf_q[l];
    int bad;
    if (dir == 0) bad = hp_chain_forward<BB>(a.Finv + (size_t)lb * n * bb, i0, i1, m, a.c);
    else bad = hp_chain_backward<BB>(a.Binv + (size_t)lb * n * bb, a.gcol + (size_t)lb * n * a.c.b, i0, i1, m, a.c);
    if (bad) atomicOr(a.status, 1);
}

// ------------------------------------------------------------------------------------------------------
// Warp-cooperative Schur chains: warp -> (strip, leaf, direction), the b x b blocks live in shared memory and the
// 32 lanes share every elimination step (the one-thread-per-chain kernel above keeps its blocks in local memory and
// is bound by the L2 traffic of those spills: 2.2 s of the 3.2 s setup at 4096^2).  Same recurrences as
// hp_chain_forward / hp_chain_backward (csrc/hp_setup_core.h), same operation order inside every entry.
// ------------------------------------------------------------------------------------------------------
struct HpLaneRow { cplx is2c, s2lo, s2hi; };                 // x2 factors of strip row k (lane k), cf. hp_strip_rows
__device__ __forceinline__ HpLaneRow hp_lane_strip_row(int k, int m, int b, const HpPml& p) {
    HpLaneRow R;
    double shift = HP_MUL((double)(m - b), p.h);
    int j = m - b + 1 + k;
    R.is2c = hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j, p.h), shift), p), p);
    R.s2lo = cinv(hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j - 1, p.h), shift), p), p));
    R.s2hi = cinv(hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j + 1, p.h), shift), p), p));
    return R;
}
// coefficients of block row i for strip row k (cf. hp_block_row): written to vec[0..5b) = L, U, sub, dia, sup
template <bool CK>
__device__ __forceinline__ void hp_lane_block_row(cplx* vec, const HpLaneRow& R, int i, int k, int m, int b, const HpStripCtx& c) {
    double ih2 = 1.0 / (c.pml.h * c.pml.h);
    cplx s1lo = c.s1t[2 * i - 1], s1hi = c.s1t[2 * i + 1], is1c = c.is1t[2 * i];
    int j = m - b + 1 + k;
    cplx c1 = cscale(ih2, cmul(s1lo, R.is2c));
    cplx c2 = cscale(ih2, cmul(s1hi, R.is2c));
    cplx c3 = cscale(ih2, cmul(R.s2lo, is1c));
    cplx c4 = cscale(ih2, cmul(R.s2hi, is1c));
    cplx c5;
    if constexpr (CK) {
        c5 = hp_kmul_sub(c.kappa_c[(size_t)(j - 1) * c.n + (i - 1)], cmul(c.omega2, cmul(is1c, R.is2c)),
                         cadd(cadd(c1, c2), cadd(c3, c4)));
    } else {
        double cv = c.c_mat[(size_t)(i - 1) * (c.n + 2) + (j - 1)];
        c5 = cscale(1.0 / (cv * cv), cmul(c.omega2, cmul(is1c, R.is2c)));
        c5 = csub(c5, cadd(cadd(c1, c2), cadd(c3, c4)));
    }
    vec[k] = c1; vec[b + k] = c2; vec[2 * b + k] = c3; vec[3 * b + k] = c5; vec[4 * b + k] = c4;
}
// in-place Gauss-Jordan inverse with partial pivoting of the b x b matrix A in shared memory (b <= 32), one warp.
// The pivot is the entry of largest modulus up to the lower 32 bits of the double (any such choice is stable).
__device__ int hp_warp_inv(cplx* A, int b, int lane, int* piv) {
    int bad = 0;
    for (int p = 0; p < b; ++p) {
        unsigned int key = 0u;
        if (lane >= p && lane < b) {
            double v = cabs2(A[lane * b + p]);
            key = (unsigned int)(__double_as_longlong(v) >> 32) + (v > 0.0 ? 1u : 0u);   // monotone in v, 0 only for v == 0
        }
        unsigned int best = __reduce_max_sync(0xffffffffu, key);
        if (best == 0u) bad = 1;
        int r = __ffs(__ballot_sync(0xffffffffu, key == best && lane >= p && lane < b)) - 1;
        if (r < 0) r = p;
        if (lane == 0) piv[p] = r;
        if (r != p && lane < b) { cplx t = A[p * b + lane]; A[p * b + lane] = A[r * b + lane]; A[r * b + lane] = t; }
        __syncwarp();
        cplx d = cinv(A[p * b + p]);
        __syncwarp();
        if (lane < b) A[p * b + lane] = cmul(lane == p ? cmake(1.0, 0.0) : A[p * b + lane], d);
        __syncwarp();
        // eliminate: every lane takes entries e = lane, lane+32, ... ; reads first, then writes
        cplx nv[(HP_BMAX * HP_BMAX + 31) / 32];
        int cnt = 0;
        for (int e = lane; e < b * b; e += 32, ++cnt) {
            int i = e / b, j = e - i * b;
            cplx cur = A[e];
            if (i != p) {
                cplx f = A[i * b + p];
                cur = cfms(f, A[p * b + j], j == p ? cmake(0.0, 0.0) : cur);
            }
            nv[cnt] = cur;
        }
        __syncwarp();
        cnt = 0;
        for (int e = lane; e < b * b; e += 32, ++cnt) A[e] = nv[cnt];
        __syncwarp();
    }
    for (int p = b - 1; p >= 0; --p) {
        int r = piv[p];
        if (r != p && lane < b) { cplx t = A[lane * b + p]; A[lane * b + p] = A[lane * b + r]; A[lane * b + r] = t; }
        __syncwarp();
    }
    return bad;
}

template <bool CK>
__global__ void __launch_bounds__(256) hp_chain_warp_kernel(HpSetupArgs a, int warps_per_block) {
    extern __shared__ double2 smw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = blockIdx.x * warps_per_block + wib;
    const int total = a.nb * a.lay.P * 2;
    if (wib >= warps_per_block || warp >= total) return;
    const int dir = warp & 1, l = (warp >> 1) % a.lay.P, lb = (warp >> 1) / a.lay.P;
    const int m = a.m0 + lb, n = a.c.n, b = a.c.b, bb = b * b;
    const int i0 = a.leaf_start[l] + 1, i1 = a.leaf_start[l] + a.leaf_q[l];
    cplx* F = smw + (size_t)wib * (4 * bb + 6 * b + 16);      // F (then G), T1, T2, Bs, vec[5b], prev[b], piv
    cplx* T1 = F + bb;
    cplx* T2 = T1 + bb;
    cplx* Bs = T2 + bb;
    cplx* vec = Bs + bb;                                     // L, U, sub, dia, sup of the current block row
    cplx* prev = vec + 5 * b;                                // U_{i-1} (forward) / L_{i+1} (backward)
    int* piv = reinterpret_cast<int*>(prev + b);
    HpLaneRow R;
    if (lane < b) R = hp_lane_strip_row(lane, m, b, a.c.pml);
    int bad = 0;
    cplx* out = (dir == 0 ? a.Finv : a.Binv) + (size_t)lb * n * bb;
    const int nsteps = i1 - i0 + 1;
    for (int st = 0; st < nsteps; ++st) {
        const int i = dir == 0 ? i0 + st : i1 - st;
        if (lane < b) hp_lane_block_row<CK>(vec, R, i, lane, m, b, a.c);
        __syncwarp();
        // F = D_i - diag(a) Xinv diag(c):  forward a = L_i, c = U_{i-1};  backward a = U_i, c = L_{i+1}
        const cplx* av = dir == 0 ? vec : vec + b;
        for (int e = lane; e < bb; e += 32) {
            int r = e / b, sc = e - r * b;
            cplx v = cmake(0.0, 0.0);
            if (r == sc) v = vec[3 * b + r];
            else if (sc == r - 1) v = vec[2 * b + r];
            else if (sc == r + 1) v = vec[4 * b + r];
            if (st > 0) v = cfms(cmul(av[r], F[e]), prev[sc], v);
            F[e] = v;
        }
        __syncwarp();
        bad |= hp_warp_inv(F, b, lane, piv);
        cplx* dst = out + (size_t)(i - 1) * bb;
        for (int e = lane; e < bb; e += 32) dst[e] = F[e];
        if (lane < b) prev[lane] = dir == 0 ? vec[b + lane] : vec[lane];
        __syncwarp();
    }
    if (dir == 1) {
        // diagonal blocks of the leaf inverse, ascending; F holds Binv[i0] = G_{i0,i0} now
        cplx* G = F;
        cplx* gcol = a.gcol + (size_t)lb * n * b;
        for (int i = i0; i <= i1; ++i) {
            if (lane < b) hp_lane_block_row<CK>(vec, R, i, lane, m, b, a.c);
            __syncwarp();
            if (i > i0) {
                const cplx* Bi = out + (size_t)(i - 1) * bb;
                for (int e = lane; e < bb; e += 32) {
                    int r = e / b, sc = e - r * b;
                    Bs[e] = Bi[e];
                    T1[e] = cmul(cmul(vec[r], G[e]), prev[sc]);
                }
                __syncwarp();
                for (int e = lane; e < bb; e += 32) {           // T2 = Bs T1
                    int r = e / b, sc = e - r * b;
                    cplx acc = cmake(0.0, 0.0);
                    for (int t = 0; t < b; ++t) acc = cfma(Bs[r * b + t], T1[t * b + sc], acc);
                    T2[e] = acc;
                }
                __syncwarp();
                for (int e = lane; e < bb; e += 32) {           // G = Bs + T2 Bs
                    int r = e / b, sc = e - r * b;
                    cplx acc = Bs[e];
                    for (int t = 0; t < b; ++t) acc = cfma(T2[r * b + t], Bs[t * b + sc], acc);
                    G[e] = acc;
                }
                __syncwarp();
            }
            if (lane < b) {
                gcol[(size_t)(i - 1) * b + lane] = G[lane * b + (b - 1)];
                prev[lane] = vec[b + lane];
            }
            __syncwarp();
        }
    }
    if (bad && lane == 0) atomicOr(a.status, 1);
}

// ------------------------------------------------------------------------------------------------------
// Register-resident Schur chains (compile-time b): one warp runs BOTH chains of a leaf, lanes 0-15 the forward
// chain, lanes 16-31 the backward one.  Lane j < B of a half keeps column j of the b x b block in registers, so a
// Gauss-Jordan step is a local pivot search in lane p, one broadcast of the pivot and of the B-1 multipliers
// (width-16 shuffles) and B-1 fused multiply-subtracts per lane; nothing of the block goes through shared memory.
// The coefficients of a block row factor into an x1 part (tables) and the x2 part of the strip row, so the
// Schur update F = D_i - diag(a) X diag(c) needs no exchange either.  The ascending recurrence of the backward
// chain (two b x b products per block row) is shared by both halves, operands broadcast from shared memory.
// Same recurrences and the same operation order inside every entry as hp_chain_warp_kernel; the shared-memory
// kernel spent its time on instruction issue (index arithmetic, shared-memory round trips, 6 warp syncs per pivot).
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ cplx hp_shfl16(cplx v, int src) {
    return cmake(__shfl_sync(0xffffffffu, v.x, src, 16), __shfl_sync(0xffffffffu, v.y, src, 16));
}

// 1/a as conj(a)/|a|^2: one division instead of the two of Smith's algorithm (the entries of the Schur blocks are of
// the order 1/h^2, far from the overflow range of |a|^2)
__device__ __forceinline__ cplx hp_crecip(cplx a) {
    const double r = 1.0 / fma(a.x, a.x, a.y * a.y);
    return cmake(a.x * r, -a.y * r);
}
#ifdef HP_PIVOT_SMITH            // developer switch: the earlier pivot rule (largest modulus, Smith's reciprocal)
#define HP_PIVOT_NORM(a) cabs2(a)
#define HP_PIVOT_INV(a) cinv(a)
#else                            // |re| + |im| is within sqrt(2) of the modulus: as good a pivot rule, one add per entry
#define HP_PIVOT_NORM(a) (fabs((a).x) + fabs((a).y))
#define HP_PIVOT_INV(a) hp_crecip(a)
#endif
// in-place inverse of the B x B matrix whose column j is A[0..B) of lane j of each half-warp (partial pivoting).
// The pivot loop is NOT unrolled (unrolled, the kernel is ~90 KB of straight-line code and stalls on instruction
// fetch): after every step the rows are rotated by one register, so that the pivot row is always A[0] and the
// body is the same code for every p; after B steps the rows are back in place.  Pivot rows are kept as 4-bit
// fields of one 64-bit word.
template <int B, bool ROLL = true>
__device__ __forceinline__ int hp_half_inv(cplx (&A)[B], int j) {
    static_assert(B <= 16, "pivot indices are packed in 4 bits");
    int bad = 0;
    unsigned long long pivs = 0ull;
    if constexpr (!ROLL) {                           // developer variant: fully unrolled pivot loop
        int piv[B];
#pragma unroll
        for (int p = 0; p < B; ++p) {
            int r_own = p;
            double best = cabs2(A[p]);
#pragma unroll
            for (int i = p + 1; i < B; ++i) {
                const double v = cabs2(A[i]);
                if (v > best) { best = v; r_own = i; }
            }
            const int r = __shfl_sync(0xffffffffu, r_own, p, 16);
            if (__shfl_sync(0xffffffffu, best, p, 16) == 0.0) bad = 1;
            piv[p] = r;
#pragma unroll
            for (int i = p + 1; i < B; ++i)
                if (i == r) { const cplx t = A[i]; A[i] = A[p]; A[p] = t; }
            const cplx d = cinv(hp_shfl16(A[p], p));
            const cplx prow = cmul(j == p ? cmake(1.0, 0.0) : A[p], d);
            A[p] = prow;
#pragma unroll
            for (int i = 0; i < B; ++i) {
                if (i == p) continue;
                const cplx f = hp_shfl16(A[i], p);
                A[i] = cfms(f, prow, j == p ? cmake(0.0, 0.0) : A[i]);
            }
        }
#pragma unroll
        for (int p = B - 1; p >= 0; --p) {
            const int r = piv[p];
            if (__any_sync(0xffffffffu, r != p)) {
                const int src = j == p ? r : (j == r ? p : j);
#pragma unroll
                for (int i = 0; i < B; ++i) A[i] = hp_shfl16(A[i], src);
            }
        }
        return bad;
    } else {
#pragma unroll 1
    for (int p = 0; p < B; ++p) {
        // logical row i >= p sits in A[i - p]; pivot search in lane p, which holds column p
        int k_own = 0;
        double best = HP_PIVOT_NORM(A[0]);
#pragma unroll
        for (int k = 1; k < B; ++k) {
            const double v = HP_PIVOT_NORM(A[k]);
            if (k < B - p && v > best) { best = v; k_own = k; }
        }
        const int kr = __shfl_sync(0xffffffffu, k_own, p, 16);
        if (__shfl_sync(0xffffffffu, best, p, 16) == 0.0) bad = 1;
        pivs |= (unsigned long long)(p + kr) << (4 * p);
        if (__any_sync(0xffffffffu, kr != 0)) {
#pragma unroll
            for (int k = 1; k < B; ++k)
                if (k == kr) { const cplx t = A[k]; A[k] = A[0]; A[0] = t; }
        }
        const cplx d = HP_PIVOT_INV(hp_shfl16(A[0], p));
        const bool isp = j == p;
        const cplx prow = cmul(isp ? cmake(1.0, 0.0) : A[0], d);
        // eliminate the other rows and rotate: new A[k-1] = updated A[k], new A[B-1] = pivot row
#pragma unroll
        for (int k = 1; k < B; ++k) {
            const cplx f = hp_shfl16(A[k], p);
            A[k - 1] = cfms(f, prow, isp ? cmake(0.0, 0.0) : A[k]);
        }
        A[B - 1] = prow;
    }
    // undo the row exchanges on the columns (columns live in lanes)
#pragma unroll 1
    for (int p = B - 1; p >= 0; --p) {
        const int r = (int)((pivs >> (4 * p)) & 15ull);
        if (__any_sync(0xffffffffu, r != p)) {
            const int src = j == p ? r : (j == r ? p : j);
#pragma unroll
            for (int i = 0; i < B; ++i) A[i] = hp_shfl16(A[i], src);
        }
    }
    return bad;
    }
}

template <int B, bool ROLL, bool CK = false>
__global__ void __launch_bounds__(128, 4) hp_chain_reg_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B, RH = (B + 1) / 2;
    __shared__ cplx s_tab[4][B];                 // 1/s2 at the strip rows (both halves work on the same strip)
    __shared__ cplx s_mat[4][3][BBc];            // ascending pass: Binv_i, T2, G (row major)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int pair = blockIdx.x * 4 + wib;
    if (pair >= a.nb * a.lay.P) return;
    const int h = lane >> 4, j = lane & 15;
    const bool act = j < B;
    const int jc = act ? j : B - 1;
    const int l = pair % a.lay.P, lb = pair / a.lay.P;
    const int m = a.m0 + lb, n = a.c.n;
    const int i0 = a.leaf_start[l] + 1, i1 = a.leaf_start[l] + a.leaf_q[l], nsteps = i1 - i0 + 1;
    const double ih2 = 1.0 / (a.c.pml.h * a.c.pml.h);
    const HpLaneRow Rj = hp_lane_strip_row(jc, m, B, a.c.pml);
    const cplx s2lo_n = hp_shfl16(Rj.s2lo, min(j + 1, 15));        // strip row j+1
    const cplx s2hi_p = hp_shfl16(Rj.s2hi, max(j - 1, 0));         // strip row j-1
    if (h == 0 && act) s_tab[wib][j] = Rj.is2c;
    __syncwarp();
    const cplx* tab = s_tab[wib];
    const int jg = m - B + 1 + jc;                                 // grid row of strip row j
    // coefficients of block row i at strip row j (cf. hp_lane_block_row): c1 = L, c2 = U, dia
    auto coeffs = [&](int i, cplx& c1, cplx& c2, cplx& dia, cplx& is1c) {
        const cplx s1lo = a.c.s1t[2 * i - 1], s1hi = a.c.s1t[2 * i + 1];
        is1c = a.c.is1t[2 * i];
        c1 = cscale(ih2, cmul(s1lo, Rj.is2c));
        c2 = cscale(ih2, cmul(s1hi, Rj.is2c));
        const cplx c3 = cscale(ih2, cmul(Rj.s2lo, is1c));
        const cplx c4 = cscale(ih2, cmul(Rj.s2hi, is1c));
        if constexpr (CK) {
            dia = hp_kmul_sub(a.c.kappa_c[(size_t)(jg - 1) * n + (i - 1)], cmul(a.c.omega2, cmul(is1c, Rj.is2c)),
                              cadd(cadd(c1, c2), cadd(c3, c4)));
        } else {
            const double cv = a.c.c_mat[(size_t)(i - 1) * (n + 2) + (jg - 1)];
            const cplx c5 = cscale(1.0 / (cv * cv), cmul(a.c.omega2, cmul(is1c, Rj.is2c)));
            dia = csub(c5, cadd(cadd(c1, c2), cadd(c3, c4)));
        }
    };

    cplx A[B];
#pragma unroll
    for (int r = 0; r < B; ++r) A[r] = cmake(0.0, 0.0);
    cplx prevj = cmake(0.0, 0.0);                                  // U_{i-1}[j] (forward) / L_{i+1}[j] (backward)
    int bad = 0;
    cplx* out = (h == 0 ? a.Finv : a.Binv) + (size_t)lb * n * BBc;
    for (int st = 0; st < nsteps; ++st) {
        const int i = h == 0 ? i0 + st : i1 - st;
        cplx c1, c2, dia, is1c;
        coeffs(i, c1, c2, dia, is1c);
        const cplx s1a = h == 0 ? a.c.s1t[2 * i - 1] : a.c.s1t[2 * i + 1];     // a_r = L_i[r] (forward) / U_i[r] (backward)
        const cplx subn = cscale(ih2, cmul(s2lo_n, is1c));                     // D[j+1][j]
        const cplx supp = cscale(ih2, cmul(s2hi_p, is1c));                     // D[j-1][j]
#pragma unroll
        for (int r = 0; r < B; ++r) {
            cplx v = cmake(0.0, 0.0);
            if (r == j) v = dia;
            else if (r == j + 1) v = subn;
            else if (r == j - 1) v = supp;
            if (st > 0) {
                const cplx av = cscale(ih2, cmul(s1a, tab[r]));
                v = cfms(cmul(av, A[r]), prevj, v);
            }
            A[r] = v;
        }
        if (!act) {                                                // idle lanes carry a zero column
#pragma unroll
            for (int r = 0; r < B; ++r) A[r] = cmake(0.0, 0.0);
        }
        bad |= hp_half_inv<B, ROLL>(A, j);
        if (act) {
            cplx* dst = out + (size_t)(i - 1) * BBc + j;
#pragma unroll
            for (int r = 0; r < B; ++r) dst[r * B] = A[r];
        }
        prevj = h == 0 ? c2 : c1;
    }
    // ---- diagonal blocks of the leaf inverse, ascending (backward chain; both halves share the products):
    //      lane (h, j) forms rows h*RH .. of column j.  G starts as Binv[i0], held by the backward half.
    cplx* Bs = s_mat[wib][0];
    cplx* T2s = s_mat[wib][1];
    cplx* Gs = s_mat[wib][2];
    cplx* gcol = a.gcol + (size_t)lb * n * B;
    const cplx* binv = a.Binv + (size_t)lb * n * BBc;
    if (h == 1 && act) {
#pragma unroll
        for (int r = 0; r < B; ++r) Gs[r * B + j] = A[r];
        if (j == B - 1)
            for (int r = 0; r < B; ++r) gcol[(size_t)(i0 - 1) * B + r] = A[r];
    }
    {   // U_{i0}[j]
        cplx c1, c2, dia, is1c;
        coeffs(i0, c1, c2, dia, is1c);
        prevj = c2;
    }
    __syncwarp();
    const int r0 = h * RH, r1 = min(B, r0 + RH);
    for (int i = i0 + 1; i <= i1; ++i) {
        cplx c1, c2, dia, is1c;
        coeffs(i, c1, c2, dia, is1c);
        const cplx s1lo = a.c.s1t[2 * i - 1];
        cplx Bcol[B], T1[B];
        if (act) {
            const cplx* Bi = binv + (size_t)(i - 1) * BBc + j;
#pragma unroll
            for (int t = 0; t < B; ++t) Bcol[t] = __ldcg(reinterpret_cast<const double2*>(Bi + t * B));
#pragma unroll
            for (int t = 0; t < B; ++t) {
                const cplx Lt = cscale(ih2, cmul(s1lo, tab[t]));
                T1[t] = cmul(cmul(Lt, Gs[t * B + j]), prevj);
            }
#pragma unroll
            for (int t = 0; t < B; ++t)
                if (t >= r0 && t < r1) Bs[t * B + j] = Bcol[t];
        }
        __syncwarp();
        if (act) {
#pragma unroll
            for (int rr = 0; rr < RH; ++rr) {
                const int r = r0 + rr;
                if (r < r1) {
                    cplx acc = cmake(0.0, 0.0);
#pragma unroll
                    for (int t = 0; t < B; ++t) acc = cfma(Bs[r * B + t], T1[t], acc);
                    T2s[r * B + j] = acc;
                }
            }
        }
        __syncwarp();
        if (act) {
#pragma unroll
            for (int rr = 0; rr < RH; ++rr) {
                const int r = r0 + rr;
                if (r < r1) {
                    cplx acc = Bs[r * B + j];
#pragma unroll
                    for (int t = 0; t < B; ++t) acc = cfma(T2s[r * B + t], Bcol[t], acc);
                    Gs[r * B + j] = acc;
                    if (j == B - 1) gcol[(size_t)(i - 1) * B + r] = acc;
                }
            }
        }
        prevj = c2;
        __syncwarp();
    }
    if (bad && lane == 0) atomicOr(a.status, 1);
}

// CTA -> (strip, leaf); thread -> leaf column r
__global__ void hp_leaf_kernel(HpSetupArgs a) {
    int l = blockIdx.x % a.lay.P, lb = blockIdx.x / a.lay.P;
    int r = threadIdx.x;
    int m = a.m0 + lb, n = a.c.n, b = a.c.b, bb = b * b;
    int q = a.leaf_q[l], K = a.lay.K;
    int rr = r < q ? r : q - 1;
    int k = ((rr + 1) * K - 1) / q;                    // part that owns column rr
    int lc0 = (q * k) / K;
    cplx* pk = hp_packet(a, lb, l * K + k);
    cplx* wrow = pk + (size_t)(rr - lc0) * a.lay.QP;
    cplx* gf = pk + a.lay.offG + (rr - lc0);
    cplx* gl = gf + (size_t)b * a.lay.CW;
    hp_leaf_column(wrow, gf, gl, a.lay.CW, a.Finv + (size_t)lb * n * bb, a.Binv + (size_t)lb * n * bb,
                   a.gcol + (size_t)lb * n * b, a.leaf_start[l] + 1, q, a.lay.QP, r, m, l > 0, l < a.lay.P - 1, a.c);
}

// The same leaf columns with the b x b propagators staged in shared memory (every thread of the block multiplies by
// the same matrix at the same step) and b a compile-time constant: 12 independent accumulation chains per thread
// instead of one.  Same operation order per entry as hp_leaf_column / hp_propagate (csrc/hp_setup_core.h).
// NT: largest CTA the instantiation is launched with (register budget: three CTAs of 128 threads per SM)
template <int B, int NT>
__global__ void __launch_bounds__(NT, NT <= 128 ? 3 : 1) hp_leaf_fast_kernel(HpSetupArgs a) {
    __shared__ cplx Ms[2][B * B];
    __shared__ cplx is2c_s[B];
    const int l = blockIdx.x % a.lay.P, lb = blockIdx.x / a.lay.P;
    const int r = threadIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int m = a.m0 + lb, n = a.c.n, bb = B * B;
    const int q = a.leaf_q[l], K = a.lay.K, i0 = a.leaf_start[l] + 1;
    const bool live = r < q, has_left = l > 0, has_right = l < a.lay.P - 1;
    const int rr = live ? r : q - 1;
    const int k = ((rr + 1) * K - 1) / q;                  // part that owns column rr
    const int lc0 = (q * k) / K;
    cplx* pk = hp_packet(a, lb, l * K + k);
    cplx* wrow = pk + (size_t)(rr - lc0) * a.lay.QP;
    cplx* gf = pk + a.lay.offG + (rr - lc0);
    cplx* gl = gf + (size_t)B * a.lay.CW;
    const size_t gstride = a.lay.CW;
    const cplx* Finv = a.Finv + (size_t)lb * n * bb;
    const cplx* Binv = a.Binv + (size_t)lb * n * bb;
    const cplx* gcol = a.gcol + (size_t)lb * n * B;
    const cplx ih2 = cmake(1.0 / (a.c.pml.h * a.c.pml.h), 0.0);
    if (tid < B) is2c_s[tid] = hp_lane_strip_row(tid, m, B, a.c.pml).is2c;
    auto loadM = [&](int buf, const cplx* src) { for (int e = tid; e < bb; e += nthr) Ms[buf][e] = src[e]; };
    // the propagator of the next step is fetched into registers before the products of this step and stored to shared
    // memory after them (the loads are L2/HBM round trips)
    constexpr int MR = (B * B + 95) / 96;                  // registers per thread: enough for CTAs of 96 threads and more
    const bool piped = nthr * MR >= bb && a.leaf_piped;    // narrow leaves (small problems) copy directly
    cplx mreg[MR];
    auto fetchM = [&](int buf, const cplx* src) {
        if (!piped) { loadM(buf, src); return; }
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = tid + u * nthr; if (e < bb) mreg[u] = src[e]; }
    };
    auto storeM = [&](int buf) {
        if (!piped) return;
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = tid + u * nthr; if (e < bb) Ms[buf][e] = mreg[u]; }
    };
    auto propagate = [&](cplx* x, const cplx* M, cplx dscale) {        // x <- -M (dscale * is2c * x)
        cplx t[B], y[B];
#pragma unroll
        for (int kk = 0; kk < B; ++kk) t[kk] = cmul(cmul(dscale, is2c_s[kk]), x[kk]);
#pragma unroll
        for (int aa = 0; aa < B; ++aa) {
            cplx acc = cmake(0.0, 0.0);
#pragma unroll
            for (int kk = 0; kk < B; ++kk) acc = cfms(M[aa * B + kk], t[kk], acc);
            y[aa] = acc;
        }
#pragma unroll
        for (int aa = 0; aa < B; ++aa) x[aa] = y[aa];
    };
    cplx x0[B], x[B];
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x0[kk] = live ? gcol[(size_t)(i0 - 1 + r) * B + kk] : cmake(0.0, 0.0);
    if (live) wrow[r] = x0[B - 1];
    // leftwards: columns q-2 .. 0, propagator Finv of block row i = i0 + col
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x[kk] = x0[kk];
    const int nst = q - 1;
    if (nst > 0) loadM(0, Finv + (size_t)(i0 + q - 2 - 1) * bb);
    __syncthreads();
    for (int s = 0; s < nst; ++s) {
        const int col = q - 2 - s, i = i0 + col;
        if (s + 1 < nst) fetchM((s + 1) & 1, Finv + (size_t)(i - 2) * bb);
        if (live && col < r) {
            propagate(x, Ms[s & 1], cmul(ih2, a.c.s1t[2 * i + 1]));
            wrow[col] = x[B - 1];
        }
        if (s + 1 < nst) storeM((s + 1) & 1);
        __syncthreads();
    }
    if (live) {
        cplx sc = cmul(ih2, a.c.s1t[2 * i0 - 1]);
#pragma unroll
        for (int kk = 0; kk < B; ++kk)
            gf[(size_t)kk * gstride] = has_left ? cmul(cmul(sc, is2c_s[kk]), x[kk]) : cmake(0.0, 0.0);
    }
    // rightwards: columns 1 .. q-1, propagator Binv of block row i = i0 + col
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x[kk] = x0[kk];
    if (nst > 0) loadM(0, Binv + (size_t)(i0 + 1 - 1) * bb);
    __syncthreads();
    for (int s = 0; s < nst; ++s) {
        const int col = 1 + s, i = i0 + col;
        if (s + 1 < nst) fetchM((s + 1) & 1, Binv + (size_t)i * bb);
        if (live && col > r) {
            propagate(x, Ms[s & 1], cmul(ih2, a.c.s1t[2 * i - 1]));
            wrow[col] = x[B - 1];
        }
        if (s + 1 < nst) storeM((s + 1) & 1);
        __syncthreads();
    }
    if (live) {
        const int it = i0 + q - 1;
        cplx sc = cmul(ih2, a.c.s1t[2 * it + 1]);
#pragma unroll
        for (int kk = 0; kk < B; ++kk)
            gl[(size_t)kk * gstride] = has_right ? cmul(cmul(sc, is2c_s[kk]), x[kk]) : cmake(0.0, 0.0);
    }
}

// Leaf generators, warp-paced: same work split as hp_leaf_fast_kernel (CTA -> (strip, leaf), thread -> leaf column r) but
// every warp stages the propagators it needs itself (cp.async into a per-warp double buffer) and walks only the
// block rows between its own columns and the leaf ends, with warp syncs only.  The CTA-wide version walks the whole
// leaf in lock step: half of the warps idle at the barrier of every step (ncu: 2.4 barrier stalls per issue).
template <int B>
__global__ void __launch_bounds__(128, 3) hp_leaf_warp_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B;
    __shared__ __align__(16) cplx Ms[4][2][BBc];
    __shared__ cplx is2c_s[B];
    const int l = blockIdx.x % a.lay.P, lb = blockIdx.x / a.lay.P;
    const int r = threadIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int m = a.m0 + lb, n = a.c.n;
    const int q = a.leaf_q[l], K = a.lay.K, i0 = a.leaf_start[l] + 1;
    const bool live = r < q, has_left = l > 0, has_right = l < a.lay.P - 1;
    if (tid < B) is2c_s[tid] = hp_lane_strip_row(tid, m, B, a.c.pml).is2c;
    __syncthreads();
    const int rmin = 32 * w, rmax = min(rmin + 31, q - 1);
    if (rmin >= q) return;                                  // warp without columns
    const int rr = live ? r : q - 1;
    const int k = ((rr + 1) * K - 1) / q;                  // part that owns column rr
    const int lc0 = (q * k) / K;
    cplx* pk = hp_packet(a, lb, l * K + k);
    cplx* wrow = pk + (size_t)(rr - lc0) * a.lay.QP;
    cplx* gf = pk + a.lay.offG + (rr - lc0);
    cplx* gl = gf + (size_t)B * a.lay.CW;
    const size_t gstride = a.lay.CW;
    const cplx* Finv = a.Finv + (size_t)lb * n * BBc;
    const cplx* Binv = a.Binv + (size_t)lb * n * BBc;
    const cplx* gcol = a.gcol + (size_t)lb * n * B;
    const cplx ih2 = cmake(1.0 / (a.c.pml.h * a.c.pml.h), 0.0);
    auto fetch = [&](int buf, const cplx* src) {           // asynchronous copy of one b x b block, 16 bytes per lane and round
        for (int e = lane; e < BBc; e += 32) {
            unsigned int dst = (unsigned int)__cvta_generic_to_shared(&Ms[w][buf][e]);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + e) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto landed = [&]() { asm volatile("cp.async.wait_group 0;" ::: "memory"); __syncwarp(); };
    auto propagate = [&](cplx* x, const cplx* M, cplx dscale) {        // x <- -M (dscale * is2c * x)
        cplx t[B], y[B];
#pragma unroll
        for (int kk = 0; kk < B; ++kk) t[kk] = cmul(cmul(dscale, is2c_s[kk]), x[kk]);
#pragma unroll
        for (int aa = 0; aa < B; ++aa) {
            cplx acc = cmake(0.0, 0.0);
#pragma unroll
            for (int kk = 0; kk < B; ++kk) acc = cfms(M[aa * B + kk], t[kk], acc);
            y[aa] = acc;
        }
#pragma unroll
        for (int aa = 0; aa < B; ++aa) x[aa] = y[aa];
    };
    cplx x0[B], x[B];
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x0[kk] = live ? gcol[(size_t)(i0 - 1 + r) * B + kk] : cmake(0.0, 0.0);
    if (live) wrow[r] = x0[B - 1];
    // leftwards: columns rmax-1 .. 0, propagator Finv of block row i = i0 + col
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x[kk] = x0[kk];
    {
        const int nst = rmax;
        if (nst > 0) fetch(0, Finv + (size_t)(i0 + rmax - 2) * BBc);
        for (int s = 0; s < nst; ++s) {
            const int col = rmax - 1 - s, i = i0 + col;
            landed();                                           // block of this step is in Ms[s & 1], the other buffer is free
            if (s + 1 < nst) fetch((s + 1) & 1, Finv + (size_t)(i - 2) * BBc);
            if (live && col < r) {
                propagate(x, Ms[w][s & 1], cmul(ih2, a.c.s1t[2 * i + 1]));
                wrow[col] = x[B - 1];
            }
        }
    }
    if (live) {
        cplx sc = cmul(ih2, a.c.s1t[2 * i0 - 1]);
#pragma unroll
        for (int kk = 0; kk < B; ++kk)
            gf[(size_t)kk * gstride] = has_left ? cmul(cmul(sc, is2c_s[kk]), x[kk]) : cmake(0.0, 0.0);
    }
    // rightwards: columns rmin+1 .. q-1, propagator Binv of block row i = i0 + col
#pragma unroll
    for (int kk = 0; kk < B; ++kk) x[kk] = x0[kk];
    {
        const int nst = q - 1 - rmin;
        __syncwarp();
        if (nst > 0) fetch(0, Binv + (size_t)(i0 + rmin) * BBc);
        for (int s = 0; s < nst; ++s) {
            const int col = rmin + 1 + s, i = i0 + col;
            landed();
            if (s + 1 < nst) fetch((s + 1) & 1, Binv + (size_t)i * BBc);
            if (live && col > r) {
                propagate(x, Ms[w][s & 1], cmul(ih2, a.c.s1t[2 * i - 1]));
                wrow[col] = x[B - 1];
            }
        }
    }
    if (live) {
        const int it = i0 + q - 1;
        cplx sc = cmul(ih2, a.c.s1t[2 * it + 1]);
#pragma unroll
        for (int kk = 0; kk < B; ++kk)
            gl[(size_t)kk * gstride] = has_right ? cmul(cmul(sc, is2c_s[kk]), x[kk]) : cmake(0.0, 0.0);
    }
}

// thread -> (strip, inner leaf, column kap of tp)
__global__ void __launch_bounds__(128) hp_corner_kernel(HpSetupArgs a) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int b = a.c.b, P = a.lay.P, bb = b * b;
    int total = a.nb * P * b;
    if (t >= total) return;
    int kap = t % b, l = (t / b) % P, lb = t / (b * P);
    if (l == 0 || l == P - 1) return;
    cplx col[HP_BMAX];
    hp_leaf_corner_tp(col, a.Binv + (size_t)lb * a.c.n * bb, a.leaf_start[l] + 1, a.leaf_q[l], a.lay.QP, kap,
                      a.m0 + lb, a.c);
    cplx* tp = a.tp + ((size_t)lb * P + l) * bb;
    for (int r = 0; r < b; ++r) tp[r * b + kap] = col[r];
}

// thread -> (strip, separator)
template <bool CK>
__global__ void __launch_bounds__(128) hp_sep_blocks_kernel(HpSetupArgs a) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int ns = a.lay.P - 1, b = a.c.b, bb = b * b, n = a.c.n;
    if (t >= a.nb * ns) return;
    int j = t % ns, lb = t / ns, m = a.m0 + lb;
    int s = a.sep[j] + 1;
    const cplx* Finv = a.Finv + (size_t)lb * n * bb;
    const cplx* Binv = a.Binv + (size_t)lb * n * bb;
    hp_sep_diag<CK>(a.Sd + ((size_t)lb * ns + j) * bb, s, m, Finv + (size_t)(s - 2) * bb, Binv + (size_t)s * bb, a.c);
    if (j + 1 < ns)
        hp_sep_offdiag(a.So + ((size_t)lb * ns + j) * bb, s, a.sep[j + 1] + 1, m,
                       a.tp + ((size_t)lb * a.lay.P + j + 1) * bb, a.c);
}

// thread -> (strip, direction)
template <int BB>
__global__ void __launch_bounds__(32) hp_sep_chain_kernel(HpSetupArgs a) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int ns = a.lay.P - 1, bb = a.c.b * a.c.b;
    if (t >= a.nb * 2) return;
    int dir = t & 1, lb = t >> 1;
    size_t o = (size_t)lb * ns * bb;
    int bad;
    if (dir == 0) bad = hp_sep_chain<BB>(a.FX + o, a.FXi + o, a.PF + o, a.Sd + o, a.So + o, ns, +1, a.c.b);
    else bad = hp_sep_chain<BB>(a.BX + o, a.BXi + o, a.PB + o, a.Sd + o, a.So + o, ns, -1, a.c.b);
    if (bad) atomicOr(a.status, 2);
}

// Separator chains on half-warps (compile-time b): half-warp -> (strip, direction), lane j keeps column j of the
// running block in registers (hp_half_inv); the operands that every lane needs (the off-diagonal block S_{j,jp},
// T1, Xinv) are broadcast from a per-half shared-memory tile.  Same recurrence and accumulation order as
// hp_sep_chain (csrc/hp_setup_core.h), which ran one thread per chain: 52 ms of latency at 4096^2.
template <int B>
__global__ void __launch_bounds__(128) hp_sep_chain_half_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B;
    __shared__ cplx s_o[8][BBc];                 // off-diagonal block of the step (as stored in So)
    __shared__ cplx s_t[8][BBc];                 // T1, then Xinv (row major)
    const int lane = threadIdx.x & 31, hw = threadIdx.x >> 4;            // half-warp in the block
    const int j = lane & 15;
    const bool act = j < B;
    const int chain = blockIdx.x * 8 + hw;
    const int ns = a.lay.P - 1;
    // idle halves of the last block follow a live chain (the shuffles and warp syncs are warp wide) without storing
    const bool real = chain < a.nb * 2;
    const int ch = real ? chain : a.nb * 2 - 1;
    const int dir = (ch & 1) ? -1 : +1, lb = ch >> 1;
    const size_t o0 = (size_t)lb * ns * BBc;
    cplx* X = (dir > 0 ? a.FX : a.BX) + o0;
    cplx* Xinv = (dir > 0 ? a.FXi : a.BXi) + o0;
    cplx* Prop = (dir > 0 ? a.PF : a.PB) + o0;
    const cplx* Sd = a.Sd + o0;
    const cplx* So = a.So + o0;
    cplx* so = s_o[hw];
    cplx* st = s_t[hw];
    const int jc = act ? j : 0;
    cplx F[B], Xi[B];
#pragma unroll
    for (int r = 0; r < B; ++r) Xi[r] = cmake(0.0, 0.0);
    int bad = 0;
    for (int step = 0; step < ns; ++step) {
        const int js = dir > 0 ? step : ns - 1 - step;
#pragma unroll
        for (int r = 0; r < B; ++r) F[r] = act ? Sd[(size_t)js * BBc + r * B + j] : cmake(0.0, 0.0);
        if (step > 0) {
            // A = S_{js,jp}: fwd So[js-1]^T, bwd So[js];  T1 = A Xinv_jp;  F -= T1 A^T
            const cplx* o = So + (size_t)(dir > 0 ? js - 1 : js) * BBc;
            __syncwarp();
            for (int e = j; e < BBc; e += 16) so[e] = o[e];
            __syncwarp();
            cplx T1[B];
#pragma unroll
            for (int r = 0; r < B; ++r) {
                cplx acc = cmake(0.0, 0.0);
#pragma unroll
                for (int t = 0; t < B; ++t) acc = cfma(dir > 0 ? so[t * B + r] : so[r * B + t], Xi[t], acc);
                T1[r] = acc;
            }
            if (act) {
#pragma unroll
                for (int r = 0; r < B; ++r) st[r * B + j] = T1[r];
            }
            __syncwarp();
            cplx Aj[B];                                  // row j of A
#pragma unroll
            for (int l = 0; l < B; ++l) Aj[l] = dir > 0 ? so[l * B + jc] : so[jc * B + l];
#pragma unroll
            for (int r = 0; r < B; ++r) {
                cplx acc = F[r];
#pragma unroll
                for (int l = 0; l < B; ++l) acc = cfms(st[r * B + l], Aj[l], acc);
                F[r] = acc;
            }
        }
        if (act && real) {
#pragma unroll
            for (int r = 0; r < B; ++r) X[(size_t)js * BBc + r * B + j] = F[r];
        }
        if (!act) {
#pragma unroll
            for (int r = 0; r < B; ++r) F[r] = cmake(0.0, 0.0);
        }
        bad |= hp_half_inv<B>(F, j);
#pragma unroll
        for (int r = 0; r < B; ++r) Xi[r] = F[r];
        if (act && real) {
#pragma unroll
            for (int r = 0; r < B; ++r) Xinv[(size_t)js * BBc + r * B + j] = F[r];
        }
        const int jn = js + dir;
        if (jn >= 0 && jn < ns) {
            // Prop_js = -Xinv_js S_{js,jn}: fwd So[js], bwd So[js-1]^T
            const cplx* o = So + (size_t)(dir > 0 ? js : js - 1) * BBc;
            __syncwarp();
            if (act) {
#pragma unroll
                for (int r = 0; r < B; ++r) st[r * B + j] = F[r];
            }
            cplx A2[B];                                  // column j of S_{js,jn}
#pragma unroll
            for (int t = 0; t < B; ++t) A2[t] = dir > 0 ? o[t * B + jc] : o[jc * B + t];
            __syncwarp();
#pragma unroll
            for (int r = 0; r < B; ++r) {
                cplx acc = cmake(0.0, 0.0);
#pragma unroll
                for (int t = 0; t < B; ++t) acc = cfms(st[r * B + t], A2[t], acc);
                if (act && real) Prop[(size_t)js * BBc + r * B + j] = acc;
            }
        }
    }
    if (bad && real && j == 0) atomicOr(a.status, 2);
}

// Corner blocks tp = G_l[(last,.),(first,kap)] (hp_leaf_corner_tp), warp -> (strip, inner leaf), lane kap < B walks
// the leaf with the backward propagators, which all 32 lanes stage in shared memory one block row ahead.
template <int B>
__global__ void __launch_bounds__(128) hp_corner_warp_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B;
    __shared__ cplx s_m[4][2][BBc];
    __shared__ cplx s_is2c[4][B];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int P = a.lay.P, n = a.c.n;
    const int w = blockIdx.x * 4 + wib;
    if (w >= a.nb * (P - 2)) return;
    const int l = 1 + w % (P - 2), lb = w / (P - 2);
    const int m = a.m0 + lb, i0 = a.leaf_start[l] + 1, q = a.leaf_q[l];
    const cplx* Binv = a.Binv + (size_t)lb * n * BBc;
    const cplx ih2 = cmake(1.0 / (a.c.pml.h * a.c.pml.h), 0.0);
    const bool act = lane < B;
    const int kap = act ? lane : 0;
    if (act) s_is2c[wib][lane] = hp_lane_strip_row(lane, m, B, a.c.pml).is2c;
    constexpr int MR = (BBc + 31) / 32;
    cplx mreg[MR];
    auto fetch = [&](const cplx* src) {
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = lane + 32 * u; if (e < BBc) mreg[u] = src[e]; }
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = lane + 32 * u; if (e < BBc) s_m[wib][buf][e] = mreg[u]; }
    };
    cplx x[B];
    const cplx* B0 = Binv + (size_t)(i0 - 1) * BBc;
#pragma unroll
    for (int r = 0; r < B; ++r) x[r] = B0[r * B + kap];
    if (q > 1) { fetch(Binv + (size_t)i0 * BBc); stash(1); }
    __syncwarp();
    for (int col = 1; col < q; ++col) {
        const int i = i0 + col;
        if (col + 1 < q) fetch(Binv + (size_t)i * BBc);
        const cplx* M = s_m[wib][col & 1];
        const cplx dscale = cmul(ih2, a.c.s1t[2 * i - 1]);
        cplx t[B], y[B];
#pragma unroll
        for (int k = 0; k < B; ++k) t[k] = cmul(cmul(dscale, s_is2c[wib][k]), x[k]);
#pragma unroll
        for (int r = 0; r < B; ++r) {
            cplx acc = cmake(0.0, 0.0);
#pragma unroll
            for (int k = 0; k < B; ++k) acc = cfms(M[r * B + k], t[k], acc);
            y[r] = acc;
        }
#pragma unroll
        for (int r = 0; r < B; ++r) x[r] = y[r];
        if (col + 1 < q) stash((col + 1) & 1);
        __syncwarp();
    }
    if (act) {
        cplx* tp = a.tp + ((size_t)lb * P + l) * BBc;
#pragma unroll
        for (int r = 0; r < B; ++r) tp[r * B + kap] = x[r];
    }
}

// The same walk with two inner leaves per warp (half-warp -> leaf, lane kap < B of the half -> source row): 24 of 32
// lanes carry a product instead of 12.  Each half stages its own propagators (its leaf, possibly one block row shorter
// than the other's) with 16 lanes; the loop runs to the longer leaf with warp-wide syncs.
template <int B>
__global__ void __launch_bounds__(128) hp_corner_half_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B;
    __shared__ cplx s_m[8][2][BBc];
    __shared__ cplx s_is2c[8][B];
    const int lane = threadIdx.x & 31, hw = threadIdx.x >> 4, j = lane & 15;
    const int P = a.lay.P, n = a.c.n;
    const int total = a.nb * (P - 2);
    const int t = blockIdx.x * 8 + hw;
    const bool real = t < total;                          // the idle half of the last warp follows the last leaf, without storing
    const int tt = real ? t : total - 1;
    const int l = 1 + tt % (P - 2), lb = tt / (P - 2);
    const int m = a.m0 + lb, i0 = a.leaf_start[l] + 1, q = a.leaf_q[l];
    const cplx* Binv = a.Binv + (size_t)lb * n * BBc;
    const cplx ih2 = cmake(1.0 / (a.c.pml.h * a.c.pml.h), 0.0);
    const bool act = j < B;
    const int kap = act ? j : 0;
    if (act) s_is2c[hw][j] = hp_lane_strip_row(j, m, B, a.c.pml).is2c;
    constexpr int MR = (BBc + 15) / 16;
    cplx mreg[MR];
    auto fetch = [&](const cplx* src) {
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = j + 16 * u; if (e < BBc) mreg[u] = src[e]; }
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int u = 0; u < MR; ++u) { const int e = j + 16 * u; if (e < BBc) s_m[hw][buf][e] = mreg[u]; }
    };
    cplx x[B];
    const cplx* B0 = Binv + (size_t)(i0 - 1) * BBc;
#pragma unroll
    for (int r = 0; r < B; ++r) x[r] = B0[r * B + kap];
    if (q > 1) { fetch(Binv + (size_t)i0 * BBc); stash(1); }
    const int qmax = max(q, __shfl_xor_sync(0xffffffffu, q, 16));
    __syncwarp();
    for (int col = 1; col < qmax; ++col) {
        const int i = i0 + col;
        const bool on = col < q;
        if (on && col + 1 < q) fetch(Binv + (size_t)i * BBc);
        if (on) {
            const cplx* M = s_m[hw][col & 1];
            const cplx dscale = cmul(ih2, a.c.s1t[2 * i - 1]);
            cplx tv[B], y[B];
#pragma unroll
            for (int k = 0; k < B; ++k) tv[k] = cmul(cmul(dscale, s_is2c[hw][k]), x[k]);
#pragma unroll
            for (int r = 0; r < B; ++r) {
                cplx acc = cmake(0.0, 0.0);
#pragma unroll
                for (int k = 0; k < B; ++k) acc = cfms(M[r * B + k], tv[k], acc);
                y[r] = acc;
            }
#pragma unroll
            for (int r = 0; r < B; ++r) x[r] = y[r];
        }
        if (on && col + 1 < q) stash((col + 1) & 1);
        __syncwarp();
    }
    if (act && real) {
        cplx* tp = a.tp + ((size_t)lb * P + l) * BBc;
#pragma unroll
        for (int r = 0; r < B; ++r) tp[r * B + kap] = x[r];
    }
}

// thread -> (strip, separator)
template <int BB>
__global__ void __launch_bounds__(64) hp_sep_diaginv_kernel(HpSetupArgs a) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int ns = a.lay.P - 1, bb = a.c.b * a.c.b;
    if (t >= a.nb * ns) return;
    size_t o = (size_t)t * bb;
    if (hp_sep_diag_inverse<BB>(a.Njj + o, a.FX + o, a.BX + o, a.Sd + o, a.c.b)) atomicOr(a.status, 4);
}

// thread -> (strip, separator, component): one row of N (= column, N is symmetric).  Classic layout: written as a row
// into the packet of the CTA that owns it.  Cluster layout: column (j, kap) belongs to cluster j, rows distributed over
// its CTAs, Np[kap][NRQ] column major.
__global__ void __launch_bounds__(128) hp_sep_rows_kernel(HpSetupArgs a, cplx* rowbuf) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    int ns = a.lay.P - 1, b = a.c.b, bb = b * b;
    if (t >= a.nb * ns * b) return;
    int kap = t % b, j = (t / b) % ns, lb = t / (b * ns);
    int row = j * b + kap;
    size_t o = (size_t)lb * ns * bb;
    if (!a.lay.colN) {
        cplx* pk = hp_packet(a, lb, row / a.lay.NR);
        cplx* nrow = pk + a.lay.offN + (size_t)(row % a.lay.NR) * a.lay.NSP;
        hp_sep_row(nrow, a.Njj + o, a.PF + o, a.PB + o, ns, j, kap, b);
    } else {
        cplx* nrow = rowbuf + (size_t)t * a.lay.NSP;
        hp_sep_row(nrow, a.Njj + o, a.PF + o, a.PB + o, ns, j, kap, b);
        const int NRQ = a.lay.NRQ;
        for (int i = 0; i < a.lay.NS; ++i) {
            cplx* pk = hp_packet(a, lb, j * a.lay.K + i / NRQ);
            pk[a.lay.offN + (size_t)kap * NRQ + (i % NRQ)] = nrow[i];
        }
    }
}

// Cluster layout, compile-time b: the same rows of N (hp_sep_row) written straight into the packets.  Column (j, kap)
// of N is contiguous in the packet of its CTA (Np[kap][NRQ]), so the b entries a thread forms per separator are one run of
// b*16 bytes; the generic kernel above goes through a row buffer and a scatter loop (two more passes over N with
// 16-byte accesses 6 KB apart).
template <int B>
__global__ void __launch_bounds__(128) hp_sep_rows_direct_kernel(HpSetupArgs a) {
    constexpr int BBc = B * B;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int ns = a.lay.P - 1;
    if (t >= a.nb * ns * B) return;
    const int kap = t % B, j = (t / B) % ns, lb = t / (B * ns);
    const size_t o = (size_t)lb * ns * BBc;
    const cplx* Njj = a.Njj + o + (size_t)j * BBc;
    const cplx* PF = a.PF + o;
    const cplx* PB = a.PB + o;
    const int NRQ = a.lay.NRQ, K = a.lay.K;
    cplx* pk0 = hp_packet(a, lb, j * K) + a.lay.offN + (size_t)kap * NRQ;     // part 0 of cluster j, column kap
    const size_t pstride = a.lay.PK;                                            // next CTA of the cluster
    auto store = [&](int i, cplx v) { const int part = i / NRQ; pk0[(size_t)part * pstride + (i - part * NRQ)] = v; };
    cplx x0[B], x[B], y[B];
#pragma unroll
    for (int r = 0; r < B; ++r) { x0[r] = Njj[r * B + kap]; store(j * B + r, x0[r]); }
#pragma unroll
    for (int r = 0; r < B; ++r) x[r] = x0[r];
    for (int jj = j - 1; jj >= 0; --jj) {
        const cplx* M = PF + (size_t)jj * BBc;
#pragma unroll
        for (int r = 0; r < B; ++r) {
            cplx acc = cmake(0.0, 0.0);
#pragma unroll
            for (int k = 0; k < B; ++k) acc = cfma(M[r * B + k], x[k], acc);
            y[r] = acc;
        }
#pragma unroll
        for (int r = 0; r < B; ++r) { x[r] = y[r]; store(jj * B + r, y[r]); }
    }
#pragma unroll
    for (int r = 0; r < B; ++r) x[r] = x0[r];
    for (int jj = j + 1; jj < ns; ++jj) {
        const cplx* M = PB + (size_t)jj * BBc;
#pragma unroll
        for (int r = 0; r < B; ++r) {
            cplx acc = cmake(0.0, 0.0);
#pragma unroll
            for (int k = 0; k < B; ++k) acc = cfma(M[r * B + k], x[k], acc);
            y[r] = acc;
        }
#pragma unroll
        for (int r = 0; r < B; ++r) { x[r] = y[r]; store(jj * B + r, y[r]); }
    }
}

// Separator recurrence rows of the cluster sweep kernel (csrc/hp_sweep4.cu).  With x3 = [x_{j-1}; x_j; x_{j+1}] of the
// previous strip of the sweep, rho_j(t) = rho_b(t) - R_j(t) x3(t-1),
//   R_j[i][0..b)   = M_j[b+i][kap]                                   (gl of leaf j from x_{j-1})
//   R_j[i][b..2b)  = M_j[b+i][b+kap] + M_{j+1}[i][kap] + cs_j [i = kap = b-1]
//   R_j[i][2b..3b) = M_{j+1}[i][b+kap]                               (gf of leaf j+1 from x_{j+1})
// M_l[r][c] = mleaf_l[c*2b + r]; cs_j = coupling of the separator column between the two grid rows of the pair.
// rsep[((m-m_lo)*2 + dir)*(P-1) + j][b][3b].  CTA -> (strip, dir, j).
__global__ void __launch_bounds__(128) hp_rsep_kernel(const cplx* __restrict__ mleaf, HpLayout lay, const int* __restrict__ sep,
        int m_lo, int m_hi, int b, double ih2, const cplx* __restrict__ s2t, const cplx* __restrict__ is1t,
        cplx* __restrict__ rsep) {
    const int ns = lay.P - 1, b2 = 2 * b, b3 = 3 * b;
    const int j = blockIdx.x % ns, dir = (blockIdx.x / ns) & 1, mi = blockIdx.x / (2 * ns);
    const int m = m_lo + mi, mprev = dir == 0 ? m - 1 : m + 1;
    if (mprev < m_lo || mprev > m_hi) return;                     // stays zero (first strip of a sweep: not used)
    const cplx* Mj = mleaf + ((size_t)(mi * 2 + dir) * lay.P + j) * b2 * b2;
    const cplx* Mj1 = Mj + (size_t)b2 * b2;
    const cplx cs = cmul(cscale(ih2, s2t[2 * (dir == 0 ? m - 1 : m) + 1]), is1t[2 * (sep[j] + 1)]);
    cplx* out = rsep + ((size_t)(mi * 2 + dir) * ns + j) * b * b3;
    for (int e = threadIdx.x; e < b * b3; e += blockDim.x) {
        const int i = e / b3, c = e - i * b3, blk = c / b, kap = c - blk * b;
        cplx v;
        if (blk == 0) v = Mj[(size_t)kap * b2 + b + i];
        else if (blk == 1) {
            v = cadd(Mj[(size_t)(b + kap) * b2 + b + i], Mj1[(size_t)kap * b2 + i]);
            if (i == b - 1 && kap == b - 1) v = cadd(v, cs);
        } else v = Mj1[(size_t)(b + kap) * b2 + i];
        out[e] = v;
    }
}

// Transfer matrices of the pipelined sweep kernel (csrc/hp_sweep.cu).  The interface data of strip m is linear
// in the separator solution x of the previous strip of the sweep:  g_l(m) = gb_l(m) + M_l(m) [x_left; x_right],
//   M_l(m)[kap'][kap] = sum_c Gc(m)[kap'][c] coef[c] Gc(mprev)[kap][c],   Gc = [Gf; Gl] of leaf l,
//   forward  (dir 0): mprev = m-1, coef[c] = A_{m,m-1}[c]   (couples grid rows m-1, m)
//   backward (dir 1): mprev = m+1, coef[c] = A_{m,m+1}[c]   (couples grid rows m, m+1)
// stored transposed, mleaf[((m-m_lo)*2 + dir)*P + l][kap][kap'], so that lanes over kap' read contiguously.
// CTA -> (strip, dir, leaf); both G blocks are staged in shared memory.
__global__ void __launch_bounds__(256) hp_mleaf_kernel(const cplx* __restrict__ packets, HpLayout lay,
        const int* __restrict__ leaf_start, const int* __restrict__ leaf_q, int m_lo, int m_hi, int b, double ih2,
        const cplx* __restrict__ s2t, const cplx* __restrict__ is1t, cplx* __restrict__ mleaf) {
    extern __shared__ double2 sm[];
    const int l = blockIdx.x % lay.P, dir = (blockIdx.x / lay.P) & 1, mi = blockIdx.x / (2 * lay.P);
    const int m = m_lo + mi, mprev = dir == 0 ? m - 1 : m + 1;
    if (mprev < m_lo || mprev > m_hi) return;                     // stays zero (never used: first strip of a sweep)
    const int q = leaf_q[l], K = lay.K, b2 = 2 * b, ls = leaf_start[l];
    cplx* Ga = sm;                       // [2b][q]  Gc(m)
    cplx* Gb = sm + (size_t)b2 * lay.QP; // [2b][q]  coef * Gc(mprev)
    const cplx rf = cscale(ih2, s2t[2 * (dir == 0 ? m - 1 : m) + 1]);
    for (int e = threadIdx.x; e < b2 * q; e += blockDim.x) {
        int kap = e / q, c = e - kap * q;
        int k = ((c + 1) * K - 1) / q, lc0 = (q * k) / K;
        size_t off = (size_t)(l * K + k) * lay.PK + lay.offG + (size_t)kap * lay.CW + (c - lc0);
        Ga[kap * lay.QP + c] = packets[(size_t)(m - m_lo) * lay.G * lay.PK + off];
        cplx coef = cmul(rf, is1t[2 * (ls + c + 1)]);
        Gb[kap * lay.QP + c] = cmul(coef, packets[(size_t)(mprev - m_lo) * lay.G * lay.PK + off]);
    }
    __syncthreads();
    cplx* out = mleaf + ((size_t)(mi * 2 + dir) * lay.P + l) * b2 * b2;
    for (int e = threadIdx.x; e < b2 * b2; e += blockDim.x) {
        int kap = e / b2, kapp = e - kap * b2;                    // out[kap][kap']
        cplx acc = cmake(0.0, 0.0);
        const cplx* ga = Ga + kapp * lay.QP;
        const cplx* gb = Gb + kap * lay.QP;
        for (int c = 0; c < q; ++c) acc = cfma(ga[c], gb[c], acc);
        out[e] = acc;
    }
}

// ------------------------------------------------------------------------------------------------------
// partition
// ------------------------------------------------------------------------------------------------------
static void hp_fill_layout(HpLayout& L, int n, int b, int P, int K, int colN) {
    int inner = n - (P - 1);
    L = HpLayout();
    L.P = P; L.K = K; L.G = P * K;
    int qmax = (inner + P - 1) / P;
    L.QP = qmax | 1;                       // row strides are odd numbers of 16-byte entries: a quarter warp that
    L.CW = ((qmax + K - 1) / K) | 1;       // reads 8 consecutive rows of Wp / Gp in shared memory hits 8 bank groups
    L.NS = b * (P - 1);
    L.NSP = L.NS > 0 ? L.NS : 1;
    L.NR = L.NS > 0 ? (L.NS + L.G - 1) / L.G : 0;
    L.offG = (size_t)L.CW * L.QP;
    L.offN = L.offG + (size_t)2 * b * L.CW;
    L.colN = colN;
    L.NCB = (b + K - 1) / K;
    L.NRQ = L.NS > 0 ? (L.NS + K - 1) / K : 0;
    L.NXG = (3 * b + K - 1) / K;
    L.PK = L.offN + (colN ? (size_t)b * L.NRQ : (size_t)L.NR * L.NSP);
}

// Choose (P, K): the sweep streams one packet per CTA and strip, so the per-CTA packet size is the time per strip;
// among the candidates that fit in memory take the smallest packet.
//   cluster layout (csrc/hp_sweep4.cu): a leaf is a cluster of K <= 4 CTAs, all P clusters must be co-resident;
//   classic layout (csrc/hp_sweep.cu, hp_sweep2.cu): G = P*K <= #SMs.
// layout_mode: 0 automatic (cluster when a partition exists), 1 classic, 2 cluster.
static int hp_choose_layout(hp_solver* s, int nstrips, int P_req, int K_req, HpLayout& best) {
    const int n = s->n, b = s->b, sms = s->num_sms;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    double budget = 0.80 * (double)free_b;
    bool found = false;
    if (s->layout_mode != 1) {
        for (int K = 1; K <= 8; ++K) {
            if (K_req > 0 ? K != K_req : (K != 1 && K != 2 && K != 4)) continue;
            int Pmin = P_req > 0 ? P_req : 1, Pmax = P_req > 0 ? P_req : std::min(std::min(sms / K, 32 * HP4_PL + 1), (n + 1) / 2);
            for (int P = Pmax; P >= Pmin; --P) {
                int inner = n - (P - 1);
                if (inner < P || inner / P < K) continue;
                HpLayout L;
                hp_fill_layout(L, n, b, P, K, 1);
                if (found && L.PK >= best.PK) continue;
                double bytes = (double)nstrips * (L.G * L.PK + (size_t)2 * (P - 1) * b * 3 * b) * sizeof(cplx);
                if (bytes > budget) continue;
                if (hp_sweep4_max_clusters(L, b) < P) continue;      // shared-memory plan + co-residency of all clusters
                best = L; found = true;
            }
        }
        if (found) return 0;
        if (s->layout_mode == 2) {
            hp_set_error("hp_precond_setup: no cluster partition of n=%d, b=%d (P=%d, K=%d requested) fits", n, b, P_req, K_req);
            return 1;
        }
    }
    int Pmin = P_req > 0 ? P_req : 1, Pmax = P_req > 0 ? P_req : std::min(sms, (n + 1) / 2);
    for (int P = Pmin; P <= Pmax; ++P) {
        int inner = n - (P - 1);
        if (inner < P) break;
        int qmin = inner / P;
        int K = K_req > 0 ? K_req : std::min(sms / P, qmin);
        if (K < 1 || K > qmin || P * K > sms) continue;
        HpLayout L;
        hp_fill_layout(L, n, b, P, K, 0);
        if (L.QP > 1024) continue;
        double bytes = (double)nstrips * L.G * L.PK * sizeof(cplx);
        if (bytes > budget) continue;
        if (!found || L.PK < best.PK) { best = L; found = true; }
    }
    if (!found) {
        hp_set_error("hp_precond_setup: no leaf/separator partition of n=%d, b=%d (P=%d, K=%d requested) fits "
                     "%d strips in %.1f GB of free device memory on %d SMs", n, b, P_req, K_req, nstrips,
                     (double)free_b / 1e9, sms);
        return 1;
    }
    return 0;
}

void hp_free_strips(hp_solver* s) {
    cudaFree(s->packets); s->packets = nullptr;
    cudaFree(s->mleaf); s->mleaf = nullptr;
    cudaFree(s->rsep); s->rsep = nullptr;
    cudaFree(s->leaf_start); s->leaf_start = nullptr;
    cudaFree(s->leaf_q); s->leaf_q = nullptr;
    cudaFree(s->sep); s->sep = nullptr;
    cudaFree(s->xch); s->xch = nullptr;
    cudaFree(s->bar); s->bar = nullptr;
    s->m_lo = 0; s->m_hi = -1; s->bytes = 0;
    for (int i = 0; i < 9; ++i) s->multi_ok[i] = 0;
    s->dmma_ok = 0;
}

// developer trace (HP_SETUP_TRACE=1): wall-clock milliseconds since the start of hp_setup_strips at the named points
struct HpTrace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    HpTrace() : on(getenv("HP_SETUP_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what, cudaStream_t st, bool sync) {
        if (!on) return;
        if (sync) cudaStreamSynchronize(st);
        double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        fprintf(stderr, "[hp_setup] %9.2f ms  %s\n", ms, what);
    }
};

int hp_setup_strips(hp_solver* s, int P_req, int K_req, int m_lo, int m_hi, cudaStream_t st) {
    HpTrace tr;
    const int n = s->n, b = s->b, bb = b * b;
    const bool ck = s->kappa_c != nullptr;                 // attenuating medium: the complex-kappa instances of the chains
    if (ck && (getenv("HP_CHAIN_THREAD") || getenv("HP_CHAIN_UNROLL"))) {
        hp_set_error("hp_precond_setup: the setup generations selected by HP_CHAIN_THREAD / HP_CHAIN_UNROLL support real media only");
        return 1;
    }
    hp_free_strips(s);
    const int nstrips = m_hi - m_lo + 1;
    HpLayout L;
    if (hp_choose_layout(s, nstrips, P_req, K_req, L)) return 1;
    s->lay = L;
    const int P = L.P, ns = P - 1;
    // leaves and separators (same arithmetic as tools/strip_model.py::partition)
    s->leaf_start_h.assign(P, 0); s->leaf_q_h.assign(P, 0); s->sep_h.assign(std::max(ns, 1), 0);
    {
        long inner = n - ns;
        int pos = 0;
        for (int l = 0; l < P; ++l) {
            int q = (int)((inner * (l + 1)) / P - (inner * l) / P);
            s->leaf_start_h[l] = pos; s->leaf_q_h[l] = q;
            pos += q;
            if (l < P - 1) { s->sep_h[l] = pos; pos += 1; }
        }
    }
    HP_CUDA(cudaMalloc(&s->leaf_start, sizeof(int) * P));
    HP_CUDA(cudaMalloc(&s->leaf_q, sizeof(int) * P));
    HP_CUDA(cudaMalloc(&s->sep, sizeof(int) * std::max(ns, 1)));
    HP_CUDA(cudaMemcpyAsync(s->leaf_start, s->leaf_start_h.data(), sizeof(int) * P, cudaMemcpyHostToDevice, st));
    HP_CUDA(cudaMemcpyAsync(s->leaf_q, s->leaf_q_h.data(), sizeof(int) * P, cudaMemcpyHostToDevice, st));
    HP_CUDA(cudaMemcpyAsync(s->sep, s->sep_h.data(), sizeof(int) * std::max(ns, 1), cudaMemcpyHostToDevice, st));
    size_t pbytes = (size_t)nstrips * L.G * L.PK * sizeof(cplx);
    tr.mark("layout chosen", st, true);
    HP_CUDA(cudaMalloc(&s->packets, pbytes));
    if (L.colN && ns > 0) HP_CUDA(cudaMalloc(&s->rsep, (size_t)nstrips * 2 * ns * b * 3 * b * sizeof(cplx)));
    tr.mark("packets allocated", st, false);
    HP_CUDA(cudaMemsetAsync(s->packets, 0, pbytes, st));
    tr.mark("packets cleared", st, true);
    size_t xch_classic = (size_t)n + (size_t)L.G * 2 * b + (size_t)L.P * 2 * b + L.NSP + L.P;
    size_t xch_cluster = ((size_t)L.G * b + (size_t)std::max(L.NS, 1) * (L.P | 1)) * 8;   // x HP_RMAX right-hand sides per launch
    s->xch_count = 4 * std::max(xch_classic, xch_cluster);
    s->bar_count = (size_t)(4 + L.P);
    HP_CUDA(cudaMalloc(&s->xch, sizeof(cplx) * s->xch_count));
    HP_CUDA(cudaMalloc(&s->bar, sizeof(unsigned int) * s->bar_count));
    HP_CUDA(cudaMemsetAsync(s->bar, 0, sizeof(unsigned int) * s->bar_count, st));
    s->m_lo = m_lo; s->m_hi = m_hi;
    s->bytes = (int64_t)pbytes;

    // batch size from the scratch footprint
    size_t per_strip = ((size_t)n * bb * 2 + (size_t)n * b + (size_t)P * bb + (size_t)9 * std::max(ns, 1) * bb +
                        (L.colN ? (size_t)L.NS * L.NSP : 0)) * sizeof(cplx);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    size_t cap_gb = 8;                                     // scratch budget (measured: 8 and 64 GB give the same kernel time, and freeing a large scratch costs wall time); HP_SCRATCH_GB overrides
    if (const char* e = getenv("HP_SCRATCH_GB")) cap_gb = (size_t)std::max(1, atoi(e));
    size_t cap = std::min<size_t>((size_t)(0.5 * (double)free_b), cap_gb << 30);
    int LB = (int)std::max<size_t>(1, std::min<size_t>((size_t)nstrips, cap / per_strip));
    HpSetupArgs a;
    a.c = hp_ctx(s); a.lay = L; a.leaf_start = s->leaf_start; a.leaf_q = s->leaf_q; a.sep = s->sep;
    a.m_lo = m_lo; a.packets = s->packets; a.status = s->status;
    a.leaf_piped = getenv("HP_LEAF_NOPIPE") ? 0 : 1;
    // released on every exit path
    struct Guard {
        hp_solver* s; cplx* scratch = nullptr; cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Guard() {
            if (e0) cudaEventDestroy(e0);
            if (e1) cudaEventDestroy(e1);
            if (scratch && s->mleaf == scratch) s->mleaf = nullptr;     // the transfer matrices lived in the scratch
            cudaFree(scratch);
        }
    } guard{s};
    cplx*& scratch = guard.scratch;
    cplx* rowbuf = nullptr;
    HP_CUDA(cudaMalloc(&scratch, per_strip * LB));
    tr.mark("scratch allocated", st, false);
    {
        cplx* p = scratch;
        a.Finv = p; p += (size_t)LB * n * bb;
        a.Binv = p; p += (size_t)LB * n * bb;
        a.gcol = p; p += (size_t)LB * n * b;
        a.tp = p; p += (size_t)LB * P * bb;
        size_t sz = (size_t)LB * std::max(ns, 1) * bb;
        a.Sd = p; p += sz; a.So = p; p += sz; a.FX = p; p += sz; a.FXi = p; p += sz; a.PF = p; p += sz;
        a.BX = p; p += sz; a.BXi = p; p += sz; a.PB = p; p += sz; a.Njj = p; p += sz;
        rowbuf = p;
    }
    HP_CUDA(cudaEventCreate(&guard.e0)); HP_CUDA(cudaEventCreate(&guard.e1));
    cudaEvent_t e0 = guard.e0, e1 = guard.e1;
    cudaEventRecord(e0, st);
    const int leaf_threads = ((L.QP + 31) / 32) * 32;
    const bool small_b = b <= 12;                          // thread-local b x b matrices sized 144 instead of HP_BMAX^2
    // warp-cooperative Schur chains: as many warps per block as fit in ~100 KB of shared memory (two blocks per SM)
    const size_t chain_per_warp = sizeof(cplx) * ((size_t)4 * bb + 6 * b + 16);
    int chain_wpb = (int)std::min<size_t>(8, (100 * 1024) / chain_per_warp);
    if (getenv("HP_CHAIN_THREAD")) chain_wpb = 0;          // developer switch: the one-thread-per-chain kernel
    const size_t chain_smem = chain_per_warp * (size_t)std::max(chain_wpb, 1);
    if (chain_wpb > 0 && chain_smem > 48 * 1024)
        HP_CUDA(cudaFuncSetAttribute(ck ? hp_chain_warp_kernel<true> : hp_chain_warp_kernel<false>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chain_smem));
    for (int m0 = m_lo; m0 <= m_hi; m0 += LB) {
        a.m0 = m0;
        a.nb = std::min(LB, m_hi - m0 + 1);
        int t1 = a.nb * P * 2;
        hp_count_launch();
        if (chain_wpb > 0 && b == 12 && !getenv("HP_CHAIN_SMEM")) {
            if (getenv("HP_CHAIN_UNROLL")) hp_chain_reg_kernel<12, false><<<(a.nb * P + 3) / 4, 128, 0, st>>>(a);
            else if (ck) hp_chain_reg_kernel<12, true, true><<<(a.nb * P + 3) / 4, 128, 0, st>>>(a);
            else hp_chain_reg_kernel<12, true><<<(a.nb * P + 3) / 4, 128, 0, st>>>(a);        // one warp per leaf: both chains
        } else if (chain_wpb > 0) {
            if (ck) hp_chain_warp_kernel<true><<<(t1 + chain_wpb - 1) / chain_wpb, 32 * chain_wpb, chain_smem, st>>>(a, chain_wpb);
            else hp_chain_warp_kernel<false><<<(t1 + chain_wpb - 1) / chain_wpb, 32 * chain_wpb, chain_smem, st>>>(a, chain_wpb);
        } else if (small_b) hp_chain_kernel<144><<<(t1 + 63) / 64, 64, 0, st>>>(a);
        else hp_chain_kernel<HP_BMAX * HP_BMAX><<<(t1 + 63) / 64, 64, 0, st>>>(a);
        hp_count_launch();
        if (b == 12 && leaf_threads <= 128 && !getenv("HP_CHAIN_THREAD") && !getenv("HP_LEAF_CTA")) hp_leaf_warp_kernel<12><<<a.nb * P, leaf_threads, 0, st>>>(a);
        else if (b == 12 && leaf_threads <= 128 && !getenv("HP_CHAIN_THREAD")) hp_leaf_fast_kernel<12, 128><<<a.nb * P, leaf_threads, 0, st>>>(a);
        else if (b == 12 && leaf_threads <= 256 && !getenv("HP_CHAIN_THREAD")) hp_leaf_fast_kernel<12, 256><<<a.nb * P, leaf_threads, 0, st>>>(a);
        else hp_leaf_kernel<<<a.nb * P, leaf_threads, 0, st>>>(a);
        if (ns > 0) {
            if (P > 2) {
                int t3 = a.nb * P * b;
                hp_count_launch();
                if (b == 12 && !getenv("HP_SETUP_THREAD") && !getenv("HP_CORNER_WARP")) hp_corner_half_kernel<12><<<(a.nb * (P - 2) + 7) / 8, 128, 0, st>>>(a);
                else if (b == 12 && !getenv("HP_SETUP_THREAD")) hp_corner_warp_kernel<12><<<(a.nb * (P - 2) + 3) / 4, 128, 0, st>>>(a);
                else hp_corner_kernel<<<(t3 + 127) / 128, 128, 0, st>>>(a);
            }
            int t4 = a.nb * ns;
            hp_count_launch();
            if (ck) hp_sep_blocks_kernel<true><<<(t4 + 127) / 128, 128, 0, st>>>(a);
            else hp_sep_blocks_kernel<false><<<(t4 + 127) / 128, 128, 0, st>>>(a);
            hp_count_launch();
            if (b == 12 && !getenv("HP_SETUP_THREAD")) hp_sep_chain_half_kernel<12><<<(a.nb * 2 + 7) / 8, 128, 0, st>>>(a);
            else if (small_b) hp_sep_chain_kernel<144><<<(a.nb * 2 + 31) / 32, 32, 0, st>>>(a); else hp_sep_chain_kernel<HP_BMAX * HP_BMAX><<<(a.nb * 2 + 31) / 32, 32, 0, st>>>(a);
            hp_count_launch();
            if (small_b) hp_sep_diaginv_kernel<144><<<(t4 + 63) / 64, 64, 0, st>>>(a); else hp_sep_diaginv_kernel<HP_BMAX * HP_BMAX><<<(t4 + 63) / 64, 64, 0, st>>>(a);
            int t7 = a.nb * ns * b;
            hp_count_launch();
            if (b == 12 && L.colN && !getenv("HP_SEP_ROWS_BUF")) hp_sep_rows_direct_kernel<12><<<(t7 + 127) / 128, 128, 0, st>>>(a);
            else hp_sep_rows_kernel<<<(t7 + 127) / 128, 128, 0, st>>>(a, rowbuf);
        }
        HP_CUDA(cudaGetLastError());
    }
    tr.mark("strip kernels done", st, true);
    {   // transfer matrices of the pipelined sweeps
        size_t mbytes = (size_t)nstrips * 2 * P * 4 * bb * sizeof(cplx);
        // cluster layout: the transfer matrices are only an intermediate of the recurrence rows and live in the scratch of
        // the strip kernels, which are done by now on this stream (an allocation and a free of 2.5 GB at this point cost
        // up to 0.5 s of wall time when the allocator had to return memory first)
        const bool m_in_scratch = L.colN && mbytes <= per_strip * (size_t)LB;
        if (m_in_scratch) s->mleaf = scratch;
        else HP_CUDA(cudaMalloc(&s->mleaf, mbytes));
        HP_CUDA(cudaMemsetAsync(s->mleaf, 0, mbytes, st));
        size_t smem = sizeof(cplx) * 2 * 2 * b * L.QP;
        HP_CUDA(cudaFuncSetAttribute(hp_mleaf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hp_count_launch(); hp_mleaf_kernel<<<nstrips * 2 * P, 256, smem, st>>>(s->packets, L, s->leaf_start, s->leaf_q, m_lo, m_hi, b,
                                                                            1.0 / (s->pml.h * s->pml.h), s->s2t, s->is1t, s->mleaf);
        HP_CUDA(cudaGetLastError());
        if (L.colN) {
            // cluster kernel: the separator recurrence rows replace the per-leaf transfer matrices
            if (ns > 0) {
                size_t rbytes = (size_t)nstrips * 2 * ns * b * 3 * b * sizeof(cplx);
                HP_CUDA(cudaMemsetAsync(s->rsep, 0, rbytes, st));
                hp_count_launch(); hp_rsep_kernel<<<nstrips * 2 * ns, 128, 0, st>>>(s->mleaf, L, s->sep, m_lo, m_hi, b,
                                                                                 1.0 / (s->pml.h * s->pml.h), s->s2t, s->is1t, s->rsep);
                HP_CUDA(cudaGetLastError());
                s->bytes += (int64_t)rbytes;
            }
            HP_CUDA(cudaStreamSynchronize(st));
            if (!m_in_scratch) HP_CUDA(cudaFree(s->mleaf));
            s->mleaf = nullptr;
        } else {
            s->bytes += (int64_t)mbytes;
        }
    }
    cudaEventRecord(e1, st);
    HP_CUDA(cudaStreamSynchronize(st));
    tr.mark("transfer matrices / recurrence rows done", st, false);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    s->setup_ms = ms;
    {
        cplx* p = scratch;
        scratch = nullptr;
        HP_CUDA(cudaFree(p));
    }
    tr.mark("scratch freed", st, false);
    return 0;                                              // the caller (hp_precond_setup) reads the status word
}
