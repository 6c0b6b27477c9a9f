// Per-task setup arithmetic of the strip solves (host/device).
//
// Replaces the reference's algo2_3 (/root/reference/code.py:345-353): instead of a sparse LU of each
// bn x bn strip operator H_m, the strip is treated as a block tridiagonal matrix over the x1 index
// (b x b blocks D_i, diagonal couplings L_i = U_{i-1}) and the restriction
// T_m = (H_m^{-1})[last row, last row] is represented by
//   * P leaves (ranges of consecutive block rows) separated by P-1 single separator block rows;
//     per leaf, samples of the Dirichlet-truncated leaf inverse G_l:
//        W  [q][q]  = G_l[(c,b),(c',b)]
//        Gf [b][q]  = cpl_left  * G_l[(first,k),(c,b)]     Gl [b][q] = cpl_right * G_l[(last,k),(c,b)]
//   * the dense inverse N = S^{-1} of the separator Schur complement S (block tridiagonal, b x b blocks).
// tools/strip_model.py is the numpy model of exactly these arrays.
//
// The functions that hold b x b matrices in thread-local arrays take the array size BB >= b*b as a template parameter
// (144 for the reference's b = 12: a quarter of the local memory of the general HP_BMAX^2 case).
//
// Every function here is the body of ONE thread of a setup kernel (csrc/hp_setup.cu); the loops over
// leaf columns are written so that the lanes of a warp walk the leaf in lock step and read the same
// b x b matrix at the same time (broadcast loads).
#pragma once
#include "hp_small.h"

struct HpStripCtx {
    int n, b;
    HpPml pml;
    cplx omega2;
    const cplx* s1t;      // s1 on the x1 half grid, t = 0..2n+2
    const cplx* is1t;     // 1/s1
    const double* c_mat;  // (n+2) x (n+2), row major, indexed [i-1][j-1] as the reference does
    const cplx* kappa_c = nullptr;   // attenuating medium: n x n complex slowness^2, grid aligned (hp_block_row<true>)
};

// Forward Schur chain of one leaf: Finv[i] = (D_i - L_i Finv[i-1] U_{i-1})^{-1}, i = i0..i1 (1-based,
// inclusive).  out points at this strip's [n][b*b] scratch.
template <int BB = HP_BMAX * HP_BMAX, bool CK = false>
HP_HD int hp_chain_forward(cplx* out, int i0, int i1, int m, const HpStripCtx& c) {
    const int b = c.b, bb = b * b;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    HpBlockRow B;
    cplx Uprev[HP_BMAX];
    cplx F[BB];
    int bad = 0;
    for (int i = i0; i <= i1; ++i) {
        hp_block_row<CK>(B, R, i, m, b, c.n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
        hp_schur_step(F, B, B.L, i > i0 ? out + (size_t)(i - 2) * bb : out, Uprev, b, i > i0);
        bad |= hp_inv_inplace(F, b);
        cplx* dst = out + (size_t)(i - 1) * bb;
        for (int e = 0; e < bb; ++e) dst[e] = F[e];
        for (int k = 0; k < b; ++k) Uprev[k] = B.U[k];
    }
    return bad;
}

// Backward Schur chain Binv[i] = (D_i - U_i Binv[i+1] L_{i+1})^{-1}, i = i1..i0, followed by the
// ascending recurrence for the diagonal blocks of the leaf inverse
//   G_{i0,i0} = Binv[i0],   G_ii = Binv_i + Binv_i L_i G_{i-1,i-1} U_{i-1} Binv_i
// of which only the last column (source in the last strip row) is kept: gcol[i][0..b).
template <int BB = HP_BMAX * HP_BMAX, bool CK = false>
HP_HD int hp_chain_backward(cplx* out, cplx* gcol, int i0, int i1, int m, const HpStripCtx& c) {
    const int b = c.b, bb = b * b;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    HpBlockRow B;
    cplx Lnext[HP_BMAX];
    cplx F[BB];
    int bad = 0;
    for (int i = i1; i >= i0; --i) {
        hp_block_row<CK>(B, R, i, m, b, c.n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
        hp_schur_step(F, B, B.U, i < i1 ? out + (size_t)i * bb : out, Lnext, b, i < i1);
        bad |= hp_inv_inplace(F, b);
        cplx* dst = out + (size_t)(i - 1) * bb;
        for (int e = 0; e < bb; ++e) dst[e] = F[e];
        for (int k = 0; k < b; ++k) Lnext[k] = B.L[k];
    }
    // diagonal blocks, ascending; only the last column g_i = G_ii[:, b-1] is propagated:
    //   g_i = Binv_i e + Binv_i L_i G_{i-1,i-1} U_{i-1} Binv_i e   needs the full G_{i-1,i-1}, so the
    //   full block is carried in G.
    cplx* G = F;
    cplx T1[BB], T2[BB];
    cplx Uprev[HP_BMAX];
    for (int i = i0; i <= i1; ++i) {
        const cplx* Bi = out + (size_t)(i - 1) * bb;
        hp_block_row<CK>(B, R, i, m, b, c.n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
        if (i == i0) {
            for (int e = 0; e < bb; ++e) G[e] = Bi[e];
        } else {
            for (int r = 0; r < b; ++r)
                for (int s = 0; s < b; ++s) T1[r * b + s] = cmul(cmul(B.L[r], G[r * b + s]), Uprev[s]);
            hp_gemm(T2, Bi, T1, b, b, b, b, b, b, +1, 0);
            for (int e = 0; e < bb; ++e) G[e] = Bi[e];
            hp_gemm(G, T2, Bi, b, b, b, b, b, b, +1, 1);
        }
        for (int k = 0; k < b; ++k) gcol[(size_t)(i - 1) * b + k] = G[k * b + (b - 1)];
        for (int k = 0; k < b; ++k) Uprev[k] = B.U[k];
    }
    return bad;
}

// x <- -M (d * x)  with M b x b row major, d a diagonal; y is scratch
HP_HD void hp_propagate(cplx* x, const cplx* M, cplx dscale, const cplx* is2c, int b) {
    cplx t[HP_BMAX], y[HP_BMAX];
    for (int k = 0; k < b; ++k) t[k] = cmul(cmul(dscale, is2c[k]), x[k]);
    for (int a = 0; a < b; ++a) {
        cplx acc = cmake(0.0, 0.0);
        for (int k = 0; k < b; ++k) acc = cfms(M[a * b + k], t[k], acc);
        y[a] = acc;
    }
    for (int a = 0; a < b; ++a) x[a] = y[a];
}

// Column r (0-based inside the leaf, r < q) of the leaf generators.  The leaf covers block rows
// i0..i0+q-1 (1-based).  Writes row r of W (wrow[0..q), W is symmetric), column r of Gf/Gl
// (gf[k*gstride], gl[k*gstride]).  has_left/has_right: a separator exists on that side, the coupling
// across the cut is folded into Gf/Gl; otherwise zeros are stored.  qloop >= q is the lock-step trip
// count (the widest leaf), so that all lanes of a warp run the same loop.
HP_HD void hp_leaf_column(cplx* wrow, cplx* gf, cplx* gl, size_t gstride, const cplx* Finv, const cplx* Binv,
                          const cplx* gcol, int i0, int q, int qloop, int r, int m, int has_left, int has_right,
                          const HpStripCtx& c) {
    const int b = c.b, bb = b * b;
    const bool live = r < q;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    const cplx ih2 = cmake(1.0 / (c.pml.h * c.pml.h), 0.0);
    cplx x0[HP_BMAX], x[HP_BMAX];
    for (int k = 0; k < b; ++k) x0[k] = live ? gcol[(size_t)(i0 - 1 + r) * b + k] : cmake(0.0, 0.0);
    if (live) wrow[r] = x0[b - 1];
    // leftwards: x_col = -Finv[col] U_col x_{col+1},  U_i[k] = s1((i+.5)h) / (h^2 s2m(j_k h))
    for (int k = 0; k < b; ++k) x[k] = x0[k];
    for (int col = qloop - 2; col >= 0; --col) {
        if (live && col < r) {
            int i = i0 + col;
            hp_propagate(x, Finv + (size_t)(i - 1) * bb, cmul(ih2, c.s1t[2 * i + 1]), R.is2c, b);
            wrow[col] = x[b - 1];
        }
    }
    if (live) {
        cplx sc = cmul(ih2, c.s1t[2 * i0 - 1]);            // L_{i0}[k] = s1((i0-.5)h)/(h^2 s2m)
        for (int k = 0; k < b; ++k)
            gf[(size_t)k * gstride] = has_left ? cmul(cmul(sc, R.is2c[k]), x[k]) : cmake(0.0, 0.0);
    }
    // rightwards: x_col = -Binv[col] L_col x_{col-1},  L_i[k] = s1((i-.5)h) / (h^2 s2m(j_k h))
    for (int k = 0; k < b; ++k) x[k] = x0[k];
    for (int col = 1; col < qloop; ++col) {
        if (live && col > r && col < q) {
            int i = i0 + col;
            hp_propagate(x, Binv + (size_t)(i - 1) * bb, cmul(ih2, c.s1t[2 * i - 1]), R.is2c, b);
            wrow[col] = x[b - 1];
        }
    }
    if (live) {
        int it = i0 + q - 1;
        cplx sc = cmul(ih2, c.s1t[2 * it + 1]);            // U_t[k]
        for (int k = 0; k < b; ++k)
            gl[(size_t)k * gstride] = has_right ? cmul(cmul(sc, R.is2c[k]), x[k]) : cmake(0.0, 0.0);
    }
}

// Column kap of the corner block tp = G_l[(last,.),(first,kap)]: start from Binv[i0][:,kap] (= G_pp
// column) and walk right.  out[a] = tp[a][kap], a < b.
HP_HD void hp_leaf_corner_tp(cplx* out, const cplx* Binv, int i0, int q, int qloop, int kap, int m,
                             const HpStripCtx& c) {
    const int b = c.b, bb = b * b;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    const cplx ih2 = cmake(1.0 / (c.pml.h * c.pml.h), 0.0);
    cplx x[HP_BMAX];
    const cplx* B0 = Binv + (size_t)(i0 - 1) * bb;
    for (int a = 0; a < b; ++a) x[a] = B0[a * b + kap];
    for (int col = 1; col < qloop; ++col) {
        if (col < q) {
            int i = i0 + col;
            hp_propagate(x, Binv + (size_t)(i - 1) * bb, cmul(ih2, c.s1t[2 * i - 1]), R.is2c, b);
        }
    }
    for (int a = 0; a < b; ++a) out[a] = x[a];
}

// ---------------------------------------------------------------------------------------------
// Separator Schur complement.  Separator j sits at block row s (1-based); the leaf on its left ends at
// s-1 (corner tt = Finv[s-1]) and the leaf on its right starts at s+1 (corner pp = Binv[s+1]).
//   S_jj     = D_s - L_s tt_left U_{s-1} - U_s pp_right L_{s+1}
//   S_j,j+1  = -U_s pt U_t           with pt = tp^T of the leaf between separators j and j+1 (t = s'-1)
// ---------------------------------------------------------------------------------------------
template <bool CK = false>
HP_HD void hp_sep_diag(cplx* S, int s, int m, const cplx* tt_left, const cplx* pp_right, const HpStripCtx& c) {
    const int b = c.b;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    HpBlockRow B;
    hp_block_row<CK>(B, R, s, m, b, c.n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
    for (int r = 0; r < b; ++r)
        for (int t = 0; t < b; ++t) {
            cplx v = cmake(0.0, 0.0);
            if (r == t) v = B.dia[r];
            else if (t == r - 1) v = B.sub[r];
            else if (t == r + 1) v = B.sup[r];
            // U_{s-1} = L_s and L_{s+1} = U_s
            v = cfms(cmul(B.L[r], tt_left[r * b + t]), B.L[t], v);
            v = cfms(cmul(B.U[r], pp_right[r * b + t]), B.U[t], v);
            S[r * b + t] = v;
        }
}

// S_{j,j+1}[a][c] = -U_s[a] tp[c][a] U_t[c]; s = separator j, s2 = separator j+1 (block rows, 1-based)
HP_HD void hp_sep_offdiag(cplx* So, int s, int s2, int m, const cplx* tp, const HpStripCtx& c) {
    const int b = c.b;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    const cplx ih2 = cmake(1.0 / (c.pml.h * c.pml.h), 0.0);
    cplx us = cmul(ih2, c.s1t[2 * s + 1]), ut = cmul(ih2, c.s1t[2 * s2 - 1]);
    for (int a = 0; a < b; ++a)
        for (int cc = 0; cc < b; ++cc) {
            cplx v = cmul(cmul(cmul(us, R.is2c[a]), tp[cc * b + a]), cmul(ut, R.is2c[cc]));
            So[a * b + cc] = cneg(v);
        }
}

// Forward chain over the separators of one strip (dir = +1) or backward chain (dir = -1):
//   fwd: X_j = S_jj - S_{j,j-1} Xinv_{j-1} S_{j-1,j},  Xinv_j,  Prop_j = -Xinv_j S_{j,j+1}
//   bwd: X_j = S_jj - S_{j,j+1} Xinv_{j+1} S_{j+1,j},  Xinv_j,  Prop_j = -Xinv_j S_{j,j-1}
// Sd [ns][b*b], So [ns-1][b*b] (So[j] = S_{j,j+1}; S_{j+1,j} is its transpose).
// X, Xinv, Prop: [ns][b*b] each.
template <int BB = HP_BMAX * HP_BMAX>
HP_HD int hp_sep_chain(cplx* X, cplx* Xinv, cplx* Prop, const cplx* Sd, const cplx* So, int ns, int dir, int b) {
    const int bb = b * b;
    cplx F[BB], T1[BB], A[BB];
    int bad = 0;
    for (int step = 0; step < ns; ++step) {
        int j = dir > 0 ? step : ns - 1 - step;
        for (int e = 0; e < bb; ++e) F[e] = Sd[(size_t)j * bb + e];
        if (step > 0) {
            int jp = j - dir;                                  // previous separator of the chain
            // A = S_{j,jp}: fwd -> S_{j,j-1} = So[j-1]^T ; bwd -> S_{j,j+1} = So[j]
            const cplx* o = So + (size_t)(dir > 0 ? j - 1 : j) * bb;
            for (int r = 0; r < b; ++r)
                for (int t = 0; t < b; ++t) A[r * b + t] = dir > 0 ? o[t * b + r] : o[r * b + t];
            hp_gemm(T1, A, Xinv + (size_t)jp * bb, b, b, b, b, b, b, +1, 0);       // S_{j,jp} Xinv_jp
            // F -= T1 * S_{jp,j} = T1 * A^T
            for (int r = 0; r < b; ++r)
                for (int t = 0; t < b; ++t) {
                    cplx acc = F[r * b + t];
                    for (int l = 0; l < b; ++l) acc = cfms(T1[r * b + l], A[t * b + l], acc);
                    F[r * b + t] = acc;
                }
        }
        for (int e = 0; e < bb; ++e) X[(size_t)j * bb + e] = F[e];
        bad |= hp_inv_inplace(F, b);
        for (int e = 0; e < bb; ++e) Xinv[(size_t)j * bb + e] = F[e];
        int jn = j + dir;                                      // next separator of the chain
        if (jn >= 0 && jn < ns) {
            // Prop_j = -Xinv_j S_{j,jn}: fwd -> S_{j,j+1} = So[j] ; bwd -> S_{j,j-1} = So[j-1]^T
            const cplx* o = So + (size_t)(dir > 0 ? j : j - 1) * bb;
            for (int r = 0; r < b; ++r)
                for (int t = 0; t < b; ++t) A[r * b + t] = dir > 0 ? o[r * b + t] : o[t * b + r];
            hp_gemm(Prop + (size_t)j * bb, F, A, b, b, b, b, b, b, -1, 0);
        }
    }
    return bad;
}

// N_jj = (FX_j + BX_j - S_jj)^{-1}
template <int BB = HP_BMAX * HP_BMAX>
HP_HD int hp_sep_diag_inverse(cplx* Njj, const cplx* FX, const cplx* BX, const cplx* Sd, int b) {
    cplx F[BB];
    for (int e = 0; e < b * b; ++e) F[e] = csub(cadd(FX[e], BX[e]), Sd[e]);
    int bad = hp_inv_inplace(F, b);
    for (int e = 0; e < b * b; ++e) Njj[e] = F[e];
    return bad;
}

// Row (j, kap) of N (= column, N is symmetric): x_j = N_jj[:, kap]; x_{j'} = PF_{j'} x_{j'+1} upwards,
// x_{j'} = PB_{j'} x_{j'-1} downwards.  nrow[0..ns*b) receives the row.  nsloop >= ns is the lock-step
// trip count.
HP_HD void hp_sep_row(cplx* nrow, const cplx* Njj, const cplx* PF, const cplx* PB, int ns, int j, int kap, int b) {
    const int bb = b * b;
    cplx x0[HP_BMAX], x[HP_BMAX], y[HP_BMAX];
    const cplx* Nj = Njj + (size_t)j * bb;
    for (int a = 0; a < b; ++a) { x0[a] = Nj[a * b + kap]; nrow[(size_t)j * b + a] = x0[a]; }
    for (int a = 0; a < b; ++a) x[a] = x0[a];
    for (int jj = j - 1; jj >= 0; --jj) {
        const cplx* M = PF + (size_t)jj * bb;
        for (int a = 0; a < b; ++a) {
            cplx acc = cmake(0.0, 0.0);
            for (int k = 0; k < b; ++k) acc = cfma(M[a * b + k], x[k], acc);
            y[a] = acc;
        }
        for (int a = 0; a < b; ++a) { x[a] = y[a]; nrow[(size_t)jj * b + a] = y[a]; }
    }
    for (int a = 0; a < b; ++a) x[a] = x0[a];
    for (int jj = j + 1; jj < ns; ++jj) {
        const cplx* M = PB + (size_t)jj * bb;
        for (int a = 0; a < b; ++a) {
            cplx acc = cmake(0.0, 0.0);
            for (int k = 0; k < b; ++k) acc = cfma(M[a * b + k], x[k], acc);
            y[a] = acc;
        }
        for (int a = 0; a < b; ++a) { x[a] = y[a]; nrow[(size_t)jj * b + a] = y[a]; }
    }
}

// coupling between block rows q and q+1 of strip m: U_q[k] = L_{q+1}[k] = 1/h^2 s1((q+.5)h)/s2m(j_k h)
HP_HD void hp_coupling(cplx* cpl, int q, int m, const HpStripCtx& c) {
    HpStripRow R;
    hp_strip_rows(R, m, c.b, c.pml);
    double ih2 = 1.0 / (c.pml.h * c.pml.h);
    cplx s = c.s1t[2 * q + 1];
    for (int k = 0; k < c.b; ++k) cpl[k] = cscale(ih2, cmul(s, R.is2c[k]));
}
