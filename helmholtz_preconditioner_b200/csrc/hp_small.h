// Small complex128 building blocks shared by every kernel of the path.
//
// Everything here is __host__ __device__ so the arithmetic can be exercised on the CPU by
// tests/host_harness.cpp (the build container has no GPU); the kernels call the same code.
//
// Reference being replaced: the numba scalar helpers sigma1/sigma2/s1/s2/s2m
// (/root/reference/code.py:11-37) and the per-point coefficient expressions of
// get_A_diag_block_coeffs / get_Hm_coeffs (code.py:82-113, 237-275).
#pragma once
#include <math.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define HP_HD __host__ __device__ __forceinline__
typedef double2 cplx;
#else
#define HP_HD inline
struct cplx { double x, y; };
#endif

#define HP_BMAX 24   // largest PML width (strip height) the small-matrix code is sized for

HP_HD cplx cmake(double re, double im) { cplx r; r.x = re; r.y = im; return r; }
HP_HD cplx cadd(cplx a, cplx b) { return cmake(a.x + b.x, a.y + b.y); }
HP_HD cplx csub(cplx a, cplx b) { return cmake(a.x - b.x, a.y - b.y); }
HP_HD cplx cneg(cplx a) { return cmake(-a.x, -a.y); }
HP_HD cplx cmul(cplx a, cplx b) { return cmake(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
HP_HD cplx cscale(double s, cplx a) { return cmake(s * a.x, s * a.y); }
// c + a*b
HP_HD cplx cfma(cplx a, cplx b, cplx c) {
    return cmake(fma(-a.y, b.y, fma(a.x, b.x, c.x)), fma(a.y, b.x, fma(a.x, b.y, c.y)));
}
// c - a*b
HP_HD cplx cfms(cplx a, cplx b, cplx c) {
    return cmake(fma(a.y, b.y, fma(-a.x, b.x, c.x)), fma(-a.y, b.x, fma(-a.x, b.y, c.y)));
}
// kappa * z for the slowness^2 of a real (double) or an attenuating (complex) medium.  With a zero imaginary part the
// complex product gives the bits of the real scaling: k*z.x - 0*z.y and k*z.y + 0*z.x round like k*z.x and k*z.y.
HP_HD cplx hp_kmul(double k, cplx z) { return cscale(k, z); }
HP_HD cplx hp_kmul(cplx k, cplx z) { return cmul(k, z); }
// kappa * z - s, the diagonal coefficient c5.  The real medium's k*z.x - s.x compiles to one fma (the product is not
// rounded), so cmul(kappa, z) - s would round differently even for Im(kappa) = 0.  The complex form is therefore
// Re(kappa) z - s + Im(kappa) (i z): its first part is the real medium's expression, and a zero imaginary part adds
// exact zeros, which keeps the bits of the real medium.
HP_HD cplx hp_kmul_sub(double k, cplx z, cplx s) { return csub(cscale(k, z), s); }
HP_HD cplx hp_kmul_sub(cplx k, cplx z, cplx s) { return cadd(csub(cscale(k.x, z), s), cscale(k.y, cmake(-z.y, z.x))); }
HP_HD double cabs2(cplx a) { return a.x * a.x + a.y * a.y; }
// Smith's algorithm, the same scheme CPython / numpy use for complex division
HP_HD cplx cdiv(cplx a, cplx b) {
    if (fabs(b.x) >= fabs(b.y)) {
        double ratio = b.y / b.x, denom = b.x + b.y * ratio;
        return cmake((a.x + a.y * ratio) / denom, (a.y - a.x * ratio) / denom);
    } else {
        double ratio = b.x / b.y, denom = b.x * ratio + b.y;
        return cmake((a.x * ratio + a.y) / denom, (a.y * ratio - a.x) / denom);
    }
}
HP_HD cplx cinv(cplx b) { return cdiv(cmake(1.0, 0.0), b); }

// ---------------------------------------------------------------------------------------------
// PML profiles.  The operation order follows the reference expressions so the branch decisions
// (x <= eta, x >= 1 - eta) and the quadratic are evaluated on identical doubles.
// ---------------------------------------------------------------------------------------------
struct HpPml {
    double cst;      // "const" of the reference
    double eta;      // PML width b*h
    double h;        // 1/(n+1)
    cplx omega;      // 2*pi*wave_num + 1j*alpha
};

#if defined(__CUDA_ARCH__)
#define HP_MUL(a, b) __dmul_rn((a), (b))
#define HP_SUB(a, b) __dsub_rn((a), (b))
#define HP_ADD(a, b) __dadd_rn((a), (b))
#else
#define HP_MUL(a, b) ((a) * (b))
#define HP_SUB(a, b) ((a) - (b))
#define HP_ADD(a, b) ((a) + (b))
#endif

HP_HD double hp_sigma1(double x, const HpPml& p) {          // code.py:11-18
    if (x <= p.eta) {
        double t = HP_SUB(x, p.eta) / p.eta;
        return HP_MUL(p.cst / p.eta, HP_MUL(t, t));
    } else if (x >= HP_SUB(1.0, p.eta)) {
        double t = HP_ADD(HP_SUB(x, 1.0), p.eta) / p.eta;
        return HP_MUL(p.cst / p.eta, HP_MUL(t, t));
    }
    return 0.0;
}
HP_HD double hp_sigma2(double x, const HpPml& p) {          // code.py:20-25
    if (x <= p.eta) {
        double t = HP_SUB(x, p.eta) / p.eta;
        return HP_MUL(p.cst / p.eta, HP_MUL(t, t));
    }
    return 0.0;
}
// 1/s = 1 + 1j*sigma/omega ; s itself is its reciprocal (code.py:27-37)
HP_HD cplx hp_inv_s(double sigma, const HpPml& p) {
    cplx q = cdiv(cmake(0.0, sigma), p.omega);
    return cmake(1.0 + q.x, q.y);
}
// grid coordinate (k + half/2)*h evaluated as the reference does: (i-.5)*h, i*h, (i+.5)*h
HP_HD double hp_coord(int twice, double h) { return HP_MUL(0.5 * (double)twice, h); }

// one entry of the half-grid tables: s1, 1/s1, s2, 1/s2 at x = t*h/2 (unshifted PML, operator A)
HP_HD void hp_table_entry(int t, const HpPml& p, cplx* s1, cplx* is1, cplx* s2, cplx* is2) {
    double x = hp_coord(t, p.h);
    cplx a = hp_inv_s(hp_sigma1(x, p), p);
    cplx c = hp_inv_s(hp_sigma2(x, p), p);
    *is1 = a; *s1 = cinv(a);
    *is2 = c; *s2 = cinv(c);
}

// ---------------------------------------------------------------------------------------------
// b x b complex matrices, row major with leading dimension HP_BMAX-free (ld = b)
// ---------------------------------------------------------------------------------------------

// In-place Gauss-Jordan inverse with partial pivoting.  Returns 0, or 1 if a pivot vanished.
HP_HD int hp_inv_inplace(cplx* A, int b) {
    int piv[2 * HP_BMAX];
    for (int p = 0; p < b; ++p) {
        int r = p;
        double best = cabs2(A[p * b + p]);
        for (int i = p + 1; i < b; ++i) {
            double v = cabs2(A[i * b + p]);
            if (v > best) { best = v; r = i; }
        }
        piv[p] = r;
        if (best == 0.0) return 1;
        if (r != p)
            for (int j = 0; j < b; ++j) { cplx t = A[p * b + j]; A[p * b + j] = A[r * b + j]; A[r * b + j] = t; }
        cplx d = cinv(A[p * b + p]);
        A[p * b + p] = cmake(1.0, 0.0);
        for (int j = 0; j < b; ++j) A[p * b + j] = cmul(A[p * b + j], d);
        for (int i = 0; i < b; ++i) {
            if (i == p) continue;
            cplx f = A[i * b + p];
            A[i * b + p] = cmake(0.0, 0.0);
            for (int j = 0; j < b; ++j) A[i * b + j] = cfms(f, A[p * b + j], A[i * b + j]);
        }
    }
    for (int p = b - 1; p >= 0; --p) {
        int r = piv[p];
        if (r != p)
            for (int i = 0; i < b; ++i) { cplx t = A[i * b + p]; A[i * b + p] = A[i * b + r]; A[i * b + r] = t; }
    }
    return 0;
}

// C (m x n) = alpha_sign * A (m x k) * B (k x n) [+ C if accumulate]; sign = +1 or -1
HP_HD void hp_gemm(cplx* C, const cplx* A, const cplx* B, int m, int k, int n, int ldc, int lda, int ldb,
                   int sign, int accumulate) {
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < n; ++j) {
            cplx acc = accumulate ? C[i * ldc + j] : cmake(0.0, 0.0);
            if (sign > 0) for (int l = 0; l < k; ++l) acc = cfma(A[i * lda + l], B[l * ldb + j], acc);
            else          for (int l = 0; l < k; ++l) acc = cfms(A[i * lda + l], B[l * ldb + j], acc);
            C[i * ldc + j] = acc;
        }
}

// ---------------------------------------------------------------------------------------------
// Strip coefficients.  A strip is the b grid rows j = m-b+1..m (k = 1..b local) with the x2 PML
// moved so that it ends on row m (s2m, code.py:35-37).  Tables over the x1 half grid are shared
// by all strips: s1t[t] = s1(t*h/2) for t = 0..2n+2 and is1t[t] = 1/s1.
// ---------------------------------------------------------------------------------------------
struct HpStripRow {          // x2-dependent factors of one strip, k = 0..b-1 local rows
    cplx is2c[HP_BMAX];      // 1/s2m(j h)
    cplx s2lo[HP_BMAX];      // s2m((j-.5) h)
    cplx s2hi[HP_BMAX];      // s2m((j+.5) h)
};

HP_HD void hp_strip_rows(HpStripRow& R, int m, int b, const HpPml& p) {
    double shift = HP_MUL((double)(m - b), p.h);                         // (m-b)*h, code.py:37
    for (int k = 0; k < b; ++k) {
        int j = m - b + 1 + k;
        R.is2c[k] = hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j, p.h), shift), p), p);
        R.s2lo[k] = cinv(hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j - 1, p.h), shift), p), p));
        R.s2hi[k] = cinv(hp_inv_s(hp_sigma2(HP_SUB(hp_coord(2 * j + 1, p.h), shift), p), p));
    }
}

// Coefficients of block row i (1-based x1 index) of a strip: tridiagonal D (sub/diag/super per k)
// and the diagonal couplings L (to i-1) and U (to i+1).   code.py:239-273
//   c1 = 1/h^2 * s1((i-.5)h)/s2m(jh)      -> L[k]
//   c2 = 1/h^2 * s1((i+.5)h)/s2m(jh)      -> U[k]
//   c3 = 1/h^2 * s2m((j-.5)h)/s1(ih)      -> sub[k]   (coupling to k-1)
//   c4 = 1/h^2 * s2m((j+.5)h)/s1(ih)      -> sup[k]   (coupling to k+1)
//   c5 = omega^2/(s1 s2m c^2) - (c1+c2+c3+c4)
// CK selects the medium: false reads the real velocity c_mat, true the complex slowness^2 kappa_c of an attenuating medium
// (grid aligned, kappa_c[(j-1) n + (i-1)] = 1/c_mat[i-1][j-1]^2, see hp_kappa_c_kernel).  The complex c5 is formed by
// hp_kmul_sub, so that a zero imaginary part gives the bits of the real medium.
struct HpBlockRow {
    cplx L[HP_BMAX], U[HP_BMAX], sub[HP_BMAX], dia[HP_BMAX], sup[HP_BMAX];
};

template <bool CK = false>
HP_HD void hp_block_row(HpBlockRow& B, const HpStripRow& R, int i, int m, int b, int n, const HpPml& p,
                        const cplx* s1t, const cplx* is1t, const double* c_mat, cplx omega2, const cplx* kappa_c = nullptr) {
    double ih2 = 1.0 / (p.h * p.h);
    cplx s1lo = s1t[2 * i - 1], s1hi = s1t[2 * i + 1], is1c = is1t[2 * i];
    for (int k = 0; k < b; ++k) {
        int j = m - b + 1 + k;
        cplx c1 = cscale(ih2, cmul(s1lo, R.is2c[k]));
        cplx c2 = cscale(ih2, cmul(s1hi, R.is2c[k]));
        cplx c3 = cscale(ih2, cmul(R.s2lo[k], is1c));
        cplx c4 = cscale(ih2, cmul(R.s2hi[k], is1c));
        cplx c5;
        if (CK) {
            c5 = hp_kmul_sub(kappa_c[(size_t)(j - 1) * n + (i - 1)], cmul(omega2, cmul(is1c, R.is2c[k])),
                             cadd(cadd(c1, c2), cadd(c3, c4)));
        } else {
            double cv = c_mat[(size_t)(i - 1) * (n + 2) + (j - 1)];      // c_mat[i-1, j-1], code.py:270
            c5 = cscale(1.0 / (cv * cv), cmul(omega2, cmul(is1c, R.is2c[k])));
            c5 = csub(c5, cadd(cadd(c1, c2), cadd(c3, c4)));
        }
        B.L[k] = c1; B.U[k] = c2; B.sub[k] = c3; B.sup[k] = c4; B.dia[k] = c5;
    }
}

// F = D_i - diag(a) * Xinv * diag(c)     (Schur complement step; Xinv is b x b)
HP_HD void hp_schur_step(cplx* F, const HpBlockRow& B, const cplx* a, const cplx* Xinv, const cplx* c, int b,
                         int have_prev) {
    for (int r = 0; r < b; ++r)
        for (int s = 0; s < b; ++s) {
            cplx v = cmake(0.0, 0.0);
            if (r == s) v = B.dia[r];
            else if (s == r - 1) v = B.sub[r];
            else if (s == r + 1) v = B.sup[r];
            if (have_prev) v = cfms(cmul(a[r], Xinv[r * b + s]), c[s], v);
            F[r * b + s] = v;
        }
}
