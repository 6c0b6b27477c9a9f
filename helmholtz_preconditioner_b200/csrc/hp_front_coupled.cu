// Coupled front block: H_F = A[:bn, :bn], the full 5-point operator of the first b grid rows (Engquist & Ying's A_FF).
//
// The reference's get_A_FF_block (/root/reference/code.py:178-183) keeps only the b diagonal blocks (csrc/hp_front.cu,
// the default).  With the couplings between the rows kept, H_F is exactly the strip operator of layer m = b
// (get_Hm(b), code.py:283-290: the moving PML of layer b is the fixed PML of the operator), and the preconditioner
// becomes the one of the paper: GMRES needs 2-5 iterations instead of 70-200 (tests/golden/large_*__pc.npz).
// algo2_4 needs the whole solve here (all b rows in, all b rows out: code.py:364, 382), not only the
// last-row restriction T_m of the strips.
//
// Ordered x1-major, H_F is block tridiagonal: n block rows (columns i of the grid) of size b, diagonal blocks D_i
// (tridiagonal, x2 couplings), off-diagonal blocks diag(l_i), diag(u_i) (x1 couplings).  One level of nested
// dissection over x1, as for the strips: P leaves separated by P-1 single separator columns.
//   setup   per leaf: forward Schur chain Sinv_i = (D_i - l_i Sinv_{i-1} u_{i-1})^-1 (block Thomas of the Dirichlet-
//           truncated leaf operator A_l); corner blocks of A_l^-1 from leaf solves with unit right-hand sides;
//           separator Schur complement (block tridiagonal, dense b x b blocks) and its chain T_s
//   solve   z_l = A_l^-1 r_l                                    (all leaves in parallel, one warp each, 2q steps)
//           S x_S = r_S - l_S z_{left,last} - u_S z_{right,first}                         (one warp, 2(P-1) steps)
//           x_l = A_l^-1 (r_l - e_first l_first x_{s_{l-1}} - e_last u_last x_{s_l})      (all leaves in parallel)
// A warp holds a b-vector one entry per lane; a b x b matrix-vector product is b shuffles and b complex multiply-adds
// per lane, the matrix row prefetched one step ahead.
#include "hp_internal.cuh"

struct HpFcArgs {
    int n, b, P, QP;
    const int *leaf_start, *leaf_q, *sep;
    const cplx* Sinv;      // [n][b*b]     forward chains of the leaves (separator columns unused)
    const cplx* LU;        // [n][2][b]    l_i (coupling to column i-1), u_i (coupling to column i+1)
    const cplx *T, *Sl, *Su;   // [P-1][b*b]
    const cplx* is1t;
};

__device__ __forceinline__ cplx fc_shfl(cplx v, int src) {
    return cmake(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src));
}
// row k of M (b entries, lane k) times the vector held one entry per lane
template <int BT>
__device__ __forceinline__ cplx fc_matvec(const cplx* m, cplx y, int b) {
    cplx a0 = cmake(0.0, 0.0), a1 = cmake(0.0, 0.0);
    constexpr int BL = BT ? BT : HP_BMAX;
#pragma unroll
    for (int c = 0; c < BL; c += 2) {
        if (BT || c < b) { a0 = cfma(m[c], fc_shfl(y, c), a0); }
        if (c + 1 < BL && (BT || c + 1 < b)) { a1 = cfma(m[c + 1], fc_shfl(y, c + 1), a1); }
    }
    return cadd(a0, a1);
}
template <int BT>
__device__ __forceinline__ void fc_load_row(cplx* m, const cplx* M, int k, int b) {
    constexpr int BL = BT ? BT : HP_BMAX;
#pragma unroll
    for (int c = 0; c < BL; ++c) m[c] = (k < b && (BT || c < b)) ? M[(size_t)k * b + c] : cmake(0.0, 0.0);
}

// right-hand side of grid column i, front row k.  rhs_mode 0: the field rows in[k*n + i]; 1: unit vector (unit_col,
// unit_row); 2: only the last row, fac * is1t[2(i+1)] * in[i]  (A_{F,b+1} u_{b+1}, code.py:381)
__device__ __forceinline__ cplx fc_rhs(const HpFcArgs& a, int rhs_mode, const cplx* in, cplx fac, int unit_col, int unit_row,
                                       int i, int k) {
    if (rhs_mode == 0) return in[(size_t)k * a.n + i];
    if (rhs_mode == 1) return (i == unit_col && k == unit_row) ? cmake(1.0, 0.0) : cmake(0.0, 0.0);
    return k == a.b - 1 ? cmul(cmul(fac, a.is1t[2 * (i + 1)]), in[i]) : cmake(0.0, 0.0);
}

// One warp per (leaf, right-hand side).  corr: subtract the couplings to the separator solution xs (field layout, valid
// at the separator columns) from the first and last column.  out_mode 0: out = solution; 1: corners[l][rhs][first|last][b];
// 2: out = base - solution.
template <int BT>
__global__ void __launch_bounds__(32) hp_fc_leaf_solve_kernel(HpFcArgs a, int rhs_mode, int corr, int out_mode, const cplx* in,
                                                              const cplx* xs, cplx* out, const cplx* base, cplx fac) {
    extern __shared__ __align__(16) unsigned char fc_smem[];
    cplx* R = reinterpret_cast<cplx*>(fc_smem);              // [q][b]: right-hand side, then w, then the solution
    const int b = BT ? BT : a.b, bb = b * b, n = a.n;
    const int l = blockIdx.x, rhs = blockIdx.y, lane = threadIdx.x, k = lane;
    const int i0 = a.leaf_start[l], q = a.leaf_q[l], i1 = i0 + q - 1;
    const int unit_col = rhs < b ? i0 : i1, unit_row = rhs < b ? rhs : rhs - b;
    for (int kk = 0; kk < b; ++kk)
        for (int t = lane; t < q; t += 32) R[(size_t)t * b + kk] = fc_rhs(a, rhs_mode, in, fac, unit_col, unit_row, i0 + t, kk);
    __syncwarp();
    if (corr && k < b) {
        if (l > 0) R[k] = cfms(a.LU[((size_t)i0 * 2) * b + k], xs[(size_t)k * n + i0 - 1], R[k]);
        if (l < a.P - 1) R[(size_t)(q - 1) * b + k] = cfms(a.LU[((size_t)i1 * 2 + 1) * b + k], xs[(size_t)k * n + i1 + 1], R[(size_t)(q - 1) * b + k]);
    }
    __syncwarp();
    constexpr int BL = BT ? BT : HP_BMAX;
    cplx m[BL], mn[BL];
    // forward elimination: w_t = Sinv_t y_t,  y_{t+1} = r_{t+1} - l_{t+1} w_t
    fc_load_row<BT>(m, a.Sinv + (size_t)i0 * bb, k, b);
    cplx y = k < b ? R[k] : cmake(0.0, 0.0);
    for (int t = 0; t < q; ++t) {
        const int i = i0 + t;
        cplx rn = cmake(0.0, 0.0), ln = cmake(0.0, 0.0);
        if (t + 1 < q) {
            fc_load_row<BT>(mn, a.Sinv + (size_t)(i + 1) * bb, k, b);
            if (k < b) { rn = R[(size_t)(t + 1) * b + k]; ln = a.LU[((size_t)(i + 1) * 2) * b + k]; }
        }
        const cplx w = fc_matvec<BT>(m, y, b);
        if (k < b) R[(size_t)t * b + k] = w;
        y = cfms(ln, w, rn);
#pragma unroll
        for (int c = 0; c < BL; ++c) m[c] = mn[c];
    }
    // back substitution: z_last = w_last,  z_t = w_t - Sinv_t (u_t z_{t+1})
    cplx z = k < b ? R[(size_t)(q - 1) * b + k] : cmake(0.0, 0.0);
    if (q > 1) fc_load_row<BT>(m, a.Sinv + (size_t)(i1 - 1) * bb, k, b);
    for (int t = q - 2; t >= 0; --t) {
        const int i = i0 + t;
        if (t > 0) fc_load_row<BT>(mn, a.Sinv + (size_t)(i - 1) * bb, k, b);
        const cplx ui = k < b ? a.LU[((size_t)i * 2 + 1) * b + k] : cmake(0.0, 0.0);
        const cplx w = k < b ? R[(size_t)t * b + k] : cmake(0.0, 0.0);
        z = csub(w, fc_matvec<BT>(m, cmul(ui, z), b));
        if (k < b) R[(size_t)t * b + k] = z;
#pragma unroll
        for (int c = 0; c < BL; ++c) m[c] = mn[c];
    }
    __syncwarp();
    if (out_mode == 1) {
        if (k < b) {
            cplx* o = out + (((size_t)l * 2 * b + rhs) * 2) * b;
            o[k] = R[k];
            o[b + k] = R[(size_t)(q - 1) * b + k];
        }
        return;
    }
    for (int kk = 0; kk < b; ++kk)
        for (int t = lane; t < q; t += 32) {
            const size_t o = (size_t)kk * n + i0 + t;
            const cplx v = R[(size_t)t * b + kk];
            out[o] = out_mode == 2 ? csub(base[o], v) : v;
        }
}

// Separator system: one warp.  zl: leaf solutions of the first pass (field layout); the separator solution is written into
// zl at the separator columns (the second pass reads it there) and into out (out_mode as above).
template <int BT>
__global__ void __launch_bounds__(32) hp_fc_schur_solve_kernel(HpFcArgs a, int rhs_mode, int out_mode, const cplx* in, cplx* zl,
                                                               cplx* out, const cplx* base, cplx fac) {
    extern __shared__ __align__(16) unsigned char fc_smem[];
    cplx* W = reinterpret_cast<cplx*>(fc_smem);              // [P-1][b]
    const int b = BT ? BT : a.b, bb = b * b, n = a.n, ns = a.P - 1, k = threadIdx.x;
    constexpr int BL = BT ? BT : HP_BMAX;
    cplx m[BL], m2[BL];
    cplx wprev = cmake(0.0, 0.0);
    for (int s = 0; s < ns; ++s) {
        const int col = a.sep[s];
        cplx y = cmake(0.0, 0.0);
        if (k < b) {
            y = fc_rhs(a, rhs_mode, in, fac, -1, -1, col, k);
            y = cfms(a.LU[((size_t)col * 2) * b + k], zl[(size_t)k * n + col - 1], y);
            y = cfms(a.LU[((size_t)col * 2 + 1) * b + k], zl[(size_t)k * n + col + 1], y);
        }
        fc_load_row<BT>(m, a.T + (size_t)s * bb, k, b);
        if (s > 0) {
            fc_load_row<BT>(m2, a.Sl + (size_t)s * bb, k, b);
            y = csub(y, fc_matvec<BT>(m2, wprev, b));
        }
        wprev = fc_matvec<BT>(m, y, b);
        if (k < b) W[(size_t)s * b + k] = wprev;
    }
    cplx x = wprev;
    for (int s = ns - 1; s >= 0; --s) {
        if (s < ns - 1) {
            fc_load_row<BT>(m2, a.Su + (size_t)s * bb, k, b);
            fc_load_row<BT>(m, a.T + (size_t)s * bb, k, b);
            const cplx t = fc_matvec<BT>(m2, x, b);
            x = csub(k < b ? W[(size_t)s * b + k] : cmake(0.0, 0.0), fc_matvec<BT>(m, t, b));
        }
        if (k < b) {
            const size_t o = (size_t)k * n + a.sep[s];
            zl[o] = x;
            out[o] = out_mode == 2 ? csub(base[o], x) : x;
        }
    }
}

// ---- setup -------------------------------------------------------------------------------------------------------
// thread -> leaf: forward Schur chain of the leaf (the strip arithmetic of csrc/hp_setup_core.h with m = b)
// (CK: attenuating medium, hp_block_row)
template <int BB, bool CK>
__global__ void hp_fc_chain_kernel(HpStripCtx c, int P, const int* leaf_start, const int* leaf_q, cplx* Sinv, int* status) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= P) return;
    if (hp_chain_forward<BB, CK>(Sinv, leaf_start[l] + 1, leaf_start[l] + leaf_q[l], c.b, c)) atomicOr(status, 16);
}
// thread -> grid column: the x1 couplings and the tridiagonal block D_i of every column
template <bool CK>
__global__ void hp_fc_coef_kernel(HpStripCtx c, cplx* LU, cplx* D3) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;      // 0-based column
    if (i >= c.n) return;
    HpStripRow R;
    hp_strip_rows(R, c.b, c.b, c.pml);
    HpBlockRow B;
    hp_block_row<CK>(B, R, i + 1, c.b, c.b, c.n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
    for (int k = 0; k < c.b; ++k) {
        LU[((size_t)i * 2) * c.b + k] = B.L[k];
        LU[((size_t)i * 2 + 1) * c.b + k] = B.U[k];
        D3[((size_t)i * 3) * c.b + k] = B.sub[k];
        D3[((size_t)i * 3 + 1) * c.b + k] = B.dia[k];
        D3[((size_t)i * 3 + 2) * c.b + k] = B.sup[k];
    }
}
// one thread: the separator Schur complement from the corner blocks of the leaf inverses, and its chain
//   Sd_s = D_s - l_s G_l[last,last] u_last(l) - u_s G_{l+1}[first,first] l_first(l+1)
//   Sl_s = -l_s G_l[last,first] l_first(l)          Su_s = -u_s G_{l+1}[first,last] u_last(l+1)
//   T_s  = (Sd_s - Sl_s T_{s-1} Su_{s-1})^-1
// corners[l][rhs][w][r]: row r of column w (0 first, 1 last) of A_l^-1 applied to the unit vector rhs (rhs < b: first
// column, row rhs; rhs >= b: last column, row rhs - b)
template <int BB>
__global__ void hp_fc_schur_factor_kernel(HpFcArgs a, const cplx* corners, const cplx* D3, cplx* T, cplx* Sl, cplx* Su, int* status) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    const int b = a.b, bb = b * b, ns = a.P - 1;
    cplx Sd[BB], X[BB], Y[BB];
    auto corner = [&](int l, int rhs, int w, int r) { return corners[(((size_t)l * 2 * b + rhs) * 2 + w) * b + r]; };
    for (int s = 0; s < ns; ++s) {
        const int col = a.sep[s], l = s, r_ = s + 1;
        const int lf = a.leaf_start[l], ll = lf + a.leaf_q[l] - 1;          // first / last column of the left leaf
        const int rf = a.leaf_start[r_], rl = rf + a.leaf_q[r_] - 1;        // of the right leaf
        const cplx* ls = a.LU + ((size_t)col * 2) * b;
        const cplx* us = a.LU + ((size_t)col * 2 + 1) * b;
        for (int r = 0; r < b; ++r)
            for (int c = 0; c < b; ++c) {
                cplx v = cmake(0.0, 0.0);
                if (r == c) v = D3[((size_t)col * 3 + 1) * b + r];
                else if (c == r - 1) v = D3[((size_t)col * 3) * b + r];
                else if (c == r + 1) v = D3[((size_t)col * 3 + 2) * b + r];
                v = cfms(cmul(ls[r], corner(l, b + c, 1, r)), a.LU[((size_t)ll * 2 + 1) * b + c], v);
                v = cfms(cmul(us[r], corner(r_, c, 0, r)), a.LU[((size_t)rf * 2) * b + c], v);
                Sd[r * b + c] = v;
                Sl[(size_t)s * bb + r * b + c] = cneg(cmul(cmul(ls[r], corner(l, c, 1, r)), a.LU[((size_t)lf * 2) * b + c]));
                Su[(size_t)s * bb + r * b + c] = cneg(cmul(cmul(us[r], corner(r_, b + c, 0, r)), a.LU[((size_t)rl * 2 + 1) * b + c]));
            }
        if (s > 0) {
            for (int e = 0; e < bb; ++e) { X[e] = Sl[(size_t)s * bb + e]; Y[e] = Su[(size_t)(s - 1) * bb + e]; }
            cplx Z[BB];
            hp_gemm(Z, X, T + (size_t)(s - 1) * bb, b, b, b, b, b, b, +1, 0);
            hp_gemm(Sd, Z, Y, b, b, b, b, b, b, -1, 1);
        }
        if (hp_inv_inplace(Sd, b)) atomicOr(status, 32);
        for (int e = 0; e < bb; ++e) T[(size_t)s * bb + e] = Sd[e];
    }
}

// ---- host --------------------------------------------------------------------------------------------------------
static HpFcArgs fc_args(const hp_solver* s) {
    HpFcArgs a;
    a.n = s->n; a.b = s->b; a.P = s->fc_P; a.QP = s->fc_QP;
    a.leaf_start = s->fc_leaf_start; a.leaf_q = s->fc_leaf_q; a.sep = s->fc_sep;
    a.Sinv = s->fc_Sinv; a.LU = s->fc_LU; a.T = s->fc_T; a.Sl = s->fc_Sl; a.Su = s->fc_Su; a.is1t = s->is1t;
    return a;
}
static size_t fc_leaf_smem(const hp_solver* s) { return sizeof(cplx) * (size_t)s->fc_QP * s->b; }

template <int BT>
static int fc_launch_leaf(const hp_solver* s, int nrhs, int rhs_mode, int corr, int out_mode, const cplx* in, const cplx* xs, cplx* out,
                          const cplx* base, cplx fac, cudaStream_t st) {
    const size_t smem = fc_leaf_smem(s);
    if (smem > 48 * 1024) HP_CUDA(cudaFuncSetAttribute(hp_fc_leaf_solve_kernel<BT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hp_count_launch();
    hp_fc_leaf_solve_kernel<BT><<<dim3(s->fc_P, nrhs), 32, smem, st>>>(fc_args(s), rhs_mode, corr, out_mode, in, xs, out, base, fac);
    HP_CUDA(cudaGetLastError());
    return 0;
}
static int fc_leaf(const hp_solver* s, int nrhs, int rhs_mode, int corr, int out_mode, const cplx* in, const cplx* xs, cplx* out,
                   const cplx* base, cplx fac, cudaStream_t st) {
    return s->b == 12 ? fc_launch_leaf<12>(s, nrhs, rhs_mode, corr, out_mode, in, xs, out, base, fac, st)
                      : fc_launch_leaf<0>(s, nrhs, rhs_mode, corr, out_mode, in, xs, out, base, fac, st);
}

// out (b rows, field layout) = H_F^-1 rhs  (out_mode 0)  or  base - H_F^-1 rhs  (out_mode 2)
int hp_front_coupled_solve(hp_solver* s, int rhs_mode, int out_mode, const cplx* in, cplx* out, const cplx* base, cplx fac,
                           cudaStream_t st) {
    cplx* zl = s->fc_work;
    if (s->fc_P == 1) return fc_leaf(s, 1, rhs_mode, 0, out_mode, in, nullptr, out, base, fac, st);
    if (fc_leaf(s, 1, rhs_mode, 0, 0, in, nullptr, zl, nullptr, fac, st)) return 2;
    const size_t smem = sizeof(cplx) * (size_t)(s->fc_P - 1) * s->b;
    hp_count_launch();
    if (s->b == 12) hp_fc_schur_solve_kernel<12><<<1, 32, smem, st>>>(fc_args(s), rhs_mode, out_mode, in, zl, out, base, fac);
    else hp_fc_schur_solve_kernel<0><<<1, 32, smem, st>>>(fc_args(s), rhs_mode, out_mode, in, zl, out, base, fac);
    HP_CUDA(cudaGetLastError());
    return fc_leaf(s, 1, rhs_mode, 1, out_mode, in, zl, out, base, fac, st);
}

void hp_front_coupled_free(hp_solver* s) {
    cudaFree(s->fc_leaf_start); cudaFree(s->fc_leaf_q); cudaFree(s->fc_sep);
    cudaFree(s->fc_Sinv); cudaFree(s->fc_LU); cudaFree(s->fc_T); cudaFree(s->fc_Sl); cudaFree(s->fc_Su); cudaFree(s->fc_work);
    s->fc_leaf_start = s->fc_leaf_q = s->fc_sep = nullptr;
    s->fc_Sinv = s->fc_LU = s->fc_T = s->fc_Sl = s->fc_Su = s->fc_work = nullptr;
    s->fc_P = 0;
}

int hp_front_coupled_setup(hp_solver* s, cudaStream_t st) {
    hp_front_coupled_free(s);
    const int n = s->n, b = s->b, bb = b * b;
    // partition: sequential depth 4 n / P (two leaf passes) + 4 P (separator chain) -> P ~ sqrt(n), at most 64 leaves of
    // at least two columns
    int P = (int)lround(sqrt((double)n));
    if (P > 64) P = 64;
    while (P > 1 && (n - (P - 1)) / P < 2) --P;
    if (const char* e = getenv("HP_FRONT_LEAVES")) P = std::max(1, std::min(atoi(e), std::max(1, (n + 1) / 3)));
    const int ns = P - 1;
    std::vector<int> ls(P), lq(P), sp(std::max(ns, 1), 0);
    int QP = 0;
    {
        long inner = n - ns;
        int pos = 0;
        for (int l = 0; l < P; ++l) {
            int q = (int)((inner * (l + 1)) / P - (inner * l) / P);
            ls[l] = pos; lq[l] = q; pos += q;
            QP = std::max(QP, q);
            if (l < P - 1) { sp[l] = pos; pos += 1; }
        }
    }
    s->fc_P = P; s->fc_QP = QP;
    int max_smem = 0, dev = 0;
    HP_CUDA(cudaGetDevice(&dev));
    HP_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (fc_leaf_smem(s) > (size_t)max_smem) { hp_set_error("coupled front block: leaf of %d columns does not fit shared memory", QP); return 1; }
    HP_CUDA(cudaMalloc(&s->fc_leaf_start, sizeof(int) * P));
    HP_CUDA(cudaMalloc(&s->fc_leaf_q, sizeof(int) * P));
    HP_CUDA(cudaMalloc(&s->fc_sep, sizeof(int) * std::max(ns, 1)));
    HP_CUDA(cudaMemcpyAsync(s->fc_leaf_start, ls.data(), sizeof(int) * P, cudaMemcpyHostToDevice, st));
    HP_CUDA(cudaMemcpyAsync(s->fc_leaf_q, lq.data(), sizeof(int) * P, cudaMemcpyHostToDevice, st));
    HP_CUDA(cudaMemcpyAsync(s->fc_sep, sp.data(), sizeof(int) * std::max(ns, 1), cudaMemcpyHostToDevice, st));
    HP_CUDA(cudaStreamSynchronize(st));                                   // the host vectors go out of scope
    HP_CUDA(cudaMalloc(&s->fc_Sinv, sizeof(cplx) * (size_t)n * bb));
    HP_CUDA(cudaMalloc(&s->fc_LU, sizeof(cplx) * (size_t)n * 2 * b));
    HP_CUDA(cudaMalloc(&s->fc_T, sizeof(cplx) * (size_t)std::max(ns, 1) * bb));
    HP_CUDA(cudaMalloc(&s->fc_Sl, sizeof(cplx) * (size_t)std::max(ns, 1) * bb));
    HP_CUDA(cudaMalloc(&s->fc_Su, sizeof(cplx) * (size_t)std::max(ns, 1) * bb));
    HP_CUDA(cudaMalloc(&s->fc_work, sizeof(cplx) * (size_t)n * b));
    HP_CUDA(cudaMemsetAsync(s->fc_Sinv, 0, sizeof(cplx) * (size_t)n * bb, st));
    cplx *D3 = nullptr, *corners = nullptr;
    struct Guard { cplx *&a, *&c; ~Guard() { cudaFree(a); cudaFree(c); } } guard{D3, corners};
    HP_CUDA(cudaMalloc(&D3, sizeof(cplx) * (size_t)n * 3 * b));
    HP_CUDA(cudaMalloc(&corners, sizeof(cplx) * (size_t)P * 2 * b * 2 * b));
    HpStripCtx c = hp_ctx(s);
    hp_count_launch();
    const bool ck = s->kappa_c != nullptr;
    if (ck) {
        if (b <= 12) hp_fc_chain_kernel<144, true><<<(P + 31) / 32, 32, 0, st>>>(c, P, s->fc_leaf_start, s->fc_leaf_q, s->fc_Sinv, s->status);
        else hp_fc_chain_kernel<HP_BMAX * HP_BMAX, true><<<(P + 31) / 32, 32, 0, st>>>(c, P, s->fc_leaf_start, s->fc_leaf_q, s->fc_Sinv, s->status);
        hp_count_launch(); hp_fc_coef_kernel<true><<<(n + 63) / 64, 64, 0, st>>>(c, s->fc_LU, D3);
    } else {
        if (b <= 12) hp_fc_chain_kernel<144, false><<<(P + 31) / 32, 32, 0, st>>>(c, P, s->fc_leaf_start, s->fc_leaf_q, s->fc_Sinv, s->status);
        else hp_fc_chain_kernel<HP_BMAX * HP_BMAX, false><<<(P + 31) / 32, 32, 0, st>>>(c, P, s->fc_leaf_start, s->fc_leaf_q, s->fc_Sinv, s->status);
        hp_count_launch(); hp_fc_coef_kernel<false><<<(n + 63) / 64, 64, 0, st>>>(c, s->fc_LU, D3);
    }
    HP_CUDA(cudaGetLastError());
    if (ns > 0) {
        if (fc_leaf(s, 2 * b, 1, 0, 1, nullptr, nullptr, corners, nullptr, cmake(0, 0), st)) return 2;
        hp_count_launch();
        if (b <= 12) hp_fc_schur_factor_kernel<144><<<1, 32, 0, st>>>(fc_args(s), corners, D3, s->fc_T, s->fc_Sl, s->fc_Su, s->status);
        else hp_fc_schur_factor_kernel<HP_BMAX * HP_BMAX><<<1, 32, 0, st>>>(fc_args(s), corners, D3, s->fc_T, s->fc_Sl, s->fc_Su, s->status);
        HP_CUDA(cudaGetLastError());
    }
    HP_CUDA(cudaStreamSynchronize(st));
    return 0;
}
