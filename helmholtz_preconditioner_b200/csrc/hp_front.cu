// Front block of the sweeping preconditioner: the first b grid rows (the fixed PML of the operator).
//
// Reference: get_A_FF_block (/root/reference/code.py:178-183) keeps only the diagonal blocks A_11..A_bb,
// so H_F is b independent complex tridiagonal systems of size n (one per grid row); the reference factors
// it with SuperLU in algo2_3 (code.py:346-347) and solves with it twice per application in algo2_4
// (code.py:364-365 and 381-384).  Here: Thomas factors computed once, one thread per grid row.
#include "hp_internal.cuh"

// factors stored [i][j] (x1 index major) so that the b threads of the solve read contiguous memory.  KT: double for a real
// medium, cplx for an attenuating one (see hp_kmul)
template <typename KT>
__global__ void hp_front_factor_kernel(int n, int b, double ih2, cplx omega2, const cplx* __restrict__ s1t,
                                       const cplx* __restrict__ is1t, const cplx* __restrict__ s2t,
                                       const cplx* __restrict__ is2t, const KT* __restrict__ kappa,
                                       cplx* __restrict__ low, cplx* __restrict__ invd, cplx* __restrict__ up,
                                       int* status) {
    int j0 = threadIdx.x;            // 0-based grid row
    if (j0 >= b) return;
    int j = j0 + 1;
    cplx is2c = is2t[2 * j];
    cplx g3 = cscale(ih2, s2t[2 * j - 1]), g4 = cscale(ih2, s2t[2 * j + 1]);
    cplx dprev = cmake(1.0, 0.0), cprev = cmake(0.0, 0.0);
    for (int i = 1; i <= n; ++i) {
        cplx is1c = is1t[2 * i];
        cplx c1 = cscale(ih2, cmul(s1t[2 * i - 1], is2c));
        cplx c2 = cscale(ih2, cmul(s1t[2 * i + 1], is2c));
        cplx c3 = cmul(g3, is1c), c4 = cmul(g4, is1c);
        cplx c5 = hp_kmul_sub(kappa[(size_t)j0 * n + (i - 1)], cmul(omega2, cmul(is1c, is2c)), cadd(cadd(c1, c2), cadd(c3, c4)));
        cplx w = cmake(0.0, 0.0), d = c5;
        if (i > 1) {
            w = cdiv(c1, dprev);
            d = cfms(w, cprev, c5);
        }
        if (d.x == 0.0 && d.y == 0.0) atomicOr(status, 8);
        size_t o = (size_t)(i - 1) * b + j0;
        low[o] = w;
        invd[o] = cinv(d);
        up[o] = c2;
        dprev = d;
        cprev = c2;
    }
}

// mode 0: out[j][.] = Tri_j^{-1} in[j][.] for the rows j = row0 .. row0 + nrows - 1  (thread per row)
// mode 1: single row j = b-1 with rhs = upc * u_next,  out[.] = base[.] - solution      (code.py:381-384)
// The recurrences are sequential in i; their operands are not, so they are fetched HP_FRONT_U steps ahead
// into registers (and a few hundred steps ahead into L2) and only the complex multiply-add chain is exposed.
#define HP_FRONT_U 16
__global__ void hp_front_solve_kernel(int n, int b, int row0, int nrows, int mode, const cplx* __restrict__ low,
                                      const cplx* __restrict__ invd, const cplx* __restrict__ up,
                                      const cplx* in, cplx* out, const cplx* base, cplx upfac,
                                      const cplx* __restrict__ is1t, cplx* work) {
    int t = threadIdx.x;
    if (t >= nrows) return;
    int j0 = row0 + t;
    const cplx* r = in + (size_t)t * n;
    cplx* y = work + (size_t)t * n;
    cplx prev = cmake(0.0, 0.0);
    for (int i0 = 0; i0 < n; i0 += HP_FRONT_U) {
        cplx rr[HP_FRONT_U], ll[HP_FRONT_U];
        if (i0 + 256 < n) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(r + i0 + 256));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(low + (size_t)(i0 + 256) * b + j0));
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k) {
            int i = i0 + k;
            if (i < n) {
                rr[k] = r[i];
                ll[k] = low[(size_t)i * b + j0];
                if (mode == 1) rr[k] = cmul(cmul(upfac, is1t[2 * (i + 1)]), rr[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k) {
            int i = i0 + k;
            if (i < n) { prev = cfms(ll[k], prev, rr[k]); rr[k] = prev; }
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k)
            if (i0 + k < n) y[i0 + k] = rr[k];
    }
    cplx xn = cmake(0.0, 0.0);
    cplx* o = out + (size_t)t * n;
    for (int i1 = n - 1; i1 >= 0; i1 -= HP_FRONT_U) {
        cplx yy[HP_FRONT_U], uu[HP_FRONT_U], dd[HP_FRONT_U], bb[HP_FRONT_U];
        if (i1 - 256 >= 0) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(up + (size_t)(i1 - 256) * b + j0));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(invd + (size_t)(i1 - 256) * b + j0));
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k) {
            int i = i1 - k;
            if (i >= 0) {
                size_t f = (size_t)i * b + j0;
                yy[k] = y[i]; uu[k] = up[f]; dd[k] = invd[f];
                if (mode == 1) bb[k] = base[i];
            }
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k) {
            int i = i1 - k;
            if (i >= 0) { xn = cmul(cfms(uu[k], xn, yy[k]), dd[k]); yy[k] = mode == 1 ? csub(bb[k], xn) : xn; }
        }
#pragma unroll
        for (int k = 0; k < HP_FRONT_U; ++k)
            if (i1 - k >= 0) o[i1 - k] = yy[k];
    }
}

// The same two recurrences as a parallel scan: both are first-order affine recurrences
//     forward   y_i = r_i - low_i y_{i-1}                      map z -> A z + C with (A, C) = (-low_i, r_i)
//     backward  x_i = (y_i - up_i x_{i+1}) invd_i                                   (A, C) = (-up_i invd_i, y_i invd_i)
// One CTA of 512 threads per grid row; a thread composes the maps of its E consecutive unknowns, the block scans the
// 1024 composed maps (warp shuffles + one shared-memory step), and the thread replays its unknowns from the value that
// enters its range.  The tridiagonal blocks are diagonally dominant (|low|, |up invd| < 1), so the composed maps only
// contract.  ~10 us instead of 1.4 ms for the sequential kernel above (n = 4096).
#define HP_FS_THREADS 512
#define HP_FS_EMAX 16
struct HpAff { cplx A, C; };
// (second o first): z -> A2 (A1 z + C1) + C2
__device__ __forceinline__ HpAff hp_aff_compose(const HpAff& second, const HpAff& first) {
    HpAff r;
    r.A = cmul(second.A, first.A);
    r.C = cfma(second.A, first.C, second.C);
    return r;
}
__device__ __forceinline__ HpAff hp_aff_shfl(const HpAff& v, int delta, bool rev) {
    HpAff r;
    if (!rev) {
        r.A.x = __shfl_up_sync(0xffffffffu, v.A.x, delta); r.A.y = __shfl_up_sync(0xffffffffu, v.A.y, delta);
        r.C.x = __shfl_up_sync(0xffffffffu, v.C.x, delta); r.C.y = __shfl_up_sync(0xffffffffu, v.C.y, delta);
    } else {
        r.A.x = __shfl_down_sync(0xffffffffu, v.A.x, delta); r.A.y = __shfl_down_sync(0xffffffffu, v.A.y, delta);
        r.C.x = __shfl_down_sync(0xffffffffu, v.C.x, delta); r.C.y = __shfl_down_sync(0xffffffffu, v.C.y, delta);
    }
    return r;
}
// value entering the range of this thread (initial state 0) given the composed map of every thread; rev: the chain
// runs from the last thread to the first.  sm: 32 HpAff.
__device__ cplx hp_aff_block_enter(HpAff mine, bool rev, HpAff* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int NW = HP_FS_THREADS / 32;
    const int vl = rev ? 31 - lane : lane, vw = rev ? NW - 1 - warp : warp;  // position along the chain
    HpAff inc = mine;                                                        // inclusive scan inside the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        HpAff o = hp_aff_shfl(inc, d, rev);
        if (vl >= d) inc = hp_aff_compose(inc, o);
    }
    if (vl == 31) sm[vw] = inc;
    __syncthreads();
    if (warp == 0) {                                                         // scan of the warp totals (forward order)
        HpAff w;
        w.A = cmake(1.0, 0.0); w.C = cmake(0.0, 0.0);
        if (lane < NW) w = sm[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            HpAff o = hp_aff_shfl(w, d, false);
            if (lane >= d) w = hp_aff_compose(w, o);
        }
        if (lane < NW) sm[lane] = w;
    }
    __syncthreads();
    HpAff prevl = hp_aff_shfl(inc, 1, rev);                                  // inclusive map of the previous lane
    cplx enter = cmake(0.0, 0.0);
    if (vw > 0) enter = sm[vw - 1].C;                                        // state after the previous warps
    if (vl > 0) enter = cfma(prevl.A, enter, prevl.C);
    __syncthreads();
    return enter;
}

__global__ void __launch_bounds__(HP_FS_THREADS) hp_front_scan_kernel(int n, int b, int row0, int mode, const cplx* __restrict__ low,
        const cplx* __restrict__ invd, const cplx* __restrict__ up, const cplx* in, cplx* out, const cplx* base,
        cplx upfac, const cplx* __restrict__ is1t) {
    __shared__ HpAff sm[32];
    const int t = blockIdx.x, j0 = row0 + t, tid = threadIdx.x;
    const int E = (n + HP_FS_THREADS - 1) / HP_FS_THREADS, i_lo = tid * E;
    const cplx* r = in + (size_t)t * n;
    cplx y[HP_FS_EMAX];
    HpAff m;
    m.A = cmake(1.0, 0.0); m.C = cmake(0.0, 0.0);
#pragma unroll
    for (int e = 0; e < HP_FS_EMAX; ++e) {
        const int i = i_lo + e;
        if (e < E && i < n) {
            cplx rr = r[i];
            if (mode == 1) rr = cmul(cmul(upfac, is1t[2 * (i + 1)]), rr);
            const cplx lo = low[(size_t)i * b + j0];
            y[e] = rr;
            m.C = cfms(lo, m.C, rr);                         // C <- r - low C
            m.A = cneg(cmul(lo, m.A));                       // A <- -low A
        }
    }
    cplx prev = hp_aff_block_enter(m, false, sm);
#pragma unroll
    for (int e = 0; e < HP_FS_EMAX; ++e) {
        const int i = i_lo + e;
        if (e < E && i < n) { prev = cfms(low[(size_t)i * b + j0], prev, y[e]); y[e] = prev; }
    }
    // backward
    m.A = cmake(1.0, 0.0); m.C = cmake(0.0, 0.0);
#pragma unroll
    for (int e = HP_FS_EMAX - 1; e >= 0; --e) {
        const int i = i_lo + e;
        if (e < E && i < n) {
            const size_t f = (size_t)i * b + j0;
            const cplx uu = up[f], dd = invd[f];
            m.C = cmul(cfms(uu, m.C, y[e]), dd);             // C <- (y - up C) invd
            m.A = cneg(cmul(cmul(uu, m.A), dd));             // A <- -up invd A
        }
    }
    cplx xn = hp_aff_block_enter(m, true, sm);
    cplx* o = out + (size_t)t * n;
#pragma unroll
    for (int e = HP_FS_EMAX - 1; e >= 0; --e) {
        const int i = i_lo + e;
        if (e < E && i < n) {
            const size_t f = (size_t)i * b + j0;
            xn = cmul(cfms(up[f], xn, y[e]), invd[f]);
            o[i] = mode == 1 ? csub(base[i], xn) : xn;
        }
    }
}

// u_row[c] -= fac * is1t[2(c+1)] * src[c]
__global__ void hp_row_couple_kernel(int n, cplx fac, const cplx* __restrict__ is1t, const cplx* __restrict__ src,
                                     cplx* __restrict__ row) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n) row[c] = cfms(cmul(fac, is1t[2 * (c + 1)]), src[c], row[c]);
}

int hp_front_setup(hp_solver* s, cudaStream_t st) {
    size_t sz = sizeof(cplx) * (size_t)s->b * s->n;
    if (!s->f_low) {
        HP_CUDA(cudaMalloc(&s->f_low, sz));
        HP_CUDA(cudaMalloc(&s->f_invd, sz));
        HP_CUDA(cudaMalloc(&s->f_up, sz));
        HP_CUDA(cudaMalloc(&s->TF, sz + sizeof(cplx) * (size_t)s->b * s->n));   // TF followed by the work rows
    }
    double ih2 = 1.0 / (s->pml.h * s->pml.h);
    hp_count_launch();
    if (s->kappa_c) hp_front_factor_kernel<<<1, 32, 0, st>>>(s->n, s->b, ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t,
                                                             (const cplx*)s->kappa_c, s->f_low, s->f_invd, s->f_up, s->status);
    else hp_front_factor_kernel<<<1, 32, 0, st>>>(s->n, s->b, ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t,
                                                  (const double*)s->kappa, s->f_low, s->f_invd, s->f_up, s->status);
    HP_CUDA(cudaGetLastError());
    if (s->front_mode == 1) return hp_front_coupled_setup(s, st);
    hp_front_coupled_free(s);
    return 0;
}

extern "C" int hp_front_begin(hp_solver* s, double* u_dev, void* stream) {
    if (!s || !s->f_low) { hp_set_error("hp_front_begin: preconditioner not set up"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    const int n = s->n, b = s->b;
    cplx* u = (cplx*)u_dev;
    cplx* work = s->TF + (size_t)b * n;
    if (s->front_mode == 1) {
        if (hp_front_coupled_solve(s, 0, 0, u, s->TF, nullptr, cmake(0, 0), st)) return 2;
    } else if (n <= HP_FS_THREADS * HP_FS_EMAX) {
        hp_count_launch();
        hp_front_scan_kernel<<<b, HP_FS_THREADS, 0, st>>>(n, b, 0, 0, s->f_low, s->f_invd, s->f_up, u, s->TF, nullptr, cmake(0, 0), s->is1t);
    } else {
        hp_count_launch();
        hp_front_solve_kernel<<<1, 32, 0, st>>>(n, b, 0, b, 0, s->f_low, s->f_invd, s->f_up, u, s->TF, nullptr, cmake(0, 0), s->is1t, work);
    }
    if (b < n) {
        // u_{b+1} -= A_{b+1,b} (T_F u_F)_b : A_{b+1,b} = diag(c3) of grid row b+1 (code.py:145-154, :365)
        double ih2 = 1.0 / (s->pml.h * s->pml.h);
        cplx fac = cscale(ih2, s->s2t_h[2 * (b + 1) - 1]);
        hp_count_launch(); hp_row_couple_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, fac, s->is1t, s->TF + (size_t)(b - 1) * n,
                                                              u + (size_t)b * n);
    }
    HP_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int hp_front_end(hp_solver* s, double* u_dev, void* stream) {
    if (!s || !s->f_low) { hp_set_error("hp_front_end: preconditioner not set up"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    const int n = s->n, b = s->b;
    cplx* u = (cplx*)u_dev;
    cplx* work = s->TF + (size_t)b * n;
    if (s->front_mode == 1) {
        // u_F = T_F u_F - H_F^{-1} [0; A_{b,b+1} u_{b+1}] with the full H_F: every row of u_F changes
        if (b < n) {
            double ih2 = 1.0 / (s->pml.h * s->pml.h);
            cplx fac = cscale(ih2, s->s2t_h[2 * b + 1]);
            return hp_front_coupled_solve(s, 2, 2, u + (size_t)b * n, u, s->TF, fac, st);
        }
        HP_CUDA(cudaMemcpyAsync(u, s->TF, sizeof(cplx) * (size_t)b * n, cudaMemcpyDeviceToDevice, st));
        return 0;
    }
    if (b > 1) HP_CUDA(cudaMemcpyAsync(u, s->TF, sizeof(cplx) * (size_t)(b - 1) * n, cudaMemcpyDeviceToDevice, st));
    if (b < n) {
        // u_b = (T_F u_F)_b - Tri_b^{-1} (A_{b,b+1} u_{b+1}) : A_{b,b+1} = diag(c4) of grid row b (code.py:131-140)
        double ih2 = 1.0 / (s->pml.h * s->pml.h);
        cplx fac = cscale(ih2, s->s2t_h[2 * b + 1]);
        hp_count_launch();
        if (n <= HP_FS_THREADS * HP_FS_EMAX)
            hp_front_scan_kernel<<<1, HP_FS_THREADS, 0, st>>>(n, b, b - 1, 1, s->f_low, s->f_invd, s->f_up, u + (size_t)b * n,
                                                            u + (size_t)(b - 1) * n, s->TF + (size_t)(b - 1) * n, fac, s->is1t);
        else
            hp_front_solve_kernel<<<1, 32, 0, st>>>(n, b, b - 1, 1, 1, s->f_low, s->f_invd, s->f_up, u + (size_t)b * n,
                                                    u + (size_t)(b - 1) * n, s->TF + (size_t)(b - 1) * n, fac, s->is1t, work);
    } else {
        HP_CUDA(cudaMemcpyAsync(u + (size_t)(b - 1) * n, s->TF + (size_t)(b - 1) * n, sizeof(cplx) * n,
                                cudaMemcpyDeviceToDevice, st));
    }
    HP_CUDA(cudaGetLastError());
    return 0;
}

// T_F u_F lives in the solver between hp_front_begin and hp_front_end; with several right-hand sides in flight
// (slab.py pipelines them through the slabs) the caller parks it in its own buffer of b*n complex numbers.
// dir 0: solver -> buf_dev, dir 1: buf_dev -> solver.
extern "C" int hp_front_tf_copy(hp_solver* s, double* buf_dev, int dir, void* stream) {
    if (!s || !s->TF) { hp_set_error("hp_front_tf_copy: preconditioner not set up"); return 1; }
    size_t sz = sizeof(cplx) * (size_t)s->b * s->n;
    HP_CUDA(cudaMemcpyAsync(dir == 0 ? (void*)buf_dev : (void*)s->TF, dir == 0 ? (const void*)s->TF : (const void*)buf_dev, sz,
                            cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}
