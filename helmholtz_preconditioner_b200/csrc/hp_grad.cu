// Inversion: the n^2-sized products of the adjoint-state gradient and of Born modelling (helmholtz_preconditioner_b200/
// inversion.py).  The reference has no counterpart; the solves these kernels sit between are the existing ones.
//
// The operator depends on the slowness^2 kappa = 1/c^2 through its diagonal only (hp_point_coef, csrc/hp_assembly.cu):
//     dA_pp / dkappa_p = w_p = omega^2 * is1t[2i] * is2t[2j],   p = (j-1) n + (i-1),
// the factor c5 multiplies kappa by.  With A u_s = f_s, the adjoint field mu_s (A mu_s = R^T conj(r_s), A is complex
// symmetric) and the misfit J = 1/2 sum_s |R u_s - d_s|^2, the gradient G = dJ/dRe kappa + i dJ/dIm kappa is
//     G_p = -conj(w_p * sum_s mu_s,p u_s,p),
// and the Born source of a perturbation dkappa is -w (.) dkappa (.) u_s.  All three kernels are plain streams (HBM-bound):
//     hp_grad_accumulate  (2R + 2) * 16 B per point  (R pairs u, mu read; acc read and written)
//     hp_grad_finish      16 + 8 + 8 B (real medium), 16 + 16 + 16 B (attenuating) per point
//     hp_born_source      (2R + 1) * 16 B per point  (dkappa read once, R fields read and written)
// Every point is computed by one thread with a fixed order of operations: the results are deterministic, and splitting
// the sources of hp_grad_accumulate over several launches (in the same order) gives the same bits.
#include "hp_internal.cuh"

#define HP_GRAD_THREADS 256
#define HP_GRAD_RMAX 8

struct HpGradSlots {               // R <= 8 field pointers by value; NULL = inactive slot
    const cplx* a[HP_GRAD_RMAX];
    const cplx* b[HP_GRAD_RMAX];
    cplx* out[HP_GRAD_RMAX];
};

// w_p = omega^2 is1(i) is2(j), i, j 1-based: the same expression hp_point_coef multiplies kappa by
__device__ __forceinline__ cplx hp_grad_w(int i, int j, cplx omega2, const cplx* __restrict__ is1t,
                                         const cplx* __restrict__ is2t) {
    return cmul(omega2, cmul(is1t[2 * i], is2t[2 * j]));
}

// principal square root (branch cut on the negative real axis); (x, 0) with x >= 0 gives (sqrt(x), 0)
__device__ __forceinline__ cplx hp_csqrt(cplx z) {
    const double r = hypot(z.x, z.y);
    if (r == 0.0) return cmake(0.0, 0.0);
    if (z.x >= 0.0) {
        const double t = sqrt(0.5 * (r + z.x));
        return cmake(t, z.y / (2.0 * t));
    }
    const double t = sqrt(0.5 * (r - z.x));
    return cmake(fabs(z.y) / (2.0 * t), copysign(t, z.y));
}

// acc[p] += u_r[p] mu_r[p] for the active slots r = 0..R-1 in slot order
__global__ void __launch_bounds__(HP_GRAD_THREADS) hp_grad_accumulate_kernel(int64_t N, int R, HpGradSlots sl,
                                                                            cplx* __restrict__ acc) {
    const int64_t p = (int64_t)blockIdx.x * HP_GRAD_THREADS + threadIdx.x;
    if (p >= N) return;
    cplx u[HP_GRAD_RMAX], m[HP_GRAD_RMAX];
#pragma unroll
    for (int r = 0; r < HP_GRAD_RMAX; ++r)           // every load issued before the first use
        if (r < R && sl.a[r]) { u[r] = __ldg(sl.a[r] + p); m[r] = __ldg(sl.b[r] + p); }
    cplx s = acc[p];
#pragma unroll
    for (int r = 0; r < HP_GRAD_RMAX; ++r)
        if (r < R && sl.a[r]) s = cfma(u[r], m[r], s);
    acc[p] = s;
}

// G = -conj(w acc), times conj(-2 kappa sqrt(kappa)) = conj(dkappa/dc) for wrt = 1, written in c_mat layout
// out[(i-1)(n+2) + (j-1)] through the 32x32 shared-memory transpose of hp_kappa_kernel; the last two rows and columns
// are exact zeros.  KT = double: real medium, out holds Re G; KT = cplx: attenuating medium, out holds G.
__device__ __forceinline__ double hp_grad_out(cplx g, double kap, int wrt) {
    return wrt ? (-2.0 * kap * sqrt(kap)) * g.x : g.x;
}
__device__ __forceinline__ cplx hp_grad_out(cplx g, cplx kap, int wrt) {
    if (!wrt) return g;
    const cplx d = cscale(-2.0, cmul(kap, hp_csqrt(kap)));
    return cmul(cmake(d.x, -d.y), g);
}
template <typename KT>
__global__ void hp_grad_finish_kernel(int n, cplx omega2, const cplx* __restrict__ is1t, const cplx* __restrict__ is2t,
                                      const KT* __restrict__ kappa, const cplx* __restrict__ acc, int wrt,
                                      KT* __restrict__ out) {
    __shared__ KT tile[32][33];
    const int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int j = j0 + r, i = i0 + threadIdx.x;        // grid-aligned read, i fastest
        if (i < n && j < n) {
            const size_t p = (size_t)j * n + i;
            const cplx w = hp_grad_w(i + 1, j + 1, omega2, is1t, is2t), a = acc[p];
            // -conj(w a), with the real part rounded the same way for both media
            const cplx g = cmake(-fma(w.x, a.x, -(w.y * a.y)), fma(w.x, a.y, w.y * a.x));
            tile[r][threadIdx.x] = hp_grad_out(g, kappa[p], wrt);
        }
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = i0 + r, j = j0 + threadIdx.x;        // c_mat layout write, j fastest
        if (i < n + 2 && j < n + 2) out[(size_t)i * (n + 2) + j] = (i < n && j < n) ? tile[threadIdx.x][r] : KT{};
    }
}

// out_r[p] = -w_p dkappa_p u_r[p] for the active slots; dkappa in c_mat layout (entry [i-1][j-1] of an (n+2)^2 array) is
// transposed once per CTA and applied to every slot.  out_r may be u_r.
__global__ void hp_born_source_kernel(int n, cplx omega2, const cplx* __restrict__ is1t, const cplx* __restrict__ is2t,
                                      const cplx* __restrict__ dkappa, int R, HpGradSlots sl) {
    __shared__ cplx tile[32][33];
    const int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int i = i0 + r, j = j0 + threadIdx.x;        // read dkappa[i][j], j fastest
        if (i < n && j < n) tile[r][threadIdx.x] = dkappa[(size_t)i * (n + 2) + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int j = j0 + r, i = i0 + threadIdx.x;        // grid-aligned, i fastest
        if (i < n && j < n) {
            const size_t p = (size_t)j * n + i;
            const cplx c = cneg(cmul(hp_grad_w(i + 1, j + 1, omega2, is1t, is2t), tile[threadIdx.x][r]));
            cplx u[HP_GRAD_RMAX];
#pragma unroll
            for (int s = 0; s < HP_GRAD_RMAX; ++s)       // every load before the first store (out_r may alias u_r)
                if (s < R && sl.a[s]) u[s] = sl.a[s][p];
#pragma unroll
            for (int s = 0; s < HP_GRAD_RMAX; ++s)
                if (s < R && sl.a[s]) sl.out[s][p] = cmul(c, u[s]);
        }
    }
}

// slot checks shared by the multi-field entry points: R in 1..8, a[r] and b[r] both NULL or both set, one slot active
static int hp_grad_slots(const char* what, int R, const double* const* a, const void* const* b, const char* an,
                         const char* bn, HpGradSlots& sl) {
    if (R < 1 || R > HP_GRAD_RMAX) { hp_set_error("%s: R must lie in 1..%d, got %d", what, HP_GRAD_RMAX, R); return 1; }
    if (!a || !b) { hp_set_error("%s: null pointer array", what); return 1; }
    int active = 0;
    for (int r = 0; r < HP_GRAD_RMAX; ++r) { sl.a[r] = sl.b[r] = nullptr; sl.out[r] = nullptr; }
    for (int r = 0; r < R; ++r) {
        if (!a[r] != !b[r]) {
            hp_set_error("%s: slot %d has %s %s but %s %s (both or neither must be NULL)", what, r, a[r] ? "a" : "no", an,
                         b[r] ? "a" : "no", bn);
            return 1;
        }
        sl.a[r] = (const cplx*)a[r];
        sl.b[r] = (const cplx*)b[r];
        sl.out[r] = (cplx*)b[r];
        active += a[r] != nullptr;
    }
    if (!active) { hp_set_error("%s: all %d slots are empty", what, R); return 1; }
    return 0;
}

extern "C" int hp_grad_accumulate(hp_solver* s, int R, const double* const* u_devs, const double* const* mu_devs,
                                  double* acc_dev, void* stream) {
    if (!s) { hp_set_error("hp_grad_accumulate: null solver"); return 1; }
    if (!acc_dev) { hp_set_error("hp_grad_accumulate: null accumulator"); return 1; }
    HpGradSlots sl;
    if (hp_grad_slots("hp_grad_accumulate", R, u_devs, (const void* const*)mu_devs, "field u", "adjoint field mu", sl)) return 1;
    const int64_t N = (int64_t)s->n * s->n;
    hp_count_launch();
    hp_grad_accumulate_kernel<<<(unsigned)((N + HP_GRAD_THREADS - 1) / HP_GRAD_THREADS), HP_GRAD_THREADS, 0,
                                (cudaStream_t)stream>>>(N, R, sl, (cplx*)acc_dev);
    HP_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int hp_grad_finish(hp_solver* s, const double* acc_dev, int wrt, double* out_dev, void* stream) {
    if (!s) { hp_set_error("hp_grad_finish: null solver"); return 1; }
    if (!acc_dev || !out_dev) { hp_set_error("hp_grad_finish: null %s", acc_dev ? "output" : "accumulator"); return 1; }
    if (wrt != 0 && wrt != 1) { hp_set_error("hp_grad_finish: wrt must be 0 (slowness^2) or 1 (velocity), got %d", wrt); return 1; }
    const int n = s->n;
    dim3 blk(32, 8), grd((n + 2 + 31) / 32, (n + 2 + 31) / 32);
    hp_count_launch();
    if (s->kappa_c) hp_grad_finish_kernel<<<grd, blk, 0, (cudaStream_t)stream>>>(
        n, s->omega2, s->is1t, s->is2t, (const cplx*)s->kappa_c, (const cplx*)acc_dev, wrt, (cplx*)out_dev);
    else hp_grad_finish_kernel<<<grd, blk, 0, (cudaStream_t)stream>>>(
        n, s->omega2, s->is1t, s->is2t, (const double*)s->kappa, (const cplx*)acc_dev, wrt, out_dev);
    HP_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int hp_born_source(hp_solver* s, int R, const double* dkappa_dev, const double* const* u_devs,
                              double* const* out_devs, void* stream) {
    if (!s) { hp_set_error("hp_born_source: null solver"); return 1; }
    if (!dkappa_dev) { hp_set_error("hp_born_source: null dkappa"); return 1; }
    HpGradSlots sl;
    if (hp_grad_slots("hp_born_source", R, u_devs, (const void* const*)out_devs, "field u", "output", sl)) return 1;
    const int n = s->n;
    dim3 blk(32, 8), grd((n + 31) / 32, (n + 31) / 32);
    hp_count_launch();
    hp_born_source_kernel<<<grd, blk, 0, (cudaStream_t)stream>>>(n, s->omega2, s->is1t, s->is2t, (const cplx*)dkappa_dev,
                                                                  R, sl);
    HP_CUDA(cudaGetLastError());
    return 0;
}
