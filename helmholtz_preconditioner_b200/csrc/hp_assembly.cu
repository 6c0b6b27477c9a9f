// Operator A: PML tables, CSR assembly and the matrix-free 5-point stencil matvec.
//
// Replaces the numba assembly loops get_A_diag_block_coeffs / get_upper_A_block / get_lower_A_block and
// the scipy glue of build_A_matrix (/root/reference/code.py:71-219).  The coefficient of grid point (i, j)
// towards its neighbours is separable,
//     c1 = s1((i-.5)h)/(h^2 s2(jh))   c2 = s1((i+.5)h)/(h^2 s2(jh))
//     c3 = s2((j-.5)h)/(h^2 s1(ih))   c4 = s2((j+.5)h)/(h^2 s1(ih))
//     c5 = omega^2/(s1 s2 c^2) - (c1+c2+c3+c4),
// so the stretching factors are evaluated once per grid line (2n+3 half-grid points per axis, kernel
// hp_tables_kernel) and the per-point work is a handful of complex multiplies: both kernels below are
// HBM-bound (CSR: 104 B written per row; matvec: 40 B per grid point, 48 B for an attenuating medium).
// The kernels that read the slowness^2 kappa = 1/c^2 are templates on its type: double for a real medium, cplx for an
// attenuating one (hp_create_complex); the real instances are the code of the real-only kernels.
#include "hp_internal.cuh"
#include <stdlib.h>

__global__ void hp_tables_kernel(int n, HpPml p, cplx* s1t, cplx* is1t, cplx* s2t, cplx* is2t) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t <= 2 * n + 2) hp_table_entry(t, p, s1t + t, is1t + t, s2t + t, is2t + t);
}

// kappa[(j-1) n + (i-1)] = 1/c_mat[i-1][j-1]^2 : the reference's transposed velocity lookup (code.py:108)
// turned into a grid-aligned array so that the stencil kernels read it coalesced.  32x32 smem transpose.
__global__ void hp_kappa_kernel(int n, const double* __restrict__ c_mat, double* __restrict__ kappa) {
    __shared__ double tile[32][33];
    int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int i = i0 + r, j = j0 + threadIdx.x;        // read c_mat[i][j], j fastest
        if (i < n && j < n) tile[r][threadIdx.x] = c_mat[(size_t)i * (n + 2) + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int j = j0 + r, i = i0 + threadIdx.x;        // write kappa[j][i], i fastest
        if (i < n && j < n) {
            double c = tile[threadIdx.x][r];
            kappa[(size_t)j * n + i] = 1.0 / (c * c);
        }
    }
}

// the same for an attenuating medium: kappa_c = 1/(c*c) with the complex multiply and Smith's division of hp_small.h, so
// that c = (cr, 0) gives (1/cr^2, 0) bit for bit.  c_mat is (n+2)^2 interleaved complex.
__global__ void hp_kappa_c_kernel(int n, const cplx* __restrict__ c_mat, cplx* __restrict__ kappa_c) {
    __shared__ cplx tile[32][33];
    int i0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int i = i0 + r, j = j0 + threadIdx.x;
        if (i < n && j < n) tile[r][threadIdx.x] = c_mat[(size_t)i * (n + 2) + j];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int j = j0 + r, i = i0 + threadIdx.x;
        if (i < n && j < n) {
            cplx c = tile[threadIdx.x][r];
            kappa_c[(size_t)j * n + i] = cinv(cmul(c, c));
        }
    }
}

// c_cplx: the (n+2)^2 complex velocity on the device for an attenuating medium (s->kappa_c set), unused otherwise
int hp_launch_tables(hp_solver* s, const cplx* c_cplx, cudaStream_t st) {
    int n = s->n, len = 2 * n + 3;
    hp_count_launch(); hp_tables_kernel<<<(len + 127) / 128, 128, 0, st>>>(n, s->pml, s->s1t, s->is1t, s->s2t, s->is2t);
    dim3 blk(32, 8), grd((n + 31) / 32, (n + 31) / 32);
    if (s->kappa_c) { hp_count_launch(); hp_kappa_c_kernel<<<grd, blk, 0, st>>>(n, c_cplx, s->kappa_c); }
    else { hp_count_launch(); hp_kappa_kernel<<<grd, blk, 0, st>>>(n, s->c_mat, s->kappa); }
    HP_CUDA(cudaGetLastError());
    return 0;
}

struct HpPointCoef { cplx c1, c2, c3, c4, c5; };

template <typename KT>
__device__ __forceinline__ HpPointCoef hp_point_coef(int i, int j, int n, double ih2, cplx omega2,
                                                     const cplx* __restrict__ s1t, const cplx* __restrict__ is1t,
                                                     const cplx* __restrict__ s2t, const cplx* __restrict__ is2t,
                                                     KT kap) {
    // i, j are 1-based grid indices
    cplx is2c = is2t[2 * j], is1c = is1t[2 * i];
    HpPointCoef c;
    c.c1 = cscale(ih2, cmul(s1t[2 * i - 1], is2c));
    c.c2 = cscale(ih2, cmul(s1t[2 * i + 1], is2c));
    c.c3 = cscale(ih2, cmul(s2t[2 * j - 1], is1c));
    c.c4 = cscale(ih2, cmul(s2t[2 * j + 1], is1c));
    c.c5 = hp_kmul_sub(kap, cmul(omega2, cmul(is1c, is2c)), cadd(cadd(c.c1, c.c2), cadd(c.c3, c.c4)));
    return c;
}

// One thread per matrix row.  Row r = (j-1) n + (i-1) stores, in ascending column order, the couplings
// to (i, j-1), (i-1, j), itself, (i+1, j), (i, j+1); neighbours outside the grid are dropped.  The row
// offset has a closed form, so indptr needs no scan.  The rows of a CTA are consecutive, hence so are their
// entries: they are assembled in shared memory and written out with consecutive threads on consecutive entries
// (a thread writing its own 3-5 entries would touch every 32-byte sector five times).
#define HP_ASM_THREADS 256
__device__ __forceinline__ int64_t hp_csr_row_offset(int64_t r, int64_t nn) {
    const int64_t j0 = r / nn, i0 = r - j0 * nn;
    return 5 * r - (r < nn ? r : nn) - (r > (nn - 1) * nn ? r - (nn - 1) * nn : 0) - (j0 + (i0 > 0 ? 1 : 0)) - j0;
}
template <typename KT>
__global__ void __launch_bounds__(HP_ASM_THREADS) hp_assemble_csr_kernel(int n, double ih2, cplx omega2,
        const cplx* __restrict__ s1t, const cplx* __restrict__ is1t, const cplx* __restrict__ s2t,
        const cplx* __restrict__ is2t, const KT* __restrict__ kappa,
        int32_t* __restrict__ indptr, int32_t* __restrict__ indices, cplx* __restrict__ data) {
    __shared__ cplx sdata[HP_ASM_THREADS * 5];
    __shared__ int32_t sidx[HP_ASM_THREADS * 5];
    const int64_t N = (int64_t)n * n, nn = n;
    const int64_t r0 = (int64_t)blockIdx.x * HP_ASM_THREADS, r = r0 + threadIdx.x;
    const int64_t rend = r0 + HP_ASM_THREADS < N ? r0 + HP_ASM_THREADS : N;
    const int64_t off0 = hp_csr_row_offset(r0, nn);
    const int64_t off1 = rend < N ? hp_csr_row_offset(rend, nn) : 5 * N - 4 * nn;
    if (r < N) {
        const int j0 = (int)(r / n), i0 = (int)(r % n);
        const int64_t off = hp_csr_row_offset(r, nn);
        HpPointCoef c = hp_point_coef(i0 + 1, j0 + 1, n, ih2, omega2, s1t, is1t, s2t, is2t, kappa[r]);
        indptr[r] = (int32_t)off;
        int o = (int)(off - off0);
        if (j0 > 0)     { sidx[o] = (int32_t)(r - n); sdata[o] = c.c3; ++o; }
        if (i0 > 0)     { sidx[o] = (int32_t)(r - 1); sdata[o] = c.c1; ++o; }
                          sidx[o] = (int32_t)r;       sdata[o] = c.c5; ++o;
        if (i0 < n - 1) { sidx[o] = (int32_t)(r + 1); sdata[o] = c.c2; ++o; }
        if (j0 < n - 1) { sidx[o] = (int32_t)(r + n); sdata[o] = c.c4; ++o; }
        if (r == N - 1) indptr[N] = (int32_t)(off0 + o);
    }
    __syncthreads();
    const int cnt = (int)(off1 - off0);
    for (int e = threadIdx.x; e < cnt; e += HP_ASM_THREADS) {
        data[off0 + e] = sdata[e];
        indices[off0 + e] = sidx[e];
    }
}

// Strip operator H_m as sorted CSR (get_Hm, /root/reference/code.py:283-290): the 5-point operator of the b grid rows
// m-b+1..m with the x2 PML moved to end on row m (s2m).  Row r = k n + (i-1) (k = 0..b-1 local grid row) holds the
// couplings to (i, k-1), (i-1, k), itself, (i+1, k), (i, k+1); the entries the reference zeroes across the row ends
// (c1_vec[n-1::n] = 0) and the ones outside the strip are not stored.  Thread -> grid column i: the coefficients come
// from the same hp_strip_rows / hp_block_row the factorisation uses (csrc/hp_setup_core.h).
__device__ __forceinline__ int64_t hp_strip_row_offset(int64_t r, int64_t nn, int64_t b) {
    const int64_t k0 = r / nn, i0 = r - k0 * nn;
    return 5 * r - (r < nn ? r : nn) - (r > (b - 1) * nn ? r - (b - 1) * nn : 0) - (k0 + (i0 > 0 ? 1 : 0)) - k0;
}
template <bool CK>
__global__ void hp_strip_csr_kernel(HpStripCtx c, int m, int32_t* __restrict__ indptr, int32_t* __restrict__ indices,
                                    cplx* __restrict__ data) {
    const int i0 = blockIdx.x * blockDim.x + threadIdx.x;       // 0-based column
    const int n = c.n, b = c.b;
    if (i0 >= n) return;
    HpStripRow R;
    hp_strip_rows(R, m, b, c.pml);
    HpBlockRow B;
    hp_block_row<CK>(B, R, i0 + 1, m, b, n, c.pml, c.s1t, c.is1t, c.c_mat, c.omega2, c.kappa_c);
    for (int k = 0; k < b; ++k) {
        const int64_t r = (int64_t)k * n + i0;
        int64_t o = hp_strip_row_offset(r, n, b);
        indptr[r] = (int32_t)o;
        if (k > 0)      { indices[o] = (int32_t)(r - n); data[o] = B.sub[k]; ++o; }
        if (i0 > 0)     { indices[o] = (int32_t)(r - 1); data[o] = B.L[k]; ++o; }
                          indices[o] = (int32_t)r;       data[o] = B.dia[k]; ++o;
        if (i0 < n - 1) { indices[o] = (int32_t)(r + 1); data[o] = B.U[k]; ++o; }
        if (k < b - 1)  { indices[o] = (int32_t)(r + n); data[o] = B.sup[k]; ++o; }
        if (r == (int64_t)b * n - 1) indptr[r + 1] = (int32_t)o;
    }
}
extern "C" int64_t hp_strip_csr_nnz(int n, int b) { return 5 * (int64_t)b * n - 2 * (int64_t)n - 2 * (int64_t)b; }
extern "C" int hp_assemble_strip_csr(hp_solver* s, int m, int32_t* indptr_dev, int32_t* indices_dev, double* data_dev, void* stream) {
    if (!s) { hp_set_error("hp_assemble_strip_csr: null solver"); return 1; }
    if (m < s->b || m > s->n) { hp_set_error("hp_assemble_strip_csr: layer m must lie in %d..%d, got %d", s->b, s->n, m); return 1; }
    hp_count_launch();
    if (s->kappa_c) hp_strip_csr_kernel<true><<<(s->n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(hp_ctx(s), m, indptr_dev, indices_dev, (cplx*)data_dev);
    else hp_strip_csr_kernel<false><<<(s->n + 63) / 64, 64, 0, (cudaStream_t)stream>>>(hp_ctx(s), m, indptr_dev, indices_dev, (cplx*)data_dev);
    HP_CUDA(cudaGetLastError());
    return 0;
}

// Matrix-free y = A x.  A CTA owns 128 consecutive x1 columns and marches over HP_SPMV_ROWS grid rows;
// each thread keeps the x2 neighbours (south, centre, north) of its column in registers, takes the x1
// neighbours from the adjacent lanes by shuffle (warp-edge lanes read them from L1/L2) and keeps the
// x1-dependent factors in registers for the whole march.  Algorithmic traffic per grid point:
// x 16 B read + y 16 B written + kappa 8 B read = 40 B (48 B with the complex kappa of an attenuating medium).
// The march length (rows per CTA) is chosen by the host so that the whole grid is ONE wave of resident CTAs
// (hp_spmv_rows): with a fixed 16 rows the 8192 CTAs of 4096^2 ran as 6.9 waves of 1184 and the last, partly filled
// wave cost 7 % of the kernel; longer marches also read fewer halo rows twice (2 per march).
#define HP_SPMV_MIN_ROWS 16
// Rows j_lo <= j < j_hi (0-based) of the grid: x and y hold those rows only (slab storage); the rows just
// outside come from the halo pointers x_south (row j_lo-1) and x_north (row j_hi), NULL on the grid boundary.
template <typename KT>
__global__ void __launch_bounds__(128) hp_stencil_matvec_kernel(int n, int j_lo, int j_hi, int rows, int pf, double ih2, cplx omega2,
        const cplx* __restrict__ s1t, const cplx* __restrict__ is1t, const cplx* __restrict__ s2t,
        const cplx* __restrict__ is2t, const KT* __restrict__ kappa,
        const cplx* __restrict__ x, const cplx* __restrict__ x_south, const cplx* __restrict__ x_north,
        cplx* __restrict__ y) {
    const int col = blockIdx.x * 128 + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int j0 = j_lo + blockIdx.y * rows;
    const bool act = col < n;
    const cplx zero = cmake(0.0, 0.0);
    cplx aW = zero, aE = zero, dI = zero, wI = zero;
    if (act) {
        aW = cscale(ih2, s1t[2 * col + 1]);       // s1((i-.5)h)/h^2, i = col+1
        aE = cscale(ih2, s1t[2 * col + 3]);       // s1((i+.5)h)/h^2
        dI = is1t[2 * col + 2];                   // 1/s1(ih)
        wI = cmul(omega2, dI);
    }
    cplx xS = zero;
    if (act) {
        if (j0 > j_lo) xS = x[(size_t)(j0 - 1 - j_lo) * n + col];
        else if (x_south) xS = x_south[col];
    }
    cplx xC = act ? x[(size_t)(j0 - j_lo) * n + col] : zero;
    const int j1 = min(j_hi, j0 + rows);
#pragma unroll 4
    const int pcols = min(128, n - (int)blockIdx.x * 128);
    for (int j = j0; j < j1; ++j) {                 // 0-based grid row, uniform over the CTA
        const size_t base = (size_t)(j - j_lo) * n;
        // HBM -> L2 a few rows ahead of the march (one bulk prefetch per row segment): the demand loads below then
        // wait for an L2 hit instead of a DRAM access, and a third of the bytes in flight per SM sustain the same bandwidth
        if (pf > 0 && threadIdx.x == 0 && j + pf < j1) {
            if (j + pf + 1 < j_hi)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(x + base + (size_t)(pf + 1) * n + blockIdx.x * 128), "r"(pcols * 16) : "memory");
            // a bulk prefetch wants 16-byte aligned rows: always so for a complex kappa, for n even for a real one
            if (sizeof(KT) == 16 || (n & 1) == 0)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(kappa + (size_t)(j + pf) * n + blockIdx.x * 128), "r"(pcols * (int)sizeof(KT)) : "memory");
        }
        cplx xN = zero;
        if (act) {
            if (j + 1 < j_hi) xN = x[base + n + col];
            else if (x_north) xN = x_north[col];
        }
        KT kap = act ? kappa[(size_t)j * n + col] : KT{};
        cplx xW, xE;
        xW.x = __shfl_up_sync(0xffffffffu, xC.x, 1);
        xW.y = __shfl_up_sync(0xffffffffu, xC.y, 1);
        xE.x = __shfl_down_sync(0xffffffffu, xC.x, 1);
        xE.y = __shfl_down_sync(0xffffffffu, xC.y, 1);
        if (lane == 0) xW = (act && col > 0) ? x[base + col - 1] : zero;
        if (lane == 31) xE = (col + 1 < n) ? x[base + col + 1] : zero;
        const cplx bJ = is2t[2 * j + 2];                       // 1/s2(jh)
        const cplx gS = cscale(ih2, s2t[2 * j + 1]);            // s2((j-.5)h)/h^2
        const cplx gN = cscale(ih2, s2t[2 * j + 3]);            // s2((j+.5)h)/h^2
        // y = c5 xC + c1 xW + c2 xE + c3 xS + c4 xN with c5 = kappa omega^2 dI bJ - (c1+c2+c3+c4)
        cplx t1 = cfma(aW, csub(xW, xC), cmul(aE, csub(xE, xC)));
        cplx t2 = cfma(gS, csub(xS, xC), cmul(gN, csub(xN, xC)));
        cplx acc = cmul(hp_kmul(kap, cmul(wI, bJ)), xC);
        acc = cfma(bJ, t1, acc);
        acc = cfma(dI, t2, acc);
        if (act) y[base + col] = acc;
        xS = xC;
        xC = xN;
    }
}

__global__ void __launch_bounds__(256) hp_csr_matvec_kernel(int64_t nrows, const int32_t* __restrict__ indptr,
        const int32_t* __restrict__ indices, const cplx* __restrict__ data, const cplx* __restrict__ x,
        cplx* __restrict__ y) {
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    cplx acc = cmake(0.0, 0.0);
    for (int32_t e = indptr[r]; e < indptr[r + 1]; ++e) acc = cfma(data[e], x[indices[e]], acc);
    y[r] = acc;
}

extern "C" int64_t hp_csr_nnz(int n) { return 5 * (int64_t)n * n - 4 * (int64_t)n; }

extern "C" int hp_assemble_csr(hp_solver* s, int32_t* indptr, int32_t* indices, double* data, void* stream) {
    if (!s) { hp_set_error("hp_assemble_csr: null solver"); return 1; }
    if (hp_csr_nnz(s->n) > 2147483647LL) { hp_set_error("hp_assemble_csr: nnz exceeds int32 indices"); return 1; }
    int64_t N = (int64_t)s->n * s->n;
    double ih2 = 1.0 / (s->pml.h * s->pml.h);
    const unsigned grd = (unsigned)((N + HP_ASM_THREADS - 1) / HP_ASM_THREADS);
    hp_count_launch();
    if (s->kappa_c) hp_assemble_csr_kernel<<<grd, HP_ASM_THREADS, 0, (cudaStream_t)stream>>>(
        s->n, ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t, (const cplx*)s->kappa_c, indptr, indices, (cplx*)data);
    else hp_assemble_csr_kernel<<<grd, HP_ASM_THREADS, 0, (cudaStream_t)stream>>>(
        s->n, ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t, (const double*)s->kappa, indptr, indices, (cplx*)data);
    HP_CUDA(cudaGetLastError());
    return 0;
}

// rows per CTA such that the grid fills the resident CTA slots of the device once (HP_SPMV_ROWS overrides)
static int hp_spmv_rows(int n, int nrows) {
    static int slots = 0, forced = -1;
    if (forced < 0) { const char* e = getenv("HP_SPMV_ROWS"); forced = e ? atoi(e) : 0; }
    if (forced > 0) return forced;
    if (!slots) {
        int dev = 0, sms = 0, per_sm = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hp_stencil_matvec_kernel<double>, 128, 0) == cudaSuccess && per_sm > 0)
            slots = sms * per_sm;
        else { cudaGetLastError(); slots = 1184; }
    }
    const int colblocks = (n + 127) / 128;
    const int rowblocks = slots / colblocks > 0 ? slots / colblocks : 1;
    const int rows = (nrows + rowblocks - 1) / rowblocks;
    return rows < HP_SPMV_MIN_ROWS ? HP_SPMV_MIN_ROWS : rows;
}

static int hp_spmv_pf() {
    static int pf = -1;
    if (pf < 0) { const char* e = getenv("HP_SPMV_PF"); pf = e ? atoi(e) : 3; }
    return pf;
}

extern "C" int hp_stencil_matvec_rows(hp_solver* s, int j_lo, int j_hi, const double* x, const double* x_south,
                                      const double* x_north, double* y, void* stream) {
    if (!s) { hp_set_error("hp_stencil_matvec: null solver"); return 1; }
    if (j_lo < 0 || j_hi > s->n || j_lo >= j_hi) { hp_set_error("hp_stencil_matvec_rows: bad row range %d..%d", j_lo, j_hi); return 1; }
    double ih2 = 1.0 / (s->pml.h * s->pml.h);
    const int rows = hp_spmv_rows(s->n, j_hi - j_lo);
    dim3 grd((s->n + 127) / 128, (j_hi - j_lo + rows - 1) / rows);
    hp_count_launch();
    if (s->kappa_c) hp_stencil_matvec_kernel<<<grd, 128, 0, (cudaStream_t)stream>>>(
        s->n, j_lo, j_hi, rows, hp_spmv_pf(), ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t, (const cplx*)s->kappa_c, (const cplx*)x,
        (const cplx*)x_south, (const cplx*)x_north, (cplx*)y);
    else hp_stencil_matvec_kernel<<<grd, 128, 0, (cudaStream_t)stream>>>(
        s->n, j_lo, j_hi, rows, hp_spmv_pf(), ih2, s->omega2, s->s1t, s->is1t, s->s2t, s->is2t, (const double*)s->kappa, (const cplx*)x,
        (const cplx*)x_south, (const cplx*)x_north, (cplx*)y);
    HP_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int hp_stencil_matvec(hp_solver* s, const double* x, double* y, void* stream) {
    if (!s) { hp_set_error("hp_stencil_matvec: null solver"); return 1; }
    return hp_stencil_matvec_rows(s, 0, s->n, x, nullptr, nullptr, y, stream);
}

extern "C" int hp_csr_matvec(int64_t nrows, const int32_t* indptr, const int32_t* indices, const double* data,
                             const double* x, double* y, void* stream) {
    hp_count_launch(); hp_csr_matvec_kernel<<<(unsigned)((nrows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        nrows, indptr, indices, (const cplx*)data, (const cplx*)x, (cplx*)y);
    HP_CUDA(cudaGetLastError());
    return 0;
}
