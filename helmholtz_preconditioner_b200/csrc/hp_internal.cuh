// Internal declarations shared by the translation units of libhelmholtz_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "hp_setup_core.h"
#include "../../include/helmholtz_b200.h"

void hp_set_error(const char* fmt, ...);
void hp_count_launch();                       // every kernel launch of the library is counted (hp_launch_count)
struct hp_solver;
void hp_profile_begin(hp_solver* s, cudaStream_t st);   // CUDA-event bracket around the sweep kernel
void hp_profile_end(hp_solver* s, cudaStream_t st, int64_t bytes);

#define HP_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            hp_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
            return 2;                                                                              \
        }                                                                                          \
    } while (0)

// x1 partition of every strip and the packed generator layout ("packets").
//
// The sweep kernel runs G = P*K CTAs; CTA g = l*K + k owns part k of leaf l (columns part c0..c1-1) and the
// rows [g*NR, (g+1)*NR) of the separator inverse N.  Per strip and CTA one contiguous packet of PK complex
// numbers holds everything that CTA streams for that strip:
//     Wp [CW][QP]   rows c0..c1-1 of W_l (zero padded)
//     Gp [2b][CW]   columns c0..c1-1 of [Gf_l; Gl_l]
//     Np [NR][NSP]  its rows of N
// Strip m (m_lo <= m <= m_hi) starts at packets + (m - m_lo) * G * PK.
struct HpLayout {
    int P = 0, K = 0, G = 0;     // leaves, parts per leaf, CTAs
    int QP = 0, CW = 0;          // widest leaf, widest part
    int NS = 0, NSP = 0, NR = 0; // separator unknowns b*(P-1), padded row length, rows of N per CTA
    size_t PK = 0;               // complex numbers per packet
    size_t offG = 0, offN = 0;   // offsets of Gp and Np inside a packet
    // cluster layout (csrc/hp_sweep4.cu): a leaf is one thread-block cluster of K CTAs, N is distributed by the columns
    // of the leaf's right separator: Np [b][NRQ] = N[rows NRQ*k .. NRQ*(k+1)-1][columns of separator l], column major
    int colN = 0;
    int NCB = 0, NRQ = 0, NXG = 0;   // ceil(b/K) separator right-hand sides, ceil(NS/K) rows of x, ceil(3b/K) gathered entries per CTA
};

struct hp_solver {
    int n = 0, b = 0;
    HpPml pml;
    cplx omega2;
    int num_sms = 0;
    // operator tables on the half grid t = 0..2n+2 (unshifted PML)
    cplx *s1t = nullptr, *is1t = nullptr, *s2t = nullptr, *is2t = nullptr;
    std::vector<cplx> s2t_h;      // host copy of s2t (couplings between grid rows are formed on the host)
    double* c_mat = nullptr;      // (n+2)^2 as given (real medium)
    double* kappa = nullptr;      // n*n, kappa[(j-1)*n + (i-1)] = 1 / c_mat[i-1][j-1]^2  (grid-aligned, real medium)
    cplx* kappa_c = nullptr;      // attenuating medium (hp_create_complex): the same n*n array, complex; c_mat and kappa stay NULL
    // strip factorisation
    HpLayout lay;
    int m_lo = 0, m_hi = -1;      // strips held by this solver
    std::vector<int> leaf_start_h, leaf_q_h, sep_h;
    int *leaf_start = nullptr, *leaf_q = nullptr, *sep = nullptr;   // device copies
    cplx* packets = nullptr;
    cplx* mleaf = nullptr;        // transfer matrices of the pipelined sweep: [strip][dir][leaf][2b][2b]
    cplx* rsep = nullptr;         // cluster kernel: separator recurrence rows R: [strip][dir][P-1][b][3b]
    int64_t bytes = 0;
    double setup_ms = 0.0;
    // front block: Thomas factors of the b tridiagonal diagonal blocks (reference H_F)
    cplx *f_low = nullptr, *f_invd = nullptr, *f_up = nullptr;   // [b][n]
    cplx* TF = nullptr;                                           // [b][n]   T_F u_F kept between the stages
    // coupled front block (csrc/hp_front_coupled.cu): H_F = A[:bn, :bn] with the couplings between the rows kept
    int front_mode = 0;           // 0 = block diagonal (reference, code.py:178-183), 1 = coupled (the paper's A_FF)
    int fc_P = 0, fc_QP = 0;      // leaves of the x1 partition, widest leaf
    int *fc_leaf_start = nullptr, *fc_leaf_q = nullptr, *fc_sep = nullptr;
    cplx *fc_Sinv = nullptr, *fc_LU = nullptr;                    // [n][b*b] leaf Schur chains, [n][2][b] x1 couplings
    cplx *fc_T = nullptr, *fc_Sl = nullptr, *fc_Su = nullptr;     // [P-1][b*b] separator chain and off-diagonal blocks
    cplx* fc_work = nullptr;                                      // [b][n] first-pass leaf solutions
    // sweep scratch
    cplx* xch = nullptr;          // exchange ring of the sweep kernel (csrc/hp_sweep.cu)
    size_t xch_count = 0, bar_count = 0;   // complex numbers of xch, words of bar (hp_context_clone allocates the same)
    int coop = 1;                 // 1: sweeps are cooperative launches (the driver checks co-residency); contexts: 0, see hp_context_clone
    int is_view = 0;              // 1: created by hp_context_clone, owns only its sweep scratch (xch, bar, TF, TFm, fc_work)
    hp_solver* parent = nullptr;  // context: the solver whose factorisation it shares
    int live_ctx = 0;             // solver: contexts cloned from it and not destroyed yet (they hold its pointers)
    long long* dbg = nullptr;     // optional per-phase cycle counters of the sweep kernel [G][8]
    int sweep_variant = 0;        // 0 = automatic; classic layout: 1 direct, 2 TMA staged, 3 pipelined; cluster layout: 4
    int layout_mode = 0;          // 0 = automatic (cluster layout when a partition exists), 1 = classic, 2 = cluster
    int multi_ok[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // multi-vector kernel with RT right-hand sides: 0 unknown, 1 fits, -1 does not
    int dmma_ok = 0;              // tensor-core kernel (8 right-hand sides): 0 unknown, 1 fits, -1 does not
    cplx* TFm = nullptr;          // [HP_RMAX][b][n] parked T_F u_F of the right-hand sides of a multi-vector application
    unsigned int* bar = nullptr;
    int* status = nullptr;        // device flag: non-zero when a pivot vanished during setup
    // optional CUDA-event timing of the sweep launches (hp_profile_enable / hp_profile_read)
    int prof_on = 0;
    std::vector<cudaEvent_t> prof_ev;   // pairs
    int prof_used = 0;
    int64_t prof_bytes = 0;
};

static inline HpStripCtx hp_ctx(const hp_solver* s) {
    HpStripCtx c;
    c.n = s->n; c.b = s->b; c.pml = s->pml; c.omega2 = s->omega2;
    c.s1t = s->s1t; c.is1t = s->is1t; c.c_mat = s->c_mat; c.kappa_c = s->kappa_c;
    return c;
}

// hp_assembly.cu
int hp_launch_tables(hp_solver* s, const cplx* c_cplx, cudaStream_t st);   // c_cplx: complex velocity (attenuating medium) or NULL
// hp_setup.cu
int hp_setup_strips(hp_solver* s, int P, int K, int m_lo, int m_hi, cudaStream_t st);
void hp_free_strips(hp_solver* s);
// hp_front.cu
int hp_front_setup(hp_solver* s, cudaStream_t st);
// hp_front_coupled.cu : out = H_F^-1 rhs (out_mode 0) or base - H_F^-1 rhs (out_mode 2) on b field rows;
// rhs_mode 0: rhs = the b rows at `in`; 2: rhs = [0; ..; 0; fac * is1t ⊙ in] (one row at `in`)
int hp_front_coupled_setup(hp_solver* s, cudaStream_t st);
void hp_front_coupled_free(hp_solver* s);
int hp_front_coupled_solve(hp_solver* s, int rhs_mode, int out_mode, const cplx* in, cplx* out, const cplx* base, cplx fac,
                           cudaStream_t st);
// hp_sweep.cu : mode 0 = forward, 1 = backward, 2 = single strip apply (vin -> yout)
int hp_sweep_launch(hp_solver* s, int mode, cplx* u, const cplx* vin, cplx* yout, int m_from, int m_to,
                    int diag_mode, cudaStream_t st);
// the same sweep for R right-hand sides in one launch (cluster layout, csrc/hp_sweep4m.cu): mode 0 forward, 1 backward
int hp_sweep_launch_multi(hp_solver* s, int mode, int R, cplx* const* um, int m_from, int m_to, int diag_mode, cudaStream_t st);
