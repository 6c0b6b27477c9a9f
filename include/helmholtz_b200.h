/* helmholtz_b200.h -- C ABI of libhelmholtz_b200.so
 *
 * B200 (sm_100a) implementation of the data-parallel hot path of bocchs/helmholtz-preconditioner
 * (reference: code.py).  Plain pointers and sizes only; no torch types.  Every entry point returns 0 on
 * success and a non-zero code on failure (hp_last_error() gives the text).  Pointers named *_dev are
 * device pointers on the solver's device; `stream` is a cudaStream_t passed as void* (NULL = default).
 * Complex numbers are interleaved (re, im) doubles, i.e. numpy complex128 / double2.
 *
 * Vector layout: the field u has n*n entries, entry (j-1)*n + (i-1) is grid point (x1 index i, x2 index j),
 * exactly the reference's f_mat.flatten() ordering (code.py:448).
 *
 * Each function cites the reference interface it replaces.
 */
#ifndef HELMHOLTZ_B200_H
#define HELMHOLTZ_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hp_solver hp_solver;

/* text of the last error raised on the calling thread */
const char* hp_last_error(void);
/* library/ABI version, and 1 if a usable CUDA device is present */
int hp_version(void);
int hp_device_ok(void);
/* number of kernel launches the library has made in this process (bench.py's gpu_launches) */
int64_t hp_launch_count(void);
/* CUDA-event timing of the sweep kernel launches (the dominant kernel): enable/reset, then read the summed
 * device time in ms, the number of launches and the algorithmic bytes they streamed (synchronises) */
int hp_profile_enable(hp_solver* s, int on);
int hp_profile_read(hp_solver* s, double* sweep_ms, int* launches, int64_t* bytes);

/* Problem definition.  Replaces the scalar set-up at code.py:442-447 (omega, h, eta) and keeps a device
 * copy of the velocity model.  c_mat is the reference's (n+2) x (n+2) row-major float64 array (init_c*_mat,
 * code.py:40-51); it is read as c_mat[i-1][j-1] like the reference does (code.py:108, 270).
 * c_is_device != 0 means c_mat already lives on the device. */
int hp_create(hp_solver** out, int n, int b, double omega_re, double omega_im, double cst,
              const double* c_mat, int c_is_device, void* stream);
/* Attenuating medium: the same problem with a complex velocity.  c_mat holds (n+2) x (n+2) complex numbers, interleaved
 * (real, imaginary) doubles in the same row-major order.  The solver keeps only the complex slowness^2
 * kappa = 1/c^2 on the grid (16 B per point) and every function below reads it: hp_assemble_csr, hp_assemble_strip_csr,
 * hp_stencil_matvec(_rows), hp_precond_setup with both front blocks, and everything that applies the preconditioner.
 * Loss means Im(omega^2 kappa) > 0 for Re omega > 0, the sign of the PML and of alpha > 0.  A velocity with zero
 * imaginary parts gives the bits of hp_create.  The setup generations selected by the developer switches
 * HP_CHAIN_THREAD and HP_CHAIN_UNROLL refuse a complex medium. */
int hp_create_complex(hp_solver** out, int n, int b, double omega_re, double omega_im, double cst,
                      const double* c_mat, int c_is_device, void* stream);
/* 1 if the solver (or the solver a context was cloned from) was made by hp_create_complex, 0 if by hp_create */
int hp_medium_is_complex(hp_solver* s);
int hp_destroy(hp_solver* s);
/* A second handle on a solver that is set up: shares the operator tables and the factorisation (read-only) and owns a
 * private copy of the sweep scratch (exchange ring, abort flags, parked front solutions T_F u_F of code.py:364), so that
 * applications of algo2_4 (code.py:356-385) issued through different contexts can be in flight on different streams at
 * once.  The reference has no counterpart (one Python thread); slab.py uses one context per group of right-hand sides.
 * `s` must outlive the context; hp_destroy(context) frees the scratch only; setup calls on a context are refused.
 * While a context of `s` is open, hp_precond_setup, hp_precond_set_front and a change of hp_set_front_mode on `s` are
 * refused too (they would replace the factorisation the context points to). */
int hp_context_clone(hp_solver* s, hp_solver** out, void* stream);

/* ---- operator A ---------------------------------------------------------------------------------- */

/* number of stored entries of A (5 n^2 - 4 n) */
int64_t hp_csr_nnz(int n);
/* build_A_matrix (code.py:202-219, with get_A_diag_block_coeffs :71-115, get_upper/lower_A_block :131-154):
 * writes sorted CSR, indptr[n*n+1] and indices[nnz] int32 (scipy's index type here), data[nnz] complex128. */
int hp_assemble_csr(hp_solver* s, int32_t* indptr_dev, int32_t* indices_dev, double* data_dev, void* stream);
/* get_Hm (code.py:283-290, with get_Hm_coeffs :224-279): the bn x bn operator of the b grid rows m-b+1..m with the x2
 * PML moved to end on row m, as sorted CSR (indptr[b*n+1], indices/data[hp_strip_csr_nnz]); b <= m <= n.  m = b is the
 * coupled front block A[:bn, :bn].  algo2_3 does not go through this matrix (the strips are factored from the same
 * coefficients in block form); it is the reference's helper, exposed for inspection and tests. */
int64_t hp_strip_csr_nnz(int n, int b);
int hp_assemble_strip_csr(hp_solver* s, int m, int32_t* indptr_dev, int32_t* indices_dev, double* data_dev, void* stream);
/* y = A x without forming A (the matvec scipy's gmres performs at code.py:516, iterative.py `matvec`) */
int hp_stencil_matvec(hp_solver* s, const double* x_dev, double* y_dev, void* stream);
/* the same for the grid rows j_lo <= j < j_hi (0-based) of a slab: x_dev/y_dev hold those rows only, x_south_dev /
 * x_north_dev are the halo rows j_lo-1 and j_hi received from the neighbouring ranks (NULL on the grid boundary) */
int hp_stencil_matvec_rows(hp_solver* s, int j_lo, int j_hi, const double* x_dev, const double* x_south_dev,
                           const double* x_north_dev, double* y_dev, void* stream);
/* y = A x from the assembled CSR arrays */
int hp_csr_matvec(int64_t nrows, const int32_t* indptr_dev, const int32_t* indices_dev, const double* data_dev,
                  const double* x_dev, double* y_dev, void* stream);

/* ---- preconditioner ------------------------------------------------------------------------------ */

/* algo2_3 (code.py:345-353): factor the front block H_F and every moving-PML strip H_m, m = m_lo..m_hi
 * (b+1 <= m_lo, m_hi <= n; pass 0,0 for all; m_lo > m_hi = front block only).  Strips outside [m_lo, m_hi]
 * belong to other ranks of a slab decomposition.  P, K choose the x1 partition of the strips (P leaves
 * separated by P-1 separator columns, K CTAs per leaf, P*K <= number of SMs); 0,0 = chosen automatically. */
int hp_precond_setup(hp_solver* s, int P, int K, int m_lo, int m_hi, void* stream);
/* bytes of device memory held by the strip factorisation, and the device time the last setup took */
int64_t hp_precond_bytes(hp_solver* s);
double hp_precond_setup_ms(hp_solver* s);
/* generator layout used by the next hp_precond_setup: 0 = automatic (cluster when a partition exists), 1 = classic
 * (one CTA per leaf part, N distributed by rows), 2 = cluster (a leaf is a thread-block cluster of K <= 8 CTAs, N
 * distributed by separator columns; fails when no such partition fits) */
int hp_set_layout_mode(hp_solver* s, int mode);
/* front block H_F factored by the next hp_precond_setup (algo2_3, code.py:346-347): 0 = the reference's
 * get_A_FF_block (code.py:178-183: only the b diagonal blocks A_11..A_bb, b independent tridiagonal systems), 1 = the
 * coupled block A[:bn, :bn] of Engquist & Ying's Algorithm 2.3/2.4, i.e. get_Hm(b) (code.py:283-290) solved in full */
int hp_set_front_mode(hp_solver* s, int mode);
/* the same switch on a solver that is already set up: factors the front block again with `mode`, keeps the strips */
int hp_precond_set_front(hp_solver* s, int mode, void* stream);
/* sweep kernel variant: 0 = automatic; classic layout: 1 = direct loads, 2 = TMA-staged block-synchronous,
 * 3 = pipelined with two hand-overs through L2 per strip; cluster layout: 4 = one hand-over through L2 per strip, the
 * exchanges inside a leaf through distributed shared memory */
int hp_set_sweep_variant(hp_solver* s, int variant);
/* 0 = fine; 1 = a sweep kernel gave up waiting for data from another CTA (a bug, never expected); synchronises */
int hp_sweep_status(hp_solver* s);

/* The three stages of algo2_4 (code.py:356-385), operating in place on the field u_dev (n*n complex):
 *   hp_front_begin   : T_F u_F = H_F^{-1} u_F kept aside, u_{b+1} -= A_{b+1,F} T_F u_F        (:364-365)
 *   hp_sweep_forward : for m = m_from..m_to     u_{m+1} -= A_{m+1,m} T_m u_m                   (:366-370)
 *   hp_sweep_backward: for m = m_from..m_to (descending, m_from >= m_to), the diagonal solve (:372-375)
 *                      fused with the upward elimination (:376-380):
 *                        diag_mode 0 (reference): u_m <- u_m - T_m (u_m + A_{m,m+1} u_{m+1})
 *                        diag_mode 1 (paper)    : u_m <- T_m (u_m - A_{m,m+1} u_{m+1})
 *   hp_front_end     : u_F <- T_F u_F - H_F^{-1} A_{F,b+1} u_{b+1}                            (:381-384)
 * hp_precond_apply runs all four on one device (u_dev <- M f_dev). */
int hp_front_begin(hp_solver* s, double* u_dev, void* stream);
int hp_sweep_forward(hp_solver* s, double* u_dev, int m_from, int m_to, void* stream);
int hp_sweep_backward(hp_solver* s, double* u_dev, int m_from, int m_to, int diag_mode, void* stream);
int hp_front_end(hp_solver* s, double* u_dev, void* stream);
/* park / restore T_F u_F (b*n complex numbers) between hp_front_begin and hp_front_end when several right-hand
 * sides are in flight: dir 0 copies solver -> buf_dev, dir 1 copies buf_dev -> solver */
int hp_front_tf_copy(hp_solver* s, double* buf_dev, int dir, void* stream);
int hp_precond_apply(hp_solver* s, const double* f_dev, double* u_dev, int diag_mode, void* stream);
/* Several right-hand sides per pass over the strip generators (algo2_4 applied to R vectors; the reference applies it to
 * one vector per call, code.py:510-511).  u_devs / f_devs: HOST arrays of R device pointers (n*n complex each); R must be
 * 1, 2, 4 or 8 and <= hp_multi_max(s) (1 when the partition of the strips does not fit the multi-vector kernel).  Per
 * right-hand side the result equals hp_sweep_forward / hp_sweep_backward / hp_precond_apply up to rounding. */
int hp_multi_max(hp_solver* s);
/* Kernel that one launch carrying R right-hand sides runs (the choice hp_sweep_forward_multi / hp_sweep_backward_multi
 * make): 2 = hp_sweep4d (FP64 tensor cores, R = 8), 1 = hp_sweep4m, 0 = none (R is not supported by this layout). */
int hp_multi_kernel(hp_solver* s, int R);
/* Masked slots: an entry u_devs[r] == NULL is an inactive slot of the launch.  Its loads read 0 and nothing is stored
 * for it; the other slots keep their index r and their results are bit for bit those of a launch of the same width in
 * which every slot is active, whatever the other slots hold.  R keeps the rules above; at least one entry must be
 * non-NULL, otherwise the call fails. */
int hp_sweep_forward_multi(hp_solver* s, int R, double* const* u_devs, int m_from, int m_to, void* stream);
int hp_sweep_backward_multi(hp_solver* s, int R, double* const* u_devs, int m_from, int m_to, int diag_mode, void* stream);
/* f_devs[r] and u_devs[r] are both NULL (inactive slot: no copy, no front solve) or both non-NULL; at least one slot must
 * be active.  Any other combination fails without launching anything. */
int hp_precond_apply_multi(hp_solver* s, int R, const double* const* f_devs, double* const* u_devs, int diag_mode, void* stream);
/* y = T_m v : last n entries of H_m^{-1} [0; v]  (lu_Hm_ra[m-b-1].solve(u_temp)[-n:], code.py:370) */
int hp_strip_apply(hp_solver* s, int m, const double* v_dev, double* y_dev, void* stream);
/* test hooks: the partition in use, and a host copy of one strip's packed generators
 * (G = P*K packets of PK complex numbers; layout in csrc/hp_internal.cuh) */
int hp_strip_layout(hp_solver* s, int* P, int* K, int* QP, int* CW, int* NS, int* NR, int64_t* PK,
                    int* leaf_start_host /* P */, int* leaf_q_host /* P */, int* sep_host /* P-1 */);
int hp_strip_packets(hp_solver* s, int m, double* packets_host);
/* cluster layout details: colN = 1 when N is stored by separator columns ([b][NRQ] per CTA), NCB/NRQ/NXG = separator
 * right-hand sides, rows of x and gathered entries per CTA */
int hp_strip_layout_ex(hp_solver* s, int* colN, int* NCB, int* NRQ, int* NXG);

/* ---- inversion (helmholtz_preconditioner_b200/inversion.py) -----------------------------------------
 * The reference has no counterpart.  With w_p = omega^2 is1(i) is2(j) = dA_pp/dkappa_p (the factor the diagonal c5
 * multiplies the slowness^2 kappa = 1/c^2 by), fields u (A u = f) and adjoint fields mu (A mu = R^T conj(r); A is complex
 * symmetric) in the vector layout above, the misfit gradient is G = -conj(w (.) sum_s mu_s (.) u_s) and the Born source
 * of a perturbation dkappa is -w (.) dkappa (.) u.  u_devs / mu_devs / out_devs are HOST arrays of R device pointers,
 * 1 <= R <= 8; a slot whose two pointers are NULL is skipped, a slot with one NULL pointer is refused, and at least one
 * slot must be active.  Each result is deterministic. */
/* acc_dev[p] += u_r[p] mu_r[p] for the active slots in the order r = 0..R-1 (n*n complex accumulator) */
int hp_grad_accumulate(hp_solver* s, int R, const double* const* u_devs, const double* const* mu_devs, double* acc_dev,
                       void* stream);
/* G = -conj(w (.) acc); wrt = 1 multiplies by conj(dkappa/dc) = conj(-2 kappa sqrt(kappa)) (principal root).  Written in
 * the c_mat layout: out_dev[(i-1)(n+2) + (j-1)] belongs to grid point (i, j), the last two rows and columns are zero.
 * (n+2)^2 float64 (Re G) for a medium made by hp_create, complex128 for one made by hp_create_complex. */
int hp_grad_finish(hp_solver* s, const double* acc_dev, int wrt, double* out_dev, void* stream);
/* out_r = -w (.) dkappa (.) u_r for the active slots; dkappa_dev is (n+2)^2 complex128 in the c_mat layout (entry
 * [i-1][j-1] for grid point (i, j); the last two rows and columns are not read).  out_devs[r] may equal u_devs[r]. */
int hp_born_source(hp_solver* s, int R, const double* dkappa_dev, const double* const* u_devs, double* const* out_devs,
                   void* stream);

/* ---- Krylov vector kernels (scipy gmres inner loop, iterative.py; called from code.py:516) -------- */

/* out_dev[0..1] = sum conj(x) y   (np.vdot) */
int hp_dotc(int64_t n, const double* x_dev, const double* y_dev, double* out_dev, void* stream);
/* out_dev[0] = ||x||_2 */
int hp_nrm2(int64_t n, const double* x_dev, double* out_dev, void* stream);
/* y += alpha x with alpha = (a_re, a_im) on the host */
int hp_axpy(int64_t n, double a_re, double a_im, const double* x_dev, double* y_dev, void* stream);
/* y += sign * alpha x, alpha (one complex number) read from device memory */
int hp_axpy_dev(int64_t n, const double* alpha_dev, double sign, const double* x_dev, double* y_dev, void* stream);
/* y = alpha x */
int hp_scale_copy(int64_t n, double a_re, double a_im, const double* x_dev, double* y_dev, void* stream);
/* Modified Gram-Schmidt of w against the rows V[0..k) (row stride ldv complex entries):
 *   hcol_dev[2*j..] = vdot(V[j], w); w -= hcol[j] V[j]   sequentially for j = 0..k-1,
 * then hcol_dev[2*k] = ||w|| (after) and hcol_dev[2*k+2] = ||w|| before orthogonalisation (h0). */
int hp_mgs(int64_t n, int k, const double* V_dev, int64_t ldv, double* w_dev, double* hcol_dev, void* stream);
/* one fused step of the same recurrence for slab-distributed vectors (the caller all-reduces the coefficient between the
 * steps): w -= (*hcoef_dev) v, then out_dev = vdot(vnext, w) over the local entries, or sum |w|^2 when vnext is NULL */
int hp_mgs_step(int64_t n, const double* hcoef_dev, const double* v_dev, double* w_dev, const double* vnext_dev,
                double* out_dev, void* stream);
/* x += sum_j y[j] V[j]   (x += y @ v[:col+1, :]); y on the host, 2*k doubles */
int hp_combine(int64_t n, int k, const double* V_dev, int64_t ldv, const double* y_host, double* x_dev,
               void* stream);

/* Block Gram-Schmidt pass on slab-distributed vectors (csrc/hp_cgs.cu): the orthogonalisation loop of scipy's gmres
 * (w -= (v_j . w) v_j for j < k; called from code.py:516) as classical Gram-Schmidt applied twice, three passes and three
 * all-reduces per Arnoldi column instead of k + 2.  For R <= 8 systems of n local entries and k <= 20 basis vectors (rows of
 * V_devs[r], leading dimension ldv complex numbers):
 *   update != 0:  w_r <- w_r - sum_j coef_devs[r][j] v_j      (k complex coefficients in device memory)
 *   dots   != 0:  out_devs[r][j] = v_j^H w_r for j < k, from the updated w_r
 *   always:       out_devs[r][k] = sum |w_r|^2 from the updated w_r  */
int hp_cgs_pass(int R, int64_t n, int k, const double* const* V_devs, int64_t ldv, double* const* w_devs,
                const double* const* coef_devs, double* const* out_devs, int update, int dots, void* stream);

/* ---- peer mailboxes (slab decomposition, helmholtz_preconditioner_b200/slab.py) --------------------------------------
 * The reference runs algo2_4 (code.py:356-385) in one process; with the grid rows cut into slabs the row handed from
 * strip m to strip m+1 (code.py:368-370, forward; 378-380, backward) crosses from one GPU to the next.  A mailbox is a
 * block of device memory [256 bytes of uint32 flags | staging rows] that the neighbouring processes map (CUDA IPC): the
 * sender stores the rows and then a sequence number, the receiver's stream waits for the number without holding an SM
 * (cuStreamWaitValue32).  handle64: the 64 bytes of the cudaIpcMemHandle_t, to be passed to the other process. */
int hp_mailbox_create(int64_t bytes, void** ptr_dev, unsigned char* handle64);
int hp_mailbox_open(const unsigned char* handle64, void** ptr_dev);
int hp_mailbox_close(void* ptr_dev);
int hp_mailbox_free(void* ptr_dev);
/* the stream waits until *(uint32*)flag_dev >= value */
int hp_stream_wait_geq(const void* flag_dev, unsigned int value, void* stream);
/* R <= 8 rows of n complex numbers: src_rows[r] -> staging_peer + r*n (complex), then *(uint32*)flag_peer = value */
int hp_handover_rows(int R, const double* const* src_rows, double* staging_peer, int64_t n, void* flag_peer,
                     unsigned int value, void* stream);
/* staging + r*n -> dst_rows[r] on this device (after hp_stream_wait_geq on the flag that guards the staging area) */
int hp_collect_rows(int R, const double* staging, double* const* dst_rows, int64_t n, void* stream);
/* *(uint32*)flags_peer[i] = value for count <= 8 flags */
int hp_signal_flags(int count, void* const* flags_peer, unsigned int value, void* stream);

#ifdef __cplusplus
}
#endif
#endif
