// C ABI glue of libhelmholtz_b200.so: solver life cycle, error text, algo2_3/algo2_4 drivers.
#include "hp_internal.cuh"

#include <stdarg.h>
#include <string.h>

static thread_local char g_err[1024] = "";

void hp_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* hp_last_error(void) { return g_err; }

#include <atomic>
static std::atomic<long long> g_launches{0};
void hp_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" int64_t hp_launch_count(void) { return (int64_t)g_launches.load(); }

void hp_profile_begin(hp_solver* s, cudaStream_t st) {
    if (!s->prof_on) return;
    if (s->prof_used + 2 > (int)s->prof_ev.size()) {
        for (int i = 0; i < 2; ++i) { cudaEvent_t e; cudaEventCreate(&e); s->prof_ev.push_back(e); }
    }
    cudaEventRecord(s->prof_ev[s->prof_used], st);
}
void hp_profile_end(hp_solver* s, cudaStream_t st, int64_t bytes) {
    if (!s->prof_on) return;
    cudaEventRecord(s->prof_ev[s->prof_used + 1], st);
    s->prof_used += 2;
    s->prof_bytes += bytes;
}
extern "C" int hp_profile_enable(hp_solver* s, int on) {
    if (!s) return 1;
    s->prof_on = on; s->prof_used = 0; s->prof_bytes = 0;
    return 0;
}
// total device time (ms) of the sweep kernel launches since hp_profile_enable, their number and the
// algorithmic bytes they streamed; synchronises the device
extern "C" int hp_profile_read(hp_solver* s, double* sweep_ms, int* launches, int64_t* bytes) {
    if (!s) return 1;
    HP_CUDA(cudaDeviceSynchronize());
    double tot = 0.0;
    for (int i = 0; i + 1 < s->prof_used; i += 2) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, s->prof_ev[i], s->prof_ev[i + 1]);
        tot += ms;
    }
    if (sweep_ms) *sweep_ms = tot;
    if (launches) *launches = s->prof_used / 2;
    if (bytes) *bytes = s->prof_bytes;
    return 0;
}
extern "C" int hp_version(void) { return 100; }

extern "C" int hp_device_ok(void) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) { cudaGetLastError(); return 0; }
    return 1;
}

// cplx_medium: c_mat holds (n+2)^2 interleaved complex numbers; the solver keeps the complex slowness^2 kappa_c only
static int hp_create_fill(hp_solver* s, int n, int b, double omega_re, double omega_im, double cst, const double* c_mat,
                          int c_is_device, int cplx_medium, cudaStream_t st) {
    s->n = n; s->b = b;
    double h = 1.0 / (double)(n + 1);                     // code.py:443
    s->pml.cst = cst; s->pml.h = h; s->pml.eta = (double)b * h;   // code.py:444
    s->pml.omega = cmake(omega_re, omega_im);             // code.py:442
    s->omega2 = cmul(s->pml.omega, s->pml.omega);
    int dev = 0;
    HP_CUDA(cudaGetDevice(&dev));
    HP_CUDA(cudaDeviceGetAttribute(&s->num_sms, cudaDevAttrMultiProcessorCount, dev));
    size_t tl = sizeof(cplx) * (size_t)(2 * n + 3);
    HP_CUDA(cudaMalloc(&s->s1t, tl)); HP_CUDA(cudaMalloc(&s->is1t, tl));
    HP_CUDA(cudaMalloc(&s->s2t, tl)); HP_CUDA(cudaMalloc(&s->is2t, tl));
    HP_CUDA(cudaMalloc(&s->status, sizeof(int)));
    HP_CUDA(cudaMemsetAsync(s->status, 0, sizeof(int), st));
    if (cplx_medium) {
        // the complex velocity is needed only to form kappa_c: a host model is staged through a temporary device copy
        const size_t cb = sizeof(cplx) * (size_t)(n + 2) * (n + 2);
        HP_CUDA(cudaMalloc(&s->kappa_c, sizeof(cplx) * (size_t)n * n));
        struct Stage { void* p = nullptr; ~Stage() { cudaFree(p); } } stage;
        const cplx* c_dev = (const cplx*)c_mat;
        if (!c_is_device) {
            HP_CUDA(cudaMalloc(&stage.p, cb));
            HP_CUDA(cudaMemcpyAsync(stage.p, c_mat, cb, cudaMemcpyHostToDevice, st));
            c_dev = (const cplx*)stage.p;
        }
        if (hp_launch_tables(s, c_dev, st)) return 2;
        s->s2t_h.resize(2 * n + 3);
        HP_CUDA(cudaMemcpyAsync(s->s2t_h.data(), s->s2t, tl, cudaMemcpyDeviceToHost, st));
        HP_CUDA(cudaStreamSynchronize(st));                // before the staging copy is freed
        return 0;
    }
    size_t cb = sizeof(double) * (size_t)(n + 2) * (n + 2);
    HP_CUDA(cudaMalloc(&s->c_mat, cb));
    HP_CUDA(cudaMalloc(&s->kappa, sizeof(double) * (size_t)n * n));
    HP_CUDA(cudaMemcpyAsync(s->c_mat, c_mat, cb, c_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    if (hp_launch_tables(s, nullptr, st)) return 2;
    s->s2t_h.resize(2 * n + 3);
    HP_CUDA(cudaMemcpyAsync(s->s2t_h.data(), s->s2t, tl, cudaMemcpyDeviceToHost, st));
    HP_CUDA(cudaStreamSynchronize(st));
    return 0;
}

static int hp_create_any(const char* what, hp_solver** out, int n, int b, double omega_re, double omega_im, double cst,
                         const double* c_mat, int c_is_device, int cplx_medium, void* stream) {
    if (!out) { hp_set_error("%s: null output", what); return 1; }
    *out = nullptr;
    if (n < 2 || b < 1 || b > HP_BMAX || b > n) {
        hp_set_error("%s: need 2 <= n, 1 <= b <= min(n, %d); got n=%d b=%d", what, HP_BMAX, n, b);
        return 1;
    }
    if (!hp_device_ok()) { hp_set_error("%s: no CUDA device (this library has no CPU path)", what); return 2; }
    cudaStream_t st = (cudaStream_t)stream;
    hp_solver* s = new hp_solver();
    int rc = hp_create_fill(s, n, b, omega_re, omega_im, cst, c_mat, c_is_device, cplx_medium, st);
    if (rc) { hp_destroy(s); return rc; }      // frees whatever was allocated before the failure
    *out = s;
    return 0;
}

extern "C" int hp_create(hp_solver** out, int n, int b, double omega_re, double omega_im, double cst,
                         const double* c_mat, int c_is_device, void* stream) {
    return hp_create_any("hp_create", out, n, b, omega_re, omega_im, cst, c_mat, c_is_device, 0, stream);
}

extern "C" int hp_create_complex(hp_solver** out, int n, int b, double omega_re, double omega_im, double cst,
                                 const double* c_mat, int c_is_device, void* stream) {
    return hp_create_any("hp_create_complex", out, n, b, omega_re, omega_im, cst, c_mat, c_is_device, 1, stream);
}

extern "C" int hp_medium_is_complex(hp_solver* s) { return s && s->kappa_c ? 1 : 0; }

// A second handle on the same operator and factorisation with its own sweep scratch (exchange ring, abort flags, parked
// front solutions): sweeps issued through different contexts may be in flight on different streams at the same time
// (slab.py: the groups of right-hand sides of the asynchronous pipeline).  Everything read-only is shared with `s`, which
// must outlive the context; hp_destroy on a context frees its scratch only.
extern "C" int hp_context_clone(hp_solver* s, hp_solver** out, void* stream) {
    if (!s || !out) { hp_set_error("hp_context_clone: null argument"); return 1; }
    *out = nullptr;
    if (!s->f_low || !s->bar) { hp_set_error("hp_context_clone: preconditioner not set up"); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    hp_solver* owner = s->is_view ? s->parent : s;
    hp_solver* c = new hp_solver(*s);
    c->is_view = 1;
    c->parent = nullptr; c->live_ctx = 0;                  // counted in the owner once the scratch exists
    // Sweeps of a context are plain cluster launches.  A cooperative launch is ordered against all other work of the process
    // on the device (measured: with the sweep of one group queued behind a stream-level wait for another GPU, the cooperative
    // launch of the next group blocks its host thread inside the launch call, and two processes then wait for each other).
    // What the cooperative attribute checks, that all P clusters fit on the device at once, was checked when the layout was
    // chosen (hp_sweep4_max_clusters / cudaOccupancyMaxActiveClusters); a sweep whose clusters are not all resident yet waits
    // for the SMs that the short kernels of other streams hold.
    c->coop = 0;
    c->xch = nullptr; c->bar = nullptr; c->TF = nullptr; c->TFm = nullptr; c->fc_work = nullptr; c->dbg = nullptr;
    c->prof_on = 0; c->prof_ev.clear(); c->prof_used = 0; c->prof_bytes = 0;
    auto fail = [&]() { hp_destroy(c); return 2; };
    const size_t sz = sizeof(cplx) * (size_t)s->b * s->n;
    if (cudaMalloc(&c->xch, sizeof(cplx) * s->xch_count) != cudaSuccess || cudaMalloc(&c->bar, sizeof(unsigned int) * s->bar_count) != cudaSuccess ||
        cudaMalloc(&c->TF, 2 * sz) != cudaSuccess || (s->fc_work && cudaMalloc(&c->fc_work, sz) != cudaSuccess) ||
        cudaMemsetAsync(c->bar, 0, sizeof(unsigned int) * s->bar_count, st) != cudaSuccess) {
        hp_set_error("hp_context_clone: allocation of the sweep scratch failed: %s", cudaGetErrorString(cudaGetLastError()));
        return fail();
    }
    c->parent = owner;
    owner->live_ctx++;
    *out = c;
    return 0;
}

// A context keeps the addresses of its owner's factorisation: refactoring the owner while one is open would leave the
// context pointing at freed memory, so the calls that replace the factorisation refuse until every context is destroyed.
static int hp_refuse_with_contexts(const hp_solver* s, const char* what) {
    if (s->live_ctx <= 0) return 0;
    hp_set_error("%s: %d context(s) made by hp_context_clone still use this factorisation; destroy them first", what, s->live_ctx);
    return 1;
}

extern "C" int hp_destroy(hp_solver* s) {
    if (!s) return 0;
    if (s->is_view) {
        if (s->parent) s->parent->live_ctx--;
        cudaFree(s->xch); cudaFree(s->bar); cudaFree(s->TF); cudaFree(s->TFm); cudaFree(s->fc_work); cudaFree(s->dbg);
        for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
        delete s;
        return 0;
    }
    hp_free_strips(s);
    cudaFree(s->s1t); cudaFree(s->is1t); cudaFree(s->s2t); cudaFree(s->is2t);
    cudaFree(s->c_mat); cudaFree(s->kappa); cudaFree(s->kappa_c); cudaFree(s->status);
    cudaFree(s->f_low); cudaFree(s->f_invd); cudaFree(s->f_up); cudaFree(s->TF); cudaFree(s->TFm);
    hp_front_coupled_free(s);
    for (cudaEvent_t e : s->prof_ev) cudaEventDestroy(e);
    delete s;
    return 0;
}

extern "C" int hp_precond_setup(hp_solver* s, int P, int K, int m_lo, int m_hi, void* stream) {
    if (!s) { hp_set_error("hp_precond_setup: null solver"); return 1; }
    if (s->is_view) { hp_set_error("hp_precond_setup: a context made by hp_context_clone shares the factorisation of its parent"); return 1; }
    if (hp_refuse_with_contexts(s, "hp_precond_setup")) return 1;
    if (m_lo == 0 && m_hi == 0) { m_lo = s->b + 1; m_hi = s->n; }
    if (m_lo < s->b + 1 || m_hi > s->n) {
        hp_set_error("hp_precond_setup: strips must lie in %d..%d, got %d..%d", s->b + 1, s->n, m_lo, m_hi);
        return 1;
    }
    cudaStream_t st = (cudaStream_t)stream;
    HP_CUDA(cudaMemsetAsync(s->status, 0, sizeof(int), st));       // pivot failures of the front block and of the strips
    if (hp_front_setup(s, st)) return 2;
    int rc = 0;
    if (m_lo > m_hi) hp_free_strips(s);                   // a rank that holds no strip (front block only)
    else rc = hp_setup_strips(s, P, K, m_lo, m_hi, st);
    if (rc) return rc;
    int status = 0;
    HP_CUDA(cudaMemcpyAsync(&status, s->status, sizeof(int), cudaMemcpyDeviceToHost, st));
    HP_CUDA(cudaStreamSynchronize(st));
    if (status) {
        hp_set_error("hp_precond_setup: a pivot vanished while factoring %s (status %d)",
                     (status & 8) ? "the front block" : "the strips", status);
        return 3;
    }
    return 0;
}

// developer hook: per-phase cycle counters of the sweep kernel.  on=1 allocates/zeroes, read copies [G][8] to host
extern "C" int hp_debug_phases(hp_solver* s, int on, long long* out_host) {
    if (!s || !s->packets) return 1;
    size_t sz = sizeof(long long) * (16 + 64 * 16) * s->lay.G;
    if (on && !s->dbg) { HP_CUDA(cudaMalloc(&s->dbg, sz)); HP_CUDA(cudaMemset(s->dbg, 0, sz)); }
    if (out_host && s->dbg) HP_CUDA(cudaMemcpy(out_host, s->dbg, sz, cudaMemcpyDeviceToHost));
    if (!on && s->dbg) { cudaFree(s->dbg); s->dbg = nullptr; }
    return 0;
}
// front block used by the next hp_precond_setup: 0 = block diagonal (the reference's get_A_FF_block), 1 = coupled
extern "C" int hp_set_front_mode(hp_solver* s, int mode) {
    if (!s || mode < 0 || mode > 1) { hp_set_error("hp_set_front_mode: mode must be 0 or 1"); return 1; }
    // the front solves read front_mode at once: switching it under a factorisation of the other mode is a refactoring
    if (mode != s->front_mode && hp_refuse_with_contexts(s, "hp_set_front_mode")) return 1;
    s->front_mode = mode;
    return 0;
}
// re-factor the front block alone with another mode; the strip factorisation is kept
extern "C" int hp_precond_set_front(hp_solver* s, int mode, void* stream) {
    if (s && s->is_view) { hp_set_error("hp_precond_set_front: not on a context made by hp_context_clone"); return 1; }
    if (s && hp_refuse_with_contexts(s, "hp_precond_set_front")) return 1;
    if (hp_set_front_mode(s, mode)) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    HP_CUDA(cudaMemsetAsync(s->status, 0, sizeof(int), st));
    if (hp_front_setup(s, st)) return 2;
    int status = 0;
    HP_CUDA(cudaMemcpyAsync(&status, s->status, sizeof(int), cudaMemcpyDeviceToHost, st));
    HP_CUDA(cudaStreamSynchronize(st));
    if (status) { hp_set_error("hp_precond_set_front: a pivot vanished while factoring the front block (status %d)", status); return 3; }
    return 0;
}
// sweep kernel: 0 = automatic; classic layout: 1 direct, 2 TMA staged, 3 pipelined; cluster layout: 4
extern "C" int hp_set_sweep_variant(hp_solver* s, int v) { if (!s) return 1; s->sweep_variant = v; return 0; }
// generator layout chosen by the next hp_precond_setup: 0 = automatic, 1 = classic (G = P*K CTAs, N by rows),
// 2 = cluster (a leaf is a thread-block cluster, N by separator columns)
extern "C" int hp_set_layout_mode(hp_solver* s, int mode) {
    if (!s || mode < 0 || mode > 2) { hp_set_error("hp_set_layout_mode: mode must be 0, 1 or 2"); return 1; }
    s->layout_mode = mode;
    return 0;
}
extern "C" int hp_strip_layout_ex(hp_solver* s, int* colN, int* NCB, int* NRQ, int* NXG) {
    if (!s || !s->packets) { hp_set_error("hp_strip_layout_ex: preconditioner not set up"); return 1; }
    if (colN) *colN = s->lay.colN; if (NCB) *NCB = s->lay.NCB; if (NRQ) *NRQ = s->lay.NRQ; if (NXG) *NXG = s->lay.NXG;
    return 0;
}
extern "C" int64_t hp_precond_bytes(hp_solver* s) { return s ? s->bytes : 0; }
extern "C" double hp_precond_setup_ms(hp_solver* s) { return s ? s->setup_ms : 0.0; }

extern "C" int hp_precond_apply(hp_solver* s, const double* f_dev, double* u_dev, int diag_mode, void* stream) {
    if (!s) { hp_set_error("hp_precond_apply: null solver"); return 1; }
    if (s->m_lo != s->b + 1 || s->m_hi != s->n) {
        if (!(s->b == s->n)) {
            hp_set_error("hp_precond_apply: solver holds strips %d..%d, needs %d..%d (use the staged calls for slabs)",
                         s->m_lo, s->m_hi, s->b + 1, s->n);
            return 1;
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int n = s->n, b = s->b;
    if (f_dev != u_dev)
        HP_CUDA(cudaMemcpyAsync(u_dev, f_dev, sizeof(cplx) * (size_t)n * n, cudaMemcpyDeviceToDevice, st));
    int rc;
    if ((rc = hp_front_begin(s, u_dev, stream))) return rc;
    if (b < n) {
        if ((rc = hp_sweep_forward(s, u_dev, b + 1, n - 1, stream))) return rc;
        if ((rc = hp_sweep_backward(s, u_dev, n, b + 1, diag_mode, stream))) return rc;
    }
    return hp_front_end(s, u_dev, stream);
}

// algo2_4 for R right-hand sides with ONE pass over the strip generators per sweep direction (csrc/hp_sweep4m.cu).
// R must be 1, 2, 4 or 8 and at most hp_multi_max(s).  Slots whose two pointers are NULL are skipped (masked).
extern "C" int hp_precond_apply_multi(hp_solver* s, int R, const double* const* f_devs, double* const* u_devs, int diag_mode,
                                      void* stream) {
    if (!s || !f_devs || !u_devs) { hp_set_error("hp_precond_apply_multi: null argument"); return 1; }
    if (s->m_lo != s->b + 1 || s->m_hi != s->n) {
        hp_set_error("hp_precond_apply_multi: solver holds strips %d..%d, needs %d..%d (use the staged calls for slabs)",
                     s->m_lo, s->m_hi, s->b + 1, s->n);
        return 1;
    }
    if (R < 1 || R > hp_multi_max(s) || (R & (R - 1))) {
        hp_set_error("hp_precond_apply_multi: R must be a power of two <= %d, got %d", hp_multi_max(s), R);
        return 1;
    }
    // a slot with f_devs[r] == u_devs[r] == NULL is inactive: the launch carries the other slots at their own indices
    int active = 0;
    for (int r = 0; r < R; ++r) {
        if (!f_devs[r] != !u_devs[r]) {
            hp_set_error("hp_precond_apply_multi: slot %d has %s input but %s output (both or neither must be NULL)", r,
                         f_devs[r] ? "an" : "no", u_devs[r] ? "an" : "no");
            return 1;
        }
        active += u_devs[r] != nullptr;
    }
    if (!active) { hp_set_error("hp_precond_apply_multi: all %d slots are empty", R); return 1; }
    cudaStream_t st = (cudaStream_t)stream;
    const int n = s->n, b = s->b;
    const size_t tf = (size_t)b * n;
    if (!s->TFm) HP_CUDA(cudaMalloc(&s->TFm, sizeof(cplx) * tf * 8));
    int rc;
    for (int r = 0; r < R; ++r) {
        if (!u_devs[r]) continue;
        if (f_devs[r] != u_devs[r])
            HP_CUDA(cudaMemcpyAsync(u_devs[r], f_devs[r], sizeof(cplx) * (size_t)n * n, cudaMemcpyDeviceToDevice, st));
        if ((rc = hp_front_begin(s, u_devs[r], stream))) return rc;
        HP_CUDA(cudaMemcpyAsync(s->TFm + r * tf, s->TF, sizeof(cplx) * tf, cudaMemcpyDeviceToDevice, st));
    }
    if (b < n) {
        if ((rc = hp_sweep_forward_multi(s, R, u_devs, b + 1, n - 1, stream))) return rc;
        if ((rc = hp_sweep_backward_multi(s, R, u_devs, n, b + 1, diag_mode, stream))) return rc;
    }
    for (int r = 0; r < R; ++r) {
        if (!u_devs[r]) continue;
        HP_CUDA(cudaMemcpyAsync(s->TF, s->TFm + r * tf, sizeof(cplx) * tf, cudaMemcpyDeviceToDevice, st));
        if ((rc = hp_front_end(s, u_devs[r], stream))) return rc;
    }
    return 0;
}

extern "C" int hp_strip_layout(hp_solver* s, int* P, int* K, int* QP, int* CW, int* NS, int* NR, int64_t* PK,
                               int* leaf_start_host, int* leaf_q_host, int* sep_host) {
    if (!s || !s->packets) { hp_set_error("hp_strip_layout: preconditioner not set up"); return 1; }
    const HpLayout& L = s->lay;
    if (P) *P = L.P; if (K) *K = L.K; if (QP) *QP = L.QP; if (CW) *CW = L.CW;
    if (NS) *NS = L.NS; if (NR) *NR = L.NR; if (PK) *PK = (int64_t)L.PK;
    if (leaf_start_host) memcpy(leaf_start_host, s->leaf_start_h.data(), sizeof(int) * L.P);
    if (leaf_q_host) memcpy(leaf_q_host, s->leaf_q_h.data(), sizeof(int) * L.P);
    if (sep_host && L.P > 1) memcpy(sep_host, s->sep_h.data(), sizeof(int) * (L.P - 1));
    return 0;
}

extern "C" int hp_strip_packets(hp_solver* s, int m, double* packets_host) {
    if (!s || !s->packets) { hp_set_error("hp_strip_packets: preconditioner not set up"); return 1; }
    if (m < s->m_lo || m > s->m_hi) { hp_set_error("hp_strip_packets: strip %d not held", m); return 1; }
    size_t cnt = (size_t)s->lay.G * s->lay.PK;
    HP_CUDA(cudaMemcpy(packets_host, s->packets + (size_t)(m - s->m_lo) * cnt, cnt * sizeof(cplx), cudaMemcpyDeviceToHost));
    return 0;
}
