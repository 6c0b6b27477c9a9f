"""Attenuating media: a complex velocity model through every layer (hp_create_complex and the complex-kappa kernels).

A. A complex c_mat equal to a real model plus 0j gives, bit for bit, what the real solver gives: CSR values, SpMV (whole
   grid and slab rows), strip operators, strip solves, M f for both diagonals and both fronts, and the 8- and 4-wide
   multi-vector sweeps (hp_sweep4d and hp_sweep4m), at n = 63 and 127 (b = 12), n = 200 (b = 20) and 4096^2.
B. A layered model attenuated by a q field (one layer at q = 10, one at q = 50, a Gaussian sponge) against the oracle,
   which handles a complex c_mat as written: CSR, A x, get_Hm, T_m v, M f / M x with 1, 4 and 8 vectors per launch, and
   the preconditioned GMRES solve.
C. The slab decomposition (two ranks on one GPU, the staged schedule driven by hand) on the attenuating model.
D. run_solver_many on the attenuating model: every source the same bits as with zero sources beside it in its slot.
E. The sign convention of fields.attenuate: loss lowers the field far from the source.
"""
import numpy as np
import pytest
import torch

from helmholtz_preconditioner_b200 import fields as hpf
from oracle import helmholtz_oracle as orc
from tests.test_gpu_large import dev
from tests.test_gpu_multi_oracle import SWEEP4D, SWEEP4M, no_dmma, relerr
from tests.test_gpu_slab_oracle import COEF, base_fields, bounds, check, make_ranks, slab_apply

pytestmark = pytest.mark.gpu

CASES = [(63, 12), (127, 12), (200, 20)]
PK = {127: (6, 4)}                # a partition on which both multi-vector kernels run (as the n = 120 slab cases)
IDS = [f"n{n}_b{b}" for n, b in CASES]


@pytest.fixture(scope="module")
def hp():
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return hp


def omega_of(n):
    return 2 * np.pi * (n / 10) + 2j


def layered(n):
    return hpf.init_layered_f1(omega_of(n), n)[0]


def q_field(n):
    """q = 10 in one layer (a band of the depth index x2), 50 in another, lossless elsewhere, plus a Gaussian sponge"""
    x = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x, x, indexing="ij")           # c_mat[i, j]: i along x1, j along x2 (depth)
    inv_q = np.zeros((n + 2, n + 2))
    inv_q[:, (n + 2) // 4:(n + 2) // 2] = 1 / 10
    inv_q[:, (n + 2) // 2:3 * (n + 2) // 4] = 1 / 50
    sponge = 0.2 * np.exp(-((xx - 0.8) ** 2 + (yy - 0.85) ** 2) / 0.01)
    inv_q += np.where(sponge > 1e-4, sponge, 0.0)
    with np.errstate(divide="ignore"):
        return np.where(inv_q > 0, 1 / np.where(inv_q > 0, inv_q, 1), np.inf)


def atten_model(hp, n):
    c = hpf.attenuate(layered(n), q_field(n))
    assert c.dtype == np.complex128 and np.all(c.imag <= 0) and np.any(c.imag < 0)
    return c


def fields_for(n, seed):
    rng = np.random.default_rng(seed)
    f = np.asarray(orc.init_f1_mat(.5, .125, omega_of(n), n), dtype=np.complex128).ravel()
    x = rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n)
    return f, x


def same(a, b, what):
    assert a.shape == b.shape and torch.equal(a, b), what


# ---------------------------------------------------------------------------------------------------------------------
# A. zero imaginary part
# ---------------------------------------------------------------------------------------------------------------------
def outputs(hp, n, b, c_mat, P=0, K=0):
    """everything the zero-imaginary-part test compares, computed by one solver (closed before returning)"""
    s = hp.HelmholtzSolver(n, b, omega_of(n), 60.0, c_mat)
    out = {}
    try:
        assert s.medium_is_complex == np.iscomplexobj(c_mat)
        f, x = (dev(v) for v in fields_for(n, n))
        A = s.assemble_csr()
        out["csr"] = (A.indptr.clone(), A.indices.clone(), A.data.clone())
        del A
        out["matvec"] = s.matvec(x)
        j0, j1 = n // 3, n // 3 + 17
        out["matvec_rows"] = s.matvec_rows(j0, j1, x[j0 * n:j1 * n].clone(), x[(j0 - 1) * n:j0 * n].clone(),
                                           x[j1 * n:(j1 + 1) * n].clone(), torch.empty((j1 - j0) * n, dtype=torch.complex128, device="cuda"))
        for m in (b, b + 1, n // 2, n):
            H = s.assemble_strip_csr(m)
            out[f"Hm{m}"] = (H.indptr.clone(), H.indices.clone(), H.data.clone())
        s.setup_preconditioner(P, K)
        v = x[:n].clone()
        for m in (b + 1, (b + 1 + n) // 2, n):
            out[f"T{m}"] = s.strip_apply(m, v)
        xs8 = [dev(w) for w in COEF @ np.array([f.cpu().numpy(), x.cpu().numpy(), (x * 1j).cpu().numpy() + 3])]
        for front in ("blockdiag", "coupled"):
            s.set_front(front)
            for diag in ("reference", "paper"):
                tag = (front, diag)
                out[tag + ("f",)] = s.precond_apply(f, diag=diag)
                out[tag + ("x",)] = s.precond_apply(x, diag=diag)
                kernels = []
                for R in (8, 4):
                    if s.multi_kernel(R):
                        outs = [torch.empty_like(f) for _ in range(R)]
                        s.precond_apply_multi(xs8[:R], outs, diag=diag)
                        out[tag + (R,)] = outs
                        kernels.append(s.multi_kernel(R))
                if s.multi_kernel(8) == SWEEP4D:
                    with no_dmma():
                        assert s.multi_kernel(8) == SWEEP4M
                        outs = [torch.empty_like(f) for _ in range(8)]
                        s.precond_apply_multi(xs8, outs, diag=diag)
                        out[tag + ("8m",)] = outs
                        kernels.append(SWEEP4M)
                out[tag + ("kernels",)] = kernels
        assert s.sweep_status() == 0
        torch.cuda.synchronize()
        return out
    finally:
        s.close()


def compare_outputs(o_real, o_cplx):
    assert o_real.keys() == o_cplx.keys()
    for k in o_real:
        a, c = o_real[k], o_cplx[k]
        if isinstance(a, (list, tuple)) and a and isinstance(a[0], torch.Tensor):
            for i, (t, u) in enumerate(zip(a, c)):
                same(t, u, (k, i))
        elif isinstance(a, torch.Tensor):
            same(a, c, k)
        else:
            assert a == c, (k, a, c)


@pytest.mark.parametrize("n,b", CASES, ids=IDS)
def test_zero_imaginary_part_is_bit_identical(hp, n, b):
    c = layered(n)
    o_real = outputs(hp, n, b, c, *PK.get(n, (0, 0)))
    o_cplx = outputs(hp, n, b, c + 0j, *PK.get(n, (0, 0)))
    compare_outputs(o_real, o_cplx)
    kernels = {k for key, v in o_real.items() if key[-1] == "kernels" for k in v}
    if n in PK:
        assert {SWEEP4D, SWEEP4M} <= kernels, kernels


def test_zero_imaginary_part_4096(hp):
    """the benchmark's layered 4096^2 model, b = 12: the real solver is closed before the complex one is set up"""
    n, b = 4096, 12
    c = layered(n)

    def run(c_mat):
        s = hp.HelmholtzSolver(n, b, omega_of(n), 60.0, c_mat)
        try:
            f, x = (dev(v) for v in fields_for(n, 5))
            A = s.assemble_csr()
            r = {"csr": A.data.clone(), "matvec": s.matvec(x)}
            del A
            H = s.assemble_strip_csr(n // 2)
            r["Hm"] = H.data.clone()
            del H
            s.setup_preconditioner(0, 0, front="coupled")
            r["T"] = s.strip_apply(n // 2, x[:n].clone())
            r["Mf"] = s.precond_apply(f, diag="paper")
            for R in (8, 4):
                assert s.multi_kernel(R), R
                outs = [torch.empty_like(f) for _ in range(R)]
                s.precond_apply_multi([f if i % 2 == 0 else x for i in range(R)], outs, diag="paper")
                r[R] = outs
            assert s.sweep_status() == 0
            torch.cuda.synchronize()
            return r
        finally:
            s.close()

    o_real = run(c)
    torch.cuda.empty_cache()
    o_cplx = run(c + 0j)
    compare_outputs(o_real, o_cplx)


# ---------------------------------------------------------------------------------------------------------------------
# B. attenuating media against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,b", CASES, ids=IDS)
def test_attenuating_operator_vs_oracle(hp, n, b):
    c = atten_model(hp, n)
    omega, const, h = omega_of(n), 60.0, 1 / (n + 1)
    eta = b * h
    s = hp.HelmholtzSolver(n, b, omega, const, c)
    try:
        assert s.medium_is_complex
        A0 = orc.build_A_matrix(b, const, eta, omega, h, n, c).tocsr()
        A0.sort_indices()
        A = s.assemble_csr()
        indptr, indices, data = (t.cpu().numpy() for t in (A.indptr, A.indices, A.data))
        assert np.array_equal(indptr, A0.indptr) and np.array_equal(indices, A0.indices)
        assert np.max(np.abs(data - A0.data) / np.abs(A0.data)) < 1e-12
        assert np.any(np.abs(A0.data.imag) > 0)
        _, x = fields_for(n, 7)
        assert relerr(s.matvec(dev(x)), A0 @ x) < 1e-13
        for m in (b, b + 1, n // 2, n):
            H0 = orc.get_Hm(m, b, const, eta, omega, h, n, c).tocsr()
            H0.sort_indices()
            ip, ix, d = hp.get_Hm(m, b, const, eta, omega, h, n, c).to_host()
            assert np.array_equal(ip, H0.indptr) and np.array_equal(ix, H0.indices), m
            assert np.max(np.abs(d - H0.data) / np.abs(H0.data)) < 1e-12, m
        HF0 = orc.get_A_FF_block(b, const, eta, omega, h, n, c).tocsr()
        HF0.sort_indices()
        HF0.eliminate_zeros()
        ip, ix, d = hp.get_A_FF_block(b, const, eta, omega, h, n, c).to_host()
        assert np.array_equal(ip, HF0.indptr) and np.array_equal(ix, HF0.indices)
        assert np.max(np.abs(d - HF0.data) / np.abs(HF0.data)) < 1e-12
    finally:
        s.close()


@pytest.mark.parametrize("n,b", CASES, ids=IDS)
def test_attenuating_preconditioner_vs_oracle(hp, n, b):
    c = atten_model(hp, n)
    omega, const, h = omega_of(n), 60.0, 1 / (n + 1)
    f, x = fields_for(n, 11)
    base = [f, x, x.conj() * 1j]
    s = hp.HelmholtzSolver(n, b, omega, const, c).setup_preconditioner()
    try:
        Pc = orc.SweepingPreconditioner(b, const, b * h, omega, h, n, c)
        rng = np.random.default_rng(3)
        for m in (b + 1, (b + 1 + n) // 2, n):
            v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
            assert relerr(s.strip_apply(m, dev(v)), Pc.T(m, v)) < 1e-12, m
        for front in ("blockdiag", "coupled"):
            s.set_front(front)
            Pc = orc.SweepingPreconditioner(b, const, b * h, omega, h, n, c, front=front)
            for diag in ("reference", "paper"):
                Pc.diag = diag
                mb = [Pc.apply(v) for v in base]
                refs8 = COEF @ np.array(mb)
                xs8 = [dev(v) for v in COEF @ np.array(base)]
                for k in range(2):
                    assert relerr(s.precond_apply(dev(base[k]), diag=diag), mb[k]) < 1e-12, (front, diag, k)
                for R in (4, 8):
                    assert s.multi_kernel(R), (R, s.layout())
                    outs = [torch.empty_like(xs8[0]) for _ in range(R)]
                    s.precond_apply_multi(xs8[:R], outs, diag=diag)
                    check(outs, list(refs8[:R]), (front, diag, f"{R} per launch"))
        assert s.sweep_status() == 0
    finally:
        s.close()


@pytest.mark.parametrize("n,b", CASES, ids=IDS)
def test_attenuating_run_solver_vs_oracle(hp, n, b):
    c = atten_model(hp, n)
    wn, const, alpha = n / 10, 60.0, 2.0
    kw = dict(c_mat=c, precond_input="vector", diag="paper", front="coupled", maxiter=60)
    r = hp.run_solver(n, b, wn, const, alpha, verbose=False, **kw)
    u0, hist0, niter0, info0 = orc.run_solver(n, b, wn, const, alpha, **kw)
    assert r.solver.medium_is_complex
    assert abs(r.niter - niter0) <= 1 and r.info == info0, (r.niter, niter0, r.info, info0)
    assert relerr(r.u, u0) < 1e-8
    r.solver.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. slab decomposition
# ---------------------------------------------------------------------------------------------------------------------
def test_attenuating_slab_vs_oracle(hp):
    n, b, const = 120, 12, 60.0
    c = atten_model(hp, n)
    omega, h = omega_of(n), 1 / (n + 1)
    f = np.asarray(orc.init_f1_mat(.5, .125, omega, n), dtype=np.complex128).ravel()
    base = base_fields(n, f)
    ranks = make_ranks(hp, n, b, omega, const, c, bounds(n, b, 2), P=6, K=4, layout="cluster")
    try:
        assert all(rk.s.medium_is_complex for rk in ranks)
        xs8 = [dev(v) for v in COEF @ np.array(base)]
        for front in ("blockdiag", "coupled"):
            ranks[0].s.set_front(front)
            Pc = orc.SweepingPreconditioner(b, const, b * h, omega, h, n, c, front=front)
            for diag in ("reference", "paper"):
                Pc.diag = diag
                refs8 = COEF @ np.array([Pc.apply(v) for v in base])
                check(slab_apply(ranks, [xs8[0]], diag), [refs8[0]], (front, diag, "single"))
                check(slab_apply(ranks, xs8, diag, [list(range(8))]), refs8, (front, diag, "8 per launch"))
                check(slab_apply(ranks, xs8[:4], diag, [list(range(4))]), refs8[:4], (front, diag, "4 per launch"))
        for rk in ranks:
            assert rk.s.sweep_status() == 0, rk.r
    finally:
        for rk in ranks:
            rk.close()


# ---------------------------------------------------------------------------------------------------------------------
# D. many sources
# ---------------------------------------------------------------------------------------------------------------------
def test_attenuating_run_solver_many(hp):
    n, b, wn, const, alpha = 127, 12, 12.7, 60.0, 2.0
    c = atten_model(hp, n)
    omega = 2 * np.pi * wn + 1j * alpha
    s = hp.HelmholtzSolver(n, b, omega, const, c).setup_preconditioner(front="coupled")
    try:
        assert s.multi_max == 8, s.layout()
        fs = [np.asarray(orc.init_f1_mat(r1, r2, omega, n), dtype=np.complex128)
              for r1, r2 in [(.5, .125), (.25, .3), (.7, .6), (.4, .85), (.1, .5)]]
        kw = dict(c_mat=c, solver=s, diag="paper", precond_input="vector", rtol=1e-6, maxiter=60, verbose=False)
        rs = hp.run_solver_many(n, b, wn, const, alpha, np.stack(fs), **kw)
        for i, f in enumerate(fs):
            alone = hp.run_solver_many(n, b, wn, const, alpha, [np.zeros_like(f)] * i + [f], **kw)[i]   # same slot, zero companions
            assert torch.equal(alone.u, rs[i].u), i
            assert alone.residuals == rs[i].residuals and alone.niter == rs[i].niter and alone.info == rs[i].info, i
            r1 = hp.run_solver(n, b, wn, const, alpha, f_mat=f, **kw)
            assert r1.info == rs[i].info and abs(r1.niter - rs[i].niter) <= 1, (i, r1.niter, rs[i].niter)
            if r1.niter == rs[i].niter:
                assert relerr(rs[i].u, r1.u.cpu().numpy()) < 1e-8, i
        assert s.sweep_status() == 0
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# E. sign convention
# ---------------------------------------------------------------------------------------------------------------------
def test_loss_lowers_the_far_field(hp):
    n, b, wn, const, alpha = 255, 12, 12.0, 60.0, 0.0
    omega = 2 * np.pi * wn + 1j * alpha
    c0 = np.ones((n + 2, n + 2))
    f = orc.init_f1_mat(.5, .5, omega, n)
    norms = {}
    for q in (np.inf, 10.0):
        c = hpf.attenuate(c0, q)
        if q == np.inf:
            assert np.array_equal(c, c0 + 0j) and not np.any(c.imag)
        r = hp.run_solver(n, b, wn, const, alpha, c_mat=c, f_mat=f, precond_input="vector", diag="paper",
                          front="coupled", rtol=1e-6, maxiter=200, verbose=False)
        assert r.info == 0, (q, r.niter)
        u = r.u.cpu().numpy().reshape(n, n)            # u[j-1, i-1]: the row index is x2
        norms[q] = np.linalg.norm(u[:n // 5])            # x2 < 0.2: more than 0.3 away from the source at x2 = 0.5
        r.solver.close()
    assert norms[10.0] < 0.5 * norms[np.inf], norms
