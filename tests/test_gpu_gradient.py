"""Inversion: the gradient and Born kernels (csrc/hp_grad.cu) and the drivers misfit_gradient / born (inversion.py).

1. The three kernels against numpy at n = 63, 127, 200 (b = 20) and 4096, R = 1, 2, 4, 8 with masked slots, for a real and
   an attenuating medium, on random inputs without symmetry (a transposed index fails).  Deterministic, and the
   accumulation gives the same bits however its sources are split into launches.
2. misfit_gradient end to end against a numpy reference built on the oracle's operator (a sparse LU of
   orc.build_A_matrix) at n = 63 and 127, real and attenuating, for both wrt.
3. A real model + 0j gives the real model's gradient bit for bit.
4. The Born/gradient identity Re sum_s r_s^H R du_s = Re <G, dkappa> at n = 255 and at the 4096^2 benchmark configuration
   with 8 and 11 sources; a dkappa applied transposed fails it.
5. A Taylor test of G against J at n = 127 on the attenuating model.
"""
import numpy as np
import pytest
import scipy.sparse.linalg as spla
import torch

from helmholtz_preconditioner_b200 import fields as hpf
from oracle import helmholtz_oracle as orc
from tests.golden.make_golden_large import load as load_fixture
from tests.test_gpu_large import MF_FILES, case_fields, dev
from tests.test_gpu_medium import atten_model, hp, layered, omega_of, q_field  # noqa: F401  (hp: fixture)

pytestmark = pytest.mark.gpu

CONST = 60.0


# ---------------------------------------------------------------------------------------------------------------------
# numpy reference
# ---------------------------------------------------------------------------------------------------------------------
def w_grid(n, b, omega, const):
    """w_p = omega^2 / (s1(i h) s2(j h)) = dA_pp/dkappa_p, flattened like the field: p = (j-1) n + (i-1)"""
    h = 1 / (n + 1)
    x = np.arange(1, n + 1) * h
    is1 = 1 / orc.s1(x, const, b * h, omega)
    is2 = 1 / orc.s2(x, const, b * h, omega)
    return (omega ** 2 * np.outer(is2, is1)).ravel()


def to_cmat(g, n):
    out = np.zeros((n + 2, n + 2), dtype=g.dtype)
    out[:n, :n] = g.reshape(n, n).T
    return out


def from_cmat(x, n):
    return np.asarray(x)[:n, :n].T.ravel()


def kappa_grid(c_mat, n):
    return 1 / from_cmat(c_mat, n) ** 2


def finish_ref(acc, n, b, omega, const, c_mat, wrt):
    G = -np.conj(w_grid(n, b, omega, const) * acc)
    if wrt == "velocity":
        k = kappa_grid(c_mat, n)
        G = np.conj(-2 * k * np.sqrt(k)) * G
    if not np.iscomplexobj(c_mat):
        G = G.real
    return to_cmat(G, n)


def ref_gradient(n, b, omega, const, c_mat, fs, idx, d_obs, wrt):
    """misfit, gradient (c_mat layout) and residuals with exact solves on the oracle's operator"""
    h = 1 / (n + 1)
    lu = spla.splu(orc.build_A_matrix(b, const, b * h, omega, h, n, c_mat).tocsc())
    acc = np.zeros(n * n, dtype=np.complex128)
    J, res = 0.0, []
    for f, d in zip(fs, d_obs):
        u = lu.solve(np.asarray(f, dtype=np.complex128).ravel())
        r = u[idx] - d
        a = np.zeros(n * n, dtype=np.complex128)
        a[idx] = np.conj(r)
        acc += lu.solve(a) * u
        J += 0.5 * np.sum(np.abs(r) ** 2)
        res.append(r)
    return J, finish_ref(acc, n, b, omega, const, c_mat, wrt), np.array(res)


def ref_data(n, b, omega, const, c_mat, fs, idx):
    h = 1 / (n + 1)
    lu = spla.splu(orc.build_A_matrix(b, const, b * h, omega, h, n, c_mat).tocsc())
    return np.array([lu.solve(np.asarray(f, dtype=np.complex128).ravel())[idx] for f in fs])


def rand_c(n, seed, complex_medium):
    rng = np.random.default_rng(seed)
    c = 1 + rng.random((n + 2, n + 2))
    return hpf.attenuate(c, 5 + 50 * rng.random((n + 2, n + 2))) if complex_medium else c


def rand_np(rng, shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


def blobs(n, seed, amp, complex_values=True, count=6):
    """a smooth random perturbation in c_mat layout without symmetry: Gaussian blobs at random centres"""
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x, x, indexing="ij")
    out = np.zeros((n + 2, n + 2), dtype=np.complex128 if complex_values else np.float64)
    for _ in range(count):
        cx, cy, sg = rng.uniform(.15, .85), rng.uniform(.15, .85), rng.uniform(.05, .15)
        a = rng.standard_normal() + (1j * rng.standard_normal() if complex_values else 0)
        out += amp * a * np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / sg ** 2)
    return out


def shots(n, omega, positions):
    return [np.asarray(hpf.init_f1_mat(p[0], p[1], omega, n), dtype=np.complex128) for p in positions]


def line_receivers(hp, n, count=20, depth=0.2):
    i = np.unique(np.linspace(1, n, count).round().astype(np.int64))
    return hp.Receivers(n, i, np.full(len(i), max(1, round(depth * (n + 1)))))


def inner(G, dk, n):
    """Re <G, dkappa> = Re sum_p conj(G_p) dkappa_p over the grid points (c_mat layout)"""
    return float(np.real(np.sum(np.conj(np.asarray(G)[:n, :n]) * np.asarray(dk)[:n, :n])))


# ---------------------------------------------------------------------------------------------------------------------
# 1. kernels
# ---------------------------------------------------------------------------------------------------------------------
KCASES = [(63, 12), (127, 12), (200, 20), (4096, 12)]
KIDS = [f"n{n}_b{b}" for n, b in KCASES]
MASKS = {1: [0], 2: [0, 1], 4: [0, 2, 3], 8: [0, 1, 3, 4, 6, 7]}      # active slots per width


def accumulate(s, us, mus, acc):
    from helmholtz_preconditioner_b200 import _lib
    _lib.check(s.lib.hp_grad_accumulate(s.handle, len(us), s._ptr_array(us), s._ptr_array(mus), acc.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream), "hp_grad_accumulate")


def finish(s, acc, wrt):
    from helmholtz_preconditioner_b200 import _lib
    out = torch.full((s.n + 2, s.n + 2), float("nan"), dtype=torch.complex128 if s.medium_is_complex else torch.float64,
                     device="cuda")
    _lib.check(s.lib.hp_grad_finish(s.handle, acc.data_ptr(), wrt, out.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "hp_grad_finish")
    return out


def born_source(s, dk, us, outs):
    from helmholtz_preconditioner_b200 import _lib
    _lib.check(s.lib.hp_born_source(s.handle, len(us), dk.data_ptr(), s._ptr_array(us), s._ptr_array(outs),
                                    torch.cuda.current_stream().cuda_stream), "hp_born_source")


def gpu_rand(n, count, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.complex(torch.randn(n * n, generator=g, device="cuda", dtype=torch.float64),
                          torch.randn(n * n, generator=g, device="cuda", dtype=torch.float64)) for _ in range(count)]


@pytest.mark.parametrize("n,b", KCASES, ids=KIDS)
@pytest.mark.parametrize("medium", ["real", "attenuating"])
def test_kernels_vs_numpy(hp, n, b, medium):
    """accumulate, finish and Born source against numpy (n <= 200) or the same arithmetic in torch on the device (4096,
    where host copies of 17 fields would take 5 GB); the finish border is exactly zero; repeated calls are bit-identical"""
    omega = omega_of(n)
    c = rand_c(n, n, medium == "attenuating")
    s = hp.HelmholtzSolver(n, b, omega, CONST, c)
    big = n > 1000
    widths = (8,) if big else (1, 2, 4, 8)
    try:
        xs = gpu_rand(n, 17, n)
        w = dev(w_grid(n, b, omega, CONST))
        # accumulate
        for R in widths:
            act = MASKS[R]
            us = [xs[r] if r in act else None for r in range(R)]
            mus = [xs[8 + r] if r in act else None for r in range(R)]
            acc0 = xs[16]
            acc = acc0.clone()
            accumulate(s, us, mus, acc)
            if big:
                ref, scale = acc0.clone(), acc0.abs()
                for r in act:
                    ref = ref + us[r] * mus[r]
                    scale = scale + us[r].abs() * mus[r].abs()
                err = float(torch.max((acc - ref).abs() / scale))
            else:
                ref, scale = acc0.cpu().numpy(), np.abs(acc0.cpu().numpy())
                for r in act:
                    u, m = us[r].cpu().numpy(), mus[r].cpu().numpy()
                    ref = ref + u * m
                    scale = scale + np.abs(u) * np.abs(m)
                err = float(np.max(np.abs(acc.cpu().numpy() - ref) / scale))
            assert err < 1e-14, (R, err)
            again = acc0.clone()
            accumulate(s, us, mus, again)
            assert torch.equal(again, acc), R
            if R > 1:                                          # the same sources split over two launches
                split = acc0.clone()
                accumulate(s, us[:R // 2], mus[:R // 2], split)
                accumulate(s, us[R // 2:], mus[R // 2:], split)
                assert torch.equal(split, acc), R
        # finish
        acc = xs[16]
        for wrt, name in ((0, "kappa"), (1, "velocity")):
            out = finish(s, acc, wrt)
            assert torch.equal(out, finish(s, acc, wrt))
            assert not torch.any(out[n:, :]) and not torch.any(out[:, n:]), "border not zero"
            # the error is measured against |G| of the complex product: Re G of a real medium may cancel
            if big:
                G = -torch.conj(w * acc)
                if wrt:
                    k = dev(kappa_grid(c, n))
                    G = torch.conj(-2 * k * torch.sqrt(k)) * G
                ref, scale = G.reshape(n, n).T, G.abs().reshape(n, n).T
                got = out[:n, :n] if s.medium_is_complex else out[:n, :n].to(torch.complex128)
                if not s.medium_is_complex:
                    ref = ref.real.to(torch.complex128)
                err = float(torch.max((got - ref).abs() / scale))
            else:
                a = acc.cpu().numpy()
                ref = finish_ref(a, n, b, omega, CONST, c, name)
                scale = np.abs(finish_ref(np.abs(a) + 0j, n, b, omega, CONST, c + 0j, name))[:n, :n]
                got = out.cpu().numpy()
                assert got.dtype == ref.dtype
                err = float(np.max(np.abs(got - ref)[:n, :n] / scale))
            assert err < 1e-14, (name, err)
        # Born source; the last two rows and columns of dkappa are NaN (never read)
        rng = np.random.default_rng(n + 1)
        dk_np = rand_np(rng, (n + 2, n + 2)) if not big else None
        dk = dev(dk_np) if not big else torch.complex(torch.randn(n + 2, n + 2, dtype=torch.float64, device="cuda"),
                                                      torch.randn(n + 2, n + 2, dtype=torch.float64, device="cuda"))
        dk[n:, :] = complex("nan")
        dk[:, n:] = complex("nan")
        dkg = dk[:n, :n].T.reshape(-1)
        for R in widths:
            act = MASKS[R]
            us = [xs[r] if r in act else None for r in range(R)]
            outs = [torch.full_like(xs[0], complex("nan")) if r in act else None for r in range(R)]
            born_source(s, dk, us, outs)
            for r in act:
                if big:
                    ref = -w * dkg * us[r]
                    err = float(torch.max((outs[r] - ref).abs() / ref.abs().clamp_min(1e-300)))
                else:
                    ref = -w.cpu().numpy() * from_cmat(dk_np, n) * us[r].cpu().numpy()
                    err = float(np.max(np.abs(outs[r].cpu().numpy() - ref) / np.maximum(np.abs(ref), 1e-300)))
                assert err < 1e-14, (R, r, err)
            again = [None if o is None else torch.empty_like(o) for o in outs]
            born_source(s, dk, us, again)
            assert all(o is None or torch.equal(o, a) for o, a in zip(outs, again)), R
            inplace = [None if u is None else u.clone() for u in us]    # out_r = u_r
            born_source(s, dk, inplace, inplace)
            assert all(o is None or torch.equal(o, a) for o, a in zip(outs, inplace)), R
    finally:
        s.close()


def test_kernel_argument_checks(hp):
    n = 40
    s = hp.HelmholtzSolver(n, 8, omega_of(n), CONST, layered(n))
    try:
        x = gpu_rand(n, 3, 1)
        acc = torch.zeros_like(x[0])
        dk = torch.zeros(n + 2, n + 2, dtype=torch.complex128, device="cuda")
        bad = [
            (lambda: accumulate(s, [], [], acc), "R must lie"),
            (lambda: accumulate(s, x[:1] * 9, x[:1] * 9, acc), "R must lie"),
            (lambda: accumulate(s, [None, None], [None, None], acc), "empty"),
            (lambda: accumulate(s, [x[0], None], [x[1], x[2]], acc), "both or neither"),
            (lambda: born_source(s, dk, [x[0]], [None]), "both or neither"),
            (lambda: born_source(s, dk, [None] * 4, [None] * 4), "empty"),
        ]
        for f, text in bad:
            with pytest.raises(hp.HelmholtzB200Error, match=text):
                f()
        st = torch.cuda.current_stream().cuda_stream
        from helmholtz_preconditioner_b200 import _lib
        for call, text in ((lambda: s.lib.hp_grad_accumulate(s.handle, 1, s._ptr_array(x[:1]), s._ptr_array(x[1:2]), None, st), "null accumulator"),
                           (lambda: s.lib.hp_grad_finish(s.handle, None, 0, acc.data_ptr(), st), "null accumulator"),
                           (lambda: s.lib.hp_grad_finish(s.handle, acc.data_ptr(), 0, None, st), "null output"),
                           (lambda: s.lib.hp_grad_finish(s.handle, acc.data_ptr(), 2, acc.data_ptr(), st), "wrt must be"),
                           (lambda: s.lib.hp_born_source(s.handle, 1, None, s._ptr_array(x[:1]), s._ptr_array(x[1:2]), st), "null dkappa")):
            assert call() != 0 and text in _lib.load().hp_last_error().decode(), text
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2./3. misfit_gradient end to end
# ---------------------------------------------------------------------------------------------------------------------
SHOTS3 = [(0.5, 0.125), (0.25, 0.3), (0.7, 0.2)]


def models(n, attenuating):
    """background and true model (the true one has a low-velocity lens just below the receivers, above the strongly
    attenuating layer of q_field, so that the residuals are a few per cent of the data), attenuated alike"""
    c0 = layered(n)
    x = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x, x, indexing="ij")
    c1 = c0 * (1 - 0.15 * np.exp(-((xx - 0.45) ** 2 + (yy - 0.3) ** 2) / 0.01))
    if attenuating:
        return hpf.attenuate(c0, q_field(n)), hpf.attenuate(c1, q_field(n))
    return c0, c1


@pytest.mark.parametrize("n", [63, 127])
@pytest.mark.parametrize("medium", ["real", "attenuating"])
def test_misfit_gradient_vs_reference(hp, n, medium):
    b, omega = 12, omega_of(n)
    c_bg, c_true = models(n, medium == "attenuating")
    fs = shots(n, omega, SHOTS3)
    rec = line_receivers(hp, n)
    idx = rec.index.cpu().numpy()
    d_obs = ref_data(n, b, omega, CONST, c_true, fs, idx)
    s = hp.HelmholtzSolver(n, b, omega, CONST, c_bg).setup_preconditioner(front="coupled")
    try:
        for wrt in ("kappa", "velocity"):
            J0, G0, r0 = ref_gradient(n, b, omega, CONST, c_bg, fs, idx, d_obs, wrt)
            res = hp.misfit_gradient(s, np.stack(fs), rec, d_obs, wrt=wrt, rtol=1e-10)
            assert all(i == 0 for i in res.forward_info + res.adjoint_info)
            assert res.grad.dtype == (torch.complex128 if medium == "attenuating" else torch.float64)
            assert abs(res.misfit - J0) <= 1e-9 * J0, (wrt, res.misfit, J0)
            G = res.grad.cpu().numpy()
            err = np.max(np.abs(G - G0)) / np.max(np.abs(G0))
            assert err < 1e-7, (wrt, err)
            assert np.linalg.norm(res.residuals.cpu().numpy() - r0) <= 1e-8 * np.linalg.norm(r0)
            assert not np.any(G[n:, :]) and not np.any(G[:, n:])
        assert s.sweep_status() == 0
    finally:
        s.close()


def test_real_medium_is_real_part_of_complex(hp):
    """wrt='kappa': Re of the gradient of c + 0j is the real medium's gradient, bit for bit"""
    n, b = 63, 12
    omega = omega_of(n)
    c_bg, c_true = models(n, False)
    fs = shots(n, omega, SHOTS3)
    rec = line_receivers(hp, n)
    d_obs = ref_data(n, b, omega, CONST, c_true, fs, rec.index.cpu().numpy())
    out = {}
    for name, c in (("real", c_bg), ("complex", c_bg + 0j)):
        s = hp.HelmholtzSolver(n, b, omega, CONST, c).setup_preconditioner(front="coupled")
        try:
            out[name] = hp.misfit_gradient(s, fs, rec, d_obs, wrt="kappa", rtol=1e-10)
        finally:
            s.close()
    assert out["complex"].grad.dtype == torch.complex128 and out["real"].grad.dtype == torch.float64
    assert torch.equal(out["complex"].grad.real.contiguous(), out["real"].grad)
    assert out["complex"].misfit == out["real"].misfit


def test_refuses_unset_solver_and_nonconvergence(hp):
    n = 63
    omega = omega_of(n)
    rec = line_receivers(hp, n)
    fs = shots(n, omega, SHOTS3)
    d = np.zeros((3, rec.nrec))
    s = hp.HelmholtzSolver(n, 12, omega, CONST, layered(n))
    try:
        with pytest.raises(hp.HelmholtzB200Error, match="set up"):
            hp.misfit_gradient(s, fs, rec, d)
        s.setup_preconditioner(front="blockdiag")
        with pytest.raises(hp.HelmholtzB200Error, match="did not converge"):
            hp.misfit_gradient(s, fs, rec, d, diag="reference", rtol=1e-12, maxiter=1)
        with pytest.raises(ValueError):
            hp.misfit_gradient(s, fs, hp.Receivers(n + 1, [1], [1]), np.zeros((3, 1)))
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. Born / gradient identity
# ---------------------------------------------------------------------------------------------------------------------
def identity_gap(hp, s, fs, rec, d_obs, dk, rtol):
    res = hp.misfit_gradient(s, fs, rec, d_obs, wrt="kappa", rtol=rtol, keep_fields=True)
    Rdu = hp.born(s, None, rec, dk, rtol=rtol, u=res.u)
    lhs = float(torch.sum(torch.conj(res.residuals) * Rdu).real.item())
    G = res.grad.cpu().numpy()
    rhs, rhs_t = inner(G, dk, s.n), inner(G, np.asarray(dk).T, s.n)
    return abs(lhs - rhs) / max(abs(lhs), abs(rhs)), abs(lhs - rhs_t) / max(abs(lhs), abs(rhs_t)), lhs, res


def test_born_identity_255(hp):
    """Observed on a B200: gap 1.3e-11, transposed dkappa 1.1 (target <= 1e-6).  Born with u solved again from f_mats
    gives the same data to 1e-8."""
    n, b = 255, 12
    omega = omega_of(n)
    c_bg = atten_model(hp, n)
    fs = shots(n, omega, SHOTS3)
    rec = line_receivers(hp, n, count=40)
    d_obs = np.zeros((len(fs), rec.nrec))
    dk = blobs(n, 7, amp=0.1)
    s = hp.HelmholtzSolver(n, b, omega, CONST, c_bg).setup_preconditioner(front="coupled")
    try:
        gap, gap_t, lhs, res = identity_gap(hp, s, fs, rec, d_obs, dk, 1e-10)
        print(f"n=255 identity gap {gap:.2e}, transposed {gap_t:.2e}")
        assert gap <= 1e-6, gap
        assert gap_t > 1e-2, gap_t
        again = hp.born(s, np.stack(fs), rec, dk, rtol=1e-10)
        ref = hp.born(s, None, rec, dk, rtol=1e-10, u=res.u)
        assert torch.linalg.norm(again - ref) <= 1e-8 * torch.linalg.norm(ref)
    finally:
        s.close()


SHOTS11 = [(0.5, 0.125), (0.2, 0.3), (0.8, 0.3), (0.35, 0.6), (0.65, 0.6), (0.5, 0.85), (0.15, 0.8), (0.85, 0.8),
           (0.3, 0.45), (0.7, 0.45), (0.25, 0.15)]


@pytest.fixture(scope="module")
def big(hp):
    """the benchmark's 4096^2 layered configuration, coupled front"""
    g = load_fixture(MF_FILES[0])
    omega, c_mat, _ = case_fields(hp, g)
    s = hp.HelmholtzSolver(int(g["n"]), int(g["b"]), omega, float(g["const"]), c_mat).setup_preconditioner(front="coupled")
    yield s, omega
    s.close()


@pytest.mark.parametrize("S", [8, 11])
def test_born_identity_4096(hp, big, S):
    """8 sources fill one wave, 11 leave three slots of the second wave empty.  Real medium, so dkappa is real.
    Observed on a B200: gap 4.2e-10 (8 sources) and 5.1e-10 (11), transposed dkappa 0.44 and 1.2 (target <= 1e-6)."""
    s, omega = big
    n = s.n
    assert s._widest() == 8
    fs = shots(n, omega, SHOTS11[:S])
    i = np.arange(1, n + 1, 16)
    rec = hp.Receivers(n, i, np.full(len(i), round(0.2 * (n + 1))))
    d_obs = np.zeros((S, rec.nrec))
    dk = blobs(n, 11, amp=0.05, complex_values=False)
    gap, gap_t, lhs, res = identity_gap(hp, s, fs, rec, d_obs, dk, 1e-10)
    print(f"n=4096 S={S} identity gap {gap:.2e}, transposed {gap_t:.2e}, forward niter {res.forward_niter}, "
          f"adjoint niter {res.adjoint_niter}")
    assert gap <= 1e-6, gap
    assert gap_t > 1e-2, gap_t
    assert s.sweep_status() == 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. Taylor test
# ---------------------------------------------------------------------------------------------------------------------
def test_taylor_127_attenuating(hp):
    """|J(kappa + eps dkappa) - J(kappa) - eps Re<G, dkappa>| falls by >= 50x per decade of eps (second order), each J from
    a fresh solver.  Observed on a B200: 2.17e-14, 2.17e-16, 2.17e-18 (100x per decade)"""
    n, b = 127, 12
    omega = omega_of(n)
    c_bg, c_true = models(n, True)
    fs = shots(n, omega, SHOTS3)
    rec = line_receivers(hp, n)
    d_obs = ref_data(n, b, omega, CONST, c_true, fs, rec.index.cpu().numpy())
    kap = 1 / c_bg ** 2
    dk = blobs(n, 5, amp=0.3 * float(np.mean(np.abs(kap))))

    def run(c):
        s = hp.HelmholtzSolver(n, b, omega, CONST, c).setup_preconditioner(front="coupled")
        try:
            return hp.misfit_gradient(s, fs, rec, d_obs, rtol=1e-12)
        finally:
            s.close()

    r0 = run(c_bg)
    slope = inner(r0.grad.cpu().numpy(), dk, n)
    rem = []
    for eps in (1e-2, 1e-3, 1e-4):
        J = run(1 / np.sqrt(kap + eps * dk)).misfit
        rem.append(abs(J - r0.misfit - eps * slope))
    print("Taylor remainders", rem, "J", r0.misfit, "slope", slope)
    assert rem[0] / rem[1] >= 50 and rem[1] / rem[2] >= 50, rem
