"""Parity at the reference's production sizes and BASELINE.json's configurations (tests/golden/large_*.npz, made by
tests/golden/make_golden_large.py from the unmodified reference and the oracle), the coupled front block, and converged
solves.  Runs on the B200 box: pytest -m gpu.

Fixture format: a field u[j, i] is stored as a few full rows, the checksum of every row with a fixed random vector z,
the checksum of every column with z2, and its norm.
"""
import glob
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import helmholtz_oracle as orc  # noqa: E402
from tests.golden.make_golden_large import load as load_fixture  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
MF_TOL = 1e-12          # north_star: preconditioned residuals within 1e-12 relative
U_TOL = 1e-8            # converged GMRES solutions (they inherit the conditioning of the Krylov recurrences)


@pytest.fixture(scope="module")
def hp():
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return hp


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(x, dtype=np.complex128))).cuda()


def case_fields(hp, g):
    n = int(g["n"])
    omega = 2 * np.pi * float(g["wave_num"]) + 1j * float(g["alpha"])
    model = str(g["model"])
    if model == "c1f1":
        c_mat, f_mat = hp.init_c1_f1(omega, n)
    elif model == "const":
        c_mat, f_mat = hp.init_const_f1(omega, n)
    else:
        c_mat, f_mat = hp.init_layered_f1(omega, n)
    return omega, c_mat, np.asarray(f_mat, dtype=np.complex128)


def x_rand(n):
    rng = np.random.default_rng(4321)          # tests/golden/make_golden_large.py::x_rand
    return rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n)


def compact_err(u_dev, g, prefix):
    """largest of the three relative errors (sampled rows, row checksums, column checksums) and the norm error"""
    n = int(g["n"])
    U = u_dev.reshape(n, n)
    z, z2 = dev(g["z"]), dev(g["z2"])
    rows = torch.from_numpy(np.asarray(g["sample_rows"])).cuda()
    got = {"rows": U[rows], "rowsum": U @ z, "colsum": z2 @ U}
    errs = {}
    for k, v in got.items():
        ref = g[f"{prefix}_{k}"]
        errs[k] = np.linalg.norm(v.cpu().numpy() - ref) / np.linalg.norm(ref)
    errs["norm"] = abs(float(torch.linalg.norm(U).item()) - float(g[f"{prefix}_norm"])) / float(g[f"{prefix}_norm"])
    return max(errs.values()), errs


REF_FILES = sorted(glob.glob(os.path.join(GOLD, "large_*__ref.npz")))
GMRES_FILES = sorted(f for f in glob.glob(os.path.join(GOLD, "large_*__*.npz")) if f[-7:-4] in ("_pb", "_pc", "_rb", "_rc"))
MF_FILES = sorted(glob.glob(os.path.join(GOLD, "large_*__mf.npz")))


def ids(files):
    return [os.path.basename(f)[6:-4] for f in files]


_solvers = {}


def solver_for(hp, g, front):
    """one factorisation per (case, front) for the whole module (the 4096^2 one holds 52 GB)"""
    key = (int(g["n"]), int(g["b"]), str(g["model"]), front)
    if key not in _solvers:
        for k in [k for k in _solvers if k[:3] != key[:3]]:       # a different problem: free the old ones first
            _solvers.pop(k).close()
        omega, c_mat, f_mat = case_fields(hp, g)
        s = hp.HelmholtzSolver(key[0], key[1], omega, float(g["const"]), c_mat)
        s.setup_preconditioner(front=front)
        _solvers[key] = s
    return _solvers[key]


@pytest.mark.parametrize("path", REF_FILES, ids=ids(REF_FILES))
def test_precond_and_operator_vs_reference(hp, path):
    """algo2_4 (code.py:356-385) and A x against the UNMODIFIED reference at n = 63, 511, 1023, 1024 (b = 20), and the
    oracle's paper-diagonal / coupled-front variants on the same inputs."""
    g = load_fixture(path)
    n = int(g["n"])
    omega, c_mat, f_mat = case_fields(hp, g)
    f, xr = dev(f_mat.ravel()), dev(x_rand(n))
    for front in ("blockdiag", "coupled"):
        s = solver_for(hp, g, front)
        if front == "blockdiag":
            e, d = compact_err(s.matvec(xr), g, "ref_Ax")
            assert e < 1e-13, ("A x", d)
            for name, v in (("ref_Mf", f), ("ref_Mx", xr)):
                e, d = compact_err(s.precond_apply(v, diag="reference"), g, name)
                assert e < MF_TOL, (name, d)
        for diag in ("reference", "paper"):
            for name, v in (("Mf", f), ("Mx", xr)):
                e, d = compact_err(s.precond_apply(v, diag=diag), g, f"orc_{front}_{diag}_{name}")
                assert e < MF_TOL, (front, diag, name, d)
        s.check_status()


@pytest.mark.parametrize("path", MF_FILES, ids=ids(MF_FILES))
def test_precond_4096_vs_oracle(hp, path):
    """M f and M x_rand at BASELINE's 4096^2 layered configuration against the oracle (SuperLU strip by strip): the error
    accumulated over the chain of 4084 strips, twice."""
    g = load_fixture(path)
    n = int(g["n"])
    omega, c_mat, f_mat = case_fields(hp, g)
    f, xr = dev(f_mat.ravel()), dev(x_rand(n))
    for front in ("blockdiag", "coupled"):
        s = solver_for(hp, g, front)
        for diag in ("reference", "paper"):
            for name, v in (("Mf", f), ("Mx", xr)):
                e, d = compact_err(s.precond_apply(v, diag=diag), g, f"orc_{front}_{diag}_{name}")
                assert e < MF_TOL, (front, diag, name, d)
        s.check_status()


@pytest.mark.parametrize("path", GMRES_FILES, ids=ids(GMRES_FILES))
def test_gmres_to_convergence(hp, path):
    """GMRES(20), rtol 1e-3, M applied to the vector it is given: iteration count +-1, exit code, history and solution
    against the oracle's run to convergence (diag = reference does not converge and is capped)."""
    g = load_fixture(path)
    n, b = int(g["n"]), int(g["b"])
    diag, front, cap = str(g["diag"]), str(g["front"]), int(g["maxiter"])
    omega, c_mat, f_mat = case_fields(hp, g)
    s = solver_for(hp, g, front)
    r = hp.run_solver(n, b, float(g["wave_num"]), float(g["const"]), float(g["alpha"]), c_mat=c_mat, f_mat=f_mat, solver=s,
                      diag=diag, precond_input="vector", rtol=1e-3, maxiter=cap, verbose=False)
    niter0, info0, hist0 = int(g["niter"]), int(g["info"]), g["hist"]
    assert abs(r.niter - niter0) <= 1, (r.niter, niter0)
    assert (r.info == 0) == (info0 == 0), (r.info, info0)
    k = min(len(hist0), r.niter)
    # Two runs whose M agree to 1e-12 stay on the same trajectory for the first restart cycles (1e-6 over 40 iterations);
    # restarted GMRES amplifies the rounding differences from cycle to cycle (1024^2, b = 20, reference front: 171
    # iterations, the histories are 7e-3 apart at the end), so the whole history gets a loose bound and the converged
    # solutions are compared at the distance of the two histories.
    hist = np.array(r.residuals[:k])
    dev_all = np.abs(hist - hist0[:k]) / hist0[:k]
    assert np.max(dev_all[:40]) < 1e-6, np.max(dev_all[:40])
    assert np.max(dev_all) < 5e-2, np.max(dev_all)
    drift = float(np.max(dev_all))
    if r.niter == niter0:
        e, d = compact_err(r.u, g, "u")
        assert e < max(U_TOL, 10 * drift), d
    if info0 == 0:
        A = s.assemble_csr()
        f = dev(f_mat.ravel())
        res = (torch.linalg.norm(f - A.matvec(r.u)) / torch.linalg.norm(f)).item()
        assert res <= 1e-3 and abs(res - float(g["true_residual"])) < max(1e-6, 10 * drift) * max(res, 1e-30) + 1e-9, (res, float(g["true_residual"]))


@pytest.mark.parametrize("n,b,model", [(20, 5, "c1f1"), (45, 12, "c2f2"), (63, 12, "c1f1"), (130, 20, "c1f2"), (300, 12, "c1f1"), (33, 24, "c2f1")])
def test_coupled_front_vs_oracle(hp, n, b, model):
    """front='coupled' (H_F = A[:bn, :bn]): M f for both diagonal modes against the oracle, partitions of 1..many leaves."""
    omega = 2 * np.pi * (n / 10) + 2j
    c_mat, f_mat = getattr(orc, "init_" + model[:2] + "_" + model[2:])(omega, n)
    h = 1 / (n + 1)
    f = np.asarray(f_mat, dtype=np.complex128).ravel()
    xr = x_rand(n)
    for leaves in (None, 1, 2, 3):
        if leaves is not None:
            os.environ["HP_FRONT_LEAVES"] = str(leaves)
        try:
            s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(front="coupled")
        finally:
            os.environ.pop("HP_FRONT_LEAVES", None)
        for diag in ("reference", "paper"):
            P = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat, diag=diag, front="coupled")
            for v in (f, xr):
                got = s.precond_apply(dev(v), diag=diag).cpu().numpy()
                ref = P.apply(v)
                assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < MF_TOL, (leaves, diag)
        s.check_status()
        s.close()


def test_front_mode_switch_restores_reference(hp):
    """a solver set up coupled and then block-diagonal again gives the reference's M f"""
    n, b = 63, 12
    omega = 2 * np.pi * 4 + 2j
    c_mat, f_mat = orc.init_c1_f1(omega, n)
    h = 1 / (n + 1)
    s = hp.HelmholtzSolver(n, b, omega, 61.0, c_mat)
    s.setup_preconditioner(front="coupled")
    s.setup_preconditioner(front="blockdiag")
    ref = orc.SweepingPreconditioner(b, 61.0, b * h, omega, h, n, c_mat).apply(f_mat.ravel())
    got = s.precond_apply(dev(f_mat.ravel())).cpu().numpy()
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < MF_TOL
    s.close()
