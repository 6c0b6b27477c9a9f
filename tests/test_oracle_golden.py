"""The oracle (oracle/helmholtz_oracle.py) against outputs of the unmodified reference
(tests/golden/*.npz, made by tests/golden/make_golden.py).  CPU only."""
import glob
import os
import re

import numpy as np
import pytest
import scipy.sparse
import scipy.sparse.linalg as spla

from oracle import helmholtz_oracle as orc
from tests.golden import make_golden_large as mgl

CASES = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_*.npz")))


def _load(path):
    g = np.load(path, allow_pickle=False)
    n, b = int(g["n"]), int(g["b"])
    omega = 2 * np.pi * float(g["wave_num"]) + 1j * float(g["alpha"])
    h = 1 / (n + 1)
    return g, dict(b=b, const=float(g["const"]), eta=b * h, omega=omega, h=h, n=n)


def relerr(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b))


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_init_and_assembly(path):
    g, p = _load(path)
    c_mat, f_mat = getattr(orc, str(g["init"]))(p["omega"], p["n"])
    assert np.array_equal(c_mat, g["c_mat"])
    assert relerr(f_mat, g["f_mat"]) < 1e-15
    A = orc.build_A_matrix(c_mat=g["c_mat"], **p)
    assert A.has_sorted_indices
    assert np.array_equal(A.indptr, g["A_indptr"])            # sparsity pattern: bit exact
    assert np.array_equal(A.indices, g["A_indices"])
    assert np.max(np.abs(A.data - g["A_data"]) / np.abs(g["A_data"])) < 1e-13   # entrywise
    y = orc.stencil_matvec(g["x_rand"], c_mat=g["c_mat"], **p)
    assert relerr(y, g["A_x_rand"]) < 1e-14


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
def test_strip_operators(path):
    g, p = _load(path)
    for tag in ("first", "mid", "last"):
        m = int(g[f"Hm_{tag}_m"])
        Hm = orc.get_Hm(m, c_mat=g["c_mat"], **p).tocsr()
        Hm.sort_indices()
        ref = scipy.sparse.csr_matrix((g[f"Hm_{tag}_data"], g[f"Hm_{tag}_indices"], g[f"Hm_{tag}_indptr"]),
                                      shape=Hm.shape)
        d = (Hm - ref)
        assert abs(d).max() / abs(ref).max() < 1e-14
        # explicit zeros of the reference (c1_vec[n-1::n] = 0) carry no coupling here either
        assert Hm.count_nonzero() == ref.count_nonzero()


GM = [p for p in CASES if "M_f" in np.load(p).files]


@pytest.mark.parametrize("path", GM, ids=[os.path.basename(p)[:-4] for p in GM])
def test_preconditioner_apply(path):
    g, p = _load(path)
    P = orc.SweepingPreconditioner(c_mat=g["c_mat"], **p)
    f_vec = g["f_mat"].flatten()
    assert relerr(P.apply(f_vec), g["M_f"]) < 1e-12
    assert relerr(P.apply(g["x_rand"]), g["M_x_rand"]) < 1e-12
    m = int(g["Hm_mid_m"])
    assert relerr(P.T(m, g["x_rand"][:p["n"]]), g["T_mid_v"]) < 1e-12


@pytest.mark.parametrize("path", GM, ids=[os.path.basename(p)[:-4] for p in GM])
def test_gmres_vector_mode(path):
    """Reference operators, M applied to its argument, 25 inner iterations: well defined, so the
    iterates and the residual history must agree tightly."""
    g, p = _load(path)
    u, hist, niter, info = orc.run_solver(p["n"], p["b"], float(g["wave_num"]), p["const"], float(g["alpha"]),
                                          getattr(orc, str(g["init"])), precond_input="vector", maxiter=25)
    assert niter == len(g["gmres_vector_hist"]) and info == int(g["gmres_vector_info"])
    assert np.allclose(hist, g["gmres_vector_hist"], rtol=1e-9, atol=0)
    assert relerr(u, g["gmres_vector_u"]) < 1e-9


@pytest.mark.parametrize("path", GM, ids=[os.path.basename(p)[:-4] for p in GM])
def test_gmres_literal_mode(path):
    """code.py:510-516 literally: M ignores its argument, so the Krylov space collapses after one
    vector and GMRES exits on a (rounding-level) breakdown.  The iteration count and exit code are
    reproducible; the returned field is an amplified rounding error and is not compared."""
    g, p = _load(path)
    u, hist, niter, info = orc.run_solver(p["n"], p["b"], float(g["wave_num"]), p["const"], float(g["alpha"]),
                                          getattr(orc, str(g["init"])))
    # the collapse is detected at inner iteration 1, 2 or 3 depending on the last bits of M f
    # (the reference itself: 1 at n=20, 3 at n=45 and n=63)
    assert 1 <= len(g["gmres_literal_hist"]) <= 3 and 1 <= niter <= 3
    assert info == int(g["gmres_literal_info"])
    assert hist[-1] < 1e-12 and g["gmres_literal_hist"][-1] < 1e-12


def test_gmres_restatement_matches_scipy():
    rng = np.random.default_rng(0)
    n = 300
    A = scipy.sparse.random(n, n, density=0.02, random_state=1) + scipy.sparse.eye(n) * 4
    A = (A + 1j * scipy.sparse.random(n, n, density=0.02, random_state=2)).tocsr()
    b = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    ilu = spla.spilu(A.tocsc(), drop_tol=1e-2)
    M = spla.LinearOperator((n, n), matvec=ilu.solve, dtype=np.complex128)
    hist = []
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        x, info = spla.gmres(A, b, M=M, rtol=1e-10, callback=lambda r: hist.append(r))
    x2, info2, hist2 = orc.gmres_scipy_restated(lambda v: A @ v, ilu.solve, b, rtol=1e-10)
    assert info == info2 and len(hist) == len(hist2)
    assert np.allclose(hist, hist2, rtol=1e-6)
    assert relerr(x2, x) < 1e-10


# ---- large fixtures (tests/golden/make_golden_large.py) -------------------------------------------------------------
LARGE = sorted(p for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "large_*.npz"))
               if not re.search(r"\.\d+\.npz$", p))                 # <name>.2.npz, ...: continuation files of <name>.npz


def test_large_fixtures_present_and_consistent():
    """every production-size case has its reference part and its converged GMRES parts; stored metadata is coherent"""
    names = {os.path.basename(p) for p in LARGE}
    for stem in ("large_n63_b12_c1f1", "large_n511_b12_c1f1", "large_n1023_b12_c1f1", "large_n1024_b20_const"):
        for part in ("ref", "pb", "pc", "rb", "rc"):
            assert f"{stem}__{part}.npz" in names, f"{stem}__{part}.npz missing"
    for p in LARGE:
        g = mgl.load(p)
        n = int(g["n"])
        assert g["z"].shape == (n,) and g["z2"].shape == (n,)
        if "hist" in g:
            assert len(g["hist"]) == int(g["niter"])
            if str(g["diag"]) == "paper":
                assert int(g["info"]) == 0 and float(g["true_residual"]) <= 1e-3       # converged solves
            else:                                                                      # code.py:372-375 as written
                assert int(g["info"]) in (0, int(g["maxiter"]))
                if str(g["front"]) == "blockdiag":
                    assert int(g["info"]) == int(g["maxiter"])                         # the reference's M: never converges
        if "oracle_vs_reference" in g:
            assert np.all(g["oracle_vs_reference"] < 1e-13)                            # oracle == unmodified reference


@pytest.mark.parametrize("part", ["pb", "pc", "rb"])
def test_large_generator_reproduces_small_case(part):
    """the committed generator, run again on the small case T, reproduces the committed fixture"""
    out = mgl.compute("T", part)
    g = mgl.load(os.path.join(os.path.dirname(__file__), "golden", f"large_n63_b12_c1f1__{part}.npz"))
    assert int(out["niter"]) == int(g["niter"]) and int(out["info"]) == int(g["info"])
    assert np.allclose(out["hist"], g["hist"], rtol=1e-9, atol=0)
    assert relerr(out["u_rows"], g["u_rows"]) < 1e-9 and relerr(out["u_rowsum"], g["u_rowsum"]) < 1e-9
