"""The multi-right-hand-side path that the benchmark times, against the oracle: the 8-wide tensor-core sweep kernel
(csrc/hp_sweep4d.cu) and the multi-vector kernel (csrc/hp_sweep4m.cu) at 4096^2 and at the edges of their partition
limits, batched GMRES (gmres_batch) against the converged fixtures, and the front block on both sides of the switch from
the parallel scan to the sequential solve (csrc/hp_front.cu, n > 8192).  Runs on the B200 box: pytest -m gpu.

Every multi-vector case states the kernel it expects (HelmholtzSolver.multi_kernel: 2 = hp_sweep4d, 1 = hp_sweep4m,
0 = one vector per launch) and fails when the partition no longer selects it.
"""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import helmholtz_oracle as orc  # noqa: E402
from tests.golden.make_golden_large import load as load_fixture  # noqa: E402
from tests.test_gpu_large import GMRES_FILES, MF_FILES, U_TOL, case_fields, compact_err, dev, ids, x_rand  # noqa: E402

TOL = 1e-12
SWEEP4D, SWEEP4M, SINGLE = 2, 1, 0


@pytest.fixture(scope="module")
def hp():
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return hp


class no_dmma:
    """HP_NO_DMMA=1 for the duration (read on every call by hp_sweep4d_supported): 8 vectors go to hp_sweep4m"""

    def __enter__(self):
        os.environ["HP_NO_DMMA"] = "1"

    def __exit__(self, *exc):
        os.environ.pop("HP_NO_DMMA", None)


def relerr(a, b):
    a = a.cpu().numpy() if isinstance(a, torch.Tensor) else a
    b = b.cpu().numpy() if isinstance(b, torch.Tensor) else b
    return np.linalg.norm(a - b) / np.linalg.norm(b)


def apply_r(s, xs, R, diag):
    """M x for every x of xs, R right-hand sides per hp_precond_apply_multi call (outputs start as NaN)"""
    outs = [torch.full_like(x, complex("nan")) for x in xs]
    for i in range(0, len(xs), R):
        s.precond_apply_multi(xs[i:i + R], outs[i:i + R], diag=diag)
    return outs


# ---------------------------------------------------------------------------------------------------------------------
# A. 4096^2: M applied to 8 different combinations of f and x_rand against the oracle's M f and M x_rand
# ---------------------------------------------------------------------------------------------------------------------
# slot k holds a_k f + b_k x_rand: extreme scales, a zero vector, two mixtures, and slot 7 repeats slot 0
SLOTS = [(1, 0), (0, 1), (2.0 ** -30 * 1j, 0), (0, -2.0 ** 30), (0, 0), (1, 0.5j), (-0.25, 1 - 1j), (1, 0)]


def check_mix(outs, coefs, g, key, what):
    """out_k against a_k M f + b_k M x_rand of the fixture: its compact form (sampled rows, row and column checksums) is
    linear in the field; per component relative to |a_k| |F| + |b_k| |X|; the norm for the pure slots"""
    n = int(g["n"])
    z, z2 = dev(g["z"]), dev(g["z2"])
    rows = torch.from_numpy(np.asarray(g["sample_rows"])).cuda()
    for k, (o, (a, b)) in enumerate(zip(outs, coefs)):
        if a == 0 and b == 0:
            assert torch.count_nonzero(o).item() == 0, (what, k, "M 0 must be exactly 0")
            continue
        U = o.reshape(n, n)
        for c, v in (("rows", U[rows]), ("rowsum", U @ z), ("colsum", z2 @ U)):
            F, X = g[f"{key}_Mf_{c}"], g[f"{key}_Mx_{c}"]
            e = np.linalg.norm(v.cpu().numpy() - (a * F + b * X)) / (abs(a) * np.linalg.norm(F) + abs(b) * np.linalg.norm(X))
            assert e < TOL, (what, k, c, e)
        if a == 0 or b == 0:
            ref = abs(a) * float(g[f"{key}_Mf_norm"]) + abs(b) * float(g[f"{key}_Mx_norm"])
            e = abs(torch.linalg.norm(o).item() - ref) / ref
            assert e < TOL, (what, k, "norm", e)


def check_slots(outs, g, key, what):
    check_mix(outs, SLOTS, g, key, what)
    assert relerr(outs[7], outs[0]) < 1e-15, (what, "slot 7 repeats slot 0")


@pytest.mark.parametrize("path", MF_FILES, ids=ids(MF_FILES))
def test_multi_4096_vs_oracle(hp, path):
    """At the benchmark's 4096^2 configuration, one factorisation, both front blocks and both diagonal modes: the
    tensor-core kernel (8 per launch), the multi-vector kernel at 8 (HP_NO_DMMA), 4 and 2 per launch (the instances
    specialised for b = 12 and clusters of 4), a batch of 11 (8 + 2 + 1) and an in-place application, against the
    oracle.  The slots differ in scale by 2^60, one is zero and one repeats another, so a slot that reads or writes
    another slot's data, or a sentinel of the exchange ring that leaks into a result, shows."""
    g = load_fixture(path)
    n = int(g["n"])
    omega, c_mat, f_mat = case_fields(hp, g)
    s = hp.HelmholtzSolver(n, int(g["b"]), omega, float(g["const"]), c_mat)
    try:
        s.setup_preconditioner()
        L = s.layout()
        assert (s.b, L["K"], L["colN"]) == (12, 4, 1), L                   # the instances specialised for (12, 4)
        f, xr = dev(f_mat.ravel()), dev(x_rand(n))
        xs = [a * f + b * xr for a, b in SLOTS]
        del f, xr
        for front in ("blockdiag", "coupled"):
            s.set_front(front)
            for diag in ("reference", "paper"):
                key = f"orc_{front}_{diag}"
                assert s.multi_kernel(8) == SWEEP4D and s.batch_kernel_name(8).startswith("hp_sweep4d_kernel")
                check_slots(apply_r(s, xs, 8, diag), g, key, (front, diag, "hp_sweep4d"))
                with no_dmma():
                    assert s.multi_kernel(8) == SWEEP4M and s.batch_kernel_name(8) == "hp_sweep4m_kernel"
                    check_slots(apply_r(s, xs, 8, diag), g, key, (front, diag, "hp_sweep4m, 8 per launch"))
                for R in (4, 2):
                    assert s.multi_kernel(R) == SWEEP4M
                    check_slots(apply_r(s, xs, R, diag), g, key, (front, diag, f"hp_sweep4m, {R} per launch"))
                # 11 pairs: one launch of 8, one of 2, one single-vector application
                order = list(range(8)) + [6, 3, 5]
                pairs = [(xs[i], torch.full_like(xs[i], complex("nan"))) for i in order]
                s.precond_apply_batch(pairs, diag=diag)
                check_slots([o for _, o in pairs[:8]], g, key, (front, diag, "batch of 11: 8"))
                check_mix([o for _, o in pairs[8:]], [SLOTS[i] for i in order[8:]], g, key, (front, diag, "batch of 11: 2 + 1"))
                del pairs
                ins = [x.clone() for x in xs]                                # in place: out_i is x_i
                s.precond_apply_multi(ins, ins, diag=diag)
                check_slots(ins, g, key, (front, diag, "in place"))
                del ins
            s.check_status()
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# B. small n, directly against the oracle, at the limits of hp_sweep4d_plan / hp_sweep4m_supported
# ---------------------------------------------------------------------------------------------------------------------
# (n, b, P, K): layout (QP, CW) it must get, kernel at 8 and at 4 per launch.  The shared-memory plans of a layout
# (B200, 227 KB per block): hp_sweep4d holds one or two strips of the W ring (S) in chunks of RC rows (NCH = 1 always:
# CW <= 32), hp_sweep4m splits a strip into NCH chunks when the ring does not fit otherwise.
EDGE_CASES = {
    "b12_K4_specialised": ((120, 12, 6, 4), (21, 5), SWEEP4D, SWEEP4M),     # the (12, 4) instances; 4d S = 2
    "b12_K1_CW31": ((127, 12, 4, 1), (31, 31), SWEEP4D, SWEEP4M),           # largest CW of both kernels (CW is odd)
    "b12_K1_CW33": ((135, 12, 4, 1), (33, 33), SINGLE, SINGLE),             # past it: one vector per launch
    "b12_K2": ((100, 12, 4, 2), (25, 13), SWEEP4D, SWEEP4M),
    "b12_K8_ring1": ((250, 12, 2, 8), (125, 17), SWEEP4D, SWEEP4M),         # 4d: S = 1; 4m at 8: NCH = 2
    "b12_P33": ((200, 12, 33, 2), (7, 3), SWEEP4D, SWEEP4M),                # P - 1 = 32 separators
    "b16": ((100, 16, 4, 4), (25, 7), SWEEP4D, SWEEP4M),                    # largest b of hp_sweep4d
    "b20_K8_nch2": ((200, 20, 2, 8), (101, 13), SWEEP4M, SWEEP4M),          # b > 16: hp_sweep4m<8>, NCH = 2
    "b20_K4": ((120, 20, 4, 4), (31, 9), SWEEP4M, SWEEP4M),                 # hp_sweep4m<8>, NCH = 1
}


def edge_solver(hp, n, b, P, K, QP, CW, c_mat, omega, m_lo=0, m_hi=0):
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(P=P, K=K, m_lo=m_lo, m_hi=m_hi, layout="cluster")
    L = s.layout()
    assert (L["colN"], L["P"], L["K"], L["QP"], L["CW"]) == (1, P, K, QP, CW), L
    return s


@pytest.mark.parametrize("case", list(EDGE_CASES), ids=list(EDGE_CASES))
def test_multi_edges_vs_oracle(hp, case):
    """8 and 4 right-hand sides per launch (and 8 through hp_sweep4m where hp_sweep4d runs) against the oracle, both
    front blocks and both diagonal modes; 8 different vectors made of f and two random fields (the oracle applies M
    to the three, M is linear)"""
    (n, b, P, K), (QP, CW), k8, k4 = EDGE_CASES[case]
    omega = 2 * np.pi * (n / 10) + 2j
    h = 1 / (n + 1)
    c_mat, f_mat = orc.init_c1_f1(omega, n)
    rng = np.random.default_rng(n + 7 * b + P)
    base = [np.asarray(f_mat, dtype=np.complex128).ravel()] + [rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n)
                                                               for _ in range(2)]
    base[0] *= np.linalg.norm(base[1]) / np.linalg.norm(base[0])
    coef = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1j, 0], [0, -2, 0.5j], [-1j, 0, 3], [0.25, -1, 1], [1, 1, -1j]])
    xs_h = coef @ np.array(base)
    xs = [dev(x) for x in xs_h]
    s = edge_solver(hp, n, b, P, K, QP, CW, c_mat, omega)
    try:
        assert (s.multi_kernel(8), s.multi_kernel(4)) == (k8, k4)
        assert s.multi_max == (8 if k8 else (4 if k4 else 1))
        for front in ("blockdiag", "coupled"):
            s.set_front(front)
            Pc = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat, front=front)
            for diag in ("reference", "paper"):
                Pc.diag = diag
                refs = coef @ np.array([Pc.apply(v) for v in base])
                runs = {}
                if k8:
                    runs["8"] = apply_r(s, xs, 8, diag)
                    if k8 == SWEEP4D:
                        with no_dmma():
                            assert s.multi_kernel(8) == SWEEP4M
                            runs["8 hp_sweep4m"] = apply_r(s, xs, 8, diag)
                else:
                    with pytest.raises(hp.HelmholtzB200Error):
                        s.precond_apply_multi(xs, [torch.empty_like(x) for x in xs], diag=diag)
                if k4:
                    runs["4"] = apply_r(s, xs, 4, diag)
                pairs = [(x, torch.full_like(x, complex("nan"))) for x in xs[:7]]
                s.precond_apply_batch(pairs, diag=diag)
                runs["batch of 7"] = [o for _, o in pairs]
                for name, outs in runs.items():
                    for k, (o, r) in enumerate(zip(outs, refs)):
                        assert relerr(o, r) < TOL, (front, diag, name, k)
            s.check_status()
    finally:
        s.close()


@pytest.mark.parametrize("nstrips", [1, 2, 3, 4, 5, 7])
def test_short_multi_sweeps_vs_single(hp, nstrips):
    """Sweeps over very few strips (ring prologues and epilogues of the 8-wide kernels): forward and both backward
    variants for 8 right-hand sides per launch (hp_sweep4d and hp_sweep4m) and 4, against the single-vector sweep on the
    same strip range"""
    n, b, P, K = 200, 12, 6, 4
    omega = 2 * np.pi * (n / 10) + 2j
    c_mat = orc.init_c1_f1(omega, n)[0]
    m_lo = 60
    m_hi = m_lo + nstrips - 1
    s = edge_solver(hp, n, b, P, K, 33, 9, c_mat, omega, m_lo=m_lo, m_hi=m_hi)
    g = torch.Generator(device="cuda").manual_seed(nstrips)
    u0 = [torch.randn(n * n, dtype=torch.complex128, device="cuda", generator=g) for _ in range(8)]

    def single(diag):
        out = []
        for u in u0:
            u = u.clone()
            s.sweep_forward(u, m_lo, m_hi)
            s.sweep_backward(u, m_hi, m_lo, diag)
            out.append(u)
        return out

    def multi(R, diag):
        us = [u.clone() for u in u0]
        for i in range(0, 8, R):
            s.sweep_forward_multi_buf(us[i:i + R], 0, m_lo, m_hi)
            s.sweep_backward_multi_buf(us[i:i + R], 0, m_hi, m_lo, diag)
        return us

    try:
        assert (s.multi_kernel(8), s.multi_kernel(4)) == (SWEEP4D, SWEEP4M)
        for diag in ("reference", "paper"):
            ref = single(diag)
            runs = {"8": multi(8, diag), "4": multi(4, diag)}
            with no_dmma():
                assert s.multi_kernel(8) == SWEEP4M
                runs["8 hp_sweep4m"] = multi(8, diag)
            for name, outs in runs.items():
                for k, (o, r) in enumerate(zip(outs, ref)):
                    assert relerr(o, r) < 1e-13, (diag, name, k)
        assert s.sweep_status() == 0
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. gmres_batch against the converged fixtures
# ---------------------------------------------------------------------------------------------------------------------
# right-hand side k is C[k] f: powers of two times unit phases (exact scalings); slot ZERO is the zero vector, which
# returns before the first iteration, so the other seven run as batches of 4 + 2 + 1 from the start
C_RHS = [1, 2j, -0.5, 2.0 ** 20 * -1j, 2.0 ** -20, -8j, 0, 0.125]
ZERO = 6

_gsolver = {}


def gmres_solver(hp, g, front):
    """one factorisation per case for the module, its front block switched as needed"""
    key = (int(g["n"]), int(g["b"]), str(g["model"]))
    s = _gsolver.get(key)
    if s is None:
        for k in list(_gsolver):
            _gsolver.pop(k).close()
        omega, c_mat, _ = case_fields(hp, g)
        s = _gsolver[key] = hp.HelmholtzSolver(key[0], key[1], omega, float(g["const"]), c_mat).setup_preconditioner(front=front)
    if s.front != front:
        s.set_front(front)
    return s


@pytest.fixture(scope="module")
def gmres_solvers():
    yield
    for k in list(_gsolver):
        _gsolver.pop(k).close()


def check_gmres_batch(g, s, f, res):
    niter0, info0, hist0 = int(g["niter"]), int(g["info"]), g["hist"]
    u0, i0, h0 = res[ZERO]
    assert i0 == 0 and h0 == [] and torch.count_nonzero(u0).item() == 0
    first = None
    for k, (c, (u, info, hist)) in enumerate(zip(C_RHS, res)):
        if k == ZERO:
            continue
        # the rules of test_gpu_large.py::test_gmres_to_convergence
        assert abs(len(hist) - niter0) <= 1, (k, len(hist), niter0)
        assert (info == 0) == (info0 == 0), (k, info, info0)
        m = min(len(hist0), len(hist))
        dev_all = np.abs(np.array(hist[:m]) - hist0[:m]) / hist0[:m]
        assert np.max(dev_all[:40]) < 1e-6, (k, np.max(dev_all[:40]))
        assert np.max(dev_all) < 5e-2, (k, np.max(dev_all))
        drift = float(np.max(dev_all))
        if len(hist) == niter0:
            e, d = compact_err(u / c, g, "u")
            assert e < max(U_TOL, 10 * drift), (k, d)
        if info0 == 0:
            r = (torch.linalg.norm(c * f - s.matvec(u)) / torch.linalg.norm(c * f)).item()
            assert r <= 1e-3 and abs(r - float(g["true_residual"])) < max(1e-6, 10 * drift) * max(r, 1e-30) + 1e-9, (k, r)
        # GMRES is invariant under scaling of the right-hand side: a slot that saw another slot's data drifts off
        if first is None:
            first = np.array(hist[:40])
        else:
            h = np.array(hist[:40])
            assert len(h) == len(first) and np.max(np.abs(h - first) / first) < 1e-10, k


def run_gmres_batch(hp, g, s, vec, **kw):
    from helmholtz_preconditioner_b200.gmres import gmres_batch
    diag = str(g["diag"])
    _, _, f_mat = case_fields(hp, g)
    f = dev(f_mat.ravel())
    bs = [c * f for c in C_RHS]
    res = gmres_batch(lambda x, o: s.matvec(x, o), lambda reqs: s.precond_apply_batch(reqs, diag=diag), bs, vec=vec, rtol=1e-3,
                      restart=20, maxiter=int(g["maxiter"]), health=s.check_status, **kw)
    check_gmres_batch(g, s, f, res)


@pytest.mark.parametrize("path", GMRES_FILES, ids=ids(GMRES_FILES))
def test_gmres_batch_to_convergence(hp, gmres_solvers, path):
    """gmres_batch as bench.py runs it (one DeviceVectors, precond_apply_batch, M applied to the vector it is given) on
    seven scaled copies of the fixture's right-hand side and a zero one, each against the oracle's converged run"""
    from helmholtz_preconditioner_b200.gmres import DeviceVectors
    g = load_fixture(path)
    s = gmres_solver(hp, g, str(g["front"]))
    run_gmres_batch(hp, g, s, DeviceVectors(int(g["n"]) ** 2, s.device))


@pytest.fixture(scope="module")
def world1():
    """a gloo process group of one rank: DeviceVectors then takes its distributed Gram-Schmidt path"""
    import torch.distributed as dist
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    yield dist.group.WORLD
    dist.destroy_process_group()


N511 = [p for p in GMRES_FILES if "_n511_" in os.path.basename(p)]


@pytest.mark.parametrize("orth", ["mgs", "cgs2"])
@pytest.mark.parametrize("path", N511, ids=ids(N511))
def test_gmres_batch_distributed_orth(hp, gmres_solvers, world1, path, orth):
    """the same with the Gram-Schmidt scalars of distributed vectors (all-reduced, batched over the systems)"""
    from helmholtz_preconditioner_b200.gmres import DeviceVectors
    g = load_fixture(path)
    n = int(g["n"])
    s = gmres_solver(hp, g, str(g["front"]))
    run_gmres_batch(hp, g, s, DeviceVectors(n * n, s.device, group=world1, orth=orth), nglobal=n * n)


# ---------------------------------------------------------------------------------------------------------------------
# D. front block: parallel scan (n <= 8192) and sequential solve (n > 8192)
# ---------------------------------------------------------------------------------------------------------------------
def front_velocity(n):
    """a velocity that varies along both axes, built on the device ((n+2)^2 doubles)"""
    x = torch.linspace(0, 1, n + 2, dtype=torch.float64, device="cuda")
    return 4 / 3 * (1 - 0.5 * torch.outer(torch.exp(-32 * (x - 0.5) ** 2), torch.exp(-8 * (x - 0.3) ** 2)))


@pytest.mark.parametrize("n,b,front", [(7681, 12, "blockdiag"), (8191, 12, "blockdiag"), (8192, 12, "blockdiag"),
                                       (8192, 12, "coupled"), (8193, 12, "blockdiag"), (8193, 12, "coupled"),
                                       (8193, 20, "blockdiag"), (11585, 12, "blockdiag")])
def test_front_block_vs_oracle(hp, n, b, front):
    """hp_front_begin (T_F u_F, and grid row b+1 updated with it) and hp_front_end (u_F) against SuperLU on the oracle's
    H_F, with the couplings of grid rows b, b+1 from the oracle's stencil coefficients.  A solver set up without strips
    holds the front block only; the front block touches the first b+1 grid rows, the row after them must stay as it was."""
    import scipy.sparse.linalg as spla
    omega = 2 * np.pi * (n / 10) + 2j
    h = 1 / (n + 1)
    const = 100.0
    c_dev = front_velocity(n)
    s = hp.HelmholtzSolver(n, b, omega, const, c_dev).setup_preconditioner(m_lo=n, m_hi=n - 1, front=front)
    try:
        c_host = np.zeros((n + 2, n + 2))
        c_host[:, :b + 2] = c_dev[:, :b + 2].cpu().numpy()                    # stencil_coeffs reads c_mat[i - 1, j - 1]
        del c_dev
        rng = np.random.default_rng(n + b)
        u_h = rng.standard_normal((b + 2, n)) + 1j * rng.standard_normal((b + 2, n))
        u = dev(u_h.ravel())
        s.front_begin(u)
        tf = s.front_tf_new()
        s.front_tf_save(tf)
        got_tf, got_u = tf.cpu().numpy(), u.cpu().numpy().reshape(b + 2, n)
        lu = spla.splu(orc.get_A_FF_block(b, const, b * h, omega, h, n, c_host, coupled=(front == "coupled")).tocsc())
        c3 = orc.stencil_coeffs([b + 1], None, b, const, b * h, omega, h, n, c_host)[2][0]     # A_{b+1,b}
        c4 = orc.stencil_coeffs([b], None, b, const, b * h, omega, h, n, c_host)[3][0]         # A_{b,b+1}
        ref_tf = lu.solve(u_h[:b].ravel())
        assert relerr(got_tf, ref_tf) < TOL, "T_F u_F"
        assert relerr(got_u[b], u_h[b] - c3 * ref_tf[-n:]) < TOL, "grid row b+1"
        assert np.array_equal(got_u[:b], u_h[:b]) and np.array_equal(got_u[b + 1], u_h[b + 1])
        # front_end with a new row b+1 (what the backward sweep leaves there)
        v = rng.standard_normal(n) + 1j * rng.standard_normal(n)
        u[b * n:(b + 1) * n] = dev(v)
        s.front_end(u)
        got_u = u.cpu().numpy().reshape(b + 2, n)
        rhs = np.zeros(b * n, dtype=np.complex128)
        rhs[-n:] = c4 * v
        ref_uF = (got_tf - lu.solve(rhs)).reshape(b, n)
        assert relerr(got_u[:b], ref_uF) < TOL, "u_F"
        assert relerr(got_u[b - 1], ref_uF[b - 1]) < TOL, "grid row b"
        assert np.array_equal(got_u[b], v) and np.array_equal(got_u[b + 1], u_h[b + 1])
        s.check_status()
    finally:
        s.close()
