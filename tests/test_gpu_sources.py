"""Several sources per call: masked right-hand-side slots in the multi-vector sweep kernels (csrc/hp_sweep4d.cu,
csrc/hp_sweep4m.cu), padded batches (precond_apply_batch(pad=True)) and run_solver_many.  Runs on the B200 box:
pytest -m gpu.

A slot whose field pointer is NULL is inactive: it reads zeros and stores nothing.  Every active slot must give the bits
it gives in a full launch of the same width, whatever the other slots hold, so that a source's solution does not depend
on which sources share its wave.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import helmholtz_oracle as orc  # noqa: E402
from tests.golden.make_golden_large import load as load_fixture  # noqa: E402
from tests.test_gpu_large import MF_FILES, U_TOL, case_fields, compact_err, dev, x_rand  # noqa: E402
from tests.test_gpu_multi_oracle import check_mix, no_dmma  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SWEEP4D, SWEEP4M = 2, 1


@pytest.fixture(scope="module")
def hp():
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return hp


def rel(a, b):
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def rand_fields(k, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(n * n, dtype=torch.complex128, device="cuda", generator=g) for _ in range(k)]


class profiled:
    """sweep launches of a solver between enter and exit (hp_profile_enable / hp_profile_read)"""

    def __init__(self, s):
        self.s = s

    def __enter__(self):
        self.s.lib.hp_profile_enable(self.s.handle, 1)
        return self

    def __exit__(self, *exc):
        ms, cnt, by = C.c_double(), C.c_int(), C.c_int64()
        self.s.lib.hp_profile_read(self.s.handle, C.byref(ms), C.byref(cnt), C.byref(by))
        self.s.lib.hp_profile_enable(self.s.handle, 0)
        self.launches = cnt.value


# ---------------------------------------------------------------------------------------------------------------------
# 1. masked launches are bit-exact
# ---------------------------------------------------------------------------------------------------------------------
LAYOUTS = [(300, 12, 6, 4), (1024, 12, 0, 0), (130, 20, 6, 5), (200, 5, 7, 2)]
_kernels_seen = set()          # (kernel, width) pairs the masked-slot tests ran


def masks(W):
    if W <= 4:
        return list(range(1, 1 << W))
    return [1 << i for i in range(W)] + [0x55, 0xAA, 0x7F, 0xFE, 0xF0, 0x0F]


def sweep_calls(s):
    """forward, backward in both diagonal modes, over all strips and over b+1..b+7"""
    n, b = s.n, s.b
    short = min(b + 7, n - 1)
    out = [("fwd", b + 1, n - 1, None), ("fwd", b + 1, short, None)]
    for diag in ("reference", "paper"):
        out += [("bwd", n, b + 1, diag), ("bwd", short, b + 1, diag)]
    return out


def run_sweep(s, call, bufs):
    kind, m_from, m_to, diag = call
    if kind == "fwd":
        s.sweep_forward_multi_buf(bufs, 0, m_from, m_to)
    else:
        s.sweep_backward_multi_buf(bufs, 0, m_from, m_to, diag=diag)


def check_masks(W, xs, ys, launch, what):
    """launch(slots) -> outputs (None for empty slots).  Reference: all W slots active with xs.  Every mask: the active
    slots, once with the others empty and once with the others holding ys, give the reference's bits."""
    full = launch(list(xs))
    for mask in masks(W):
        act = [r for r in range(W) if mask >> r & 1]
        got = launch([xs[r] if r in act else None for r in range(W)])
        mixed = launch([xs[r] if r in act else ys[r] for r in range(W)])
        for r in act:
            assert torch.equal(got[r], full[r]), (what, hex(mask), r, "empty companions")
            assert torch.equal(mixed[r], full[r]), (what, hex(mask), r, "other companions")
        for r in range(W):
            if r not in act:
                assert got[r] is None
    again = launch(list(xs))                 # the exchange ring and the abort flags are left clean
    for r in range(W):
        assert torch.equal(again[r], full[r]), (what, r, "full launch after masked ones")


def masked_widths(s):
    """(width, label, env) of every launch kind this layout runs: 2, 4, 8 up to multi_max, and 8 through hp_sweep4m"""
    out = []
    for W in (2, 4, 8):
        if W <= s.multi_max:
            out.append((W, None))
    if s.multi_max == 8 and s.multi_kernel(8) == SWEEP4D:
        with no_dmma():
            if s.multi_kernel(8) == SWEEP4M:
                out.append((8, "no_dmma"))
    return out


@pytest.mark.parametrize("n,b,P,K", LAYOUTS)
def test_masked_slots_bit_exact(hp, n, b, P, K):
    omega = 2 * np.pi * (n / 10) + 2j
    c_mat = orc.init_c1_f1(omega, n)[0]
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(P=P, K=K, layout="cluster")
    try:
        assert s.multi_max >= 2, s.layout()
        for W, env in masked_widths(s):
            ctx = no_dmma() if env else _null()
            with ctx:
                kern = s.multi_kernel(W)
                assert kern in (SWEEP4D, SWEEP4M)
                _kernels_seen.add((kern, W))
                xs, ys = rand_fields(W, n, 11 * W + 1), rand_fields(W, n, 11 * W + 2)
                for call in sweep_calls(s):
                    def launch(slots, call=call):
                        bufs = [None if x is None else x.clone() for x in slots]
                        run_sweep(s, call, bufs)
                        return bufs
                    check_masks(W, xs, ys, launch, (n, W, kern, call))
                for front in ("blockdiag", "coupled"):
                    s.set_front(front)
                    for diag in ("reference", "paper"):
                        def launch(slots, diag=diag):
                            outs = [None if x is None else torch.full_like(x, complex("nan")) for x in slots]
                            s.precond_apply_slots([None if x is None else (x, o) for x, o in zip(slots, outs)], diag=diag)
                            return outs
                        check_masks(W, xs, ys, launch, (n, W, kern, front, diag))
                assert s.sweep_status() == 0
    finally:
        s.close()


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


def test_masked_kernels_covered():
    """the layouts above ran hp_sweep4d and hp_sweep4m at 2, 4 and 8 right-hand sides per launch"""
    if not _kernels_seen:
        pytest.skip("run together with test_masked_slots_bit_exact")
    assert {(SWEEP4D, 8), (SWEEP4M, 8), (SWEEP4M, 4), (SWEEP4M, 2)} <= _kernels_seen, _kernels_seen


# ---------------------------------------------------------------------------------------------------------------------
# 2. masked launches against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_masked_vs_oracle_small(hp):
    n, b = 150, 12
    omega = 2 * np.pi * 15 + 2j
    c_mat, f_mat = orc.init_c2_f2(omega, n)
    h = 1 / (n + 1)
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(layout="cluster")
    try:
        W = s.multi_max
        assert W >= 4, s.layout()
        active = {8: [0, 3, 6], 4: [0, 2, 3]}[W]
        rng = np.random.default_rng(7)
        xs = [f_mat.ravel().astype(np.complex128)] + [rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n) for _ in active[1:]]
        for front in ("blockdiag", "coupled"):
            s.set_front(front)
            for diag in ("reference", "paper"):
                P = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat, diag=diag, front=front)
                slots = [None] * W
                for r, x in zip(active, xs):
                    d = torch.from_numpy(x).cuda()
                    slots[r] = (d, torch.full_like(d, complex("nan")))
                s.precond_apply_slots(slots, diag=diag)
                for r, x in zip(active, xs):
                    ref = P.apply(x)
                    e = np.linalg.norm(slots[r][1].cpu().numpy() - ref) / np.linalg.norm(ref)
                    assert e < 1e-12, (front, diag, r, e)
        assert s.sweep_status() == 0
    finally:
        s.close()


@pytest.fixture(scope="module")
def big(hp):
    """the benchmark's 4096^2 layered configuration with its oracle fixture (one factorisation for the module)"""
    g = load_fixture(MF_FILES[0])
    omega, c_mat, f_mat = case_fields(hp, g)
    s = hp.HelmholtzSolver(int(g["n"]), int(g["b"]), omega, float(g["const"]), c_mat).setup_preconditioner()
    yield g, s, c_mat, f_mat
    s.close()


def test_masked_4096_vs_oracle(hp, big):
    """an 8-wide hp_sweep4d launch with slots 0, 3 and 7 active holding f, x_rand and f + x_rand"""
    g, s, _, f_mat = big
    n = s.n
    assert s.multi_kernel(8) == SWEEP4D
    f, xr = dev(f_mat.ravel()), dev(x_rand(n))
    ins = {0: f, 3: xr, 7: f + xr}
    coefs = [(1, 0), (0, 1), (1, 1)]
    for front in ("blockdiag", "coupled"):
        s.set_front(front)
        for diag in ("reference", "paper"):
            slots = [(ins[r], torch.full_like(f, complex("nan"))) if r in ins else None for r in range(8)]
            s.precond_apply_slots(slots, diag=diag)
            check_mix([slots[r][1] for r in (0, 3, 7)], coefs, g, f"orc_{front}_{diag}", (front, diag, "masked hp_sweep4d"))
            del slots
    assert s.sweep_status() == 0


# ---------------------------------------------------------------------------------------------------------------------
# 3. padded batches
# ---------------------------------------------------------------------------------------------------------------------
def test_padded_batch(hp):
    n, b = 1024, 12
    omega = 2 * np.pi * (n / 10) + 2j
    c_mat = hp.init_layered_f1(omega, n)[0]
    s = hp.HelmholtzSolver(n, b, omega, 100.0, c_mat).setup_preconditioner()
    try:
        assert s.multi_max == 8, s.layout()
        xs = rand_fields(11, n, 3)
        for diag in ("reference", "paper"):
            singles = [s.precond_apply(x, diag=diag) for x in xs]
            for S in (3, 5, 7, 11):
                pairs = [(x, torch.full_like(x, complex("nan"))) for x in xs[:S]]
                with profiled(s) as p:
                    s.precond_apply_batch(pairs, diag=diag, pad=True)
                assert p.launches == 2 * math.ceil(S / 8), (S, p.launches)
                for (_, o), ref in zip(pairs, singles):
                    assert rel(o, ref) < 1e-13, (diag, S)
        outs = [torch.empty_like(x) for x in xs[:8]]
        with pytest.raises(hp.HelmholtzB200Error):
            s.precond_apply_slots([None] * 8)
        with pytest.raises(hp.HelmholtzB200Error):
            s.precond_apply_slots([None])
        with pytest.raises(hp.HelmholtzB200Error):
            s.precond_apply_multi([None] + xs[1:8], outs)
        with pytest.raises(hp.HelmholtzB200Error):
            s.precond_apply_slots([(x, o) for x, o in zip(xs[:3], outs[:3])])
        with pytest.raises(hp.HelmholtzB200Error):
            s.sweep_forward_multi_buf([None] * 8, 0, b + 1, n - 1)
        assert s.sweep_status() == 0
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4.-7. run_solver_many
# ---------------------------------------------------------------------------------------------------------------------
N511 = {"coupled": os.path.join(GOLD, "large_n511_b12_c1f1__pc.npz"), "blockdiag": os.path.join(GOLD, "large_n511_b12_c1f1__pb.npz")}
# shot positions (fr1, fr2) of init_f1_mat; the first is init_c1_f1's source, the fixture's f
SHOTS = [(0.5, 0.125), (0.2, 0.3), (0.8, 0.3), (0.35, 0.6), (0.65, 0.6), (0.5, 0.85), (0.15, 0.8), (0.85, 0.8)]
OTHER_SHOTS = [(0.3, 0.45), (0.7, 0.45), None, (0.25, 0.15), (0.75, 0.15), (0.5, 0.7), (0.4, 0.9)]     # None: a zero source

_s511 = {}


def solver_511(hp, front):
    if front not in _s511:
        g = load_fixture(N511[front])
        omega, c_mat, _ = case_fields(hp, g)
        s = hp.HelmholtzSolver(int(g["n"]), int(g["b"]), omega, float(g["const"]), c_mat).setup_preconditioner(front=front)
        _s511[front] = (g, s, c_mat)
    return _s511[front]


def shots(hp, g, positions):
    n = int(g["n"])
    omega = 2 * np.pi * float(g["wave_num"]) + 1j * float(g["alpha"])
    return [np.zeros((n, n)) if p is None else hp.init_f1_mat(p[0], p[1], omega, n) for p in positions]


def problem(g):
    return int(g["n"]), int(g["b"]), float(g["wave_num"]), float(g["const"]), float(g["alpha"])


def count_rounds(s):
    """wrap s.precond_apply_slots: the widths of the launches a solve asks for"""
    widths = []
    orig = s.precond_apply_slots

    def counted(slots, diag="reference"):
        widths.append(len(slots))
        return orig(slots, diag=diag)
    s.precond_apply_slots = counted
    return widths


def compare_to_single(rs, singles, what):
    for i, (r, r0) in enumerate(zip(rs, singles)):
        assert r.info == r0.info, (what, i, r.info, r0.info)
        assert abs(r.niter - r0.niter) <= 1, (what, i, r.niter, r0.niter)
        if r.niter == r0.niter:                    # one iteration more or less ends elsewhere inside the tolerance
            assert rel(r.u, r0.u) < U_TOL, (what, i, rel(r.u, r0.u))


@pytest.mark.parametrize("front", ["coupled", "blockdiag"])
def test_run_solver_many_vs_run_solver(hp, front):
    g, s, c_mat = solver_511(hp, front)
    args = problem(g)
    assert s.multi_max == 8, s.layout()
    fs = shots(hp, g, SHOTS)
    kw = dict(c_mat=c_mat, solver=s, diag="paper", precond_input="vector", rtol=1e-3, maxiter=int(g["maxiter"]), verbose=False)
    singles = [hp.run_solver(*args, f_mat=f, **kw) for f in fs]
    widths = count_rounds(s)
    try:
        with profiled(s) as p:
            rs = hp.run_solver_many(*args, np.stack(fs), **kw)
    finally:
        del s.precond_apply_slots
    assert len(rs) == len(fs)
    assert widths and set(widths) == {8}, widths
    assert p.launches == 2 * len(widths), (p.launches, len(widths))
    compare_to_single(rs, singles, front)
    # the fixture's source against the oracle's converged solve (tests/test_gpu_large.py::test_gmres_to_convergence)
    r = rs[0]
    niter0, info0, hist0 = int(g["niter"]), int(g["info"]), g["hist"]
    assert abs(r.niter - niter0) <= 1 and (r.info == 0) == (info0 == 0), (r.niter, niter0, r.info, info0)
    k = min(len(hist0), r.niter)
    drift = float(np.max(np.abs(np.array(r.residuals[:k]) - hist0[:k]) / hist0[:k]))
    assert drift < 5e-2, drift
    if r.niter == niter0:
        e, d = compact_err(r.u, g, "u")
        assert e < max(U_TOL, 10 * drift), d
    if front == "blockdiag":
        assert len({r.niter for r in rs}) >= 2, [r.niter for r in rs]      # the ragged path ran
    for r in rs:
        assert r.init_time >= 0 and r.solve_time > 0 and r.solve_time == rs[0].solve_time


def test_run_solver_many_independent_of_companions(hp):
    g, s, c_mat = solver_511(hp, "blockdiag")
    args = problem(g)
    fs, others = shots(hp, g, SHOTS), shots(hp, g, OTHER_SHOTS)
    kw = dict(c_mat=c_mat, solver=s, diag="paper", precond_input="vector", rtol=1e-3, maxiter=int(g["maxiter"]), verbose=False)
    a = hp.run_solver_many(*args, [fs[0]] + fs[1:], **kw)
    b = hp.run_solver_many(*args, [fs[0]] + others, **kw)
    c = hp.run_solver_many(*args, fs[1:] + [others[0], fs[0]], **kw)          # ninth: second wave, slot 0
    assert len(c) == 9
    for r in (b[0], c[8]):
        assert torch.equal(r.u, a[0].u)
        assert r.residuals == a[0].residuals and r.niter == a[0].niter and r.info == a[0].info
    z = b[1 + OTHER_SHOTS.index(None)]
    assert z.niter == 0 and z.info == 0 and torch.count_nonzero(z.u).item() == 0
    for i in range(1, 8):                                                     # the same sources in other slots
        assert a[i].info == c[i - 1].info and abs(a[i].niter - c[i - 1].niter) <= 1
    assert s.sweep_status() == 0


def test_run_solver_many_rhs_input(hp):
    """precond_input='rhs' (the reference as written): M f of a wave in one masked launch, copied on every request"""
    g, s, c_mat = solver_511(hp, "blockdiag")
    args = problem(g)
    fs = shots(hp, g, SHOTS[:5])
    kw = dict(c_mat=c_mat, solver=s, diag="reference", precond_input="rhs", maxiter=2, verbose=False)
    singles = [hp.run_solver(*args, f_mat=f, **kw) for f in fs]
    widths = count_rounds(s)
    try:
        rs = hp.run_solver_many(*args, torch.from_numpy(np.stack(fs)).reshape(len(fs), -1), **kw)
    finally:
        del s.precond_apply_slots
    assert widths == [8], widths
    # With M x = M f for every x the Krylov space has one direction: the second Arnoldi vector is M f minus its own
    # projection, i.e. rounding, and the history entries (already relative to ||f||) sit at 1e-15.  Their leading digits
    # come from the rounding of M f, which the 8-wide tensor-core sweep and the single-vector sweep do differently, and
    # whether Arnoldi stops with h1 <= eps h0 after one column or two is decided at that level too.  So the histories are
    # compared in units of ||f||, over the iterations both runs made.
    for i, (r, r0) in enumerate(zip(rs, singles)):
        assert r.info == r0.info and abs(r.niter - r0.niter) <= 1, (i, r.info, r0.info, r.niter, r0.niter)
        k = min(r.niter, r0.niter)
        h, h0 = np.array(r.residuals[:k]), np.array(r0.residuals[:k])
        assert k >= 1 and np.all(np.abs(h - h0) <= 1e-12 * np.maximum(np.abs(h0), 1.0)), (i, h, h0)


def test_run_solver_many_4096(hp, big):
    """the benchmark's configuration, paper diagonal with the coupled front, eight shot positions"""
    g, s, c_mat, _ = big
    s.set_front("coupled")
    args = problem(g)
    fs = shots(hp, g, SHOTS)
    kw = dict(c_mat=c_mat, solver=s, diag="paper", precond_input="vector", rtol=1e-3, verbose=False)
    singles = []
    for f in fs:
        r0 = hp.run_solver(*args, f_mat=f, **kw)
        singles.append(r0)
    rs = hp.run_solver_many(*args, fs, **kw)
    for r in rs:
        assert r.info == 0
    compare_to_single(rs, singles, "4096")
    assert s.sweep_status() == 0


def teardown_module():
    for _, s, _ in _s511.values():
        s.close()
    _s511.clear()
