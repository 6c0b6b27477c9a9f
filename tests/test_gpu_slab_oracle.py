"""The slab-decomposed path (helmholtz_preconditioner_b200/slab.py) against the oracle, on one GPU.

A. W solvers, one per rank, each holding its own strips only, driven through the staged schedule of
   SlabSolver.precond_apply / precond_apply_batch by hand (the hand-overs are torch copies).  Every slab buffer sits
   inside G guard rows on each side; the guards, the ghost row j0-1 of every rank and the ghost row n of the last rank
   hold a NaN sentinel that no kernel may read (the result would be NaN) or write (the bits would change).  The staged
   kernels get a base pointer outside the slab buffer (HelmholtzSolver._base), so a kernel that touches a row it must
   not shows here, inside memory the test owns.
B. hp_stencil_matvec_rows with halo rows from separate tensors and the slab inside a NaN guard.
C. the peer hand-over kernels of csrc/hp_peer.cu in one process.
D. solver contexts swept concurrently on three streams, parked front solutions, and the refusal to refactor a solver
   whose contexts are open.
E. the production SlabSolver with a HelmholtzSolver backend over gloo, two and three processes sharing GPU 0.
Runs on the B200 box: pytest -m gpu.
"""
import ctypes as C
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

pytestmark = pytest.mark.gpu

from oracle import helmholtz_oracle as orc  # noqa: E402
from tests.golden.make_golden_large import load as load_fixture  # noqa: E402
from tests.test_gpu_large import MF_FILES, case_fields, dev, ids, x_rand  # noqa: E402
from tests.test_gpu_multi_oracle import SLOTS, SWEEP4D, SWEEP4M, check_slots, no_dmma, relerr  # noqa: E402

TOL = 1e-12             # M x
SPMV_TOL = 1e-13        # A x
G = 3                   # guard rows on each side of a slab buffer
SENT = 0x7FF40000DEADBEEF   # a signalling NaN with a payload: any arithmetic on it gives another bit pattern

# eight right-hand sides made of three base fields (the oracle applies M to the three; M is linear): single fields,
# mixtures, extreme scales and a zero slot
COEF = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [1, 1j, 0], [0, -2.0 ** 30, 0], [0, 0, 0], [2.0 ** -30 * 1j, 0, 0],
                 [0.25, -1, 1]])
ORDER11 = list(range(8)) + [6, 3, 5]                 # a batch of 11: one launch of 8, one of 2, one single application


@pytest.fixture(scope="module")
def hp():
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return hp


def sentinel_fill(t):
    t.view(torch.int64).fill_(SENT)
    return t


def intact(t):
    return bool((t.view(torch.int64) == SENT).all())


def guarded(rows, n):
    """(allocation, view): `rows` rows of n complex numbers with G sentinel rows on each side"""
    full = sentinel_fill(torch.empty((rows + 2 * G) * n, dtype=torch.complex128, device="cuda"))
    return full, full[G * n:(G + rows) * n]


# ---------------------------------------------------------------------------------------------------------------------
# A. in-process slab emulation
# ---------------------------------------------------------------------------------------------------------------------
class SlabRank:
    """One rank of a slab decomposition: a solver holding the strips m = max(b+1, j0+1) .. min(n, j1) (as
    distributed_gmres_setup sets it up) and guarded buffers of rows j0-1 .. j1 (as SlabSolver.buf)."""

    def __init__(self, hp, n, b, omega, const, c_mat, R, r, P=0, K=0, layout="auto"):
        self.n, self.b, self.r, self.W = n, b, r, len(R) - 1
        self.j0, self.j1 = R[r], R[r + 1]
        self.rows = self.j1 - self.j0
        self.m_lo, self.m_hi = max(b + 1, self.j0 + 1), min(n, self.j1)
        self.s = hp.HelmholtzSolver(n, b, omega, const, c_mat).setup_preconditioner(P, K, self.m_lo, self.m_hi, layout=layout)
        self.full, self.bufs, self.tfs = [], [], []

    def reserve(self, k):
        while len(self.bufs) < k:
            full, buf = guarded(self.rows + 2, self.n)
            self.full.append(full)
            self.bufs.append(buf)
        while self.r == 0 and len(self.tfs) < k:
            self.tfs.append(self.s.front_tf_new())

    def row(self, j, i):
        """global row j (j0-1 <= j <= j1) of buffer i"""
        o = (j - self.j0 + 1) * self.n
        return self.bufs[i][o:o + self.n]

    def own(self, i):
        return self.bufs[i][self.n:(self.rows + 1) * self.n]

    def sentinels(self, i):
        n = self.n
        regs = [("guard below", self.full[i][:G * n]), ("guard above", self.full[i][(G + self.rows + 2) * n:]),
                (f"ghost row {self.j0 - 1}", self.bufs[i][:n])]
        if self.r == self.W - 1:
            regs.append((f"ghost row {self.j1}", self.bufs[i][(self.rows + 1) * n:]))
        return regs

    def close(self):
        self.s.close()


def make_ranks(hp, n, b, omega, const, c_mat, R, **kw):
    return [SlabRank(hp, n, b, omega, const, c_mat, R, r, **kw) for r in range(len(R) - 1)]


def batch_groups(s, R):
    """the groups of right-hand sides per launch of precond_apply_batch"""
    groups, i = [], 0
    while i < R:
        g = s.batch_group(R - i)
        groups.append(list(range(i, i + g)))
        i += g
    return groups


def slab_apply(ranks, xs, diag, groups=None, trace=None):
    """M x for every global field x of xs through the staged calls of every rank, in the order of
    SlabSolver.precond_apply (one right-hand side) and precond_apply_batch (several, T_F u_F parked per right-hand side).
    groups: lists of indices of xs swept by one launch (default: as precond_apply_batch splits them).  trace, if a dict,
    receives the global fields after the forward chain and after the backward chain, rank by rank."""
    n, W, R = ranks[0].n, len(ranks), len(xs)
    if groups is None:
        groups = batch_groups(ranks[0].s, R)
    for rk in ranks:
        rk.reserve(R)
        for i, x in enumerate(xs):
            sentinel_fill(rk.full[i])
            rk.own(i).copy_(x[rk.j0 * n:rk.j1 * n])
            if rk.r < W - 1:                                  # initial values of the first row of the next slab
                rk.row(rk.j1, i).copy_(x[rk.j1 * n:(rk.j1 + 1) * n])

    def sweep(rk, forward):
        s, row0 = rk.s, rk.j0 - 1
        lo, hi = (rk.m_lo, min(rk.m_hi, n - 1)) if forward else (rk.m_hi, rk.m_lo)
        if (lo > hi) if forward else (hi > lo):
            return
        for grp in groups:
            bufs = [rk.bufs[i] for i in grp]
            if forward:
                if len(grp) > 1:
                    s.sweep_forward_multi_buf(bufs, row0, lo, hi)
                else:
                    s.sweep_forward_buf(bufs[0], row0, lo, hi)
            else:
                if len(grp) > 1:
                    s.sweep_backward_multi_buf(bufs, row0, lo, hi, diag)
                else:
                    s.sweep_backward_buf(bufs[0], row0, lo, hi, diag)

    def snapshot(key):
        if trace is not None:
            trace[key] = [[rk.bufs[i][n:(rk.rows + 2 if rk.r < W - 1 else rk.rows + 1) * n].clone() for i in range(R)]
                          for rk in ranks]

    for rk in ranks:                                         # forward chain
        if rk.r == 0:
            for i in range(R):
                rk.s.front_begin_buf(rk.bufs[i], rk.j0 - 1)
                if R > 1:
                    rk.s.front_tf_save(rk.tfs[i])
        else:
            for i in range(R):
                rk.row(rk.j0, i).copy_(ranks[rk.r - 1].row(rk.j0, i))
        sweep(rk, True)
    snapshot("forward")
    for rk in reversed(ranks):                               # backward chain
        if rk.r < W - 1:
            for i in range(R):
                rk.row(rk.j1, i).copy_(ranks[rk.r + 1].row(rk.j1, i))
        sweep(rk, False)
    snapshot("backward")
    rk = ranks[0]
    for i in range(R):
        if R > 1:
            rk.s.front_tf_load(rk.tfs[i])
        rk.s.front_end_buf(rk.bufs[i], rk.j0 - 1)
    outs = [torch.cat([rk.own(i) for rk in ranks]) for i in range(R)]
    for rk in ranks:
        for i in range(R):
            for name, reg in rk.sentinels(i):
                assert intact(reg), (f"rank {rk.r} [{rk.j0}, {rk.j1})", f"right-hand side {i}", name, "was read or written")
    return outs


def oracle_stages(Pc, x):
    """the oracle's field after the forward chain, after the backward chain (rows below b untouched until the front
    solve) and at the end (SweepingPreconditioner.apply, step by step)"""
    b, n = Pc.b, Pc.n
    u = np.array(x, dtype=np.complex128).reshape(n, n).copy()
    TF = Pc.lu_HF.solve(u[:b].ravel())
    u[b] = u[b] - Pc.lo[b] * TF[-n:]
    for m in range(b + 1, n):
        u[m] = u[m] - Pc.lo[m] * Pc.T(m, u[m - 1])
    fwd = u.copy()
    for m in range(b + 1, n + 1):
        t = Pc.T(m, u[m - 1])
        u[m - 1] = (u[m - 1] - t) if Pc.diag == "reference" else t
    for m in range(n - 1, b, -1):
        u[m - 1] = u[m - 1] - Pc.T(m, Pc.up[m - 1] * u[m])
    bwd = u.copy()
    return fwd, bwd, Pc.apply(x).reshape(n, n)


def problem(n):
    omega = 2 * np.pi * (n / 10) + 2j
    c_mat, f_mat = orc.init_c1_f1(omega, n)
    return omega, c_mat, np.asarray(f_mat, dtype=np.complex128).ravel()


def base_fields(n, f):
    rng = np.random.default_rng(n + 11)
    r1, r2 = (rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n) for _ in range(2))
    return [f * (np.linalg.norm(r1) / np.linalg.norm(f)), r1, r2]


def check(outs, refs, what):
    for k, (o, r) in enumerate(zip(outs, refs)):
        o = o.cpu().numpy()
        if not np.any(r):
            assert np.all(o == 0), (what, k, "M 0 must be exactly 0")
            continue
        assert np.all(np.isfinite(o)), (what, k, "non-finite result")
        e = relerr(o, r)
        assert e < TOL, (what, k, e)


def run_slab_case(hp, n, b, R, P=0, K=0, layout="auto", kernels=None, variants=(0,), const=60.0):
    """M x of the slab decomposition R against the oracle: both front blocks, both diagonal modes; single right-hand
    sides (random, source, 2^30 and 2^-30 scales, zero), R = 8, 4, 2 per launch and a batch of 11 when the layout carries
    several per launch (kernels = expected (multi_kernel(8), multi_kernel(4), multi_kernel(2)))"""
    omega, c_mat, f = problem(n)
    h = 1 / (n + 1)
    base = base_fields(n, f)
    ranks = make_ranks(hp, n, b, omega, const, c_mat, R, P=P, K=K, layout=layout)
    try:
        strips = [m for rk in ranks for m in range(rk.m_lo, rk.m_hi + 1)]
        assert strips == list(range(b + 1, n + 1)), "every strip has exactly one owner"
        if kernels is not None:
            for rk in ranks:
                assert tuple(rk.s.multi_kernel(k) for k in (8, 4, 2)) == kernels, (rk.r, rk.s.layout())
        xs8 = [dev(v) for v in COEF @ np.array(base)]
        singles = [(1, 1), (1, 0), (2.0 ** 30, 1), (2.0 ** -30, 0), (0, 1)]        # (scale, base index)
        xs1 = [dev(a * base[k]) for a, k in singles]
        for front in ("blockdiag", "coupled"):
            ranks[0].s.set_front(front)
            Pc = orc.SweepingPreconditioner(b, const, b * h, omega, h, n, c_mat, front=front)
            for diag in ("reference", "paper"):
                Pc.diag = diag
                mb = [Pc.apply(v) for v in base]
                refs1 = [a * mb[k] for a, k in singles]
                refs8 = COEF @ np.array(mb)
                for v in variants:
                    for rk in ranks:
                        rk.s.set_sweep_variant(v)
                    tag = (front, diag, f"variant {v}")
                    for k, x in enumerate(xs1):
                        check(slab_apply(ranks, [x], diag), [refs1[k]], tag + (f"single {singles[k]}",))
                    check(slab_apply(ranks, [xs8[i] for i in ORDER11], diag), [refs8[i] for i in ORDER11], tag + ("batch of 11",))
                if kernels is not None:
                    for per in (8, 4, 2):
                        grp = [list(range(i, i + per)) for i in range(0, 8, per)]
                        check(slab_apply(ranks, xs8, diag, grp), refs8, (front, diag, f"{per} per launch"))
                    if kernels[0] == SWEEP4D:
                        with no_dmma():
                            assert ranks[0].s.multi_kernel(8) == SWEEP4M
                            check(slab_apply(ranks, xs8, diag, [list(range(8))]), refs8, (front, diag, "8 per launch, hp_sweep4m"))
        for rk in ranks:
            assert rk.s.sweep_status() == 0, rk.r
    finally:
        for rk in ranks:
            rk.close()


def bounds(n, b, W, **kw):
    from helmholtz_preconditioner_b200.slab import slab_bounds
    return slab_bounds(n, b, W, **kw)


# (n, b, R or W, P, K, layout, expected kernels at 8/4/2 per launch, sweep variants)
SLAB_CASES = {
    "n120_b12_K4_W2": (120, 12, 2, 6, 4, "cluster", (SWEEP4D, SWEEP4M, SWEEP4M), (0,)),       # the (12, 4) instances
    "n120_b12_K4_W3": (120, 12, 3, 6, 4, "cluster", (SWEEP4D, SWEEP4M, SWEEP4M), (0,)),
    "n200_b20_K8_W2": (200, 20, 2, 2, 8, "cluster", (SWEEP4M, SWEEP4M, SWEEP4M), (0,)),      # hp_sweep4m<8>, NCH = 2
    "n40_b5_classic_W3": (40, 5, 3, 0, 0, "classic", None, (1, 2, 3)),
    "n120_thin": (120, 12, [0, 13, 14, 60, 120], 6, 4, "cluster", (SWEEP4D, SWEEP4M, SWEEP4M), (0,)),   # 1 strip, 1 row
    "n120_front_equiv": (120, 12, ("fe", 3, 20), 6, 4, "cluster", (SWEEP4D, SWEEP4M, SWEEP4M), (4,)),
}


@pytest.mark.parametrize("case", list(SLAB_CASES), ids=list(SLAB_CASES))
def test_slab_precond_vs_oracle(hp, case):
    n, b, R, P, K, layout, kernels, variants = SLAB_CASES[case]
    if isinstance(R, int):
        R = bounds(n, b, R)
    elif isinstance(R, tuple):
        R = bounds(n, b, R[1], front_equiv=R[2])
        assert R[1] < n // 3, R                                      # rank 0 gets fewer rows than its share
    run_slab_case(hp, n, b, R, P, K, layout, kernels, variants)


def test_slab_stages_vs_oracle(hp):
    """the rows of every rank after the forward chain and after the backward chain against the oracle's sweep, for one
    and for eight right-hand sides per launch: a failure names the rank and the stage"""
    n, b = 120, 12
    omega, c_mat, f = problem(n)
    h = 1 / (n + 1)
    base = base_fields(n, f)
    R = bounds(n, b, 3)
    ranks = make_ranks(hp, n, b, omega, 60.0, c_mat, R, P=6, K=4, layout="cluster")
    try:
        Pc = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat)
        for diag in ("reference", "paper"):
            Pc.diag = diag
            st = [oracle_stages(Pc, v) for v in base]
            for xs, idx in (([dev(base[1])], [1]), ([dev(v) for v in base] * 2 + [dev(base[0]), dev(base[1])], [0, 1, 2] * 2 + [0, 1])):
                trace = {}
                outs = slab_apply(ranks, xs, diag, [list(range(len(xs)))], trace=trace)
                for stage, si in (("forward", 0), ("backward", 1)):
                    for rk, per in zip(ranks, trace[stage]):
                        hi = rk.j1 + 1 if rk.r < len(ranks) - 1 else rk.j1           # with the ghost row above
                        for i, got in zip(idx, per):
                            ref = st[i][si][rk.j0:hi].ravel()
                            e = relerr(got.cpu().numpy(), ref)
                            assert e < TOL, (diag, stage, f"rank {rk.r} rows [{rk.j0}, {hi})", len(xs), e)
                check(outs, [st[i][2].ravel() for i in idx], (diag, "final", len(xs)))
    finally:
        for rk in ranks:
            rk.close()


@pytest.mark.parametrize("W", [2, 4, 8])
@pytest.mark.parametrize("path", MF_FILES, ids=ids(MF_FILES))
def test_slab_4096_vs_oracle(hp, path, W):
    """what bench.py --gpus W computes per rank: the 4096^2 layered configuration cut into W slabs, the 8 slots of
    test_gpu_multi_oracle.py in one launch of the tensor-core kernel per rank and direction, both front blocks, both
    diagonal modes, against the oracle fixture"""
    g = load_fixture(path)
    n, b = int(g["n"]), int(g["b"])
    omega, c_mat, f_mat = case_fields(hp, g)
    R = bounds(n, b, W)
    ranks = make_ranks(hp, n, b, omega, float(g["const"]), c_mat, R)
    try:
        for rk in ranks:
            L = rk.s.layout()
            assert (L["K"], L["colN"]) == (4, 1) and rk.s.multi_kernel(8) == SWEEP4D, (rk.r, L)
        f, xr = dev(f_mat.ravel()), dev(x_rand(n))
        xs = [a * f + c * xr for a, c in SLOTS]
        del f, xr
        for front in ("blockdiag", "coupled"):
            ranks[0].s.set_front(front)
            for diag in ("reference", "paper"):
                outs = slab_apply(ranks, xs, diag, [list(range(8))])
                check_slots(outs, g, f"orc_{front}_{diag}", (front, diag, f"W = {W}"))
                del outs
        for rk in ranks:
            assert rk.s.sweep_status() == 0, rk.r
    finally:
        for rk in ranks:
            rk.close()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# B. hp_stencil_matvec_rows with halo rows
# ---------------------------------------------------------------------------------------------------------------------
def stencil_rows(p, x, j0, j1):
    """rows j0 <= j < j1 of A x from the oracle's stencil coefficients; x holds rows j0-1 .. j1 (None outside the grid)"""
    n = p["n"]
    c1, c2, c3, c4, c5 = orc.stencil_coeffs(np.arange(j0 + 1, j1 + 1), None, **p)
    south, u, north = x
    y = c5 * u
    y[:, 1:] += c1[:, 1:] * u[:, :-1]
    y[:, :-1] += c2[:, :-1] * u[:, 1:]
    y[1:] += c3[1:] * u[:-1]
    y[:-1] += c4[:-1] * u[1:]
    if south is not None:
        y[0] += c3[0] * south
    if north is not None:
        y[-1] += c4[-1] * north
    return y.ravel()


@pytest.mark.parametrize("n", [127, 128, 129, 300, 4096])
def test_matvec_rows_halos_vs_oracle(hp, n):
    """A x on slabs of 1, 2, 15, 16, 17 and 33 rows (around the 16-row minimum march of hp_spmv_rows; at 4096 also 2000
    rows, a march longer than 16 with the L2 prefetch near the slab's end) at the bottom, inside and at the top of the
    grid.  The slab sits inside NaN guard rows: rows j0-1 and j1 must come from the halo tensors, NULL on the boundary;
    the output's guard must stay untouched."""
    b = 12
    omega = 2 * np.pi * (min(n, 300) / 10) + 2j
    h = 1 / (n + 1)
    c_mat = orc.init_c1_mat(.5, .5, n)
    p = dict(b=b, const=60.0, eta=b * h, omega=omega, h=h, n=n, c_mat=c_mat)
    rng = np.random.default_rng(n)
    heights = [1, 2, 15, 16, 17, 33] + ([2000] if n == 4096 else [])
    full_x = full_y = None
    if n <= 300:
        full_x = (rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)))
        full_y = orc.stencil_matvec(full_x.ravel(), **p).reshape(n, n)
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat)
    try:
        for hgt in heights:
            for j0 in sorted({0, n // 2 - hgt // 2, n - hgt}):
                j1 = j0 + hgt
                if full_x is not None:
                    rows = full_x[max(j0 - 1, 0):j1 + 1]
                else:
                    shape = (min(j1 + 1, n) - max(j0 - 1, 0), n)
                    rows = rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
                south = rows[0] if j0 > 0 else None
                north = rows[-1] if j1 < n else None
                own = rows[(1 if j0 > 0 else 0):(1 if j0 > 0 else 0) + hgt]
                ref = full_y[j0:j1].ravel() if full_y is not None else stencil_rows(p, (south, own.copy(), north), j0, j1)
                if full_y is not None and hgt == 17:
                    assert relerr(stencil_rows(p, (south, own.copy(), north), j0, j1), ref) < 1e-15
                xfull, xs = guarded(hgt, n)
                xs.copy_(dev(own.ravel()))
                yfull, ys = guarded(hgt, n)
                halo_s = dev(south) if south is not None else None
                halo_n = dev(north) if north is not None else None
                s.matvec_rows(j0, j1, xs, halo_s, halo_n, ys)
                got = ys.cpu().numpy()
                what = (n, f"rows [{j0}, {j1})")
                assert np.all(np.isfinite(got)), what + ("a row next to the slab was read instead of a halo",)
                assert relerr(got, ref) < SPMV_TOL, what + (relerr(got, ref),)
                assert intact(yfull[:G * n]) and intact(yfull[(G + hgt) * n:]), what + ("the output's guard was written",)
                assert intact(xfull[:G * n]) and intact(xfull[(G + hgt) * n:]), what + ("the input's guard was written",)
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# C. peer hand-over kernels (csrc/hp_peer.cu) in one process: the local mailbox stands in for the peer's mapping
# ---------------------------------------------------------------------------------------------------------------------
RMAX = 8
FILL = 0xA5


class _DeviceBytes:
    """a torch view of device memory that the library allocated"""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 3,
                                         "strides": None}


class Mailbox:
    """[256 bytes of flags | forward staging [RMAX][n] | backward staging [RMAX][n]] as slab.PeerMailbox lays it out"""

    def __init__(self, n):
        from helmholtz_preconditioner_b200 import _lib
        self.lib, self.check, self.n = _lib.require_device(), _lib.check, n
        self.nbytes = 256 + 2 * RMAX * n * 16
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        self.check(self.lib.hp_mailbox_create(self.nbytes, C.byref(ptr), handle), "hp_mailbox_create")
        self.ptr = ptr.value
        self.mem = torch.as_tensor(_DeviceBytes(self.ptr, self.nbytes), device="cuda")
        assert self.mem.data_ptr() == self.ptr
        self.flags = self.mem[:256].view(torch.int32)
        self.stage = self.mem[256:]

    def staging(self, which):
        return self.ptr + 256 + which * RMAX * self.n * 16

    def stage_bytes(self, which, R):
        o = which * RMAX * self.n * 16
        return o, o + R * self.n * 16

    def handover(self, which, rows, seq, stream):
        arr = (C.c_void_p * len(rows))(*[t.data_ptr() for t in rows])
        self.check(self.lib.hp_handover_rows(len(rows), arr, self.staging(which), self.n, self.ptr + 4 * which, seq, stream),
                   "hp_handover_rows")

    def wait(self, which, seq, stream):
        self.check(self.lib.hp_stream_wait_geq(self.ptr + 4 * which, seq, stream), "hp_stream_wait_geq")

    def collect(self, which, rows, stream):
        arr = (C.c_void_p * len(rows))(*[t.data_ptr() for t in rows])
        self.check(self.lib.hp_collect_rows(len(rows), self.staging(which), arr, self.n, stream), "hp_collect_rows")

    def close(self):
        torch.cuda.synchronize()
        del self.mem, self.flags, self.stage
        self.lib.hp_mailbox_free(self.ptr)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def rand_rows(R, n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.randn(n, dtype=torch.complex128, device="cuda", generator=g) for _ in range(R)]


@pytest.mark.parametrize("n", [1, 5, 1023, 1024, 1025, 4096])
def test_handover_collect_rows(hp, n):
    """R = 1..8 rows through hp_handover_rows -> hp_stream_wait_geq -> hp_collect_rows, alternately through the forward
    and the backward staging area: rows arrive bit for bit, the flag holds the sequence number, the other flags, the
    staging bytes beyond R n and the guard rows around every destination row are unchanged"""
    mb = Mailbox(n)
    try:
        flags = np.zeros(64, dtype=np.int32)
        for R in range(1, RMAX + 1):
            which, seq = R % 2, 100 + R
            mb.stage.fill_(FILL)
            src = rand_rows(R, n, 1000 * n + R)
            dst = [guarded(1, n) for _ in range(R)]
            torch.cuda.synchronize()
            mb.handover(which, src, seq, _stream())
            mb.wait(which, seq, _stream())
            mb.collect(which, [d for _, d in dst], _stream())
            torch.cuda.synchronize()
            flags[which] = seq
            assert np.array_equal(mb.flags.cpu().numpy(), flags), (R, "flags")
            lo, hi = mb.stage_bytes(which, R)
            want = torch.cat([t.view(torch.uint8) for t in src])
            assert torch.equal(mb.stage[lo:hi], want), (R, "staging")
            assert bool((mb.stage[:lo] == FILL).all()) and bool((mb.stage[hi:] == FILL).all()), (R, "staging beyond R n")
            for r, ((full, d), t) in enumerate(zip(dst, src)):
                assert torch.equal(d.view(torch.int64), t.view(torch.int64)), (R, r, "row")
                assert intact(full[:G * n]) and intact(full[(G + 1) * n:]), (R, r, "guard of the destination row")
    finally:
        mb.close()


def test_signal_flags(hp):
    """hp_signal_flags sets exactly the `count` flags it is given"""
    from helmholtz_preconditioner_b200 import _lib
    lib = _lib.require_device()
    flags = torch.empty(64, dtype=torch.int32, device="cuda")
    for count in range(1, 9):
        flags.fill_(-7)
        arr = (C.c_void_p * count)(*[flags.data_ptr() + 4 * (3 * i + 1) for i in range(count)])
        _lib.check(lib.hp_signal_flags(count, arr, 500 + count, _stream()), "hp_signal_flags")
        want = torch.full_like(flags, -7)
        want[[3 * i + 1 for i in range(count)]] = 500 + count
        assert torch.equal(flags, want), count


def test_wait_holds_collect_until_handover(hp):
    """the hand-over is enqueued first, on stream B behind a long sleep; stream A waits for its sequence number and then
    collects.  The staging area holds a sentinel until the hand-over, so a collect that did not wait returns it."""
    n, R = 4096, RMAX
    mb = Mailbox(n)
    try:
        warm = rand_rows(R, n, 1)                            # every kernel of the exchange has run once (lazy loading)
        mb.handover(0, warm, 1, _stream())
        mb.wait(0, 1, _stream())
        mb.collect(0, [torch.empty_like(t) for t in warm], _stream())
        mb.stage.fill_(FILL)
        src = rand_rows(R, n, 2)
        dst = [sentinel_fill(torch.empty_like(t)) for t in src]
        a, b = torch.cuda.Stream(), torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(b):
            torch.cuda._sleep(200_000_000)
            mb.handover(0, src, 2, b.cuda_stream)
        with torch.cuda.stream(a):
            mb.wait(0, 2, a.cuda_stream)
            mb.collect(0, dst, a.cuda_stream)
        torch.cuda.synchronize()
        assert mb.flags[0].item() == 2
        for r, (d, t) in enumerate(zip(dst, src)):
            assert torch.equal(d.view(torch.int64), t.view(torch.int64)), (r, "collected before the hand-over arrived")
    finally:
        mb.close()


# ---------------------------------------------------------------------------------------------------------------------
# D. solver contexts and parked front solutions
# ---------------------------------------------------------------------------------------------------------------------
def test_concurrent_contexts_vs_oracle(hp):
    """three contexts of one solver (n = 250, P = 2, K = 8: three sweeps fit on the device at once) on three streams,
    released together: each runs precond_apply_multi and the staged 8-wide sweeps on its own 8 right-hand sides.  A
    context that shared exchange ring, flags or parked front solutions with another would mix their data."""
    n, b, P, K = 250, 12, 2, 8
    omega, c_mat, f = problem(n)
    h = 1 / (n + 1)
    base = base_fields(n, f)
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(P, K, layout="cluster")
    ctxs = []
    try:
        L = s.layout()
        assert (L["P"], L["K"], L["QP"], L["CW"]) == (2, 8, 125, 17) and s.multi_kernel(8) == SWEEP4D, L
        ctxs = [s.clone_context() for _ in range(3)]
        Pc = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat)
        mb = {}
        for diag in ("reference", "paper"):
            Pc.diag = diag
            mb[diag] = np.array([Pc.apply(v) for v in base])
        coefs = [np.roll(COEF, 3 * c, axis=0) * (1j ** c) for c in range(3)]         # different data per context
        xs = [[dev(v) for v in cf @ np.array(base)] for cf in coefs]
        outs = [[sentinel_fill(torch.empty_like(x)) for x in row] for row in xs]
        us = [[x.clone() for x in row] for row in xs]
        tfs = [[c.front_tf_new() for _ in range(8)] for c in ctxs]
        streams = [torch.cuda.Stream() for _ in ctxs]
        torch.cuda.synchronize()
        gate = torch.cuda.Event()
        torch.cuda._sleep(100_000_000)                       # everything below is enqueued before any of it starts
        gate.record()

        def on(c, fn):
            with torch.cuda.stream(streams[c]):
                fn(ctxs[c])

        for c in range(3):
            on(c, lambda ctx: torch.cuda.current_stream().wait_event(gate))
        for c in range(3):
            on(c, lambda ctx, c=c: ctx.precond_apply_multi(xs[c], outs[c], diag="reference"))
        for c in range(3):
            def begin(ctx, c=c):
                for k in range(8):
                    ctx.front_begin(us[c][k])
                    ctx.front_tf_save(tfs[c][k])
            on(c, begin)
        for c in range(3):
            on(c, lambda ctx, c=c: ctx.sweep_forward_multi_buf(us[c], 0, b + 1, n - 1))
        for c in range(3):
            on(c, lambda ctx, c=c: ctx.sweep_backward_multi_buf(us[c], 0, n, b + 1, "paper"))
        for c in range(3):
            def end(ctx, c=c):
                for k in range(8):
                    ctx.front_tf_load(tfs[c][k])
                    ctx.front_end(us[c][k])
            on(c, end)
        torch.cuda.synchronize()
        assert [ctx.sweep_status() for ctx in ctxs] == [0, 0, 0]
        for c in range(3):
            check(outs[c], coefs[c] @ mb["reference"], (f"context {c}", "precond_apply_multi"))
            check(us[c], coefs[c] @ mb["paper"], (f"context {c}", "staged sweeps"))
    finally:
        for ctx in ctxs:
            ctx.close()
        s.close()


@pytest.mark.parametrize("front", ["blockdiag", "coupled"])
def test_parked_front_solution(hp, front):
    """T_F u_F parked with front_tf_save survives hp_front_begin of another right-hand side: front_tf_load + front_end
    finish the first application as the oracle does"""
    n, b = 120, 12
    omega, c_mat, f = problem(n)
    h = 1 / (n + 1)
    base = base_fields(n, f)
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner(6, 4, layout="cluster", front=front)
    try:
        Pc = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat, front=front)
        for diag in ("reference", "paper"):
            Pc.diag = diag
            u1, u2 = dev(base[1]), dev(base[2])
            t = s.front_tf_new()
            s.front_begin(u1)
            s.front_tf_save(t)
            s.sweep_forward(u1, b + 1, n - 1)
            s.sweep_backward(u1, n, b + 1, diag)
            s.front_begin(u2)                                # replaces the solver's own T_F u_F
            s.front_tf_load(t)
            s.front_end(u1)
            check([u1], [Pc.apply(base[1])], (front, diag))
        assert s.sweep_status() == 0
    finally:
        s.close()


def test_refactor_refused_while_contexts_are_open(hp):
    """hp_precond_setup, hp_precond_set_front and a change of the front mode on a solver with open contexts would leave
    the contexts pointing at freed memory: they are refused, the solver keeps working, and they work again once every
    context (also a context cloned from a context) is closed"""
    n, b = 40, 5
    omega, c_mat, f = problem(n)
    h = 1 / (n + 1)
    x = dev(f)
    ref = {fr: orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat, front=fr).apply(f) for fr in ("blockdiag", "coupled")}
    s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat).setup_preconditioner()
    try:
        c1 = s.clone_context()
        c2 = c1.clone_context()
        for _ in range(2):
            for call in (lambda: s.setup_preconditioner(), lambda: s.set_front("coupled"),
                         lambda: s.setup_preconditioner(front="coupled")):
                with pytest.raises(hp.HelmholtzB200Error, match="context"):
                    call()
            assert s.front == "blockdiag"
            check([s.precond_apply(x)], [ref["blockdiag"]], "the solver after a refused call")
            c1.close()                                       # c2 still holds the factorisation
        c2.close()
        s.set_front("coupled")
        check([s.precond_apply(x)], [ref["coupled"]], "set_front after the contexts are closed")
        s.setup_preconditioner(front="blockdiag")
        check([s.precond_apply(x)], [ref["blockdiag"]], "setup after the contexts are closed")
    finally:
        s.close()


# ---------------------------------------------------------------------------------------------------------------------
# E. the production SlabSolver on the GPU, ranks in processes that share GPU 0
# ---------------------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        return sk.getsockname()[1]


def _slab_fields(n, k):
    rng = np.random.default_rng(k + 17)
    return [rng.standard_normal((n, n)) + 1j * rng.standard_normal((n, n)) for _ in range(k)]


def _slab_worker(rank, world, port, n, b, ret):
    import faulthandler
    import sys
    faulthandler.dump_traceback_later(300, exit=True, file=sys.stderr)
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
        torch.cuda.set_device(0)
        dev0 = torch.device("cuda:0")
        import helmholtz_preconditioner_b200 as hp
        from helmholtz_preconditioner_b200.slab import SlabSolver, slab_bounds

        class HostStaged(SlabSolver):
            """point-to-point messages through host copies (gloo carries no device tensors)"""
            keep = []

            def _send(self, t, dst):
                dist.send(t.cpu(), dst)

            def _recv(self, t, src):
                c = torch.empty(t.shape, dtype=t.dtype)
                dist.recv(c, src)
                t.copy_(c)

            def _exchange(self, ops):
                if not ops:
                    return
                cpu, back = [], []
                for q in ops:
                    t = q.tensor.cpu() if q.op is dist.isend else torch.empty(q.tensor.shape, dtype=q.tensor.dtype)
                    cpu.append(dist.P2POp(q.op, t, q.peer, q.group))
                    if q.op is dist.irecv:
                        back.append((q.tensor, t))
                for w in dist.batch_isend_irecv(cpu):
                    w.wait()
                for dst, t in back:
                    dst.copy_(t)

            def _post(self, ops):
                cpu = [dist.P2POp(q.op, q.tensor.cpu(), q.peer, q.group) for q in ops]
                self.keep += cpu
                return dist.batch_isend_irecv(cpu)

        omega, c_mat, _ = problem(n)
        R = slab_bounds(n, b, world)
        j0, j1 = R[rank], R[rank + 1]
        s = hp.HelmholtzSolver(n, b, omega, 60.0, c_mat, device=dev0)
        s.setup_preconditioner(6, 4, max(b + 1, j0 + 1), min(n, j1), layout="cluster")
        S = HostStaged(s, n, b, rank, world, None, device=dev0)
        xs = [torch.from_numpy(np.ascontiguousarray(x[j0:j1].ravel())).to(dev0) for x in _slab_fields(n, 11)]
        res = {}
        for diag in ("reference", "paper"):
            out = torch.full_like(xs[0], complex("nan"))
            S.precond_apply(xs[0], out, diag=diag)
            res[f"M1_{diag}"] = [out.cpu().numpy()]
            pairs = [(x, torch.full_like(x, complex("nan"))) for x in xs]
            S.precond_apply_batch(pairs, diag=diag)
            res[f"M11_{diag}"] = [o.cpu().numpy() for _, o in pairs]
        out = torch.full_like(xs[0], complex("nan"))
        S.matvec(xs[0], out)
        res["A1"] = [out.cpu().numpy()]
        pairs = [(x, torch.full_like(x, complex("nan"))) for x in xs[:3]]
        S.matvec_batch(pairs)
        res["A3"] = [o.cpu().numpy() for _, o in pairs]
        torch.cuda.synchronize()
        res["status"] = s.sweep_status()
        res["groups"] = [len(g) for g in batch_groups(s, 11)]
        s.close()
        ret[rank] = res
        faulthandler.cancel_dump_traceback_later()
        dist.destroy_process_group()
    except Exception as e:                                   # noqa: BLE001 - reported to the parent
        import traceback
        ret[rank] = dict(error=traceback.format_exc())
        raise e


@pytest.mark.parametrize("world", [2, 3])
def test_slab_solver_processes_vs_oracle(hp, world):
    """SlabSolver.precond_apply, precond_apply_batch (11 right-hand sides: 8 + 2 + 1 per launch), matvec and matvec_batch
    with the HelmholtzSolver backend of every rank (row views, base pointers row0 = j0-1, group splitting) against the
    oracle"""
    n, b = 120, 12
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_slab_worker, args=(world, _free_port(), n, b, ret), nprocs=world, join=True)
    for r in range(world):
        assert "error" not in ret[r], ret[r].get("error")
        assert ret[r]["status"] == 0 and ret[r]["groups"] == [8, 2, 1], (r, ret[r]["status"], ret[r]["groups"])
    omega, c_mat, _ = problem(n)
    h = 1 / (n + 1)
    xs = _slab_fields(n, 11)
    glob = {k: [np.concatenate([ret[r][k][i] for r in range(world)]) for i in range(len(ret[0][k]))]
            for k in ret[0] if k not in ("status", "groups")}
    Pc = orc.SweepingPreconditioner(b, 60.0, b * h, omega, h, n, c_mat)
    for diag in ("reference", "paper"):
        Pc.diag = diag
        refs = [Pc.apply(x.ravel()) for x in xs]
        for k, (o, r) in enumerate(zip(glob[f"M1_{diag}"] + glob[f"M11_{diag}"], refs[:1] + refs)):
            assert np.all(np.isfinite(o)) and relerr(o, r) < TOL, (world, diag, k, relerr(o, r))
    p = dict(b=b, const=60.0, eta=b * h, omega=omega, h=h, n=n, c_mat=c_mat)
    for k, (o, x) in enumerate(zip(glob["A1"] + glob["A3"], xs[:1] + xs[:3])):
        r = orc.stencil_matvec(x.ravel(), **p)
        assert np.all(np.isfinite(o)) and relerr(o, r) < SPMV_TOL, (world, "A x", k, relerr(o, r))
