"""Golden fixtures at the reference's production sizes and at BASELINE.json's configurations.

Run in the build container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden_large.py A ref          # one (case, part); see CASES / PARTS below
    python tests/golden/make_golden_large.py all            # everything, sequentially (hours on one core)

Cases
    T  run_solver(63, 12, 4, 61, 2, init_c1_f1)              code.py:570 (small; tests regenerate it and compare)
    A  run_solver(511, 12, 64, 81, 2, init_c1_f1)            code.py:584
    B  run_solver(1023, 12, 128, 100, 2, init_c1_f1)         code.py:589
    C  1024^2, constant velocity, 10 points per wavelength, PML width 20   (BASELINE.json configs[1])
    D  4096^2, layered velocity, 10 points per wavelength, PML width 12    (BASELINE.json configs[2]; M f only)

Parts (A, B, C)
    ref  algo2_4 of the UNMODIFIED reference (imported from /root/reference/code.py as in make_golden.py) on f and
         on a random vector, next to the oracle's four (front, diag) variants on the same inputs; the oracle's
         (blockdiag, reference) result is asserted equal to the reference's to 1e-13 before anything is written
    pb pc rb rc   GMRES(20), rtol 1e-3, preconditioner applied to the vector it is given (precond_input='vector'),
         diag = p(aper) | r(eference, code.py:372-375), front = b(lockdiag, code.py:178-183) | c(oupled);
         diag = paper runs to convergence; diag = reference does not converge in any useful number of iterations
         (blockdiag: never; coupled: 439 iterations at n = 63) and is capped, the cap is stored
Part (D)
    mf   M f and M x_rand for the four variants; the strip factorisations do not fit in memory at this size
         (~160 GB), so every strip is factorised twice (forward pass, backward pass) and dropped

Full fields are too large to commit (16 MB each at 1023^2), so a field u[j, i] is stored as: a few full rows, the
checksum of every row with a fixed random vector z (u @ z), the checksum of every column (z2 @ u), and its norm.
No committed file exceeds 1 MB: a fixture larger than that is split into <name>.npz, <name>.2.npz, ... (write / load).
"""
import glob
import os
import sys
import time

import numpy as np
import scipy.sparse.linalg as spla

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

from oracle import helmholtz_oracle as orc  # noqa: E402

CASES = {
    "T": dict(n=63, b=12, wave_num=4.0, const=61.0, alpha=2.0, model="c1f1", cap_rb=40),    # small: the tests regenerate it
    "A": dict(n=511, b=12, wave_num=64.0, const=81.0, alpha=2.0, model="c1f1", cap_rb=40),
    "B": dict(n=1023, b=12, wave_num=128.0, const=100.0, alpha=2.0, model="c1f1", cap_rb=40),
    "C": dict(n=1024, b=20, wave_num=102.4, const=100.0, alpha=2.0, model="const", cap_rb=40),
    "D": dict(n=4096, b=12, wave_num=409.6, const=100.0, alpha=2.0, model="layered"),
}
PARTS = {"pb": ("paper", "blockdiag"), "pc": ("paper", "coupled"), "rb": ("reference", "blockdiag"),
         "rc": ("reference", "coupled")}


def fields(case):
    """Inputs of a case.  The layered / constant models are the package's closed-form input generators
    (helmholtz_preconditioner_b200/fields.py: numpy only, no device code)."""
    from helmholtz_preconditioner_b200 import fields as F
    p = CASES[case]
    omega = 2 * np.pi * p["wave_num"] + 1j * p["alpha"]
    n = p["n"]
    if p["model"] == "c1f1":
        c_mat, f_mat = orc.init_c1_f1(omega, n)
    elif p["model"] == "const":
        c_mat, f_mat = F.init_const_f1(omega, n)
    else:
        c_mat, f_mat = F.init_layered_f1(omega, n)
    return omega, c_mat, np.asarray(f_mat, dtype=np.complex128)


def checks(n):
    rng = np.random.default_rng(20261018)
    z = np.exp(2j * np.pi * rng.random(n))
    z2 = np.exp(2j * np.pi * rng.random(n))
    return z, z2


def sample_rows(n, b):
    stride = 128 if n <= 2048 else 2048
    return np.array(sorted(set([0, b - 1, b, b + 1, n // 2, n - 2, n - 1] + list(range(0, n, stride)))))


def compact(prefix, vec, n, b, out):
    U = np.asarray(vec).reshape(n, n)
    z, z2 = checks(n)
    rows = sample_rows(n, b)
    out[prefix + "_rows"] = U[rows]
    out[prefix + "_rowsum"] = U @ z
    out[prefix + "_colsum"] = z2 @ U
    out[prefix + "_norm"] = np.linalg.norm(U)


def header(case):
    p = CASES[case]
    n, b = p["n"], p["b"]
    z, z2 = checks(n)
    return dict(n=n, b=b, wave_num=p["wave_num"], const=p["const"], alpha=p["alpha"], model=p["model"],
                sample_rows=sample_rows(n, b), z=z, z2=z2)


def x_rand(n):
    rng = np.random.default_rng(4321)
    return rng.standard_normal(n * n) + 1j * rng.standard_normal(n * n)


PART_BYTES = 900_000


def write(path, out):
    """np.savez_compressed of the arrays of `out`, in order, spread over path, path[:-4] + '.2.npz', ... so that no file
    holds more than PART_BYTES of array data"""
    for old in glob.glob(glob.escape(path[:-4]) + ".[0-9]*.npz"):
        os.remove(old)
    parts, size = [{}], 0
    for k, v in out.items():
        nb = np.asarray(v).nbytes
        if parts[-1] and size + nb > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = v
        size += nb
    for i, arrays in enumerate(parts):
        np.savez_compressed(path if i == 0 else f"{path[:-4]}.{i + 1}.npz", **arrays)


def load(path):
    """the arrays of a fixture written by write(), as one dict"""
    out, i = dict(np.load(path)), 2
    while os.path.exists(f"{path[:-4]}.{i}.npz"):
        out.update(np.load(f"{path[:-4]}.{i}.npz"))
        i += 1
    return out


def save(case, part, out):
    p = CASES[case]
    name = f"large_n{p['n']}_b{p['b']}_{p['model']}__{part}.npz"
    write(os.path.join(HERE, name), out)
    print("written", name, {k: getattr(v, "shape", v) for k, v in out.items() if not k.endswith(("_rows", "sum"))}, flush=True)


def relerr(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(np.asarray(b))


def part_ref(case):
    from make_golden import load_reference
    ref = load_reference()
    p = CASES[case]
    n, b, const = p["n"], p["b"], p["const"]
    omega, c_mat, f_mat = fields(case)
    h = 1 / (n + 1)
    eta = b * h
    f_vec = f_mat.flatten()
    xr = x_rand(n)
    t0 = time.time()
    lu_HF, lu_Hm_ra = ref.algo2_3(b, const, eta, omega, h, n, c_mat)
    A_b1F = ref.get_A_b1F_block(b, const, eta, omega, h, n, c_mat)
    A_Fb1 = ref.get_A_Fb1_block(b, const, eta, omega, h, n, c_mat)
    up_A_ra, lo_A_ra = [], []
    for i in range(1, n):
        up_A_ra.append(ref.get_A_block(i, i + 1, b, const, eta, omega, h, n, c_mat))
        lo_A_ra.append(ref.get_A_block(i + 1, i, b, const, eta, omega, h, n, c_mat))
    args = (b, n, lu_HF, A_b1F, A_Fb1, up_A_ra, lo_A_ra, lu_Hm_ra)
    print(f"reference algo2_3: {time.time() - t0:.1f} s", flush=True)
    out = header(case)
    t0 = time.time()
    Mf = np.asarray(ref.algo2_4(f_vec, *args)).ravel()
    out["t_algo2_4_reference_s"] = time.time() - t0
    Mx = np.asarray(ref.algo2_4(xr, *args)).ravel()
    compact("ref_Mf", Mf, n, b, out)
    compact("ref_Mx", Mx, n, b, out)
    A = ref.build_A_matrix(b, const, eta, omega, h, n, c_mat).tocsr()
    compact("ref_Ax", A @ xr, n, b, out)
    del lu_HF, lu_Hm_ra, args
    for front in ("blockdiag", "coupled"):
        P = orc.SweepingPreconditioner(b, const, eta, omega, h, n, c_mat, diag="reference", front=front)
        for diag in ("reference", "paper"):
            P.diag = diag
            of, ox = P.apply(f_vec), P.apply(xr)
            if (front, diag) == ("blockdiag", "reference"):
                e1, e2 = relerr(of, Mf), relerr(ox, Mx)
                print("oracle vs reference algo2_4:", e1, e2, flush=True)
                assert e1 < 1e-13 and e2 < 1e-13
                out["oracle_vs_reference"] = np.array([e1, e2])
            compact(f"orc_{front}_{diag}_Mf", of, n, b, out)
            compact(f"orc_{front}_{diag}_Mx", ox, n, b, out)
        del P
    return out


def part_gmres(case, part):
    diag, front = PARTS[part]
    p = CASES[case]
    n, b = p["n"], p["b"]
    omega, c_mat, f_mat = fields(case)
    cap = p["cap_rb"] if diag == "reference" else 2000
    t0 = time.time()
    u, hist, niter, info = orc.run_solver(n, b, p["wave_num"], p["const"], p["alpha"], c_mat=c_mat, f_mat=f_mat,
                                          diag=diag, front=front, precond_input="vector", rtol=1e-3, maxiter=cap)
    dt = time.time() - t0
    h = 1 / (n + 1)
    A = orc.build_A_matrix(b, p["const"], b * h, omega, h, n, c_mat)
    fv = f_mat.flatten()
    out = header(case)
    out.update(diag=diag, front=front, maxiter=cap, rtol=1e-3, hist=np.array(hist), niter=niter, info=info,
               true_residual=np.linalg.norm(fv - A @ u) / np.linalg.norm(fv), oracle_seconds=dt)
    compact("u", u, n, b, out)
    print(case, part, "niter", niter, "info", info, "true residual", out["true_residual"], f"{dt:.0f} s", flush=True)
    return out


def part_mf_streamed(case):
    """algo2_4 (code.py:356-385) for several vectors and the four (front, diag) variants at a size whose strip
    factorisations cannot be held: ascending pass = forward sweep, descending pass = diagonal + backward sweep."""
    p = CASES[case]
    n, b, const = p["n"], p["b"], p["const"]
    omega, c_mat, f_mat = fields(case)
    h = 1 / (n + 1)
    eta = b * h
    inputs = [f_mat.flatten(), x_rand(n)]
    fronts = ("blockdiag", "coupled")
    diags = ("reference", "paper")
    _, _, c3, c4, _ = orc.stencil_coeffs(np.arange(1, n + 1), None, b, const, eta, omega, h, n, c_mat)
    lo, up = c3, c4
    # forward state: U[f][k] = (n, n) field of front f, input k
    U = [[np.array(x, dtype=np.complex128).reshape(n, n).copy() for x in inputs] for _ in fronts]
    TF = [[None] * len(inputs) for _ in fronts]
    luF = []
    for fi, front in enumerate(fronts):
        HF = orc.get_A_FF_block(b, const, eta, omega, h, n, c_mat, coupled=(front == "coupled")).tocsc()
        luF.append(spla.splu(HF))
        for k in range(len(inputs)):
            TF[fi][k] = luF[fi].solve(U[fi][k][:b].ravel())
            U[fi][k][b] = U[fi][k][b] - lo[b] * TF[fi][k][-n:]                           # code.py:365
    nv = len(fronts) * len(inputs)
    t0 = time.time()
    for m in range(b + 1, n):                                                         # code.py:366-370
        lu = spla.splu(orc.get_Hm(m, b, const, eta, omega, h, n, c_mat).tocsc())
        rhs = np.zeros((b * n, nv), dtype=np.complex128)
        for fi in range(len(fronts)):
            for k in range(len(inputs)):
                rhs[-n:, fi * len(inputs) + k] = U[fi][k][m - 1]
        sol = lu.solve(rhs)[-n:]
        for fi in range(len(fronts)):
            for k in range(len(inputs)):
                U[fi][k][m] = U[fi][k][m] - lo[m] * sol[:, fi * len(inputs) + k]
        if (m - b) % 200 == 0:
            print(f"forward strip {m}/{n}  {time.time() - t0:.0f} s", flush=True)
    # descending pass: diagonal (code.py:372-375) and backward sweep (code.py:376-380) share the factorisation of strip m
    W = {(fi, k, d): U[fi][k].copy() for fi in range(len(fronts)) for k in range(len(inputs)) for d in diags}
    keys = sorted(W)
    for m in range(n, b, -1):
        lu = spla.splu(orc.get_Hm(m, b, const, eta, omega, h, n, c_mat).tocsc())
        rhs = np.zeros((b * n, 2 * len(keys)), dtype=np.complex128)
        for c, key in enumerate(keys):
            rhs[-n:, 2 * c] = W[key][m - 1]
            if m <= n - 1:
                rhs[-n:, 2 * c + 1] = up[m - 1] * W[key][m]
        sol = lu.solve(rhs)[-n:]
        for c, key in enumerate(keys):
            t = sol[:, 2 * c]
            W[key][m - 1] = (W[key][m - 1] - t) if key[2] == "reference" else t
            if m <= n - 1:
                W[key][m - 1] = W[key][m - 1] - sol[:, 2 * c + 1]
        if (n - m) % 200 == 0:
            print(f"backward strip {m}/{n}  {time.time() - t0:.0f} s", flush=True)
    out = header(case)
    for (fi, k, d) in keys:
        u = W[(fi, k, d)]
        Au = np.zeros(b * n, dtype=np.complex128)                                     # code.py:381-384
        Au[-n:] = up[b - 1] * u[b]
        u[:b] = (TF[fi][k] - luF[fi].solve(Au)).reshape(b, n)
        compact(f"orc_{fronts[fi]}_{d}_{'Mf' if k == 0 else 'Mx'}", u.ravel(), n, b, out)
    out["oracle_seconds"] = time.time() - t0
    return out


def compute(case, part):
    if case == "D":
        assert part == "mf"
        return part_mf_streamed(case)
    if part == "ref":
        return part_ref(case)
    return part_gmres(case, part)


def run(case, part):
    save(case, part, compute(case, part))


if __name__ == "__main__":
    if sys.argv[1] == "all":
        for c in "TABC":
            for pt in ("ref", "pb", "pc", "rb", "rc"):
                run(c, pt)
        run("D", "mf")
    else:
        run(sys.argv[1], sys.argv[2])
