"""Velocity models and sources of the reference (host side, numpy): /root/reference/code.py:39-66, 390-408.

These produce the *inputs* of the hot path (an (n+2)^2 velocity array and an n^2 source); they are O(n^2)
host arithmetic done once and are kept in the reference's own form so that user-supplied models drop in."""
import numpy as np


def init_c1_mat(r1, r2, n):
    """code.py:40-44 -- Gaussian low-velocity lens centred at (r1, r2)."""
    x_i = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x_i, x_i)
    return 4 / 3 * (1 - .5 * np.exp(-32 * ((xx - r1) ** 2 + (yy - r2) ** 2)))


def init_c2_mat(n):
    """code.py:47-51 -- vertical wave guide."""
    x_i = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x_i, x_i)
    return 4 / 3 * (1 - .5 * np.exp(-32 * ((xx - .5) ** 2)))


def init_f1_mat(r1, r2, omega, n):
    """code.py:54-58 -- narrow Gaussian point source."""
    x_i = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x_i[1:-1], x_i[1:-1])
    return np.exp(-(4 * omega / np.pi) ** 2 * ((xx - r1) ** 2 + (yy - r2) ** 2))


def init_f2_mat(r1, r2, d1, d2, omega, n):
    """code.py:61-66 -- Gaussian wave packet travelling in direction (d1, d2)."""
    x_i = np.linspace(0, 1, n + 2)
    xx, yy = np.meshgrid(x_i[1:-1], x_i[1:-1])
    return np.exp(-4 * omega * ((xx - r1) ** 2 + (yy - r2) ** 2)) * np.exp(1j * omega * (xx * d1 + yy * d2))


def init_c1_f1(omega, n, cr1=.5, cr2=.5, fr1=.5, fr2=.125):
    """code.py:390-393."""
    return init_c1_mat(cr1, cr2, n), init_f1_mat(fr1, fr2, omega, n)


def init_c1_f2(omega, n, cr1=.5, cr2=.5, fr1=.125, fr2=.125, d1=1 / 2 ** .5, d2=1 / 2 ** .5):
    """code.py:395-398."""
    return init_c1_mat(cr1, cr2, n), init_f2_mat(fr1, fr2, d1, d2, omega, n)


def init_c2_f1(omega, n, r1=.5, r2=.5):
    """code.py:400-403."""
    return init_c2_mat(n), init_f1_mat(r1, r2, omega, n)


def init_c2_f2(omega, n, r1=.5, r2=.5, d1=1 / 2 ** .5, d2=1 / 2 ** .5):
    """code.py:405-408."""
    return init_c2_mat(n), init_f2_mat(r1, r2, d1, d2, omega, n)


def init_const_f1(omega, n, c0=1.0, fr1=.5, fr2=.125):
    """Constant velocity c0 with the reference's point source (BASELINE config: constant-velocity 2D)."""
    return np.full((n + 2, n + 2), float(c0)), init_f1_mat(fr1, fr2, omega, n)


def init_layered_f1(omega, n, layers=8, c_lo=1.0, c_hi=2.0, fr1=.5, fr2=.125, seed=0):
    """Synthetic layered velocity model (BASELINE config: heterogeneous layered 2D): `layers` horizontal layers
    (constant along x1) with velocities drawn in [c_lo, c_hi], slightly smoothed across the interfaces.
    Stored in the reference's c_mat convention (read as c_mat[i-1, j-1], code.py:108)."""
    rng = np.random.default_rng(seed)
    vel = c_lo + (c_hi - c_lo) * rng.random(layers)
    x_i = np.linspace(0, 1, n + 2)
    edges = np.linspace(0, 1, layers + 1)
    prof = np.zeros(n + 2)
    w = 2.0 / (n + 1)
    for k in range(layers):
        lo, hi = edges[k], edges[k + 1]
        prof += vel[k] * 0.5 * (np.tanh((x_i - lo) / w) - np.tanh((x_i - hi) / w))
    prof[prof < c_lo * 0.5] = c_lo
    c_mat = np.tile(prof[None, :], (n + 2, 1))     # varies with the second index = x2 (depth)
    return c_mat, init_f1_mat(fr1, fr2, omega, n)


def attenuate(c_mat, q):
    """Attenuating medium from a velocity model and a quality factor: returns c_mat / sqrt(1 + 1j/q), complex.

    q is a scalar or an array of c_mat's shape; np.inf means lossless (the result then has a zero imaginary part).
    Sign convention: the solver's PML, s = 1/(1 + i sigma/omega), and a damping alpha > 0 in
    omega = 2 pi wave_num + 1j alpha both make loss Im(omega^2 kappa) > 0 for Re omega > 0, with the slowness^2
    kappa = 1/c^2.  Here kappa = (1 + 1j/q)/c_mat^2, so Im(kappa) > 0 for 0 < q < inf: a wave decays as it travels.
    Pass the result as c_mat to HelmholtzSolver, run_solver, run_solver_many or any other entry point."""
    c = np.asarray(c_mat)
    q = np.asarray(q, dtype=np.float64)
    if q.ndim and q.shape != c.shape:
        raise ValueError(f"q must be a scalar or of c_mat's shape {c.shape}, got {q.shape}")
    return c / np.sqrt(1 + 1j / q)
