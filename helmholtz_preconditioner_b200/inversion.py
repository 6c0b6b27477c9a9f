"""Inversion for the medium (full-waveform inversion): data misfit at receivers, its adjoint-state gradient, and Born
(linearised) modelling, for many sources of one medium on one device.

Conventions (see INTEGRATION.md, "Inversion"):
- kappa = 1/c^2 is the slowness^2 the operator reads; c_mat is read transposed, so grid point (i, j) (1-based) takes
  c_mat[i-1, j-1].  Gradients and perturbations use the same (n+2, n+2) c_mat layout: grad[i-1, j-1] belongs to (i, j),
  and the last two rows and columns of a gradient are zero.
- The misfit is J = 1/2 sum_s |R u_s - d_s|^2 with A u_s = f_s and R the sampling at the receivers.
- The gradient is G = dJ/dRe kappa + i dJ/dIm kappa, so that dJ = Re sum_p conj(G_p) dkappa_p.  For a real medium it is
  Re G (float64).  wrt='velocity' gives conj(dkappa/dc) G with dkappa/dc = -2 kappa sqrt(kappa), the principal root.
- A is complex symmetric, so the adjoint field is a forward solve: A mu_s = R^T conj(r_s), r_s = R u_s - d_s, and
  G = -conj(w (.) sum_s mu_s (.) u_s) with w = dA_pp/dkappa_p = omega^2 is1(i) is2(j).

The sources run in waves of as many as one sweep launch carries (as in solver.run_solver_many).  The n^2-sized products
are the kernels of csrc/hp_grad.cu; sampling and injection at the receivers are nrec-sized torch indexing.
"""
import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .gmres import DeviceVectors
from .solver import DIAG_MODES, _as_device_field, _ptr, _solve_wave, _source_fields, _stream

WRT = {"kappa": 0, "velocity": 1}


class Receivers:
    """The grid points (i[k], j[k]) (1-based, 1 <= i, j <= n) at which every source's field is recorded.

    index is the int64 tensor of field positions (j-1) n + (i-1) (the f_mat.flatten() ordering), on `device` (default:
    the current CUDA device when there is one, else the host; the drivers move it to the solver's device)."""

    def __init__(self, n, i, j, device=None):
        i, j = np.asarray(i), np.asarray(j)
        if i.ndim != 1 or j.ndim != 1 or i.shape != j.shape:
            raise ValueError(f"i and j must be 1-D and of equal length, got shapes {i.shape} and {j.shape}")
        if i.size == 0:
            raise ValueError("no receivers")
        if not (np.issubdtype(i.dtype, np.integer) and np.issubdtype(j.dtype, np.integer)):
            raise ValueError("receiver indices must be integers")
        n = int(n)
        bad = (i < 1) | (i > n) | (j < 1) | (j > n)
        if bad.any():
            k = int(np.flatnonzero(bad)[0])
            raise ValueError(f"receiver {k} at (i, j) = ({i[k]}, {j[k]}) lies outside the grid 1..{n}")
        p = (j.astype(np.int64) - 1) * n + (i.astype(np.int64) - 1)
        _, first, counts = np.unique(p, return_index=True, return_counts=True)
        if (counts > 1).any():
            k = int(np.sort(first[counts > 1])[0])
            raise ValueError(f"receiver ({i[k]}, {j[k]}) appears more than once")
        self.n, self.i, self.j = n, i.astype(np.int64), j.astype(np.int64)
        if device is None and torch.cuda.is_available():
            device = torch.device(f"cuda:{torch.cuda.current_device()}")
        self.index = torch.from_numpy(p).to(device if device is not None else "cpu")

    @property
    def nrec(self):
        return int(self.index.numel())

    def __len__(self):
        return self.nrec

    def on(self, device):
        """index on `device` (moved there once)"""
        if self.index.device != torch.device(device):
            self.index = self.index.to(device)
        return self.index

    def sample(self, u):
        """R u: the field u (n*n,) at the receivers, (nrec,)"""
        return u.reshape(-1)[self.on(u.device)]

    def inject(self, r, out=None):
        """R^T conj(r): conj(r) scattered into a zeroed field (n*n,) complex128 (the adjoint source)"""
        if out is None:
            out = torch.zeros(self.n * self.n, dtype=torch.complex128, device=r.device)
        else:
            out.zero_()
        out[self.on(out.device)] = r.conj()
        return out


@dataclass
class GradientResult:
    misfit: float                   # J = 1/2 sum_s |R u_s - d_s|^2
    grad: torch.Tensor              # (n+2, n+2) in c_mat layout: float64 for a real medium, complex128 for an attenuating one
    residuals: torch.Tensor         # (S, nrec) complex128: R u_s - d_s
    forward_niter: list             # per source: GMRES iterations and exit code of the forward solve
    forward_info: list
    adjoint_niter: list             # ... and of the adjoint solve
    adjoint_info: list
    times: dict = field(default_factory=dict)   # wall seconds: forward, adjoint and kernels (accumulate, finish, sampling)
    u: list = field(default=None, repr=False)   # the forward fields (n*n,) when keep_fields=True (born(..., u=...))


def _count(f_mats):
    if isinstance(f_mats, (list, tuple)):
        return len(f_mats)
    if getattr(f_mats, "ndim", 0) < 2:
        raise ValueError("f_mats must be (S, n, n), (S, n*n) or a list of fields")
    return int(f_mats.shape[0])


def _items(f_mats):
    return list(f_mats) if isinstance(f_mats, (list, tuple)) else [f_mats[i] for i in range(f_mats.shape[0])]


def _check_solver(solver, receivers, what):
    _lib.require_device()
    if solver is None or not getattr(solver, "handle", None):
        raise _lib.HelmholtzB200Error(f"{what}: no solver")
    if (solver.m_lo, solver.m_hi) != (solver.b + 1, solver.n):
        raise _lib.HelmholtzB200Error(f"{what}: the solver must be set up on all strips (setup_preconditioner()), "
                                      f"it holds strips {solver.m_lo}..{solver.m_hi}")
    if receivers.n != solver.n:
        raise ValueError(f"{what}: receivers are for n = {receivers.n}, the solver has n = {solver.n}")
    solver._on_device()


def _solve(s, fs, vec, diag, rtol, restart, maxiter, what):
    """one wave, precond_input='vector'; raise if a solve did not converge (a gradient would be silently wrong)"""
    outs = _solve_wave(s, fs, s._widest(), vec, diag, "vector", rtol, restart, maxiter)
    for k, (_, info, _) in enumerate(outs):
        if info != 0:
            raise _lib.HelmholtzB200Error(f"{what} solve of wave source {k} did not converge (info {info}); raise maxiter or "
                                          "rtol")
    return outs


def misfit_gradient(solver, f_mats, receivers, d_obs, *, wrt="kappa", diag="paper", rtol=1e-6, restart=20, maxiter=None,
                    keep_fields=False):
    """Misfit J = 1/2 sum_s |R u_s - d_s|^2 and its gradient for the sources f_mats of solver's medium.

    solver: a HelmholtzSolver set up with setup_preconditioner() (front='coupled' converges in a few iterations).
    f_mats: (S, n, n) or (S, n*n) array or tensor, or a list of S fields.  receivers: Receivers.  d_obs: (S, nrec) observed
    data.  wrt: 'kappa' (slowness^2 1/c^2) or 'velocity' (c).  diag, rtol, restart, maxiter: those of run_solver_many;
    the solves apply the preconditioner to the GMRES vector (precond_input='vector').  keep_fields=True keeps the forward
    fields in the result (GradientResult.u) for born(..., u=...).

    Sources run in waves of one sweep launch: each wave is solved forward, then adjoint, then added to the gradient, so
    about three fields per wave slot are alive at a time.  Raises HelmholtzB200Error if a solve does not converge."""
    if wrt not in WRT:
        raise ValueError(f"wrt must be 'kappa' or 'velocity', got {wrt!r}")
    if diag not in DIAG_MODES:
        raise ValueError(f"diag must be one of {sorted(DIAG_MODES)}, got {diag!r}")
    S = _count(f_mats)
    if tuple(d_obs.shape) != (S, receivers.nrec):
        raise ValueError(f"d_obs must be (S, nrec) = ({S}, {receivers.nrec}), got {tuple(d_obs.shape)}")
    _check_solver(solver, receivers, "misfit_gradient")
    s = solver
    n, dev = s.n, s.device
    d = _as_device_field(d_obs, dev).reshape(S, receivers.nrec)
    items = _items(f_mats)
    W = s._widest()
    vec = DeviceVectors(n * n, dev, restart=restart)
    acc = torch.zeros(n * n, dtype=torch.complex128, device=dev)
    res = torch.empty(S, receivers.nrec, dtype=torch.complex128, device=dev)
    fwd_it, fwd_info, adj_it, adj_info, kept = [], [], [], [], []
    times = {"forward": 0.0, "adjoint": 0.0, "kernels": 0.0}
    for w0 in range(0, S, W):
        t0 = time.time()
        fs = _source_fields(items[w0:w0 + W], n, dev)
        outs = _solve(s, fs, vec, diag, rtol, restart, maxiter, "forward")
        del fs
        us = [u for u, _, _ in outs]
        fwd_it += [len(h) for _, _, h in outs]
        fwd_info += [info for _, info, _ in outs]
        torch.cuda.synchronize(dev)
        t1 = time.time()
        adj = []
        for k, u in enumerate(us):
            res[w0 + k] = receivers.sample(u) - d[w0 + k]
            adj.append(receivers.inject(res[w0 + k]))
        torch.cuda.synchronize(dev)
        t2 = time.time()
        outs = _solve(s, adj, vec, diag, rtol, restart, maxiter, "adjoint")
        del adj
        mus = [m for m, _, _ in outs]
        adj_it += [len(h) for _, _, h in outs]
        adj_info += [info for _, info, _ in outs]
        torch.cuda.synchronize(dev)
        t3 = time.time()
        _lib.check(s.lib.hp_grad_accumulate(s.handle, len(us), s._ptr_array(us), s._ptr_array(mus), _ptr(acc), _stream()),
                   "hp_grad_accumulate")
        if keep_fields:
            kept += us
        del us, mus
        torch.cuda.synchronize(dev)
        t4 = time.time()
        times["forward"] += t1 - t0
        times["adjoint"] += t3 - t2
        times["kernels"] += (t2 - t1) + (t4 - t3)
    t0 = time.time()
    grad = torch.empty(n + 2, n + 2, dtype=torch.complex128 if s.medium_is_complex else torch.float64, device=dev)
    _lib.check(s.lib.hp_grad_finish(s.handle, _ptr(acc), WRT[wrt], _ptr(grad), _stream()), "hp_grad_finish")
    misfit = 0.5 * float(torch.sum(res.real ** 2 + res.imag ** 2).item())
    times["kernels"] += time.time() - t0
    return GradientResult(misfit, grad, res, fwd_it, fwd_info, adj_it, adj_info, times, kept if keep_fields else None)


def born(solver, f_mats, receivers, dkappa, *, diag="paper", rtol=1e-6, restart=20, maxiter=None, u=None):
    """Born (linearised) data R du_s for a slowness^2 perturbation dkappa: du_s = A^-1 (-w (.) dkappa (.) u_s), with
    w = dA_pp/dkappa_p.  Returns an (S, nrec) complex128 device tensor.

    dkappa: (n+2, n+2) in c_mat layout (entry [i-1, j-1] for grid point (i, j); the last two rows and columns are not
    read), real or complex.  u: the forward fields A u_s = f_s, (S, n*n) or a list of (n*n,) device fields (for instance
    misfit_gradient(..., keep_fields=True).u); without it they are solved here from f_mats (which may be None when u is
    given).  The other arguments mean what they mean for misfit_gradient."""
    if diag not in DIAG_MODES:
        raise ValueError(f"diag must be one of {sorted(DIAG_MODES)}, got {diag!r}")
    if u is None and f_mats is None:
        raise ValueError("born needs f_mats or u")
    S = _count(u if u is not None else f_mats)
    if u is not None and f_mats is not None and _count(f_mats) != S:
        raise ValueError(f"u holds {S} fields, f_mats {_count(f_mats)}")
    _check_solver(solver, receivers, "born")
    s = solver
    n, dev = s.n, s.device
    if tuple(dkappa.shape) != (n + 2, n + 2):
        raise ValueError(f"dkappa must be ({n + 2}, {n + 2}) like c_mat, got {tuple(dkappa.shape)}")
    dk = _as_device_field(dkappa, dev)
    items = _items(u if u is not None else f_mats)
    W = s._widest()
    vec = DeviceVectors(n * n, dev, restart=restart)
    out = torch.empty(S, receivers.nrec, dtype=torch.complex128, device=dev)
    for w0 in range(0, S, W):
        if u is None:
            us = [x for x, _, _ in _solve(s, _source_fields(items[w0:w0 + W], n, dev), vec, diag, rtol, restart, maxiter,
                                          "forward")]
        else:
            us = _source_fields(items[w0:w0 + W], n, dev)
        srcs = [torch.empty_like(x) for x in us]
        _lib.check(s.lib.hp_born_source(s.handle, len(us), _ptr(dk), s._ptr_array(us), s._ptr_array(srcs), _stream()),
                   "hp_born_source")
        del us
        outs = _solve(s, srcs, vec, diag, rtol, restart, maxiter, "Born")
        del srcs
        for k, (du, _, _) in enumerate(outs):
            out[w0 + k] = receivers.sample(du)
    return out
