"""Restarted, left-preconditioned GMRES on the device, following scipy.sparse.linalg.gmres.

Reference call site: /root/reference/code.py:516
    u, exit_code = scipy.sparse.linalg.gmres(A, f_vec, M=M, tol=1e-3, callback=counter_prec)
i.e. scipy's defaults restart=20, maxiter=10*N, x0=0, atol=0 and the legacy callback (called once per inner
iteration with the preconditioned residual estimate divided by ||b||).  The control flow below follows
scipy/sparse/linalg/_isolve/iterative.py (scipy 1.11+: modified Gram-Schmidt Arnoldi, Givens rotations,
inner tolerance adaptation ptol), so that iteration counts match the reference.

The n^2-sized work (matvec, preconditioner, dot products, axpys) runs in the CUDA kernels of
libhelmholtz_b200.so; only the (restart+1)^2 Hessenberg arithmetic is done on the host.  With a process
group, vectors are slab-distributed and the dot products are all-reduced (NCCL).
"""
import math

import numpy as np
import torch

from . import _lib


_TRACE = bool(__import__("os").environ.get("HP_GMRES_TRACE"))     # developer switch: one line per served round of gmres_batch


def _ptr(t):
    return t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def lartg(f, g):
    """Givens rotation with LAPACK zlartg semantics: real c, complex s, [c s; -conj(s) c] [f; g] = [r; 0]."""
    f, g = complex(f), complex(g)
    if g == 0:
        return 1.0, 0j, f
    if f == 0:
        d = abs(g)
        return 0.0, g.conjugate() / d, d
    f1 = abs(f)
    h = math.hypot(f1, abs(g))
    c = f1 / h
    fs = f / f1
    return c, fs * g.conjugate() / h, fs * h


class CommStats:
    """how many collective / point-to-point calls the host issued (bench.py reports them per step)"""
    calls = 0


class DeviceVectors:
    """Krylov vector kernels on (a slab of) the field; reductions are summed over `group` if given."""

    def __init__(self, nloc, device, group=None, restart=20, orth=None):
        """orth: orthogonalisation of DISTRIBUTED vectors: "mgs" = modified Gram-Schmidt as scipy does it (k + 2 all-reduces
        per Arnoldi column, fused axpy + next dot passes), "cgs2" = classical Gram-Schmidt applied twice (csrc/hp_cgs.cu:
        3 block passes and 3 all-reduces per column, the Hessenberg entries agree with MGS to 1e-13).  Default: HP_ORTH or
        "mgs": measured in the group pipeline of bench.py, cgs2 is slower (N = 2: 128 vs 132 iters/s, N = 4: 250 vs 283) - the
        register-heavy block passes run at lower occupancy than the fused MGS passes (98 % of HBM peak) and the saved
        all-reduces do not pay for it.  Vectors on one device always use the fused MGS kernels."""
        import os
        self.lib = _lib.require_device()
        self.nloc, self.device, self.group = nloc, torch.device(device), group
        self.orth = orth or os.environ.get("HP_ORTH", "mgs")
        self.cgs = None                                      # coefficient block of the cgs2 passes, [3][R][k + 1]
        self.scal = torch.zeros(max(64, restart + 3), dtype=torch.complex128, device=device)
        self.scalb = None                                    # scalars of a batch of systems, [restart + 3][R]
        self._pin = None                                     # pinned host buffer of _host()

    def reserve(self, restart):
        """hp_mgs writes restart + 2 scalars (coefficients, norm after, norm before)"""
        if self.scal.numel() < restart + 3:
            self.scal = torch.zeros(restart + 3, dtype=torch.complex128, device=self.device)

    def _batch_scal(self, rows, R):
        if self.scalb is None or self.scalb.shape[0] < rows or self.scalb.shape[1] != R:
            self.scalb = torch.zeros((max(rows, self.scal.numel()), R), dtype=torch.complex128, device=self.device)
        return self.scalb

    def _host(self, t):
        """device scalars -> numpy, through a pinned buffer and a wait on the current stream only.  A copy to pageable
        memory (.cpu(), .item()) returns when the copy is done and holds a lock of the driver until then: with several
        host threads on one device (slab.GroupPipeline) a thread that waits that way for another GPU keeps the other
        threads from launching the work that GPU is waiting for (measured at N = 2)."""
        t = t.contiguous()
        m = t.numel()
        if self._pin is None or self._pin.numel() < m:
            self._pin = torch.empty(max(m, 1024), dtype=torch.complex128).pin_memory()
        h = self._pin[:m]
        h.copy_(t.reshape(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return h.numpy().reshape(t.shape).copy()

    def _all_reduce(self, t):
        import torch.distributed as dist
        CommStats.calls += 1
        dist.all_reduce(torch.view_as_real(t), group=self.group)

    def norm(self, x):
        if self.group is None:
            _lib.check(self.lib.hp_nrm2(self.nloc, _ptr(x), _ptr(self.scal), _stream()), "hp_nrm2")
            return float(self._host(self.scal[:1])[0].real)
        _lib.check(self.lib.hp_dotc(self.nloc, _ptr(x), _ptr(x), _ptr(self.scal), _stream()), "hp_dotc")
        self._all_reduce(self.scal[:1])
        return math.sqrt(float(self._host(self.scal[:1])[0].real))

    def norm_batch(self, xs):
        """norms of several vectors with one all-reduce and one copy to the host"""
        R = len(xs)
        sc = self._batch_scal(1, R)[0]
        for i, x in enumerate(xs):
            if self.group is None:
                _lib.check(self.lib.hp_nrm2(self.nloc, _ptr(x), _ptr(sc[i:]), _stream()), "hp_nrm2")
            else:
                _lib.check(self.lib.hp_dotc(self.nloc, _ptr(x), _ptr(x), _ptr(sc[i:]), _stream()), "hp_dotc")
        if self.group is not None:
            self._all_reduce(sc[:R])
        v = self._host(sc[:R]).real
        return [float(t) for t in (v if self.group is None else np.sqrt(v))]

    def scale_copy(self, a, x, y):
        a = complex(a)
        _lib.check(self.lib.hp_scale_copy(self.nloc, a.real, a.imag, _ptr(x), _ptr(y), _stream()), "hp_scale_copy")

    def axpy(self, a, x, y):
        a = complex(a)
        _lib.check(self.lib.hp_axpy(self.nloc, a.real, a.imag, _ptr(x), _ptr(y), _stream()), "hp_axpy")

    def mgs(self, V, k, w):
        """Modified Gram-Schmidt of w against V[0..k): returns (h[0..k), ||w|| after, ||w|| before)."""
        return self.mgs_batch([(V, k, w)])[0]

    def mgs_batch(self, items):
        """The same for several systems that are at the same Arnoldi column k: items = [(V, k, w), ...].  Distributed
        vectors: the coefficients stay on the device (dot -> all-reduce -> fused axpy + next dot), ONE all-reduce per
        column for all systems (R x 16 bytes) instead of one per system, and one copy to the host at the end."""
        R = len(items)
        k = items[0][1]
        assert all(it[1] == k for it in items)
        if self.group is None:
            if R == 1:
                V, _, w = items[0]
                _lib.check(self.lib.hp_mgs(self.nloc, k, _ptr(V), V.stride(0), _ptr(w), _ptr(self.scal), _stream()), "hp_mgs")
                h = self._host(self.scal[:k + 2])
                return [(h[:k].copy(), float(h[k].real), float(h[k + 1].real))]
            sc = self._batch_scal(k + 2, R)                  # system i uses column i ... stored row-wise per system below
            flat = sc.view(-1)
            for i, (V, _, w) in enumerate(items):           # hp_mgs writes k + 2 consecutive scalars per system
                _lib.check(self.lib.hp_mgs(self.nloc, k, _ptr(V), V.stride(0), _ptr(w), _ptr(flat[i * (k + 2):]), _stream()), "hp_mgs")
            h = self._host(flat[:R * (k + 2)]).reshape(R, k + 2)
            return [(h[i, :k].copy(), float(h[i, k].real), float(h[i, k + 1].real)) for i in range(R)]
        lib, n = self.lib, self.nloc
        if self.orth == "cgs2" and k <= 20:
            return self._cgs2_batch(items)
        sc = self._batch_scal(k + 2, R)                      # sc[j][i]: coefficient j of system i; rows k, k+1: |w|^2 after, before
        for i, (V, _, w) in enumerate(items):
            _lib.check(lib.hp_dotc(n, _ptr(w), _ptr(w), _ptr(sc[k + 1, i:]), _stream()), "hp_dotc")
            if k > 0:
                _lib.check(lib.hp_dotc(n, _ptr(V[0]), _ptr(w), _ptr(sc[0, i:]), _stream()), "hp_dotc")
        for j in range(k):
            self._all_reduce(sc[j, :R])
            for i, (V, _, w) in enumerate(items):            # w -= h_j v_j and the next local dot in one pass
                nxt = _ptr(V[j + 1]) if j + 1 < k else 0
                _lib.check(lib.hp_mgs_step(n, _ptr(sc[j, i:]), _ptr(V[j]), _ptr(w), nxt, _ptr(sc[j + 1, i:]), _stream()), "hp_mgs_step")
        if k == 0:
            for i, (V, _, w) in enumerate(items):
                _lib.check(lib.hp_dotc(n, _ptr(w), _ptr(w), _ptr(sc[0, i:]), _stream()), "hp_dotc")
        self._all_reduce(sc[k:k + 2, :R].reshape(-1) if sc.shape[1] == R else sc[k:k + 2, :R].contiguous())
        h = self._host(sc[:k + 2, :R])
        return [(h[:k, i].copy(), math.sqrt(float(h[k, i].real)), math.sqrt(float(h[k + 1, i].real))) for i in range(R)]

    def _cgs2_batch(self, items):
        """mgs_batch for distributed vectors with classical Gram-Schmidt applied twice: per pass one launch per 8 systems
        and ONE all-reduce of (k + 1) numbers per system for all of them"""
        import ctypes as C
        k, R = items[0][1], len(items)
        m = k + 1                                            # pass p, system i: D[p, i * m : (i + 1) * m] = k coefficients, |w|^2
        if self.cgs is None or self.cgs.shape[1] < R * 21:
            self.cgs = torch.zeros((3, max(R, 8) * 21), dtype=torch.complex128, device=self.device)
        D = self.cgs
        arr = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])                        # noqa: E731
        ldv = items[0][0].stride(0)
        for p, (upd, dots) in enumerate(((0, 1), (1, 1), (1, 0))):
            for i0 in range(0, R, 8):
                idx = range(i0, min(R, i0 + 8))
                coef = arr([D[p - 1, i * m:] for i in idx]) if upd else None
                _lib.check(self.lib.hp_cgs_pass(len(idx), self.nloc, k, arr([items[i][0] for i in idx]), ldv, arr([items[i][2] for i in idx]),
                                                coef, arr([D[p, i * m:] for i in idx]), upd, dots, _stream()), "hp_cgs_pass")
            self._all_reduce(D[p, :R * m])
        h = self._host(D[:, :R * m]).reshape(3, R, m)
        return [((h[0, i, :k] + h[1, i, :k]).copy(), math.sqrt(float(h[2, i, k].real)), math.sqrt(float(h[0, i, k].real))) for i in range(R)]

    def combine(self, V, y, x):
        """x += sum_j y[j] V[j]."""
        y = np.ascontiguousarray(np.asarray(y, dtype=np.complex128))
        _lib.check(self.lib.hp_combine(self.nloc, len(y), _ptr(V), V.stride(0), y.ctypes.data, _ptr(x), _stream()),
                   "hp_combine")


def _serve(req, matvec, psolve, vec):
    kind = req[0]
    if kind == "M":
        psolve(req[1], req[2])
    elif kind == "A":
        matvec(req[1], req[2])
    elif kind == "norm":
        return vec.norm(req[1])
    elif kind == "mgs":
        return vec.mgs(req[1], req[2], req[3])
    return None


def gmres(matvec, psolve, b, *, vec, rtol=1e-5, atol=0.0, restart=20, maxiter=None, callback=None, nglobal=None,
          health=None):
    """scipy.sparse.linalg.gmres(A, b, M=M, rtol=..., restart=..., maxiter=..., callback=...) on device vectors.

    matvec(x, out), psolve(x, out): device operators writing into `out`.  b: device vector (local slab).
    Returns (x, info, hist): hist holds what scipy hands to the legacy callback, one entry per inner iteration.
    """
    gen = gmres_steps(b, vec=vec, rtol=rtol, atol=atol, restart=restart, maxiter=maxiter, callback=callback,
                      nglobal=nglobal, health=health)
    try:
        req = next(gen)
        while True:
            req = gen.send(_serve(req, matvec, psolve, vec))
    except StopIteration as done:
        return done.value


def gmres_batch(matvec, psolve_batch, bs, *, vec, matvec_batch=None, with_index=False, **kw):
    """The same iteration for several right-hand sides advanced in lock step.  Every round collects the pending request of
    each unfinished system and serves them together: preconditioner requests go to psolve_batch as a list (one
    multi-right-hand-side sweep on one GPU; pipelined through the slabs in slab.py), operator requests to matvec_batch
    (halo rows of all systems in one exchange), norms and Gram-Schmidt steps to the batched reductions of DeviceVectors
    (one all-reduce per Arnoldi column for all systems).  Returns [(x, info, hist), ...] in the order of `bs`.
    with_index=True: psolve_batch receives (i, x, out) triples, i the index of the system in `bs` (a caller can then
    keep every system in its own slot of the sweep launch); default: (x, out) pairs."""
    gens = [gmres_steps(b, vec=vec, **kw) for b in bs]
    results = [None] * len(bs)
    reqs = {}

    def advance(i, value=None, first=False):
        try:
            reqs[i] = next(gens[i]) if first else gens[i].send(value)
        except StopIteration as done:
            results[i] = done.value
            reqs.pop(i, None)

    for i in range(len(gens)):
        advance(i, first=True)
    while reqs:
        by_kind = {}
        for i in sorted(reqs):
            key = reqs[i][0] if reqs[i][0] != "mgs" else ("mgs", reqs[i][2])
            by_kind.setdefault(key, []).append(i)
        key, idx = next(iter(by_kind.items()))              # lock step: normally a single kind per round
        kind = key if isinstance(key, str) else key[0]
        if _TRACE:
            import sys
            import threading
            print(f"[gmres_batch {threading.current_thread().name}] {key} x{len(idx)}", file=sys.stderr, flush=True)
        if kind == "M":
            psolve_batch([(i, reqs[i][1], reqs[i][2]) if with_index else (reqs[i][1], reqs[i][2]) for i in idx])
            vals = [None] * len(idx)
        elif kind == "A":
            if matvec_batch is not None:
                matvec_batch([(reqs[i][1], reqs[i][2]) for i in idx])
            else:
                for i in idx:
                    matvec(reqs[i][1], reqs[i][2])
            vals = [None] * len(idx)
        elif kind == "norm":
            vals = vec.norm_batch([reqs[i][1] for i in idx])
        else:
            vals = vec.mgs_batch([(reqs[i][1], reqs[i][2], reqs[i][3]) for i in idx])
        for i, v in zip(idx, vals):
            advance(i, v)
    return results


def gmres_steps(b, *, vec, rtol=1e-5, atol=0.0, restart=20, maxiter=None, callback=None, nglobal=None, health=None):
    """Generator form of gmres().  Yields a request whenever something outside the local vector arithmetic is needed
    and receives its result through send():
        ("M", x, out)  out = M x          ("A", x, out)  out = A x
        ("norm", x) -> ||x||              ("mgs", V, k, w) -> (h[0..k), ||w|| after, ||w|| before)
    so that a driver can serve the requests of several systems together (gmres_batch).  Returns (x, info, hist)
    through StopIteration.  health(): called at every restart boundary (the host is in sync with the device there
    anyway); raises if a kernel of the operators reported a fault."""
    nloc = b.numel()
    n = nglobal if nglobal is not None else nloc
    dev = b.device
    x = torch.zeros_like(b)
    hist = []
    bnrm2 = yield ("norm", b)
    if bnrm2 == 0:
        return x, 0, hist
    atol = max(float(atol), float(rtol) * bnrm2)
    eps = np.finfo(np.float64).eps
    if maxiter is None:
        maxiter = n * 10
    restart = min(restart, n)
    vec.reserve(restart)
    V = torch.empty((restart + 1, nloc), dtype=torch.complex128, device=dev)
    r = torch.empty_like(b)
    av = torch.empty_like(b)
    w = torch.empty_like(b)
    yield ("M", b, w)
    Mb_nrm2 = yield ("norm", w)
    ptol_max_factor = 1.0
    ptol = Mb_nrm2 * min(ptol_max_factor, atol / bnrm2)
    presid = 0.0
    hh = np.zeros((restart, restart + 1), dtype=np.complex128)
    givens = np.zeros((restart, 2), dtype=np.complex128)
    inner_iter = 0
    rnorm = math.inf
    for iteration in range(maxiter):
        if iteration == 0:
            vec.scale_copy(1.0, b, r)
            if bnrm2 < atol:
                return x, 0, hist
        yield ("M", r, V[0])
        tmp = yield ("norm", V[0])
        vec.scale_copy(1.0 / tmp, V[0], V[0])
        S = np.zeros(restart + 1, dtype=np.complex128)
        S[0] = tmp
        breakdown = False
        col = 0
        for col in range(restart):
            yield ("A", V[col], av)
            yield ("M", av, w)
            hcol, h1, h0 = yield ("mgs", V, col + 1, w)
            hh[col, :col + 1] = hcol
            hh[col, col + 1] = h1
            if h1 <= eps * h0:
                hh[col, col + 1] = 0
                breakdown = True
                vec.scale_copy(1.0, w, V[col + 1])
            else:
                vec.scale_copy(1.0 / h1, w, V[col + 1])
            for k in range(col):
                c, s = givens[k, 0], givens[k, 1]
                n0, n1 = hh[col, k], hh[col, k + 1]
                hh[col, k], hh[col, k + 1] = c * n0 + s * n1, -np.conj(s) * n0 + c * n1
            c, s, mag = lartg(hh[col, col], hh[col, col + 1])
            givens[col, :] = [c, s]
            hh[col, col], hh[col, col + 1] = mag, 0
            tmp = -np.conjugate(s) * S[col]
            S[col], S[col + 1] = c * S[col], tmp
            presid = abs(tmp)
            inner_iter += 1
            hist.append(presid / bnrm2)
            if callback is not None:
                callback(presid / bnrm2)
            if inner_iter == maxiter:
                break
            if presid <= ptol or breakdown:
                break
        if hh[col, col] == 0:
            S[col] = 0
        y = np.zeros(col + 1, dtype=np.complex128)
        y[:] = S[:col + 1]
        for k in range(col, 0, -1):
            if y[k] != 0:
                y[k] /= hh[k, k]
                tmp = y[k]
                y[:k] -= tmp * hh[k, :k]
        if y[0] != 0:
            y[0] /= hh[0, 0]
        vec.combine(V, y, x)
        yield ("A", x, av)
        vec.scale_copy(-1.0, av, r)
        vec.axpy(1.0, b, r)
        rnorm = yield ("norm", r)
        if health is not None:
            health()
        if inner_iter == maxiter:
            return x, (0 if rnorm <= atol else maxiter), hist
        if rnorm <= atol:
            break
        elif breakdown:
            break
        elif presid <= ptol:
            ptol_max_factor = max(eps, 0.25 * ptol_max_factor)
        else:
            ptol_max_factor = min(1.0, 1.5 * ptol_max_factor)
        ptol = presid * min(ptol_max_factor, atol / rnorm)
    info = 0 if rnorm <= atol else maxiter
    return x, info, hist
