"""Host-side mirror of the reference's entry points (/root/reference/code.py) over libhelmholtz_b200.so.

Same names, argument order and meaning as the reference for the hot path:

    build_A_matrix(b, const, eta, omega, h, n, c_mat)          code.py:202-219   -> DeviceCSR
    algo2_3(b, const, eta, omega, h, n, c_mat)                 code.py:345-353   -> (front, strips) handles
    algo2_4(f_vec, b, n, lu_HF, ..., lu_Hm_ra)                 code.py:356-385   -> M f
    run_solver(n, b, wave_num, const, alpha, init_func, ...)   code.py:424-541   -> SolveResult

PyTorch is used for device buffers and streams only; every n^2-sized operation is a kernel of the library.
There is no CPU path: without the library or a CUDA device these functions raise.
"""
import ctypes as C
import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib, fields
from .gmres import DeviceVectors, gmres, gmres_batch

DIAG_MODES = {"reference": 0, "paper": 1}
LAYOUT_MODES = {"auto": 0, "classic": 1, "cluster": 2}
FRONT_MODES = {"blockdiag": 0, "coupled": 1}
HP_RMAX = 8                       # right-hand sides of the widest sweep launch (csrc/hp_sweep_common.cuh)


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _as_device_field(x, device):
    """complex128 contiguous device tensor from numpy / torch input (host->device copy if needed)."""
    if isinstance(x, torch.Tensor):
        return x.to(device=device, dtype=torch.complex128).contiguous().reshape(-1)
    a = np.ascontiguousarray(np.asarray(x, dtype=np.complex128)).reshape(-1)
    return torch.from_numpy(a).to(device)


def _is_complex_medium(c_mat):
    """True for a velocity model of complex dtype (an attenuating medium), judged by the dtype alone."""
    if isinstance(c_mat, torch.Tensor):
        return c_mat.is_complex()
    return np.iscomplexobj(c_mat)


class HelmholtzSolver:
    """One problem instance on one device: owns the hp_solver handle (tables, velocity, factorisation).

    Arguments are the reference's: n interior points per side, b PML width in points, omega complex angular
    frequency (2*pi*wave_num + 1j*alpha, code.py:442), const the PML strength, c_mat the (n+2)^2 velocity.
    A c_mat of complex dtype (numpy, or a torch tensor on the host or the device) is an attenuating medium
    (hp_create_complex, see fields.attenuate); a real dtype gives the lossless path."""

    def __init__(self, n, b, omega, const, c_mat, device=None):
        cplx_medium = _is_complex_medium(c_mat)
        if cplx_medium and tuple(c_mat.shape) != (n + 2, n + 2):
            raise ValueError(f"c_mat must be ({n + 2}, {n + 2}) like the reference's init_c*_mat, got {tuple(c_mat.shape)}")
        self.lib = _lib.require_device()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        if self.device.index is None:
            self.device = torch.device(f"cuda:{torch.cuda.current_device()}")
        self.n, self.b, self.omega, self.const = int(n), int(b), complex(omega), float(const)
        self.h = 1 / (n + 1)
        self.eta = b * self.h
        create = self.lib.hp_create
        if cplx_medium:
            create = self.lib.hp_create_complex
            if isinstance(c_mat, torch.Tensor) and c_mat.is_cuda:
                c_dev = c_mat.to(dtype=torch.complex128).contiguous()
                cptr, on_dev = c_dev.data_ptr(), 1
            else:
                c_np = c_mat.detach().resolve_conj().numpy() if isinstance(c_mat, torch.Tensor) else c_mat
                c_host = np.ascontiguousarray(np.asarray(c_np, dtype=np.complex128))
                cptr, on_dev = c_host.ctypes.data, 0
        elif isinstance(c_mat, torch.Tensor) and c_mat.is_cuda:
            c_dev = c_mat.to(dtype=torch.float64).contiguous()
            cptr, on_dev = c_dev.data_ptr(), 1
        else:
            c_host = np.ascontiguousarray(np.asarray(c_mat, dtype=np.float64))
            cptr, on_dev = c_host.ctypes.data, 0
        shape = tuple(c_mat.shape)
        if shape != (n + 2, n + 2):
            raise ValueError(f"c_mat must be ({n + 2}, {n + 2}) like the reference's init_c*_mat, got {shape}")
        h = C.c_void_p()
        what = "hp_create_complex" if cplx_medium else "hp_create"
        with torch.cuda.device(self.device):
            _lib.check(create(C.byref(h), self.n, self.b, self.omega.real, self.omega.imag, self.const,
                              cptr, on_dev, _stream()), what)
        self.handle = h
        self.m_lo, self.m_hi = 0, -1
        self.max_group = 8            # cap on the right-hand sides per sweep launch (1 = one launch per vector)

    @property
    def medium_is_complex(self):
        """True when the solver holds an attenuating (complex) medium, made from a c_mat of complex dtype."""
        return bool(self.lib.hp_medium_is_complex(self.handle))

    def clone_context(self):
        """A second handle on this solver's operator and factorisation with private sweep scratch (hp_context_clone):
        preconditioner applications issued through different contexts may be in flight on different CUDA streams at the
        same time (one context per group of right-hand sides in slab.GroupPipeline).  Close the contexts before the
        solver they were cloned from."""
        self._on_device()
        c = object.__new__(HelmholtzSolver)
        c.__dict__.update(self.__dict__)
        h = C.c_void_p()
        _lib.check(self.lib.hp_context_clone(self.handle, C.byref(h), _stream()), "hp_context_clone")
        c.handle = h
        c.parent = self                                      # keeps the owner of the factorisation alive
        return c

    def close(self):
        if getattr(self, "handle", None):
            self.lib.hp_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- operator -------------------------------------------------------------------------------------
    def assemble_csr(self):
        """build_A_matrix: sorted CSR on the device (int32 indices, complex128 values)."""
        self._on_device()
        n = self.n
        N = n * n
        nnz = self.lib.hp_csr_nnz(n)
        indptr = torch.empty(N + 1, dtype=torch.int32, device=self.device)
        indices = torch.empty(nnz, dtype=torch.int32, device=self.device)
        data = torch.empty(nnz, dtype=torch.complex128, device=self.device)
        _lib.check(self.lib.hp_assemble_csr(self.handle, _ptr(indptr), _ptr(indices), _ptr(data), _stream()),
                   "hp_assemble_csr")
        return DeviceCSR(self, indptr, indices, data)

    def assemble_strip_csr(self, m):
        """get_Hm(m): the strip operator of layer m as sorted CSR on the device (code.py:283-290)."""
        self._on_device()
        n, b = self.n, self.b
        nnz = self.lib.hp_strip_csr_nnz(n, b)
        indptr = torch.empty(b * n + 1, dtype=torch.int32, device=self.device)
        indices = torch.empty(nnz, dtype=torch.int32, device=self.device)
        data = torch.empty(nnz, dtype=torch.complex128, device=self.device)
        _lib.check(self.lib.hp_assemble_strip_csr(self.handle, int(m), _ptr(indptr), _ptr(indices), _ptr(data), _stream()),
                   "hp_assemble_strip_csr")
        return DeviceCSR(self, indptr, indices, data, shape=(b * n, b * n))

    def matvec(self, x, out=None):
        """y = A x, matrix free."""
        self._on_device()
        if out is None:
            out = torch.empty_like(x)
        _lib.check(self.lib.hp_stencil_matvec(self.handle, _ptr(x), _ptr(out), _stream()), "hp_stencil_matvec")
        return out

    def matvec_rows(self, j_lo, j_hi, x, south, north, out):
        _lib.check(self.lib.hp_stencil_matvec_rows(self.handle, j_lo, j_hi, _ptr(x), _ptr(south), _ptr(north),
                                                   _ptr(out), _stream()), "hp_stencil_matvec_rows")
        return out

    # ---- preconditioner -------------------------------------------------------------------------------
    def setup_preconditioner(self, P=0, K=0, m_lo=0, m_hi=0, layout="auto", front="blockdiag"):
        """algo2_3.  (m_lo, m_hi) = (0, 0): all strips b+1..n; otherwise the strips of this rank's slab.
        layout: "auto" (cluster when a partition exists), "classic", "cluster" (include/helmholtz_b200.h).
        front: "blockdiag" = the reference's H_F (code.py:178-183, only the diagonal blocks), "coupled" = the full
        A[:bn, :bn] of the paper (2-5 GMRES iterations instead of 70-200 with diag='paper')."""
        self._on_device()
        _lib.check(self.lib.hp_set_front_mode(self.handle, FRONT_MODES[front]), "hp_set_front_mode")
        self.front = front
        _lib.check(self.lib.hp_set_layout_mode(self.handle, LAYOUT_MODES[layout]), "hp_set_layout_mode")
        _lib.check(self.lib.hp_precond_setup(self.handle, P, K, m_lo, m_hi, _stream()), "hp_precond_setup")
        if m_lo == 0 and m_hi == 0:
            m_lo, m_hi = self.b + 1, self.n
        self.m_lo, self.m_hi = m_lo, m_hi
        return self

    def set_front(self, front):
        """switch the front block of a solver that is set up ("blockdiag" | "coupled"); the strips are kept"""
        self._on_device()
        _lib.check(self.lib.hp_precond_set_front(self.handle, FRONT_MODES[front], _stream()), "hp_precond_set_front")
        self.front = front
        return self

    def set_sweep_variant(self, variant):
        """0 = automatic; classic layout: 1 direct, 2 TMA staged, 3 pipelined; cluster layout: 4."""
        _lib.check(self.lib.hp_set_sweep_variant(self.handle, int(variant)), "hp_set_sweep_variant")
        return self

    def sweep_status(self):
        """0 = fine (synchronises the device)."""
        return int(self.lib.hp_sweep_status(self.handle))

    def check_status(self):
        """Raise if a sweep kernel gave up waiting for another CTA since the setup (its output is then garbage).
        Synchronises the device; called where the host waits for the device anyway (GMRES restart boundaries, the end
        of run_solver, algo2_4)."""
        st = self.sweep_status()
        if st:
            raise _lib.HelmholtzB200Error(
                f"sweep kernel fault (status {st}): a CTA timed out waiting for exchange data; results since the last "
                "setup_preconditioner() are invalid")

    def _on_device(self):
        """every call runs on the current device and stream: refuse a solver that lives elsewhere"""
        if torch.cuda.current_device() != self.device.index:
            raise _lib.HelmholtzB200Error(
                f"solver lives on {self.device}, current device is cuda:{torch.cuda.current_device()} "
                "(wrap the call in torch.cuda.device(solver.device))")

    @property
    def precond_bytes(self):
        return int(self.lib.hp_precond_bytes(self.handle))

    @property
    def setup_ms(self):
        return float(self.lib.hp_precond_setup_ms(self.handle))

    def layout(self):
        P, K, QP, CW, NS, NR = (C.c_int() for _ in range(6))
        PK = C.c_int64()
        _lib.check(self.lib.hp_strip_layout(self.handle, C.byref(P), C.byref(K), C.byref(QP), C.byref(CW), C.byref(NS),
                                            C.byref(NR), C.byref(PK), None, None, None), "hp_strip_layout")
        ls = (C.c_int * P.value)()
        lq = (C.c_int * P.value)()
        sp = (C.c_int * max(P.value - 1, 1))()
        _lib.check(self.lib.hp_strip_layout(self.handle, None, None, None, None, None, None, None, ls, lq, sp),
                   "hp_strip_layout")
        colN, NCB, NRQ, NXG = (C.c_int() for _ in range(4))
        _lib.check(self.lib.hp_strip_layout_ex(self.handle, C.byref(colN), C.byref(NCB), C.byref(NRQ), C.byref(NXG)),
                   "hp_strip_layout_ex")
        return dict(P=P.value, K=K.value, G=P.value * K.value, QP=QP.value, CW=CW.value, NS=NS.value, NR=NR.value,
                    PK=PK.value, leaf_start=np.array(ls[:]), q=np.array(lq[:]), sep=np.array(sp[:P.value - 1]),
                    colN=colN.value, NCB=NCB.value, NRQ=NRQ.value, NXG=NXG.value)

    def strip_packets(self, m):
        L = self.layout()
        out = np.zeros((L["G"], L["PK"]), dtype=np.complex128)
        _lib.check(self.lib.hp_strip_packets(self.handle, m, out.ctypes.data), "hp_strip_packets")
        return L, out

    def strip_apply(self, m, v, out=None):
        """T_m v: last n entries of H_m^{-1} [0; v]  (code.py:368-370)."""
        self._on_device()
        if out is None:
            out = torch.empty_like(v)
        _lib.check(self.lib.hp_strip_apply(self.handle, m, _ptr(v), _ptr(out), _stream()), "hp_strip_apply")
        return out

    def precond_apply(self, f, out=None, diag="reference"):
        """algo2_4: out = M f."""
        self._on_device()
        if out is None:
            out = torch.empty_like(f)
        _lib.check(self.lib.hp_precond_apply(self.handle, _ptr(f), _ptr(out), DIAG_MODES[diag], _stream()),
                   "hp_precond_apply")
        return out

    @property
    def multi_max(self):
        """right-hand sides one sweep launch can carry with the partition in use (1, 2, 4 or 8)"""
        return int(self.lib.hp_multi_max(self.handle))

    def batch_group(self, R):
        """right-hand sides one sweep launch carries when R are in flight"""
        g = 1
        while g * 2 <= min(R, self.multi_max, self.max_group):
            g *= 2
        return g

    def multi_kernel(self, R):
        """sweep kernel of one launch carrying R right-hand sides: 2 = hp_sweep4d (tensor cores, R = 8), 1 = hp_sweep4m,
        0 = none (this layout cannot carry R per launch)"""
        return int(self.lib.hp_multi_kernel(self.handle, int(R)))

    def batch_kernel_name(self, R):
        g = self.batch_group(R)
        if g > 1:
            return "hp_sweep4d_kernel (FP64 tensor cores, 8 right-hand sides)" if self.multi_kernel(g) == 2 else "hp_sweep4m_kernel"
        return "hp_sweep4_kernel" if self.layout()["colN"] else "hp_sweep2_kernel"

    @staticmethod
    def _ptr_array(ts):
        return (C.c_void_p * len(ts))(*[0 if t is None else t.data_ptr() for t in ts])

    def precond_apply_multi(self, fs, outs, diag="reference"):
        """algo2_4 on R = len(fs) vectors with one pass over the strip generators per sweep (R in {1, 2, 4, 8}).
        fs[i] = outs[i] = None leaves slot i of the launch empty (masked)."""
        self._on_device()
        _lib.check(self.lib.hp_precond_apply_multi(self.handle, len(fs), self._ptr_array(fs), self._ptr_array(outs), DIAG_MODES[diag],
                                                   _stream()), "hp_precond_apply_multi")
        return outs

    def precond_apply_slots(self, slots, diag="reference"):
        """out = M x for every entry (x, out) of `slots` in ONE launch per sweep direction, entry i in slot i of the
        launch; None entries are empty slots.  len(slots) is the launch width (1, or a power of two the layout can carry,
        multi_kernel(len(slots)) != 0).  An active slot's result does not depend on what the other slots hold."""
        if len(slots) == 1:
            if slots[0] is None:
                raise _lib.HelmholtzB200Error("precond_apply_slots: the only slot of the launch is empty")
            self.precond_apply(slots[0][0], out=slots[0][1], diag=diag)
            return
        self.precond_apply_multi([None if p is None else p[0] for p in slots], [None if p is None else p[1] for p in slots],
                                 diag=diag)

    def _widest(self):
        """right-hand sides of the widest launch in use (multi_max, capped by max_group)"""
        return self.batch_group(HP_RMAX)

    def precond_apply_batch(self, pairs, diag="reference", pad=False):
        """out_i = M x_i for every (x_i, out_i) of `pairs`.  pad=False: in groups of batch_group() right-hand sides per
        launch (7 pairs: launches of 4 + 2 + 1).  pad=True: the widest launch takes min(remaining, widest) pairs and is
        padded with empty slots up to the smallest width that holds them and that the layout supports (7 pairs: one
        8-wide launch with one empty slot; 3 pairs: one 4-wide launch)."""
        i = 0
        if pad:
            cap = self._widest()
            while i < len(pairs):
                take = min(len(pairs) - i, cap)
                w = 1
                while w < take or (w > 1 and w < cap and not self.multi_kernel(w)):
                    w *= 2
                self.precond_apply_slots(list(pairs[i:i + take]) + [None] * (w - take), diag=diag)
                i += take
            return
        while i < len(pairs):
            g = self.batch_group(len(pairs) - i)
            if g == 1:
                self.precond_apply(pairs[i][0], out=pairs[i][1], diag=diag)
            else:
                self.precond_apply_multi([p[0] for p in pairs[i:i + g]], [p[1] for p in pairs[i:i + g]], diag=diag)
            i += g

    def sweep_forward_multi_buf(self, bufs, row0, m_from, m_to):
        """one multi-vector forward sweep over strips m_from..m_to; a None entry is an empty slot"""
        arr = (C.c_void_p * len(bufs))(*[0 if t is None else self._base(t, row0) for t in bufs])
        _lib.check(self.lib.hp_sweep_forward_multi(self.handle, len(bufs), arr, m_from, m_to, _stream()), "hp_sweep_forward_multi")

    def sweep_backward_multi_buf(self, bufs, row0, m_from, m_to, diag="reference"):
        arr = (C.c_void_p * len(bufs))(*[0 if t is None else self._base(t, row0) for t in bufs])
        _lib.check(self.lib.hp_sweep_backward_multi(self.handle, len(bufs), arr, m_from, m_to, DIAG_MODES[diag], _stream()),
                   "hp_sweep_backward_multi")

    # staged calls on a slab buffer whose first row is global row `row0` (slab decomposition, slab.py): the
    # kernels index the field by absolute row, so they get the address global row 0 would have
    def _base(self, buf, row0):
        return buf.data_ptr() - row0 * self.n * 16

    def front_begin_buf(self, buf, row0):
        _lib.check(self.lib.hp_front_begin(self.handle, self._base(buf, row0), _stream()), "hp_front_begin")

    def front_end_buf(self, buf, row0):
        _lib.check(self.lib.hp_front_end(self.handle, self._base(buf, row0), _stream()), "hp_front_end")

    def front_tf_new(self):
        """buffer that can park T_F u_F of one right-hand side (front_tf_save / front_tf_load)"""
        return torch.empty(self.b * self.n, dtype=torch.complex128, device=self.device)

    def front_tf_save(self, t):
        _lib.check(self.lib.hp_front_tf_copy(self.handle, _ptr(t), 0, _stream()), "hp_front_tf_copy")

    def front_tf_load(self, t):
        _lib.check(self.lib.hp_front_tf_copy(self.handle, _ptr(t), 1, _stream()), "hp_front_tf_copy")

    def sweep_forward_buf(self, buf, row0, m_from, m_to):
        _lib.check(self.lib.hp_sweep_forward(self.handle, self._base(buf, row0), m_from, m_to, _stream()), "hp_sweep_forward")

    def sweep_backward_buf(self, buf, row0, m_from, m_to, diag="reference"):
        _lib.check(self.lib.hp_sweep_backward(self.handle, self._base(buf, row0), m_from, m_to, DIAG_MODES[diag], _stream()),
                   "hp_sweep_backward")

    # staged calls (slab decomposition)
    def front_begin(self, u):
        _lib.check(self.lib.hp_front_begin(self.handle, _ptr(u), _stream()), "hp_front_begin")

    def front_end(self, u):
        _lib.check(self.lib.hp_front_end(self.handle, _ptr(u), _stream()), "hp_front_end")

    def sweep_forward(self, u, m_from, m_to):
        _lib.check(self.lib.hp_sweep_forward(self.handle, _ptr(u), m_from, m_to, _stream()), "hp_sweep_forward")

    def sweep_backward(self, u, m_from, m_to, diag="reference"):
        _lib.check(self.lib.hp_sweep_backward(self.handle, _ptr(u), m_from, m_to, DIAG_MODES[diag], _stream()),
                   "hp_sweep_backward")


class DeviceCSR:
    """What build_A_matrix returns: the operator as sorted CSR arrays in device memory."""

    def __init__(self, solver, indptr, indices, data, shape=None):
        self.solver, self.indptr, self.indices, self.data = solver, indptr, indices, data
        self.shape = shape if shape is not None else (solver.n ** 2, solver.n ** 2)

    def matvec(self, x, out=None):
        x = _as_device_field(x, self.solver.device)
        if out is None:
            out = torch.empty_like(x)
        _lib.check(self.solver.lib.hp_csr_matvec(self.shape[0], _ptr(self.indptr), _ptr(self.indices), _ptr(self.data),
                                                 _ptr(x), _ptr(out), _stream()), "hp_csr_matvec")
        return out

    __matmul__ = matvec

    def to_host(self):
        """(indptr, indices, data) as numpy arrays (scipy.sparse.csr_matrix takes them as is)."""
        return self.indptr.cpu().numpy(), self.indices.cpu().numpy(), self.data.cpu().numpy()


# ------------------------------------------------------------------------------------------------------
# reference-named functions
# ------------------------------------------------------------------------------------------------------
def _solver_for(b, const, eta, omega, h, n, c_mat, device=None):
    if abs(h - 1 / (n + 1)) > 1e-15 or abs(eta - b * h) > 1e-15:
        raise ValueError("h and eta must be 1/(n+1) and b*h as in the reference (code.py:443-444)")
    return HelmholtzSolver(n, b, omega, const, c_mat, device=device)


def build_A_matrix(b, const, eta, omega, h, n, c_mat, device=None):
    """code.py:202-219."""
    return _solver_for(b, const, eta, omega, h, n, c_mat, device).assemble_csr()


def get_Hm(m, b, const, eta, omega, h, n, c_mat, device=None):
    """code.py:283-290: the strip operator of layer m (DeviceCSR, bn x bn)."""
    return _solver_for(b, const, eta, omega, h, n, c_mat, device).assemble_strip_csr(m)


def get_A_FF_block(b, const, eta, omega, h, n, c_mat, device=None, coupled=False):
    """code.py:178-183.  The reference keeps only the diagonal blocks (b tridiagonal systems); coupled=True is the full
    A[:bn, :bn] = get_Hm(b).  Returned as DeviceCSR; the block-diagonal form drops the couplings between the rows."""
    A = _solver_for(b, const, eta, omega, h, n, c_mat, device).assemble_strip_csr(b)
    if coupled:
        return A
    indptr, indices, data = A.to_host()
    rows = np.repeat(np.arange(b * n), np.diff(indptr))
    keep = np.abs(indices - rows) <= 1                              # code.py:180-182: block_diag of the A_ii
    ip = np.zeros(b * n + 1, dtype=np.int32)
    np.cumsum(np.bincount(rows[keep], minlength=b * n), out=ip[1:])
    dev = A.solver.device
    return DeviceCSR(A.solver, torch.from_numpy(ip).to(dev), torch.from_numpy(indices[keep]).to(dev),
                     torch.from_numpy(data[keep]).to(dev), shape=A.shape)


def algo2_3(b, const, eta, omega, h, n, c_mat, device=None, P=0, K=0, layout="auto", front="blockdiag"):
    """code.py:345-353.  Returns (lu_HF, lu_Hm_ra): both are the same factorisation handle here."""
    s = _solver_for(b, const, eta, omega, h, n, c_mat, device).setup_preconditioner(P, K, layout=layout, front=front)
    return s, s


def algo2_4(f_vec, b, n, lu_HF, A_b1F=None, A_Fb1=None, up_A_ra=None, lo_A_ra=None, lu_Hm_ra=None, diag="reference"):
    """code.py:356-385.  The coupling blocks A_b1F, A_Fb1, up_A_ra, lo_A_ra of the reference signature are
    implied by the solver handle and ignored.  Returns M f as an (n, n) device tensor like the reference's u."""
    s = lu_HF
    f = _as_device_field(f_vec, s.device)
    u = s.precond_apply(f, diag=diag).reshape(n, n)
    s.check_status()
    return u


@dataclass
class SolveResult:
    u: torch.Tensor                 # solution field, (n*n,) complex128 on the device (reference: u)
    residuals: list                 # what scipy hands to the callback, one per inner iteration
    niter: int                      # counter_prec.niter of the reference
    info: int                       # exit_code of scipy gmres
    init_time: float                # "Initialization time" (code.py:522)
    solve_time: float               # "GMRES solve time"    (code.py:523)
    solver: object = field(default=None, repr=False)

    def __iter__(self):             # the reference returns (init_time_length, solve_time_length)
        return iter((self.init_time, self.solve_time))


def run_solver(n, b, wave_num, const, alpha, init_func=fields.init_c1_f1, plot_solution=False, *, c_mat=None,
               f_mat=None, diag="reference", precond_input="rhs", front="blockdiag", rtol=1e-3, restart=20, maxiter=None,
               device=None, P=0, K=0, verbose=True, solver=None):
    """code.py:424-541 (the preconditioned solve; plotting is not part of this package).

    precond_input='rhs' is the reference as written: its LinearOperator ignores the vector it is given and
    always returns algo2_4(f_vec) (code.py:510-511).  'vector' applies the preconditioner to the argument.
    diag='reference' keeps u_m <- u_m - T_m u_m (code.py:372-375); 'paper' is Engquist-Ying's u_m <- T_m u_m.
    front='blockdiag' is the reference's H_F (code.py:178-183); 'coupled' keeps the couplings between its rows.
    The reference as written (rhs / reference / blockdiag) does not converge (info != 0); vector / paper converges,
    with front='coupled' in a handful of iterations.  A solver passed in keeps the front block it was set up with.
    """
    lib = _lib.require_device()   # noqa: F841  (fail before any host work if the device path is missing)
    t0 = time.time()
    omega = 2 * np.pi * wave_num + 1j * alpha          # code.py:442
    if c_mat is None or f_mat is None:
        c0, f0 = init_func(omega, n)
        c_mat = c0 if c_mat is None else c_mat
        f_mat = f0 if f_mat is None else f_mat
    s = solver if solver is not None else HelmholtzSolver(n, b, omega, const, c_mat, device=device)
    f = _as_device_field(f_mat, s.device)                # f_mat.flatten(), code.py:448
    if solver is None:
        s.setup_preconditioner(P, K, front=front)        # algo2_3, code.py:496
    torch.cuda.synchronize(s.device)
    t1 = time.time()
    vec = DeviceVectors(n * n, s.device, restart=restart)
    Mf = None
    if precond_input == "rhs":
        Mf = s.precond_apply(f, diag=diag)

        def psolve(x, out):
            # code.py:510-511: matvec=lambda x: algo2_4(f_vec, ...) -- the argument is ignored; algo2_4 is
            # deterministic, so its result is computed once and copied
            vec.scale_copy(1.0, Mf, out)
    elif precond_input == "vector":
        def psolve(x, out):
            s.precond_apply(x, out=out, diag=diag)
    else:
        raise ValueError("precond_input must be 'rhs' or 'vector'")
    u, info, hist = gmres(lambda x, out: s.matvec(x, out), psolve, f, vec=vec, rtol=rtol, restart=restart,
                          maxiter=maxiter, health=s.check_status)
    s.check_status()
    t2 = time.time()
    if verbose:
        print("GMRES iterations with preconditioner: " + str(len(hist)))      # code.py:520
        print("Initialization time = " + str(t1 - t0))
        print("GMRES solve time = " + str(t2 - t1))
    return SolveResult(u, hist, len(hist), info, t1 - t0, t2 - t1, s)


def _source_fields(f_mats, n, device):
    """(S, n, n) / (S, n*n) array or tensor, or a list of (n, n) / (n*n,) fields -> list of (n*n,) device tensors"""
    items = list(f_mats) if isinstance(f_mats, (list, tuple)) else [f_mats[i] for i in range(f_mats.shape[0])]
    fs = [_as_device_field(f, device) for f in items]
    for i, f in enumerate(fs):
        if f.numel() != n * n:
            raise ValueError(f"source {i} has {f.numel()} entries, expected n*n = {n * n}")
    return fs


def _solve_wave(s, wave, W, vec, diag, precond_input, rtol, restart, maxiter):
    """One wave of at most W = s._widest() sources (device fields) by batched GMRES, source i pinned to slot i of every
    sweep launch, converged or idle slots left empty.  Returns gmres_batch's [(u, info, hist)] after checking the sweep
    status.  Shared by run_solver_many and the inversion drivers (inversion.py)."""
    Mf = None
    if precond_input == "rhs":
        # as in run_solver, M f is computed once and copied: one launch for the whole wave
        Mf = [torch.empty_like(f) for f in wave]
        s.precond_apply_slots([(f, m) for f, m in zip(wave, Mf)] + [None] * (W - len(wave)), diag=diag)

    def psolve_batch(reqs):
        if Mf is not None:
            for i, _, out in reqs:
                vec.scale_copy(1.0, Mf[i], out)
            return
        slots = [None] * W
        for i, x, out in reqs:
            slots[i] = (x, out)
        s.precond_apply_slots(slots, diag=diag)

    outs = gmres_batch(lambda x, out: s.matvec(x, out), psolve_batch, wave, vec=vec, with_index=True, rtol=rtol,
                       restart=restart, maxiter=maxiter, health=s.check_status)
    s.check_status()
    return outs


def run_solver_many(n, b, wave_num, const, alpha, f_mats, init_func=fields.init_c1_f1, *, c_mat=None, diag="reference",
                    precond_input="rhs", front="blockdiag", rtol=1e-3, restart=20, maxiter=None, device=None, P=0, K=0,
                    verbose=True, solver=None):
    """run_solver for several sources (right-hand sides) of one medium: the solver is set up once, and the sources are
    solved in waves of as many as one sweep launch carries (multi_max; 1 = one source at a time).

    f_mats: (S, n, n) or (S, n*n) array or tensor, or a list of such fields.  c_mat defaults to init_func's.  The other
    arguments mean what they mean for run_solver.  Within a wave, source i always occupies slot i of the sweep launch;
    the slots of sources that have converged, or that do not ask for M x in a round, are left empty.  So every
    preconditioner round is one launch per sweep direction, and a source's result does not depend on which sources
    share its wave (bit for bit, given its slot).

    Returns one SolveResult per source in input order: init_time is the shared set-up time, solve_time the wall time of
    the source's wave; u, residuals, niter and info are the source's own."""
    _lib.require_device()
    t0 = time.time()
    omega = 2 * np.pi * wave_num + 1j * alpha
    if c_mat is None and solver is None:
        c_mat = init_func(omega, n)[0]
    s = solver if solver is not None else HelmholtzSolver(n, b, omega, const, c_mat, device=device)
    fs = _source_fields(f_mats, n, s.device)
    if solver is None:
        s.setup_preconditioner(P, K, front=front)
    if precond_input not in ("rhs", "vector"):
        raise ValueError("precond_input must be 'rhs' or 'vector'")
    torch.cuda.synchronize(s.device)
    t1 = time.time()
    W = s._widest()
    vec = DeviceVectors(n * n, s.device, restart=restart)
    results = []
    for w0 in range(0, len(fs), W):
        tw = time.time()
        outs = _solve_wave(s, fs[w0:w0 + W], W, vec, diag, precond_input, rtol, restart, maxiter)
        t_wave = time.time() - tw
        for j, (u, info, hist) in enumerate(outs):
            results.append(SolveResult(u, hist, len(hist), info, t1 - t0, t_wave, s))
            if verbose:
                print(f"source {w0 + j}: GMRES iterations with preconditioner: {len(hist)} (info {info})")
    if verbose:
        print("Initialization time = " + str(t1 - t0))
        print("GMRES solve time = " + str(time.time() - t1))
    return results
