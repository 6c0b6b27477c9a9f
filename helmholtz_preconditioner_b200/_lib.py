"""ctypes binding of libhelmholtz_b200.so (include/helmholtz_b200.h).

There is no CPU path: importing the package works anywhere (so that the host logic can be tested), but
every compute entry point raises if the library or a CUDA device is missing.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HELMHOLTZ_B200_LIB", os.path.join(HERE, "libhelmholtz_b200.so"))   # env override: developer builds

_vp, _i, _i64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_double
_ip = C.POINTER(C.c_int)

# name -> (restype, argtypes); mirrors include/helmholtz_b200.h one to one
SIGNATURES = {
    "hp_last_error": (C.c_char_p, []),
    "hp_version": (_i, []),
    "hp_device_ok": (_i, []),
    "hp_launch_count": (_i64, []),
    "hp_profile_enable": (_i, [_vp, _i]),
    "hp_profile_read": (_i, [_vp, C.POINTER(_d), _ip, C.POINTER(_i64)]),
    "hp_create": (_i, [C.POINTER(_vp), _i, _i, _d, _d, _d, _vp, _i, _vp]),
    "hp_create_complex": (_i, [C.POINTER(_vp), _i, _i, _d, _d, _d, _vp, _i, _vp]),
    "hp_medium_is_complex": (_i, [_vp]),
    "hp_destroy": (_i, [_vp]),
    "hp_context_clone": (_i, [_vp, C.POINTER(_vp), _vp]),
    "hp_cgs_pass": (_i, [_i, _i64, _i, C.POINTER(_vp), _i64, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _i, _i, _vp]),
    "hp_mailbox_create": (_i, [_i64, C.POINTER(_vp), _vp]),
    "hp_mailbox_open": (_i, [_vp, C.POINTER(_vp)]),
    "hp_mailbox_close": (_i, [_vp]),
    "hp_mailbox_free": (_i, [_vp]),
    "hp_stream_wait_geq": (_i, [_vp, C.c_uint, _vp]),
    "hp_handover_rows": (_i, [_i, C.POINTER(_vp), _vp, _i64, _vp, C.c_uint, _vp]),
    "hp_collect_rows": (_i, [_i, _vp, C.POINTER(_vp), _i64, _vp]),
    "hp_signal_flags": (_i, [_i, C.POINTER(_vp), C.c_uint, _vp]),
    "hp_csr_nnz": (_i64, [_i]),
    "hp_assemble_csr": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "hp_strip_csr_nnz": (_i64, [_i, _i]),
    "hp_assemble_strip_csr": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "hp_stencil_matvec": (_i, [_vp, _vp, _vp, _vp]),
    "hp_stencil_matvec_rows": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hp_csr_matvec": (_i, [_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hp_precond_setup": (_i, [_vp, _i, _i, _i, _i, _vp]),
    "hp_debug_phases": (_i, [_vp, _i, _vp]),
    "hp_sweep_status": (_i, [_vp]),
    "hp_set_sweep_variant": (_i, [_vp, _i]),
    "hp_set_layout_mode": (_i, [_vp, _i]),
    "hp_set_front_mode": (_i, [_vp, _i]),
    "hp_precond_set_front": (_i, [_vp, _i, _vp]),
    "hp_strip_layout_ex": (_i, [_vp, _ip, _ip, _ip, _ip]),
    "hp_precond_bytes": (_i64, [_vp]),
    "hp_precond_setup_ms": (_d, [_vp]),
    "hp_front_begin": (_i, [_vp, _vp, _vp]),
    "hp_front_tf_copy": (_i, [_vp, _vp, _i, _vp]),
    "hp_sweep_forward": (_i, [_vp, _vp, _i, _i, _vp]),
    "hp_sweep_backward": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "hp_front_end": (_i, [_vp, _vp, _vp]),
    "hp_precond_apply": (_i, [_vp, _vp, _vp, _i, _vp]),
    "hp_multi_max": (_i, [_vp]),
    "hp_multi_kernel": (_i, [_vp, _i]),
    "hp_sweep_forward_multi": (_i, [_vp, _i, C.POINTER(_vp), _i, _i, _vp]),
    "hp_sweep_backward_multi": (_i, [_vp, _i, C.POINTER(_vp), _i, _i, _i, _vp]),
    "hp_precond_apply_multi": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_vp), _i, _vp]),
    "hp_strip_apply": (_i, [_vp, _i, _vp, _vp, _vp]),
    "hp_strip_layout": (_i, [_vp, _ip, _ip, _ip, _ip, _ip, _ip, C.POINTER(_i64), _ip, _ip, _ip]),
    "hp_strip_packets": (_i, [_vp, _i, _vp]),
    "hp_grad_accumulate": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_vp), _vp, _vp]),
    "hp_grad_finish": (_i, [_vp, _vp, _i, _vp, _vp]),
    "hp_born_source": (_i, [_vp, _i, _vp, C.POINTER(_vp), C.POINTER(_vp), _vp]),
    "hp_dotc": (_i, [_i64, _vp, _vp, _vp, _vp]),
    "hp_nrm2": (_i, [_i64, _vp, _vp, _vp]),
    "hp_axpy": (_i, [_i64, _d, _d, _vp, _vp, _vp]),
    "hp_axpy_dev": (_i, [_i64, _vp, _d, _vp, _vp, _vp]),
    "hp_scale_copy": (_i, [_i64, _d, _d, _vp, _vp, _vp]),
    "hp_mgs": (_i, [_i64, _i, _vp, _i64, _vp, _vp, _vp]),
    "hp_mgs_step": (_i, [_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hp_combine": (_i, [_i64, _i, _vp, _i64, _vp, _vp, _vp]),
}

_lib = None


class HelmholtzB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (no CUDA call is made)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HelmholtzB200Error(
                f"{LIB_PATH} is missing: build it with `python -m helmholtz_preconditioner_b200.build` "
                "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc, what=""):
    if rc != 0:
        raise HelmholtzB200Error(f"{what} failed (code {rc}): {load().hp_last_error().decode()}")


def require_device():
    lib = load()
    if not lib.hp_device_ok():
        raise HelmholtzB200Error("no CUDA device: helmholtz_preconditioner_b200 has no CPU path")
    return lib
