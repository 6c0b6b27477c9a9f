"""B200-native implementation of the hot path of bocchs/helmholtz-preconditioner (code.py): PML Helmholtz
assembly, matrix-free stencil SpMV, moving-PML sweeping preconditioner and preconditioned GMRES, as
hand-written sm_100a CUDA kernels behind a C ABI (include/helmholtz_b200.h)."""
from ._lib import HelmholtzB200Error, LIB_PATH, load  # noqa: F401
from .fields import (attenuate, init_c1_f1, init_c1_f2, init_c1_mat, init_c2_f1, init_c2_f2, init_c2_mat,  # noqa: F401
                     init_const_f1, init_f1_mat, init_f2_mat, init_layered_f1)


def __getattr__(name):
    # solver.py needs torch; keep `import helmholtz_preconditioner_b200` light for the host-only tests
    if name in ("HelmholtzSolver", "DeviceCSR", "SolveResult", "run_solver", "run_solver_many", "build_A_matrix", "algo2_3", "algo2_4", "get_Hm", "get_A_FF_block"):
        from . import solver
        return getattr(solver, name)
    if name in ("Receivers", "GradientResult", "misfit_gradient", "born"):
        from . import inversion
        return getattr(inversion, name)
    if name in ("gmres", "gmres_batch", "DeviceVectors", "lartg"):
        import importlib
        return getattr(importlib.import_module(__name__ + ".gmres"), name)
    raise AttributeError(name)
