"""run_solver_many (several sources in one call) on a machine without a CUDA device: the package exports it, and it
fails loudly instead of falling back to a CPU path.  No compute call is made here."""
import pytest


def test_run_solver_many_exported():
    import helmholtz_preconditioner_b200 as hp
    from helmholtz_preconditioner_b200 import solver
    assert hp.run_solver_many is solver.run_solver_many


def test_run_solver_many_no_cpu_fallback():
    import numpy as np
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import helmholtz_preconditioner_b200 as hp
    hp.load()
    with pytest.raises(hp.HelmholtzB200Error):
        hp.run_solver_many(20, 5, 3, 30, 2, np.zeros((2, 20, 20)))
