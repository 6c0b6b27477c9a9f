"""Inversion on the host side: the lazy exports, Receivers validation, and the argument checks misfit_gradient and born make
before any device work."""
import numpy as np
import pytest
import torch

import helmholtz_preconditioner_b200 as hp


def test_lazy_exports():
    from helmholtz_preconditioner_b200 import inversion
    for name in ("Receivers", "GradientResult", "misfit_gradient", "born"):
        assert getattr(hp, name) is getattr(inversion, name)


def test_receivers_index_and_validation():
    n = 10
    r = hp.Receivers(n, [1, 10, 3], [1, 2, 10], device="cpu")
    assert r.nrec == len(r) == 3
    assert r.index.dtype == torch.int64 and r.index.tolist() == [0, 1 * n + 9, 9 * n + 2]
    u = torch.arange(n * n, dtype=torch.float64).to(torch.complex128)
    assert r.sample(u).tolist() == [0, 19, 92]
    a = r.inject(torch.tensor([1 + 2j, 3 - 1j, -1j], dtype=torch.complex128))
    assert a.shape == (n * n,) and torch.count_nonzero(a).item() == 3
    assert a[19].item() == 3 + 1j and a[92].item() == 1j                 # conj(r) scattered into zeros
    for i, j in (([0], [1]), ([1], [11]), ([11], [1]), ([1], [0])):       # outside 1..n
        with pytest.raises(ValueError):
            hp.Receivers(n, i, j, device="cpu")
    with pytest.raises(ValueError):
        hp.Receivers(n, [2, 3, 2], [4, 4, 4], device="cpu")              # duplicate
    with pytest.raises(ValueError):
        hp.Receivers(n, [1, 2], [1], device="cpu")                       # unequal lengths
    with pytest.raises(ValueError):
        hp.Receivers(n, [], [], device="cpu")
    with pytest.raises(ValueError):
        hp.Receivers(n, [1.5], [2], device="cpu")


def _no_device():
    if torch.cuda.is_available():
        pytest.skip("GPU present")


def test_bad_arguments_raise_value_error():
    n, S = 12, 3
    rec = hp.Receivers(n, np.arange(1, 6), np.full(5, 2), device="cpu")
    f = np.zeros((S, n, n))
    with pytest.raises(ValueError):
        hp.misfit_gradient(None, f, rec, np.zeros((S, 4)))
    with pytest.raises(ValueError):
        hp.misfit_gradient(None, f, rec, np.zeros((S + 1, 5)))
    with pytest.raises(ValueError):
        hp.misfit_gradient(None, f, rec, np.zeros((S, 5)), wrt="c")
    with pytest.raises(ValueError):
        hp.misfit_gradient(None, f, rec, np.zeros((S, 5)), diag="none")
    with pytest.raises(ValueError):
        hp.born(None, None, rec, np.zeros((n + 2, n + 2)))


def test_without_device_raises():
    _no_device()
    n, S = 12, 2
    rec = hp.Receivers(n, [3, 4], [5, 5])
    with pytest.raises(hp.HelmholtzB200Error):
        hp.misfit_gradient(None, np.zeros((S, n, n)), rec, np.zeros((S, 2)))
    with pytest.raises(hp.HelmholtzB200Error):
        hp.born(None, np.zeros((S, n, n)), rec, np.zeros((n + 2, n + 2)))
