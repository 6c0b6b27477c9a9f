"""Attenuating media on the host side: fields.attenuate and the checks HelmholtzSolver makes before any device work."""
import warnings

import numpy as np
import pytest
import torch

import helmholtz_preconditioner_b200 as hp
from helmholtz_preconditioner_b200 import fields


def test_attenuate_formula():
    c = fields.init_layered_f1(2 * np.pi * 3 + 1j, 30)[0]
    for q in (10.0, 50.0):
        a = fields.attenuate(c, q)
        assert a.dtype == np.complex128 and a.shape == c.shape
        assert np.array_equal(a, c / np.sqrt(1 + 1j / q))
        kappa = 1 / a ** 2
        assert np.allclose(kappa, (1 + 1j / q) / c ** 2, rtol=1e-14)
        assert np.all(kappa.imag > 0)                    # loss: Im(omega^2 kappa) > 0 for a real positive omega
    q = np.full(c.shape, np.inf)
    q[:, 5:9] = 10.0
    a = fields.attenuate(c, q)
    assert np.array_equal(a[:, 5:9], c[:, 5:9] / np.sqrt(1 + 0.1j))
    assert np.array_equal(a[:, 9:], c[:, 9:] + 0j) and not np.any(a.imag[:, 9:])


def test_attenuate_lossless_is_the_real_model():
    c = fields.init_c1_mat(.5, .5, 20)
    a = fields.attenuate(c, np.inf)
    assert np.iscomplexobj(a) and np.array_equal(a.real, c) and not np.any(a.imag)


def test_attenuate_q_shape():
    with pytest.raises(ValueError):
        fields.attenuate(np.ones((5, 5)), np.ones((4, 4)))


def _no_device():
    if torch.cuda.is_available():
        pytest.skip("GPU present")


@pytest.mark.parametrize("make", [lambda c: c, lambda c: c.astype(np.complex64), torch.from_numpy],
                         ids=["numpy", "complex64", "torch"])
def test_complex_model_without_device_raises(make):
    _no_device()
    c = make(fields.attenuate(np.ones((22, 22)), 10.0))
    with warnings.catch_warnings():
        warnings.simplefilter("error")                  # a ComplexWarning would mean the imaginary part was dropped
        with pytest.raises(hp.HelmholtzB200Error):
            hp.HelmholtzSolver(20, 5, 2 * np.pi * 3 + 2j, 30.0, c)
        with pytest.raises(hp.HelmholtzB200Error):
            hp.run_solver(20, 5, 3, 30, 2, c_mat=c, verbose=False)


@pytest.mark.parametrize("make", [lambda c: c, torch.from_numpy], ids=["numpy", "torch"])
def test_complex_model_of_wrong_shape(make):
    c = make(fields.attenuate(np.ones((21, 22)), 10.0))
    with pytest.raises(ValueError):
        hp.HelmholtzSolver(20, 5, 2 * np.pi * 3 + 2j, 30.0, c)

