"""CPU checks of SmoothNMF.abundance_uncertainty: where it exists, what scikit-learn's estimator checks see, the ctypes
signature of its C-ABI entry point, the argument errors that come before any device work (on a machine without a GPU a
call that got as far as the device raises espm_b200's "needs a CUDA device" error instead), and the NumPy oracle of its
formulas that the GPU tests compare against."""
import contextlib
import ctypes
import io
import os
import re

import numpy as np
import pytest
from sklearn.exceptions import NotFittedError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _est(**kw):
    from espm_b200 import SmoothNMF
    with contextlib.redirect_stdout(io.StringIO()):
        return SmoothNMF(**kw)


def _fake_fitted(n=40, m=5, k=3, p=12, **kw):
    """An estimator with the fitted attributes abundance_uncertainty reads, without running a fit."""
    est = _est(n_components=k, **kw)
    rng = np.random.default_rng(0)
    est.G_ = rng.uniform(0.1, 1.0, size=(n, m))
    est.W_ = rng.uniform(0.1, 1.0, size=(m, k))
    est.H_ = rng.uniform(0.1, 1.0, size=(k, p))
    est._identity_G = False
    return est


def information_oracle(X, GW, H, ls):
    """(p, k, k) fp64 F_j[a, b] = sum_c x_cj g_ca g_cb / y_cj^2 with g = max(GW, ls), h = max(H, ls), y = g h."""
    X = np.asarray(X, dtype=np.float64)
    g = np.maximum(np.asarray(GW, np.float64), ls)
    Y = g @ np.maximum(np.asarray(H, np.float64), ls)
    Wt = X / Y ** 2                                            # (n, p)
    return np.einsum("cj,ca,cb->jab", Wt, g, g)


def covariance_oracle(F, simplex):
    """(p, k, k) F_j^-1, projected onto sum_a h_a = 1 with ``simplex``: Fi - (Fi 1)(Fi 1)^T / (1^T Fi 1)."""
    Fi = np.linalg.inv(F)
    if not simplex:
        return Fi
    v = Fi.sum(2)
    return Fi - v[:, :, None] * v[:, None, :] / v.sum(1)[:, None, None]


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_method_exists_for_both_layouts(hspy_comp):
    assert callable(getattr(_est(hspy_comp=hspy_comp), "abundance_uncertainty", None))


def test_abundance_uncertainty_is_exported():
    import espm_b200
    assert "AbundanceUncertainty" in espm_b200.__all__
    assert espm_b200.AbundanceUncertainty._fields == ("std", "covariance", "information")


def _check_names(est):
    from sklearn.utils.estimator_checks import estimator_checks_generator
    names = []
    for _, check in estimator_checks_generator(est, legacy=True):
        fn = check
        while hasattr(fn, "func"):
            fn = fn.func
        names.append(fn.__name__)
    return names


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_estimator_checks_are_unchanged(monkeypatch, hspy_comp):
    from espm_b200 import SmoothNMF
    with_method = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    monkeypatch.delattr(SmoothNMF, "abundance_uncertainty")
    without = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    assert with_method and with_method == without


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_unfitted_raises_before_device_work(hspy_comp):
    with pytest.raises(NotFittedError):
        _est(hspy_comp=hspy_comp).abundance_uncertainty(np.ones((40, 12)))


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_channel_count_must_match_the_fitted_model(hspy_comp):
    est = _fake_fitted(n=40, hspy_comp=hspy_comp)
    X = np.ones((39, 12))
    with pytest.raises(ValueError, match="39 channels.*40"):
        est.abundance_uncertainty(X.T if hspy_comp else X)


def test_pixel_count_must_match_H_when_H_is_omitted():
    est = _fake_fitted(n=40, p=12)
    with pytest.raises(ValueError, match="13 pixels.*12"):
        est.abundance_uncertainty(np.ones((40, 13)))


@pytest.mark.parametrize("shape", [(3, 12), (2, 13), (13, 3)])
def test_H_shape_is_checked(shape):
    est = _fake_fitted(n=40, k=3, p=12)
    with pytest.raises(ValueError, match="H has shape"):
        est.abundance_uncertainty(np.ones((40, 13)), H=np.ones(shape))


@pytest.mark.parametrize("simplex_H", [False, True])
def test_valid_call_reaches_the_device(simplex_H):
    import torch
    from espm_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("this machine has a GPU: the call would run")
    est = _fake_fitted(n=40, k=3, p=12, simplex_H=simplex_H)
    with pytest.raises(_lib.EspmError, match="needs a CUDA device"):
        est.abundance_uncertainty(np.ones((40, 13)), H=np.ones((3, 13)))


def test_lib_signature_matches_header():
    from espm_b200 import _lib
    header = open(os.path.join(ROOT, "include", "espm_b200.h")).read()
    m = re.search(r"int\s+espm_abundance_info\(([^)]*)\);", header)
    assert m
    args = [a.strip() for a in m.group(1).split(",")]
    ctype = {"const espm_state* st": ctypes.POINTER(_lib.EspmState), "int simplex": ctypes.c_int,
             "double* out": ctypes.c_void_p, "void* stream": ctypes.c_void_p}
    restype, argtypes = _lib._EXPORTS["espm_abundance_info"]
    assert restype is ctypes.c_int
    assert argtypes == [ctype[a] for a in args]


@pytest.mark.parametrize("k", [2, 3, 5])
def test_oracle_is_consistent(k):
    """F is symmetric positive definite for data with counts; the unconstrained C is its inverse; the simplex C has
    C 1 = 0 and equals U (U^T F U)^-1 U^T for an orthonormal basis U of the null space of 1^T (the covariance of the
    k - 1 free coordinates, mapped back)."""
    rng = np.random.default_rng(k)
    n, p = 60, 9
    GW = rng.uniform(0.0, 1.0, size=(n, k))
    GW[:, 0] = 0.0                                             # a clamped column: g = ls there
    H = rng.dirichlet(np.ones(k), size=p).T
    X = rng.poisson(200.0 * np.maximum(GW, 1e-3) @ H).astype(np.float64)
    F = information_oracle(X, GW, H, 1e-3)
    assert F.shape == (p, k, k)
    assert np.allclose(F, np.swapaxes(F, 1, 2), rtol=1e-14, atol=0)
    assert np.all(np.linalg.eigvalsh(F) > 0)
    C = covariance_oracle(F, False)
    assert np.allclose(np.einsum("jab,jbc->jac", C, F), np.eye(k)[None], atol=1e-10)
    Cs = covariance_oracle(F, True)
    scale = np.abs(C).max(axis=(1, 2))                        # the projection's rounding is relative to F^-1
    assert np.all(np.abs(Cs.sum(2)).max(1) <= 1e-12 * scale)
    Q, _ = np.linalg.qr(np.concatenate([np.ones((k, 1)), rng.normal(size=(k, k - 1))], axis=1))
    U = Q[:, 1:]                                              # orthonormal, orthogonal to 1
    ref = U[None] @ np.linalg.inv(U.T[None] @ F @ U[None]) @ U.T[None]
    assert np.max(np.abs(Cs - ref)) <= 1e-10 * scale.max()
    assert np.all(np.diagonal(Cs, axis1=1, axis2=2) < np.diagonal(C, axis1=1, axis2=2))
