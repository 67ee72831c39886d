"""CPU checks of SmoothNMF.goodness_of_fit: where it exists, what scikit-learn's estimator checks see, the ctypes
signatures of its C-ABI entry points, and the argument errors that come before any device work (on a machine without a
GPU a call that got as far as the device raises espm_b200's "needs a CUDA device" error instead)."""
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
    """An estimator with the fitted attributes goodness_of_fit reads, without running a fit."""
    est = _est(n_components=k, **kw)
    rng = np.random.default_rng(0)
    est.G_ = rng.uniform(0.1, 1.0, size=(n, m))
    est.W_ = rng.uniform(0.1, 1.0, size=(m, k))
    est.H_ = rng.uniform(0.1, 1.0, size=(k, p))
    est._identity_G = False
    return est


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_method_exists_for_both_layouts(hspy_comp):
    assert callable(getattr(_est(hspy_comp=hspy_comp), "goodness_of_fit", None))


def test_fit_statistics_is_exported():
    import espm_b200
    assert "FitStatistics" in espm_b200.__all__
    assert espm_b200.FitStatistics._fields == ("pixel_counts", "pixel_model", "pixel_kl", "pixel_chi2",
                                               "channel_counts", "channel_model", "channel_kl", "channel_chi2")


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
    monkeypatch.delattr(SmoothNMF, "goodness_of_fit")
    without = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    assert with_method and with_method == without


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_unfitted_raises_before_device_work(hspy_comp):
    with pytest.raises(NotFittedError):
        _est(hspy_comp=hspy_comp).goodness_of_fit(np.ones((40, 12)))


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_channel_count_must_match_the_fitted_model(hspy_comp):
    est = _fake_fitted(n=40, hspy_comp=hspy_comp)
    X = np.ones((39, 12))
    with pytest.raises(ValueError, match="39 channels.*40"):
        est.goodness_of_fit(X.T if hspy_comp else X)


def test_pixel_count_must_match_H_when_H_is_omitted():
    est = _fake_fitted(n=40, p=12)
    with pytest.raises(ValueError, match="13 pixels.*12"):
        est.goodness_of_fit(np.ones((40, 13)))


@pytest.mark.parametrize("shape", [(3, 12), (2, 13), (13, 3)])
def test_H_shape_is_checked(shape):
    est = _fake_fitted(n=40, k=3, p=12)
    with pytest.raises(ValueError, match="H has shape"):
        est.goodness_of_fit(np.ones((40, 13)), H=np.ones(shape))


def test_valid_call_reaches_the_device():
    import torch
    from espm_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("this machine has a GPU: the call would run")
    est = _fake_fitted(n=40, k=3, p=12)
    with pytest.raises(_lib.EspmError, match="needs a CUDA device"):
        est.goodness_of_fit(np.ones((40, 13)), H=np.ones((3, 13)))


def _header_signature(name):
    header = open(os.path.join(ROOT, "include", "espm_b200.h")).read()
    m = re.search(r"int\s+%s\(([^)]*)\);" % name, header)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


def test_lib_signatures_match_header():
    from espm_b200 import _lib
    ctype = {"const espm_state* st": ctypes.POINTER(_lib.EspmState), "int64_t* bytes_out": ctypes.POINTER(ctypes.c_int64),
             "double* pixel_out": ctypes.c_void_p, "double* channel_out": ctypes.c_void_p,
             "void* scratch": ctypes.c_void_p, "void* stream": ctypes.c_void_p}
    for name in ("espm_fit_stats_scratch", "espm_fit_stats"):
        restype, argtypes = _lib._EXPORTS[name]
        assert restype is ctypes.c_int
        assert argtypes == [ctype[a] for a in _header_signature(name)], name
