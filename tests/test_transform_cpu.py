"""CPU checks of SmoothNMF.transform: where it exists, what scikit-learn's estimator checks see, the C-ABI flag of the
H-only loop, and the argument errors that must come before any device work (this box has no GPU: a call that got as
far as the device would raise espm_b200's "needs a CUDA device" error instead)."""
import contextlib
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


def _fake_fitted(n=40, m=5, k=3, **kw):
    """An estimator with the fitted attributes transform reads, without running a fit."""
    est = _est(n_components=k, hspy_comp=True, **kw)
    rng = np.random.default_rng(0)
    est.G_ = rng.uniform(0.1, 1.0, size=(n, m))
    est.W_ = rng.uniform(0.1, 1.0, size=(m, k))
    est.H_ = rng.uniform(0.1, 1.0, size=(k, 12))
    est._identity_G = False
    return est


def test_transform_exists_only_with_hspy_comp():
    assert not hasattr(_est(), "transform")
    assert hasattr(_est(hspy_comp=True), "transform")
    est = _est()
    est.set_params(hspy_comp=True)
    assert hasattr(est, "transform")


def test_estimator_checks_add_no_transformer_checks():
    from sklearn.utils.estimator_checks import estimator_checks_generator
    names = []
    for _, check in estimator_checks_generator(_est(n_components=3), legacy=True):
        fn = check
        while hasattr(fn, "func"):
            fn = fn.func
        names.append(fn.__name__)
    assert names
    assert not [nm for nm in names if nm.startswith("check_transformer")]


def test_h_only_flag_matches_header():
    from espm_b200 import _lib
    header = open(os.path.join(ROOT, "include", "espm_b200.h")).read()
    m = re.search(r"#define\s+ESPM_FLAG_H_ONLY\s+\(1u << (\d+)\)", header)
    assert m and (1 << int(m.group(1))) == _lib.FLAG_H_ONLY
    others = [int(b) for name, b in re.findall(r"#define\s+ESPM_FLAG_(\w+)\s+\(1u << (\d+)\)", header)
              if name != "H_ONLY"]
    assert int(m.group(1)) not in others


def test_unfitted_raises_before_device_work():
    est = _est(hspy_comp=True)
    with pytest.raises(NotFittedError):
        est.transform(np.ones((10, 40)))


@pytest.mark.parametrize("kw, word", [
    (dict(algo="bmd"), "bmd"),
    (dict(algo="projected_gradient", simplex_W=False), "projected_gradient"),
    (dict(algo="l2_surrogate", l2=True), "l2"),
    (dict(linesearch=True, lambda_L=1.0), "linesearch"),
])
def test_unsupported_options_raise_before_device_work(kw, word):
    est = _fake_fitted(**kw)
    with pytest.raises(NotImplementedError, match=word):
        est.transform(np.ones((12, 40)))


def test_channel_count_must_match_the_fitted_model():
    est = _fake_fitted(n=40)
    with pytest.raises(ValueError, match="40"):
        est.transform(np.ones((12, 39)))


def test_initial_h_shape_is_checked():
    est = _fake_fitted(n=40, k=3)
    with pytest.raises(ValueError, match="H has shape"):
        est.transform(np.ones((12, 40)), H=np.ones((3, 11)))


def test_laplacian_shape_mismatch_raises_check_shape_2d_message():
    est = _fake_fitted(lambda_L=1.0, shape_2d=(3, 4))
    # the fitted shape_2d does not describe 15 pixels and no shape is given
    with pytest.raises(ValueError, match="does not match the number of pixels 15"):
        est.transform(np.ones((15, 40)))
    # an explicit shape that does not match either
    with pytest.raises(ValueError, match="does not match the number of pixels 15"):
        est.transform(np.ones((15, 40)), shape_2d=(4, 4))
