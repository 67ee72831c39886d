"""CPU checks of SmoothNMF.residual_components: the export, the ctypes signatures of its C-ABI entry points, the argument
errors that come before any device work (on a machine without a GPU a call that got as far as the device raises
espm_b200's "needs a CUDA device" error instead), and the host driver (``host.residual_components``) with NumPy
operators standing in for the two device products, against ``np.linalg.svd`` of a dense R."""
import contextlib
import ctypes
import io

import numpy as np
import pytest
from sklearn.exceptions import NotFittedError


def _est(**kw):
    from espm_b200 import SmoothNMF
    with contextlib.redirect_stdout(io.StringIO()):
        return SmoothNMF(**kw)


def _fake_fitted(n=40, m=5, k=3, p=30, **kw):
    """An estimator with the fitted attributes residual_components reads, without running a fit."""
    est = _est(n_components=k, **kw)
    rng = np.random.default_rng(0)
    est.G_ = rng.uniform(0.1, 1.0, size=(n, m))
    est.W_ = rng.uniform(0.1, 1.0, size=(m, k))
    est.H_ = rng.uniform(0.1, 1.0, size=(k, p))
    est._identity_G = False
    est.physics_model_ = None
    return est


# ---------------------------------------------------------------------------------------------------- oracles
def pearson_residual(X, GW, H, ls):
    """(n, p) fp64 R = (x - y) / sqrt(y) with g = max(GW, ls), h = max(H, ls), y = g h."""
    y = np.maximum(np.asarray(GW, np.float64), ls) @ np.maximum(np.asarray(H, np.float64), ls)
    return (np.asarray(X, np.float64) - y) / np.sqrt(y)


def subspace_angle(A, B):
    """Sine of the largest principal angle between the column spaces of A and B (orthonormal columns, same count):
    ||(I - A A^T) B||_2, accurate for small angles, where arccos of the cosines is not."""
    return float(np.linalg.norm(B - A @ (A.T @ B), 2))


def _gapped(n=120, p=300, rank=4, seed=0):
    """R with singular values 40, 30, 20, 10 and then 1 / (1 + i) (a clear gap after the 4th)."""
    rng = np.random.default_rng(seed)
    U = np.linalg.qr(rng.standard_normal((n, n)))[0]
    V = np.linalg.qr(rng.standard_normal((p, n)))[0]
    s = np.concatenate([[40.0, 30.0, 20.0, 10.0][:rank], 1.0 / (1.0 + np.arange(n - rank))])
    return (U * s) @ V.T


def _operators(R, blocks=None):
    """The three callables of host.residual_components for R (n, p), with the pixels split into ``blocks`` (fake ranks):
    left returns the list of per-rank P blocks, right and gram add the per-rank blocks in rank order."""
    p = R.shape[1]
    cuts = [0, p] if blocks is None else blocks
    parts = [R[:, a:b] for a, b in zip(cuts[:-1], cuts[1:])]

    def left(Q):
        return [(Rb.T @ Q).T for Rb in parts]

    def right(Ps):
        out = parts[0] @ Ps[0].T
        for Rb, Pb in zip(parts[1:], Ps[1:]):
            out = out + Rb @ Pb.T
        return out

    def gram(Ps):
        out = Ps[0] @ Ps[0].T
        for Pb in Ps[1:]:
            out = out + Pb @ Pb.T
        return out
    return left, right, gram


def _run(R, rank, n_iter, seed=1, blocks=None):
    from espm_b200.host import RESID_OVERSAMPLE, residual_components
    Q0 = np.random.RandomState(seed).standard_normal((R.shape[0], rank + RESID_OVERSAMPLE))
    left, right, gram = _operators(R, blocks)
    s, spectra, V, Ps = residual_components(left, right, gram, Q0, rank, n_iter)
    maps = np.concatenate([V.T @ Pb for Pb in Ps], axis=1)
    return s, spectra, maps


# ---------------------------------------------------------------------------------------------------- host driver
def test_driver_matches_dense_svd():
    R = _gapped()
    s, spectra, maps = _run(R, 4, 7)
    U, S, Vt = np.linalg.svd(R, full_matrices=False)
    assert s.shape == (4,) and spectra.shape == (120, 4) and maps.shape == (4, 300)
    assert np.all(np.diff(s) < 0)
    assert np.max(np.abs(s - S[:4]) / S[:4]) <= 1e-10
    assert subspace_angle(spectra, U[:, :4]) <= 1e-8
    assert subspace_angle(maps.T, Vt[:4].T) <= 1e-8
    assert np.allclose(spectra.T @ spectra, np.eye(4), atol=1e-12)
    assert np.allclose(maps @ maps.T, np.eye(4), atol=1e-10)
    # each triplet, with signs: R v_i = s_i u_i
    assert np.max(np.abs(R @ maps.T - spectra * s)) <= 1e-8 * s[0]


def test_driver_sign_convention():
    R = _gapped(seed=3)
    for seed in range(4):                                   # the start's sign pattern must not show through
        s, spectra, maps = _run(R, 4, 7, seed=seed)
        lead = spectra[np.argmax(np.abs(spectra), axis=0), np.arange(4)]
        assert np.all(lead > 0)
        U, S, Vt = np.linalg.svd(R, full_matrices=False)
        flip = np.sign(U[np.argmax(np.abs(U[:, :4]), axis=0), np.arange(4)])
        assert np.allclose(spectra, U[:, :4] * flip, atol=1e-8)
        assert np.allclose(maps, Vt[:4] * flip[:, None], atol=1e-8)


def test_driver_iteration_count():
    """n_iter = 1 is one range-finder pass (Q from R R^T Q0): with r = rank + 10 and a gap of 10x to the tail it already
    finds the top.  n_iter = 0 projects R on the random start only: values below the true ones, never above."""
    R = _gapped()
    S = np.linalg.svd(R, compute_uv=False)[:4]
    s, _, _ = _run(R, 4, 1)
    assert np.max(np.abs(s - S) / S) <= 1e-2
    s0, spectra0, _ = _run(R, 4, 0)
    assert np.all(s0 <= S * (1 + 1e-12)) and np.allclose(spectra0.T @ spectra0, np.eye(4), atol=1e-12)


def test_fake_ranks_combine_in_rank_order():
    """Two fake ranks, each holding half the pixels: every rank's view is built from the same rank-ordered sums, so the
    ranks agree bit for bit, and with a single rank the result is the same to rounding."""
    R = _gapped(p=301)
    blocks = [0, 150, 301]
    a = _run(R, 4, 7, blocks=blocks)
    b = _run(R, 4, 7, blocks=blocks)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    one = _run(R, 4, 7)
    assert np.max(np.abs(a[0] - one[0]) / one[0]) <= 1e-12
    assert np.max(np.abs(a[1] - one[1])) <= 1e-10
    assert np.max(np.abs(a[2] - one[2])) <= 1e-10


def test_driver_on_a_pearson_residual():
    """A planted missing phase in a Poisson image: the host driver on the dense Pearson residual of the 3-phase truth
    finds the 4th phase's spectrum and map."""
    rng = np.random.default_rng(5)
    n, p, k = 80, 400, 4
    x = np.linspace(0, 1, n)
    GW = np.stack([np.exp(-0.5 * ((x - c) / 0.03) ** 2) + 0.05 for c in (0.2, 0.4, 0.6, 0.8)], 1) * 50.0
    H = rng.dirichlet(np.ones(k), size=p).T
    X = rng.poisson(GW @ H).astype(np.float64)
    R = pearson_residual(X, GW[:, :3], H[:3], 1e-14)
    s, spectra, maps = _run(R, 2, 7)
    assert s[0] > 3 * s[1]
    assert np.argmax(spectra[:, 0]) in range(int(0.75 * n), int(0.85 * n) + 1)
    assert abs(np.corrcoef(maps[0], H[3])[0, 1]) >= 0.8


# ---------------------------------------------------------------------------------------------------- interface
def test_exported():
    import espm_b200
    from espm_b200 import ResidualComponents, SmoothNMF
    assert "ResidualComponents" in espm_b200.__all__
    assert ResidualComponents._fields == ("singular_values", "spectra", "maps")
    assert callable(SmoothNMF.residual_components)


def test_ctypes_signatures():
    from espm_b200 import _lib
    st = ctypes.POINTER(_lib.EspmState)
    i32, i64, vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p
    assert _lib._EXPORTS["espm_resid_left_scratch"] == (ctypes.c_int, [st, i32, ctypes.POINTER(i64)])
    assert _lib._EXPORTS["espm_resid_right_scratch"] == (ctypes.c_int, [st, i32, ctypes.POINTER(i64)])
    assert _lib._EXPORTS["espm_resid_left"] == (ctypes.c_int, [st, vp, i32, vp, vp, vp])
    assert _lib._EXPORTS["espm_resid_right"] == (ctypes.c_int, [st, vp, i32, vp, vp, vp])


def test_not_fitted():
    with pytest.raises(NotFittedError):
        _est(n_components=3).residual_components(np.ones((40, 30)))


@pytest.mark.parametrize("hspy_comp", [False, True])
@pytest.mark.parametrize("kw, msg", [
    (dict(rank=0), "rank must be between 1 and"),
    (dict(rank=-2), "rank must be between 1 and"),
    (dict(rank=21), r"min\(n, p\) - 10 = 20"),
    (dict(rank=2.0), "rank must be an integer"),
    (dict(rank=True), "rank must be an integer"),
    (dict(rank="3"), "rank must be an integer"),
    (dict(n_iter=-1), "n_iter must be an integer >= 0"),
    (dict(n_iter=1.5), "n_iter must be an integer >= 0"),
    (dict(random_state="seed"), "cannot be used to seed"),
])
def test_argument_errors_before_device_work(kw, msg, hspy_comp, monkeypatch):
    from espm_b200.engine import FitEngine
    est = _fake_fitted(hspy_comp=hspy_comp)
    called = []
    monkeypatch.setattr(FitEngine, "for_statistics", classmethod(lambda *a, **k: called.append(1)))
    X = np.ones((30, 40)) if hspy_comp else np.ones((40, 30))
    with pytest.raises(ValueError, match=msg):
        est.residual_components(X, **kw)
    assert not called


def test_rank_bound_uses_the_smaller_side():
    from espm_b200.engine import FitEngine
    est = _fake_fitted(n=40, p=25)
    with pytest.raises(ValueError, match=r"= 15, got 16"):
        est.residual_components(np.ones((40, 25)), rank=16)
    # rank 15 passes the argument checks and goes on to the engine
    seen = []

    def fake(cls, *a, **k):
        seen.append(a[0].shape)
        raise RuntimeError("stop")
    import unittest.mock
    with unittest.mock.patch.object(FitEngine, "for_statistics", classmethod(fake)):
        with pytest.raises(RuntimeError, match="stop"):
            est.residual_components(np.ones((40, 25)), rank=15, random_state=0)
    assert seen == [(40, 25)]


@pytest.mark.parametrize("kw, msg", [
    (dict(H=np.ones((2, 30))), "H has shape"),
    (dict(X=np.ones((39, 30))), "X has 39 channels"),
    (dict(X=np.ones((40, 31))), "pass the maps of this image as H"),
])
def test_shape_errors_of_goodness_of_fit(kw, msg):
    est = _fake_fitted()
    X = kw.pop("X", np.ones((40, 30)))
    with pytest.raises(ValueError, match=msg):
        est.residual_components(X, rank=2, **kw)


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_estimator_checks_are_unchanged(monkeypatch, hspy_comp):
    from espm_b200 import SmoothNMF
    from test_phase_uncertainty_cpu import _check_names
    with_method = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    monkeypatch.delattr(SmoothNMF, "residual_components")
    without = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    assert with_method and with_method == without


def test_valid_call_reaches_the_device():
    import torch
    from espm_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("this machine has a GPU: the call would run")
    est = _fake_fitted()
    with pytest.raises(_lib.EspmError, match="needs a CUDA device"):
        est.residual_components(np.ones((40, 30)), rank=2)
