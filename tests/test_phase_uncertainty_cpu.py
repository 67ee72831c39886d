"""CPU checks of SmoothNMF.phase_uncertainty: where it exists, what scikit-learn's estimator checks see, the ctypes
signatures of its C-ABI entry points, the argument errors that come before any device work (on a machine without a GPU a
call that got as far as the device raises espm_b200's "needs a CUDA device" error instead), and the host algebra
(``host.phase_covariance``) against dense NumPy oracles of its formulas, which the GPU tests compare against too."""
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
    """An estimator with the fitted attributes phase_uncertainty reads, without running a fit."""
    est = _est(n_components=k, **kw)
    rng = np.random.default_rng(0)
    est.G_ = rng.uniform(0.1, 1.0, size=(n, m))
    est.W_ = rng.uniform(0.1, 1.0, size=(m, k))
    est.H_ = rng.uniform(0.1, 1.0, size=(k, p))
    est._identity_G = False
    est.physics_model_ = None
    return est


# ---------------------------------------------------------------------------------------------------- oracles
def channel_information_oracle(X, GW, H, ls):
    """(n, k, k) fp64 A_c[a, b] = sum_j x_cj h_aj h_bj / y_cj^2 with g = max(GW, ls), h = max(H, ls), y = g h."""
    X = np.asarray(X, dtype=np.float64)
    g = np.maximum(np.asarray(GW, np.float64), ls)
    h = np.maximum(np.asarray(H, np.float64), ls)
    Wt = X / (g @ h) ** 2
    return np.einsum("cj,aj,bj->cab", Wt, h, h)


def pack(A):
    """(n, k, k) -> (k(k+1)/2, n) packed upper triangles, row by row (the device layout)."""
    iu = np.triu_indices(A.shape[1])
    return np.ascontiguousarray(A[:, iu[0], iu[1]].T)


def dense_information(X, G, W, H, ls):
    """F = J^T diag(x / y^2) J with J[(c, j), (e, a)] = dy_cj / dW_ea = G_ce h_aj (the clamped model, factors fixed);
    (m k, m k), index e k + a."""
    g = np.maximum(G @ W, ls)
    h = np.maximum(H, ls)
    y = g @ h
    n, m = G.shape
    k = W.shape[1]
    J = np.einsum("ce,aj->cjea", G, h).reshape(n * X.shape[1], m * k)
    return J.T @ ((X / y ** 2).reshape(-1)[:, None] * J)


def constraint_matrix(free, rows):
    """(r, m k) rows of the simplex constraints over the free entries; a column without a free entry has none."""
    m, k = free.shape
    in_S = np.zeros(m, dtype=bool)
    if rows is not None:
        in_S[rows] = True
    out = []
    for a in range(k):
        r = np.zeros((m, k))
        r[in_S & free[:, a], a] = 1.0
        if r.any():
            out.append(r.reshape(-1))
    return np.array(out).reshape(-1, m * k)


def nullspace_covariance(F, free, rows):
    """C = U (U^T F U)^-1 U^T, U an orthonormal basis of the free directions that satisfy the constraints."""
    mk = F.shape[0]
    P = np.eye(mk)[:, free.reshape(-1)]                       # free coordinates
    Acon = constraint_matrix(free, rows) @ P
    if Acon.shape[0]:
        _, s, Vt = np.linalg.svd(Acon)
        N = Vt[Acon.shape[0]:].T
    else:
        N = np.eye(P.shape[1])
    U = P @ N
    return U @ np.linalg.inv(U.T @ F @ U) @ U.T


def _problem(n=30, m=4, k=3, p=50, seed=0, counts=400.0):
    rng = np.random.default_rng(seed)
    G = rng.uniform(0.0, 1.0, size=(n, m))
    W = rng.uniform(0.05, 1.0, size=(m, k))
    W /= W.sum(0, keepdims=True)
    H = rng.uniform(0.0, 1.0, size=(k, p))
    H[0, ::5] = 0.0                                           # clamped to log_shift
    X = rng.poisson(counts * np.maximum(G @ W, 1e-3) @ np.maximum(H, 1e-3)).astype(np.float64)
    return X, G, W, H


# ---------------------------------------------------------------------------------------------------- estimator
@pytest.mark.parametrize("hspy_comp", [False, True])
def test_method_exists_for_both_layouts(hspy_comp):
    assert callable(getattr(_est(hspy_comp=hspy_comp), "phase_uncertainty", None))


def test_phase_uncertainty_is_exported():
    import espm_b200
    assert "PhaseUncertainty" in espm_b200.__all__
    assert espm_b200.PhaseUncertainty._fields == ("std", "covariance", "information", "spectrum_std")


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
    monkeypatch.delattr(SmoothNMF, "phase_uncertainty")
    without = _check_names(_est(n_components=3, hspy_comp=hspy_comp))
    assert with_method and with_method == without


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_unfitted_raises_before_device_work(hspy_comp):
    with pytest.raises(NotFittedError):
        _est(hspy_comp=hspy_comp).phase_uncertainty(np.ones((40, 12)))


@pytest.mark.parametrize("hspy_comp", [False, True])
def test_channel_count_must_match_the_fitted_model(hspy_comp):
    est = _fake_fitted(n=40, hspy_comp=hspy_comp)
    X = np.ones((39, 12))
    with pytest.raises(ValueError, match="39 channels.*40"):
        est.phase_uncertainty(X.T if hspy_comp else X)


def test_pixel_count_must_match_H_when_H_is_omitted():
    est = _fake_fitted(n=40, p=12)
    with pytest.raises(ValueError, match="13 pixels.*12"):
        est.phase_uncertainty(np.ones((40, 13)))


@pytest.mark.parametrize("shape", [(3, 12), (2, 13), (13, 3)])
def test_H_shape_is_checked(shape):
    est = _fake_fitted(n=40, k=3, p=12)
    with pytest.raises(ValueError, match="H has shape"):
        est.phase_uncertainty(np.ones((40, 13)), H=np.ones(shape))


@pytest.mark.parametrize("simplex_W", [False, True])
def test_valid_call_reaches_the_device(simplex_W):
    import torch
    from espm_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("this machine has a GPU: the call would run")
    est = _fake_fitted(n=40, k=3, p=12, simplex_W=simplex_W)
    with pytest.raises(_lib.EspmError, match="needs a CUDA device"):
        est.phase_uncertainty(np.ones((40, 13)), H=np.ones((3, 13)))


@pytest.mark.parametrize("name, ctype_of", [
    ("espm_phase_info_scratch", {"int64_t* bytes_out": "i64p"}),
    ("espm_phase_info", {"double* out": "vp", "void* scratch": "vp", "void* stream": "vp"}),
])
def test_lib_signature_matches_header(name, ctype_of):
    from espm_b200 import _lib
    header = open(os.path.join(ROOT, "include", "espm_b200.h")).read()
    m = re.search(r"int\s+%s\(([^)]*)\);" % name, header)
    assert m
    args = [a.strip() for a in m.group(1).split(",")]
    kinds = {"vp": ctypes.c_void_p, "i64p": ctypes.POINTER(ctypes.c_int64)}
    ctype = {"const espm_state* st": ctypes.POINTER(_lib.EspmState)}
    ctype.update({a: kinds[v] for a, v in ctype_of.items()})
    restype, argtypes = _lib._EXPORTS[name]
    assert restype is ctypes.c_int
    assert argtypes == [ctype[a] for a in args]


# ---------------------------------------------------------------------------------------------------- host algebra
def test_per_channel_information_assembles_the_dense_jacobian_information():
    X, G, W, H = _problem()
    from espm_b200.host import phase_covariance
    A = channel_information_oracle(X, G @ W, H, 1e-3)
    F = dense_information(X, G, W, H, 1e-3)
    m, k = W.shape
    _, _, info, _ = phase_covariance(pack(A), G, np.ones((m, k), bool), None)
    assert info.shape == (m, k, m, k)
    assert np.max(np.abs(info.reshape(m * k, m * k) - F)) <= 1e-12 * np.abs(F).max()


@pytest.mark.parametrize("with_fixed", [False, True])
def test_constrained_covariance_matches_the_nullspace_formula(with_fixed):
    from espm_b200.host import phase_covariance
    X, G, W, H = _problem(seed=1)
    m, k = W.shape
    free = np.ones((m, k), bool)
    if with_fixed:
        free[1, 0] = free[3, 2] = False
    rows = np.array([0, 2, 3])                               # a physical model's simplex rows
    std, C, info, spec = phase_covariance(pack(channel_information_oracle(X, G @ W, H, 1e-3)), G, free, rows)
    F = info.reshape(m * k, m * k)
    Cf = C.reshape(m * k, m * k)
    ref = nullspace_covariance(F, free, rows)
    scale = np.abs(np.linalg.inv(F[np.ix_(free.reshape(-1), free.reshape(-1))])).max()
    assert np.max(np.abs(Cf - ref)) <= 1e-10 * scale
    assert np.max(np.abs(constraint_matrix(free, rows) @ Cf)) <= 1e-10 * scale
    assert np.array_equal(Cf, Cf.T)
    assert np.allclose(std, np.sqrt(np.diag(ref)).reshape(m, k), rtol=1e-8, atol=1e-12 * np.sqrt(scale))
    assert np.all(std[~free] == 0.0) and np.all(C[~free] == 0.0) and np.all(C[:, :, ~free] == 0.0)
    for a in range(k):
        band = np.sqrt(np.einsum("ce,ef,cf->c", G, C[:, a, :, a], G))
        assert np.allclose(spec[:, a], band, rtol=1e-10, atol=0)


@pytest.mark.parametrize("simplex", [False, True])
@pytest.mark.parametrize("with_fixed", [False, True])
def test_identity_G_blocks_equal_the_dense_projection(simplex, with_fixed):
    from espm_b200.host import phase_covariance, unpack_triangles
    n, k = 12, 3
    X, _, W, H = _problem(n=n, m=n, k=k, p=80, seed=2)
    G = np.eye(n)
    free = np.ones((n, k), bool)
    if with_fixed:
        free[2, 1] = free[5, :] = False
    rows = np.arange(n) if simplex else None
    A = channel_information_oracle(X, W, H, 1e-3)
    std, C, info, spec = phase_covariance(pack(A), None, free, rows)
    assert std.shape == (n, k) and C.shape == (n, k, k) and info.shape == (n, k, k) and spec.shape == (n, k)
    F = dense_information(X, G, W, H, 1e-3)
    ref = nullspace_covariance(F, free, rows).reshape(n, k, n, k)
    blocks = np.stack([ref[c, :, c, :] for c in range(n)])
    scale = np.abs(blocks).max()
    assert np.max(np.abs(C - blocks)) <= 1e-10 * scale
    assert np.array_equal(info, unpack_triangles(pack(A), k))
    assert np.array_equal(spec, std)
    assert np.all(std[~free] == 0.0)
    assert np.allclose(std, np.sqrt(np.einsum("caa->ca", blocks)), rtol=1e-8, atol=1e-12)


def test_singular_information_is_nan():
    from espm_b200.host import phase_covariance
    X, G, W, H = _problem(seed=3)
    m, k = W.shape
    G[:, 1] = G[:, 0]                                         # two identical elements: F is singular
    std, C, info, spec = phase_covariance(pack(channel_information_oracle(X, G @ W, H, 1e-3)), G,
                                          np.ones((m, k), bool), np.arange(m))
    assert np.all(np.isnan(std)) and np.all(np.isnan(C)) and np.all(np.isnan(spec))
    assert np.all(np.isfinite(info))


@pytest.mark.parametrize("simplex", [False, True])
def test_identity_G_channel_without_counts_is_nan_there_only(simplex):
    """The channel is NaN; under simplex_W the others equal the projection with that channel's entries fixed."""
    from espm_b200.host import phase_covariance
    n, k = 10, 3
    X, _, W, H = _problem(n=n, m=n, k=k, p=80, seed=4)
    X[6] = 0.0
    rows = np.arange(n) if simplex else None
    A = channel_information_oracle(X, W, H, 1e-3)
    std, C, _, _ = phase_covariance(pack(A), None, np.ones((n, k), bool), rows)
    assert np.all(np.isnan(std[6])) and np.all(np.isnan(C[6]))
    rest = np.arange(n) != 6
    assert np.all(np.isfinite(std[rest])) and np.all(np.isfinite(C[rest]))
    free = np.ones((n, k), bool)
    free[6] = False
    _, ref, _, _ = phase_covariance(pack(A), None, free, rows)
    assert np.array_equal(C[rest], ref[rest])


def test_all_entries_fixed_gives_zero_covariance():
    from espm_b200.host import phase_covariance
    X, G, W, H = _problem(seed=5)
    m, k = W.shape
    std, C, _, spec = phase_covariance(pack(channel_information_oracle(X, G @ W, H, 1e-3)), G,
                                       np.zeros((m, k), bool), np.arange(m))
    assert np.all(std == 0.0) and np.all(C == 0.0) and np.all(spec == 0.0)
