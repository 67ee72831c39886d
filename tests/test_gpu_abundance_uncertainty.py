"""SmoothNMF.abundance_uncertainty on the device (espm_abundance_info) against NumPy fp64:

    F_j[a, b] = sum_c x_cj g_ca g_cb / y_cj^2,  g = max(G W, ls),  y = g max(H, ls),
    C_j = F_j^-1, or with simplex_H  F_j^-1 - (F_j^-1 1)(F_j^-1 1)^T / (1^T F_j^-1 1),  std = sqrt(diag C_j).

``information`` is compared entry by entry with the oracle of F (every term is >= 0, so a relative bound holds for
every entry).  ``covariance`` and ``std`` are compared with NumPy's inverse and projection of the device's own F, to
1e-10 of max |F_j^-1| (the projection cancels entries of that size), which keeps F_j's conditioning out of the
tolerance."""
import contextlib
import io
import os
import socket
import sys

import numpy as np
import pytest

from test_abundance_uncertainty_cpu import covariance_oracle, information_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, M = 160, 6
SHAPE, NEW_SHAPE = (13, 11), (12, 14)


def _G(seed=5, n=N):
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 1, n)
    G = np.zeros((n, M))
    for j in range(M - 2):
        c, s = rng.uniform(0.05, 0.95), rng.uniform(0.01, 0.04)
        G[:, j] = np.exp(-0.5 * ((x - c) / s) ** 2)
    G[:, M - 2] = np.exp(-3 * x) + 0.05
    G[:, M - 1] = (1 - x) * 0.5 + 0.05
    return G


def _image(seed, shape, G, k, counts=20.0):
    rng = np.random.default_rng(seed)
    p = shape[0] * shape[1]
    Wt = np.random.default_rng(11).uniform(size=(G.shape[1], k))
    Ht = rng.uniform(size=(k, p)) ** 2
    Ht /= Ht.sum(0, keepdims=True)
    lam = G @ Wt @ Ht
    return rng.poisson(lam / lam.sum(0, keepdims=True) * counts).astype(np.float64)


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def _fit(k=3, identity_G=False, dtype=np.float64, hspy_comp=False, counts=2000.0, **kw):
    """(fitted estimator, X (n, p) it was fitted on).  With identity G the k phases are k free spectra: F has full rank
    for every k (G W of rank <= M = 6 otherwise)."""
    from espm_b200 import SmoothNMF
    if kw.get("simplex_H"):
        kw.setdefault("simplex_W", False)                 # with both, the estimator drops simplex_H (as the reference)
    G = _G()
    X = _image(1, SHAPE, np.eye(N) if identity_G else G, k, counts).astype(dtype)
    m = N if identity_G else M
    W0 = np.random.default_rng(3).uniform(0.05, 1.0, size=(m, k)).astype(dtype)
    H0 = np.random.default_rng(4).uniform(0.05, 1.0, size=(k, X.shape[1]))
    H0 = (H0 / H0.sum(0, keepdims=True)).astype(dtype)
    est = SmoothNMF(n_components=k, G=None if identity_G else G.astype(dtype), hspy_comp=hspy_comp, max_iter=10,
                    tol=0, no_stop_criterion=True, verbose=0, **kw)
    _quiet(est.fit_transform, X.T if hspy_comp else X, W=W0, H=H0)
    return est, X


def _GW(est):
    return est.W_ if est._identity_G else est.G_ @ est.W_


def _check(u, X, GW, H, ls, simplex, tol_info):
    k, p = np.shape(H)
    assert u.std.shape == (k, p) and u.covariance.shape == (p, k, k) and u.information.shape == (p, k, k)
    for a in u:
        assert a.dtype == np.float64
    F = information_oracle(X, GW, H, ls)
    err = np.max(np.abs(u.information - F) / np.maximum(np.abs(F), 1e-300))
    assert err <= tol_info, "information: %.3e > %.1e" % (err, tol_info)
    assert np.array_equal(u.information, np.swapaxes(u.information, 1, 2))
    assert np.all(np.isfinite(u.std)), "singular pixels: %s" % np.flatnonzero(~np.isfinite(u.std[0]))
    C = covariance_oracle(u.information, simplex)
    scale = np.abs(covariance_oracle(u.information, False)).max(axis=(1, 2))     # max |F_j^-1|
    cerr = np.max(np.abs(u.covariance - C).max(axis=(1, 2)) / scale)
    assert cerr <= 1e-10, "covariance: %.3e" % cerr
    assert np.array_equal(u.covariance, np.swapaxes(u.covariance, 1, 2))
    serr = np.max(np.abs(u.std - np.sqrt(np.diagonal(C, axis1=1, axis2=2)).T) / np.sqrt(scale))
    assert serr <= 1e-10, "std: %.3e" % serr
    if simplex:
        assert np.max(np.abs(u.covariance.sum(2)).max(1) / scale) <= 1e-10


CASES = {
    "simplex_H_lap_mu": dict(simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE),
    "no_simplex": dict(),
    "identity_G": dict(identity_G=True),
    "normalize": dict(normalize=True, simplex_H=True),
    "hspy_comp": dict(hspy_comp=True, simplex_H=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_fp64_matches_oracle(case):
    kw = CASES[case]
    est, X = _fit(**kw)
    Xin = X.T if kw.get("hspy_comp") else X
    u = _quiet(est.abundance_uncertainty, Xin)
    assert est.simplex_H == bool(kw.get("simplex_H"))
    _check(u, X, _GW(est), est.H_, est.log_shift, est.simplex_H, 1e-12)


@pytest.mark.parametrize("k", [2, 3, 4, 5, 6, 8, 12, 16])
@pytest.mark.parametrize("simplex_H", [False, True], ids=["free", "simplex"])
def test_every_padded_k(k, simplex_H):
    est, X = _fit(k=k, identity_G=True, simplex_H=simplex_H, counts=20000.0)
    assert est.simplex_H == simplex_H
    _check(est.abundance_uncertainty(X), X, _GW(est), est.H_, est.log_shift, simplex_H, 1e-12)


@pytest.mark.parametrize("k", [4, 8])
def test_fp32_matches_oracle_on_rounded_inputs(k):
    est, X = _fit(k=k, dtype=np.float32, identity_G=k > 6, simplex_H=True)
    assert est.W_.dtype == np.float32
    u = est.abundance_uncertainty(X)
    GW = est.W_ if est._identity_G else est.G_.astype(np.float32) @ est.W_.astype(np.float32)
    _check(u, X, GW, est.H_.astype(np.float32), est.log_shift, True, 2e-5)


def test_hspy_comp_layout_gives_identical_arrays():
    est, X = _fit(simplex_H=True, mu=0.05)
    est_h, X_h = _fit(simplex_H=True, mu=0.05, hspy_comp=True)
    a = est.abundance_uncertainty(X)
    b = est_h.abundance_uncertainty(X_h.T)
    assert np.array_equal(est.H_, est_h.H_)
    for f in a._fields:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


def _recording_storage(monkeypatch):
    """Records the X storage of every engine abundance_uncertainty builds."""
    from espm_b200.engine import FitEngine
    seen = []
    make = FitEngine.for_statistics

    def wrapped(*a, **kw):
        eng = make(*a, **kw)
        seen.append(eng.x_storage)
        return eng
    monkeypatch.setattr(FitEngine, "for_statistics", wrapped)
    return seen


@pytest.mark.parametrize("storage", ["uint8", "uint16"])
def test_compact_storage_equals_dense(storage, monkeypatch):
    import espm_b200
    est, X = _fit(dtype=np.float32, simplex_H=True, counts=200.0)
    seen = _recording_storage(monkeypatch)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = "dense"
        dense = est.abundance_uncertainty(X)
        espm_b200.config.x_storage = storage
        compact = est.abundance_uncertainty(X)
    finally:
        espm_b200.config.x_storage = keep
    assert seen == ["dense", storage]
    for f in dense._fields:
        assert np.allclose(getattr(compact, f), getattr(dense, f), rtol=1e-6, atol=0), f


# (X storage, arithmetic) pairs of the kernel instances: f64 / f64 (16-channel stages), f32 / f32, uint8 / f32,
# uint16 / f32, f32 / f64
PAIRS = {"f64": (np.float64, np.float64, "dense"), "f32": (np.float32, np.float32, "dense"),
         "uint8": (np.float32, np.float32, "uint8"), "uint16": (np.float32, np.float32, "uint16"),
         "f32_storage_f64_arith": (np.float32, np.float64, "dense")}


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("n", [150, 161])
@pytest.mark.parametrize("simplex", [False, True], ids=["free", "simplex"])
def test_padded_channels_never_count(pair, n, simplex):
    """n not a multiple of 32 (nor of 16): the pad channels of the last stage hold x = 0 and must reach no sum; p = 143
    also leaves pad pixels in the last tile."""
    import espm_b200
    from espm_b200 import _lib as L
    from espm_b200.engine import FitEngine
    xdt, cdt, storage = PAIRS[pair]
    k = 5
    G = _G(n=n)
    X = _image(7, SHAPE, G, k, counts=3000.0)
    rng = np.random.default_rng(8)
    W = rng.uniform(0.05, 1.0, size=(M, k))
    H = rng.uniform(0.05, 1.0, size=(k, X.shape[1]))
    H[1, ::4] = 0.0                                          # clamped to log_shift
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X.astype(xdt), G.astype(cdt), W.astype(cdt), H.astype(cdt), log_shift=1e-3)
        assert eng.x_storage == storage
        assert eng.c_code == (L.F64 if cdt == np.float64 else L.F32)
        assert eng.st.n_pad > n
        out = eng.abundance_information(simplex).cpu().numpy()
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    nt = k * (k + 1) // 2
    assert out.shape == (k + 2 * nt, X.shape[1])
    iu = np.triu_indices(k)
    F = information_oracle(X.astype(xdt), G.astype(cdt) @ W.astype(cdt), H.astype(cdt), 1e-3)
    got = out[k + nt:].T
    err = np.max(np.abs(got - F[:, iu[0], iu[1]]) / F[:, iu[0], iu[1]])
    assert err <= (1e-12 if cdt == np.float64 else 2e-5), err
    Fd = np.zeros_like(F)
    Fd[:, iu[0], iu[1]] = got
    Fd[:, iu[1], iu[0]] = got
    C = covariance_oracle(Fd, simplex)
    scale = np.abs(covariance_oracle(Fd, False)).max(axis=(1, 2))
    assert np.max(np.abs(out[k:k + nt].T - C[:, iu[0], iu[1]]).max(1) / scale) <= 1e-10
    assert np.max(np.abs(out[:k] - np.sqrt(np.diagonal(C, axis1=1, axis2=2)).T) / np.sqrt(scale)) <= 1e-10


def test_pixel_without_counts_is_nan_there_only():
    est, X = _fit(simplex_H=True)
    X = X.copy()
    X[:, 17] = 0.0
    u = est.abundance_uncertainty(X)
    bad = np.zeros(X.shape[1], bool)
    bad[17] = True
    assert np.all(np.isnan(u.std[:, bad])) and np.all(np.isnan(u.covariance[bad]))
    assert np.all(np.isfinite(u.std[:, ~bad])) and np.all(np.isfinite(u.covariance[~bad]))
    assert np.all(u.information[17] == 0.0)
    _check(type(u)(u.std[:, ~bad], u.covariance[~bad], u.information[~bad]), X[:, ~bad], _GW(est), est.H_[:, ~bad],
           est.log_shift, True, 1e-12)


def test_new_image_with_transformed_maps():
    est, _ = _fit(hspy_comp=True, simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE)
    XB = _image(2, NEW_SHAPE, _G(), 3, counts=2000.0)
    H = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE).T
    u = est.abundance_uncertainty(XB.T, H=H)
    assert u.std.shape == (3, XB.shape[1])
    _check(u, XB, _GW(est), H, est.log_shift, True, 1e-12)


def test_no_side_effects_and_deterministic():
    est, X = _fit(simplex_H=True, mu=0.05)
    _ = est.X_                                           # materialise the lazy attribute too
    before = {k: v for k, v in est.__dict__.items()}
    copies = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in before.items()}
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        a = est.abundance_uncertainty(X)
        b = est.abundance_uncertainty(X)
    assert out.getvalue() == ""
    assert set(est.__dict__) == set(before)
    for k, v in est.__dict__.items():
        assert v is before[k], k
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, copies[k]), k
    for f in a._fields:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


def test_invalid_data_raises_fit_errors():
    est, X = _fit()
    for bad, msg in ((np.nan, "NaN"), (np.inf, "infinity"), (-1.0, "Negative")):
        Xb = X.copy()
        Xb[3, 7] = bad
        with pytest.raises(ValueError, match=msg):
            est.abundance_uncertainty(Xb)


# ---------------------------------------------------------------------------------------------------- calibration
@pytest.mark.parametrize("simplex_H", [False, True], ids=["free", "simplex"])
def test_std_is_calibrated(simplex_H):
    """4000 pixels share one interior H_true (every phase >= 0.15) at ~1e4 counts per pixel; with lambda_L = mu = 0 the
    pixels are independent, so the spread of the fitted H_ across pixels is the sampling spread of the per-pixel maximum
    likelihood estimate, whose asymptotic standard deviation is what ``std`` reports.  The empirical standard deviation of
    4000 samples has a relative sampling error of 1 / sqrt(2 * 3999) = 1.1 %; the MLE's deviation from its Gaussian limit
    at 1e4 counts, and evaluating F at the estimate instead of the truth, add well under 1 %.  10 % is thus about nine
    standard errors of the check itself, while a wrong factor (a missing x / y, the unprojected simplex covariance, or the
    expected instead of observed information off by the square root of the count scale) moves the ratio by far more."""
    from espm_b200 import SmoothNMF
    n, k, p, counts = N, 3, 4000, 1e4
    x = np.linspace(0, 1, n)
    W = np.stack([np.exp(-0.5 * ((x - c) / 0.05) ** 2) + 0.05 for c in (0.2, 0.5, 0.8)], axis=1)
    h_true = np.array([0.45, 0.35, 0.2])
    W *= counts / (W @ h_true).sum()                         # sum_c (W h_true)_c = counts
    lam = np.repeat((W @ h_true)[:, None], p, axis=1)
    X = np.random.default_rng(12).poisson(lam).astype(np.float64)
    H0 = np.repeat(np.full((k, 1), 1.0 / k), p, axis=1)
    est = SmoothNMF(n_components=k, G=None, fixed_W=W, simplex_H=simplex_H, simplex_W=False, lambda_L=0.0, mu=0.0,
                    max_iter=3000, tol=0, no_stop_criterion=True, verbose=0)
    _quiet(est.fit_transform, X, W=W, H=H0)
    u = est.abundance_uncertainty(X)
    assert np.all(np.isfinite(u.std))
    emp = est.H_.std(axis=1, ddof=1)
    pred = u.std.mean(axis=1)
    assert np.max(np.abs(est.H_.mean(1) - h_true) / h_true) < 0.01
    ratio = emp / pred
    assert np.all(np.abs(ratio - 1) <= 0.10), ratio


# ---------------------------------------------------------------------------------------------------- full size
@pytest.mark.parametrize("storage", ["dense", "uint8"])
def test_c3_against_numpy_sample(storage):
    import torch
    import espm_b200
    from espm_b200 import synth
    from espm_b200.engine import FitEngine
    nx = ny = 512
    n, k, seed, ls = 2048, 4, 93, 1e-14
    prob = synth.make_problem(nx, ny, n, k, 12, seed=seed)
    G = prob["G_full"].astype(np.float32)
    X = synth.poisson_X_torch(prob, 0, nx * ny, seed, torch.device("cuda", 0), torch.float32)
    GWt = prob["G_full"] @ prob["W_true"]                 # model = the Poisson mean of X
    W = (prob["W_true"] / GWt.sum(0) * prob["dens"] * prob["counts"]).astype(np.float32)
    H = prob["H_true"].astype(np.float32)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X, G, W, H, log_shift=ls)
        assert eng.x_storage == storage
        out = eng.abundance_information(True).cpu().numpy()
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    sample = np.sort(np.random.default_rng(7).choice(nx * ny, 4096, replace=False))
    Xs = X[:, torch.from_numpy(sample).to(X.device)].cpu().numpy()
    del X, eng
    nt = k * (k + 1) // 2
    iu = np.triu_indices(k)
    F = information_oracle(Xs, G @ W, H[:, sample], ls)[:, iu[0], iu[1]]
    got = out[k + nt:, sample].T
    assert np.max(np.abs(got - F) / F) <= 2e-5
    # some pixels of this image have cond(F_j) up to ~1e10, where the fp32 rounding of F (~1e-6) can make F_j
    # indefinite and the pixel is reported singular; every pixel with cond(F_j) < 1e4 must have finite errors
    Ff = np.zeros((sample.size, k, k))
    Ff[:, iu[0], iu[1]] = F
    Ff[:, iu[1], iu[0]] = F
    ev = np.linalg.eigvalsh(Ff)
    well = ev[:, -1] < 1e4 * ev[:, 0]
    assert well.mean() > 0.5
    assert np.all(np.isfinite(out[:k, sample[well]]))


# ---------------------------------------------------------------------------------------------------- sharded
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out_dir, peer):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    tests = os.path.join(ROOT, "tests")
    if tests not in sys.path:
        sys.path.insert(0, tests)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["ESPM_B200_PEER"] = "1" if peer else "0"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import espm_b200
        est, X = _fit(simplex_H=True, mu=0.05)               # the fit is sharded as well
        s = est.abundance_uncertainty(X)
        keep = espm_b200.config.distributed
        espm_b200.config.distributed = False
        u = est.abundance_uncertainty(X)
        espm_b200.config.distributed = keep
        res = {}
        for f in s._fields:
            res["s_" + f], res["u_" + f] = getattr(s, f), getattr(u, f)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False], ids=["peer-memory", "nccl"])
def test_sharded_abundance_uncertainty(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer), nprocs=2, join=True)
    res = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    from espm_b200 import AbundanceUncertainty
    for f in AbundanceUncertainty._fields:
        assert np.array_equal(res[0]["s_" + f], res[1]["s_" + f]), f
        assert np.array_equal(res[0]["s_" + f], res[0]["u_" + f]), f
