"""SmoothNMF.phase_uncertainty on the device (espm_phase_info) against NumPy fp64:

    A_c[a, b] = sum_j x_cj h_aj h_bj / y_cj^2,  g = max(G W, ls),  h = max(H, ls),  y = g h,
    F[(e,a),(f,b)] = sum_c G_ce G_cf A_c[a, b],  C = the constrained inverse of F on the free entries.

``information`` (through A) is compared entry by entry with the oracle (every term is >= 0, so a relative bound holds
for every entry).  ``covariance`` and ``std`` are compared with the null-space formula of the CPU tests evaluated on the
device's own F, to 1e-10 of max |F_phi^-1|, which keeps F's conditioning out of the tolerance."""
import contextlib
import io
import os
import socket
import sys

import numpy as np
import pytest

from test_gpu_abundance_uncertainty import PAIRS, SHAPE, NEW_SHAPE, N, M, _G, _image, _quiet
from test_phase_uncertainty_cpu import (channel_information_oracle, constraint_matrix, nullspace_covariance, pack)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class FakeModel:
    """A physical model whose simplex rows are all but the last two (the background columns), as test_gpu_parity.py."""
    def __init__(self, G):
        self.G = G

    def NMF_initialize_W(self, D):
        return np.abs(np.linalg.lstsq(self.G, D, rcond=None)[0])

    def NMF_simplex(self):
        return list(range(self.G.shape[1] - 2))

    def NMF_update(self, W=None):
        return self.G


def _fit(k=3, identity_G=False, dtype=np.float64, hspy_comp=False, counts=2000.0, physics=False, n=N, **kw):
    """(fitted estimator, X (n, p) it was fitted on)."""
    from espm_b200 import SmoothNMF
    G = _G(n=n)
    X = _image(1, SHAPE, np.eye(n) if identity_G else G, k, counts).astype(dtype)
    m = n if identity_G else M
    W0 = np.random.default_rng(3).uniform(0.05, 1.0, size=(m, k))
    W0 = (W0 / W0.sum(0, keepdims=True)).astype(dtype)
    H0 = np.random.default_rng(4).uniform(0.05, 1.0, size=(k, X.shape[1])).astype(dtype)
    Gin = None if identity_G else (FakeModel(G.astype(dtype)) if physics else G.astype(dtype))
    est = SmoothNMF(n_components=k, G=Gin, hspy_comp=hspy_comp, max_iter=10, tol=0, no_stop_criterion=True, verbose=0,
                    **kw)
    _quiet(est.fit_transform, X.T if hspy_comp else X, W=W0, H=H0)
    return est, X


def _free_rows(est):
    m, k = est.W_.shape
    free = np.ones((m, k), bool) if est.fixed_W is None else np.asarray(est.fixed_W) < 0
    rows = None
    if est.simplex_W:
        rows = np.arange(m) if est.physics_model_ is None else np.asarray(est.physics_model_.NMF_simplex())
    return free, rows


def _GW(est):
    return est.W_ if est._identity_G else est.G_ @ est.W_


def _check(u, est, X, H, tol_A):
    """A against the oracle, C / std / spectrum_std against the null-space formula on the device's own F."""
    m, k = est.W_.shape
    n = X.shape[0]
    free, rows = _free_rows(est)
    for a in u:
        assert a.dtype == np.float64
    A = channel_information_oracle(X, _GW(est), H, est.log_shift)
    if est._identity_G:
        assert u.std.shape == (n, k) and u.covariance.shape == (n, k, k) and u.information.shape == (n, k, k)
        Ad = u.information
        F = np.zeros((n * k, n * k))
        for c in range(n):
            F[c * k:(c + 1) * k, c * k:(c + 1) * k] = Ad[c]
        G = np.eye(n)
    else:
        assert u.std.shape == (m, k) and u.covariance.shape == (m, k, m, k) and u.information.shape == (m, k, m, k)
        F = u.information.reshape(m * k, m * k)
        Ad = None
        G = est.G_
    assert u.spectrum_std.shape == (n, k)
    got = pack(Ad) if Ad is not None else None
    if got is None:                                   # real G: F = sum_c G_ce G_cf A_c from the oracle's A
        Fo = np.einsum("ce,cf,cab->eafb", G, G, A).reshape(m * k, m * k)
        err = np.max(np.abs(F - Fo) / np.maximum(np.abs(Fo), 1e-300))
    else:
        ref = pack(A)
        err = np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300))
    assert err <= tol_A, "information: %.3e > %.1e" % (err, tol_A)
    assert np.all(np.isfinite(u.std))
    C = nullspace_covariance(F, free, rows)
    phi = free.reshape(-1)
    scale = np.abs(np.linalg.inv(F[np.ix_(phi, phi)])).max()
    if est._identity_G:
        Cd = np.stack([C[c * k:(c + 1) * k, c * k:(c + 1) * k] for c in range(n)])
        cerr = np.max(np.abs(u.covariance - Cd)) / scale
    else:
        cerr = np.max(np.abs(u.covariance.reshape(m * k, m * k) - C)) / scale
        Acon = constraint_matrix(free, rows)
        if Acon.shape[0]:
            assert np.max(np.abs(Acon @ u.covariance.reshape(m * k, m * k))) <= 1e-10 * scale
    assert cerr <= 1e-10, "covariance: %.3e" % cerr
    serr = np.max(np.abs(u.std.reshape(-1) - np.sqrt(np.maximum(np.diag(C), 0.0)))) / np.sqrt(scale)
    assert serr <= 1e-10, "std: %.3e" % serr
    assert np.all(u.std[~free] == 0.0)
    Cr = C.reshape(m, k, m, k)
    var = np.stack([np.einsum("ce,ef,cf->c", G, Cr[:, a, :, a], G) for a in range(k)], 1)
    assert np.max(np.abs(u.spectrum_std ** 2 - var)) <= 1e-9 * scale * np.abs(G).sum(1).max() ** 2


CASES = {
    "simplex_W_all_rows": dict(),
    "simplex_W_physics_rows": dict(physics=True),
    "simplex_H": dict(simplex_H=True, simplex_W=False, lambda_L=2.0, mu=0.05, shape_2d=SHAPE),
    "identity_G_free": dict(identity_G=True, simplex_W=False),
    "identity_G_simplex_W": dict(identity_G=True),
    "fixed_W": dict(fixed_W=np.where(np.arange(M * 3).reshape(M, 3) % 5 == 0, 0.3, -1.0)),
    "normalize": dict(normalize=True),
    "hspy_comp": dict(hspy_comp=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_fp64_matches_oracle(case):
    kw = dict(CASES[case])
    est, X = _fit(**kw)
    u = _quiet(est.phase_uncertainty, X.T if kw.get("hspy_comp") else X)
    if case == "simplex_W_physics_rows":
        assert est.physics_model_ is not None and est.simplex_W
    _check(u, est, X, est.H_, 1e-12)


@pytest.mark.parametrize("k", [2, 3, 4, 5, 6, 8, 12, 16])
def test_every_padded_k(k):
    est, X = _fit(k=k, identity_G=True, n=64, counts=20000.0)
    _check(est.phase_uncertainty(X), est, X, est.H_, 1e-12)


@pytest.mark.parametrize("k", [4, 8])
def test_fp32_matches_oracle_on_rounded_inputs(k):
    est, X = _fit(k=k, dtype=np.float32, identity_G=True, n=64, counts=20000.0)
    assert est.W_.dtype == np.float32
    u = est.phase_uncertainty(X)
    A = channel_information_oracle(X, est.W_.astype(np.float32), est.H_.astype(np.float32), est.log_shift)
    ref = pack(A)
    assert np.max(np.abs(pack(u.information) - ref) / ref) <= 2e-5


def _recording_storage(monkeypatch):
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
    est, X = _fit(dtype=np.float32, counts=200.0)
    seen = _recording_storage(monkeypatch)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = "dense"
        dense = est.phase_uncertainty(X)
        espm_b200.config.x_storage = storage
        compact = est.phase_uncertainty(X)
    finally:
        espm_b200.config.x_storage = keep
    assert seen == ["dense", storage]
    for f in dense._fields:
        assert np.allclose(getattr(compact, f), getattr(dense, f), rtol=1e-6, atol=0), f


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("n", [150, 161])
def test_padded_channels_and_pixels_never_count(pair, n):
    """n not a multiple of 32 (nor of 16): the pad channels of the last stage hold x = 0 and are not returned; p = 143
    leaves pad pixels in the last tile, whose h = log_shift gives y > 0 and x = 0."""
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
        assert eng.st.n_pad > n and eng.p_loc % 128 != 0
        before = eng.n_launches
        out = eng.phase_information().cpu().numpy()
        assert eng.n_launches == before + 3
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    ref = pack(channel_information_oracle(X.astype(xdt), G.astype(cdt) @ W.astype(cdt), H.astype(cdt), 1e-3))
    assert out.shape == ref.shape == (k * (k + 1) // 2, n)
    assert np.max(np.abs(out - ref) / ref) <= (1e-12 if cdt == np.float64 else 2e-5)


def test_channel_without_counts_is_nan_there_only():
    from espm_b200.host import phase_covariance
    est, X = _fit(identity_G=True)
    X = X.copy()
    X[5] = 0.0
    u = est.phase_uncertainty(X)
    bad = np.arange(X.shape[0]) == 5
    assert np.all(np.isnan(u.std[bad])) and np.all(np.isnan(u.covariance[bad]))
    assert np.all(np.isfinite(u.std[~bad])) and np.all(np.isfinite(u.covariance[~bad]))
    assert np.all(u.information[5] == 0.0)
    A = channel_information_oracle(X, est.W_, est.H_, est.log_shift)
    assert np.max(np.abs(pack(u.information)[:, ~bad] - pack(A)[:, ~bad]) / pack(A)[:, ~bad]) <= 1e-12
    # the other channels: as if channel 5 were fixed (left out of M), from the device's own A
    free = np.ones(est.W_.shape, bool)
    free[5] = False
    _, C, _, _ = phase_covariance(pack(u.information), None, free, np.arange(X.shape[0]))
    assert np.allclose(u.covariance[~bad], C[~bad], rtol=1e-12, atol=0)


def test_new_image_with_transformed_maps():
    est, _ = _fit(hspy_comp=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE)
    XB = _image(2, NEW_SHAPE, _G(), 3, counts=2000.0)
    H = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE).T
    u = est.phase_uncertainty(XB.T, H=H)
    _check(u, est, XB, H, 1e-12)


def test_no_side_effects_and_deterministic():
    est, X = _fit(mu=0.05)
    _ = est.X_
    before = {k: v for k, v in est.__dict__.items()}
    copies = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in before.items()}
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        a = est.phase_uncertainty(X)
        b = est.phase_uncertainty(X)
    assert out.getvalue() == ""
    assert set(est.__dict__) == set(before)
    for k, v in est.__dict__.items():
        assert v is before[k], k
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, copies[k]), k
    for f in a._fields:
        assert np.array_equal(getattr(a, f), getattr(b, f), equal_nan=True), f


def test_invalid_data_raises_fit_errors():
    est, X = _fit()
    for bad, msg in ((np.nan, "NaN"), (np.inf, "infinity"), (-1.0, "Negative")):
        Xb = X.copy()
        Xb[3, 7] = bad
        with pytest.raises(ValueError, match=msg):
            est.phase_uncertainty(Xb)


# ---------------------------------------------------------------------------------------------------- calibration
def test_std_is_calibrated_identity_G():
    """Identity G with the maps fixed to H_true and no W constraint: every channel's row of W is estimated from its own
    counts only, so with all 2000 channels sharing one true row w, the fitted rows are 2000 independent samples of the
    maximum likelihood estimate of w, whose asymptotic standard deviation is what ``std`` reports.  The empirical
    standard deviation of 2000 samples has a relative sampling error of 1 / sqrt(2 * 1999) = 1.6 %; at ~1e4 counts per
    channel the MLE's deviation from its Gaussian limit, and evaluating A_c at the estimate, add well under 1 %.  10 %
    is thus about six standard errors of the check, while a wrong factor (a missing x / y, the expected instead of the
    observed information) moves the ratio by far more."""
    from espm_b200 import SmoothNMF
    n, k, p = 2000, 3, 400
    rng = np.random.default_rng(21)
    H = rng.dirichlet(np.full(k, 1.0), size=p).T
    w = np.array([0.45, 0.35, 0.2]) * (1e4 / H.sum(1).mean())  # ~1e4 counts per channel
    X = rng.poisson(np.repeat((w @ H)[None], n, axis=0)).astype(np.float64)
    W0 = np.full((n, k), w.mean())
    est = SmoothNMF(n_components=k, G=None, fixed_H=H, simplex_W=False, simplex_H=False, lambda_L=0.0, mu=0.0,
                    max_iter=3000, tol=0, no_stop_criterion=True, verbose=0)
    _quiet(est.fit_transform, X, W=W0, H=H.copy())
    u = est.phase_uncertainty(X, H=H)
    assert np.all(np.isfinite(u.std))
    assert np.max(np.abs(est.W_.mean(0) - w) / w) < 0.01
    ratio = est.W_.std(axis=0, ddof=1) / u.std.mean(axis=0)
    assert np.all(np.abs(ratio - 1) <= 0.10), ratio


def test_std_is_calibrated_real_G_simplex_W():
    """Real G of six separated peaks, maps fixed to H_true, simplex_W over all rows: 300 Poisson redraws of one image,
    each fitted; the spread of W_ across the redraws is the sampling spread of the constrained estimate, which ``std``
    (the projected bound) predicts.  The peaks keep F well conditioned, so that 400 multiplicative updates converge in
    every direction (nearly collinear columns, as the two smooth backgrounds of ``_G``, converge too slowly and leave
    the redraws closer together than the bound).  300 samples give the empirical standard deviation a relative sampling error of 1 / sqrt(598) = 4.1 %; the
    band, 15 %, is about 3.6 of those; ``std`` is averaged over every tenth redraw, so its own spread adds little."""
    from espm_b200 import SmoothNMF
    k, reps = 3, 300
    x = np.linspace(0, 1, N)
    G = np.stack([np.exp(-0.5 * ((x - c) / 0.05) ** 2) + 0.02 for c in np.linspace(0.1, 0.9, M)], axis=1)
    rng = np.random.default_rng(31)
    W = rng.uniform(0.3, 1.0, size=(M, k))
    W /= W.sum(0, keepdims=True)
    H = rng.dirichlet(np.ones(k), size=SHAPE[0] * SHAPE[1]).T * 300.0
    lam = G @ W @ H
    fits, stds = [], []
    for r in range(reps):
        X = np.random.default_rng(1000 + r).poisson(lam).astype(np.float64)
        est = SmoothNMF(n_components=k, G=G, fixed_H=H, simplex_W=True, lambda_L=0.0, mu=0.0, max_iter=400, tol=0,
                        no_stop_criterion=True, verbose=0)
        _quiet(est.fit_transform, X, W=np.full((M, k), 1.0 / M), H=H.copy())
        fits.append(est.W_.copy())
        if r % 10 == 0:
            stds.append(est.phase_uncertainty(X, H=H).std)
    fits, pred = np.array(fits), np.mean(stds, axis=0)
    assert np.all(np.isfinite(pred))
    ratio = fits.std(axis=0, ddof=1) / pred
    assert np.all(np.abs(ratio - 1) <= 0.15), ratio


# ---------------------------------------------------------------------------------------------------- full size
@pytest.mark.parametrize("storage", ["dense", "uint8"])
def test_c3_against_chunked_numpy(storage):
    import torch
    import espm_b200
    from espm_b200 import synth
    from espm_b200.engine import FitEngine
    nx = ny = 512
    n, k, seed, ls = 2048, 4, 93, 1e-14
    prob = synth.make_problem(nx, ny, n, k, 12, seed=seed)
    G = prob["G_full"].astype(np.float32)
    X = synth.poisson_X_torch(prob, 0, nx * ny, seed, torch.device("cuda", 0), torch.float32)
    GWt = prob["G_full"] @ prob["W_true"]
    W = (prob["W_true"] / GWt.sum(0) * prob["dens"] * prob["counts"]).astype(np.float32)
    H = prob["H_true"].astype(np.float32)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X, G, W, H, log_shift=ls)
        assert eng.x_storage == storage
        out = eng.phase_information().cpu().numpy()
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    g = np.maximum(G.astype(np.float64) @ W.astype(np.float64), ls)
    Hc = np.maximum(H.astype(np.float64), ls)
    iu = np.triu_indices(k)
    ref = np.zeros((n, iu[0].size))
    for a in range(0, nx * ny, 16384):
        h = Hc[:, a:a + 16384]
        x = X[:, a:a + 16384].double().cpu().numpy()
        ref += (x / (g @ h) ** 2) @ (h[iu[0]] * h[iu[1]]).T
    del X, eng
    ref = ref.T
    live = ref > 0
    assert live.any()
    assert np.all(out[~live] == 0.0)
    assert np.max(np.abs(out[live] - ref[live]) / ref[live]) <= 2e-5


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
        est, X = _fit(mu=0.05)                               # the fit is sharded as well
        s = est.phase_uncertainty(X)
        keep = espm_b200.config.distributed
        espm_b200.config.distributed = False
        u = est.phase_uncertainty(X)
        espm_b200.config.distributed = keep
        res = {}
        for f in s._fields:
            res["s_" + f], res["u_" + f] = getattr(s, f), getattr(u, f)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False], ids=["peer-memory", "nccl"])
def test_sharded_phase_uncertainty(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer), nprocs=2, join=True)
    res = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    from espm_b200 import PhaseUncertainty
    for f in PhaseUncertainty._fields:
        assert np.array_equal(res[0]["s_" + f], res[1]["s_" + f]), f
        a, b = res[0]["s_" + f], res[0]["u_" + f]
        assert np.max(np.abs(a - b)) <= 1e-12 * np.abs(b).max(), f
