"""SmoothNMF.residual_components on the device (espm_resid_left / espm_resid_right) against NumPy fp64:

    g = max(G W, ls),  h = max(H, ls),  y = g h,  R = (x - y) / sqrt(y),
    left = (R^T Q)^T (r, p),  right = R P^T (n, r).

The products are compared entry by entry.  Their terms have mixed signs, so the tolerance scales with the sum of the
absolute terms, with |R| replaced by a = (x + y) / sqrt(y) (resid.cuh): 1e-12 in fp64 and the header's bound in fp32.
The whole call is compared with the same randomized subspace iteration run on a dense NumPy R from the same start, and,
with enough iterations to converge, with np.linalg.svd of R."""
import contextlib
import io
import os
import socket
import sys

import numpy as np
import pytest

from test_gpu_abundance_uncertainty import M, N, NEW_SHAPE, PAIRS, SHAPE, _G, _fit, _GW, _image, _quiet
from test_residual_components_cpu import pearson_residual, subspace_angle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U24 = 2.0 ** -24
RSQ = 2.0 ** -22.9


def _bounds(kp, m=1):
    """(E_L, E_R) of resid.cuh for padded width kp; m - 1 more ulps of y when the device forms G W from an m-column G."""
    return (kp + 14 + m - 1) * U24 + RSQ, (kp + 261 + m - 1) * U24 + RSQ


def _engine(X, G, W, H, ls, storage):
    import espm_b200
    from espm_b200.engine import FitEngine
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X, G, W, H, log_shift=ls)
        assert eng.x_storage == storage
    finally:
        espm_b200.config.x_storage = keep
    return eng


def _products(eng, Q, P):
    return eng.residual_left(Q).cpu().numpy(), eng.residual_right(P).cpu().numpy()


# ---------------------------------------------------------------------------------------------------- products
@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("k, identity", [(1, False), (4, False), (8, True)], ids=["k1", "k4", "k8_identity"])
def test_products_match_numpy(pair, k, identity):
    """n = 161 (pad channels in the last stage) and p = 143 (pad pixels in the last tile); r = 1, 7, 16 and 21 (two
    launches of 16 columns)."""
    xdt, cdt, storage = PAIRS[pair]
    n, ls = 161, 1e-3
    G = np.eye(n) if identity else _G(n=n)
    X = _image(7, SHAPE, G, k, counts=3000.0).astype(xdt)
    rng = np.random.default_rng(8)
    W = rng.uniform(0.05, 1.0, size=(G.shape[1], k)).astype(cdt)
    H = rng.uniform(0.05, 1.0, size=(k, X.shape[1]))
    H[0, ::4] = 0.0                                          # clamped to log_shift
    H = H.astype(cdt)
    eng = _engine(X, None if identity else G.astype(cdt), W, H, ls, storage)
    try:
        assert eng.st.n_pad > n and eng.p_loc % 128 != 0
        GW = W.astype(np.float64) if identity else G.astype(cdt).astype(np.float64) @ W.astype(np.float64)
        R = pearson_residual(X, GW, H, ls)
        y = np.maximum(GW.astype(np.float64), ls) @ np.maximum(H.astype(np.float64), ls)
        A = (X.astype(np.float64) + y) / np.sqrt(y)
        e_l, e_r = (1e-12, 1e-12) if cdt == np.float64 else _bounds(eng.st.kp, 1 if identity else M)
        for r in (1, 7, 16, 21):
            Q = rng.standard_normal((n, r))
            P = rng.standard_normal((r, X.shape[1]))
            before = eng.n_launches
            left, right = _products(eng, Q, P)
            blocks = -(-r // 16)
            assert eng.n_launches == before + 5 * blocks
            assert left.shape == (r, X.shape[1]) and right.shape == (n, r)
            err_l = np.abs(left - (R.T @ Q).T) / (A.T @ np.abs(Q)).T
            err_r = np.abs(right - R @ P.T) / (A @ np.abs(P).T)
            assert err_l.max() <= e_l, "left r=%d: %.3e > %.3e" % (r, err_l.max(), e_l)
            assert err_r.max() <= e_r, "right r=%d: %.3e > %.3e" % (r, err_r.max(), e_r)
            again = _products(eng, Q, P)
            assert np.array_equal(again[0], left) and np.array_equal(again[1], right)
    finally:
        eng.close()


@pytest.mark.parametrize("storage", ["uint8", "uint16"])
def test_compact_storage_gives_the_dense_bits(storage):
    G = _G()
    X = _image(7, SHAPE, G, 4, counts=200.0).astype(np.float32)
    rng = np.random.default_rng(9)
    W = rng.uniform(0.05, 1.0, size=(M, 4)).astype(np.float32)
    H = rng.uniform(0.05, 1.0, size=(4, X.shape[1])).astype(np.float32)
    Q = rng.standard_normal((N, 21))
    P = rng.standard_normal((21, X.shape[1]))
    out = {}
    for s in ("dense", storage):
        eng = _engine(X, G.astype(np.float32), W, H, 1e-3, s)
        try:
            out[s] = _products(eng, Q, P)
        finally:
            eng.close()
    assert np.array_equal(out["dense"][0], out[storage][0])
    assert np.array_equal(out["dense"][1], out[storage][1])


# ---------------------------------------------------------------------------------------------------- end to end
def _dense_run(R, rank, n_iter, random_state):
    """The host driver on a dense R from the start the estimator draws."""
    from sklearn.utils import check_random_state
    from espm_b200.host import RESID_OVERSAMPLE, residual_components
    Q0 = check_random_state(random_state).standard_normal((R.shape[0], rank + RESID_OVERSAMPLE))
    s, spectra, V, P = residual_components(lambda Q: (R.T @ Q).T, lambda P: R @ P.T, lambda P: P @ P.T, Q0, rank,
                                           n_iter)
    return s, spectra, V.T @ P


def _check(rc, R, rank, n_iter, seed, fp32):
    n, p = R.shape
    assert rc.singular_values.shape == (rank,) and rc.spectra.shape == (n, rank) and rc.maps.shape == (rank, p)
    for a in rc:
        assert a.dtype == np.float64
    assert np.all(np.diff(rc.singular_values) <= 0)
    lead = rc.spectra[np.argmax(np.abs(rc.spectra), axis=0), np.arange(rank)]
    assert np.all(lead > 0)
    assert np.allclose(rc.spectra.T @ rc.spectra, np.eye(rank), atol=1e-10)
    assert np.allclose(rc.maps @ rc.maps.T, np.eye(rank), atol=1e-8)
    # the same iteration on the dense R
    s, spectra, maps = _dense_run(R, rank, n_iter, seed)
    tol = 1e-4 if fp32 else 1e-10
    assert np.max(np.abs(rc.singular_values - s) / s) <= tol
    # against the SVD: after n_iter = 150 iterations even the near-degenerate top of a pure-noise residual of this size
    # has converged (to 1e-14 in NumPy)
    U, S, Vt = np.linalg.svd(R, full_matrices=False)
    assert np.max(np.abs(rc.singular_values - S[:rank]) / S[:rank]) <= (1e-4 if fp32 else 1e-8)
    atol = 1e-3 if fp32 else 1e-6
    assert subspace_angle(rc.spectra, U[:, :rank]) <= atol
    assert subspace_angle(rc.maps.T, Vt[:rank].T) <= atol
    # Frobenius norm of R is the total chi-square
    assert S[0] ** 2 <= np.sum(R ** 2)


CASES = {
    "default": dict(),
    "hspy_comp": dict(hspy_comp=True),
    "normalize": dict(normalize=True),
    "identity_G": dict(identity_G=True),
    "simplex_H": dict(simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE),
    "fp32": dict(dtype=np.float32),
}


@pytest.mark.parametrize("case", list(CASES))
def test_end_to_end_matches_dense_svd(case):
    kw = dict(CASES[case])
    est, X = _fit(**kw)
    rc = est.residual_components(X.T if kw.get("hspy_comp") else X, rank=4, n_iter=150, random_state=5)
    R = pearson_residual(X, _GW(est), est.H_, est.log_shift)
    _check(rc, R, 4, 150, 5, kw.get("dtype") == np.float32)


def test_new_image_with_transformed_maps():
    est, _ = _fit(hspy_comp=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE)
    XB = _image(2, NEW_SHAPE, _G(), 3, counts=2000.0)
    H = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE).T
    rc = est.residual_components(XB.T, rank=3, H=H, n_iter=150, random_state=np.random.RandomState(2))
    _check(rc, pearson_residual(XB, _GW(est), H, est.log_shift), 3, 150, np.random.RandomState(2), False)


def test_no_side_effects_and_deterministic():
    est, X = _fit(mu=0.05)
    _ = est.X_
    before = {k: v for k, v in est.__dict__.items()}
    copies = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in before.items()}
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        a = est.residual_components(X, rank=3, random_state=1)
        b = est.residual_components(X, rank=3, random_state=1)
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
            est.residual_components(Xb, rank=2)


# ---------------------------------------------------------------------------------------------------- planted phase
def _planted(seed=41, side=40, n=160, counts=4000.0):
    """Four phases, each with a line of its own (Gaussian columns 0-3 of G) on the two backgrounds; phase 3 lives in a
    disk only.  Returns (G, W_true, H_true, X, line channels of phase 3)."""
    x = np.linspace(0, 1, n)
    centers = [0.15, 0.35, 0.55, 0.75]
    G = np.stack([np.exp(-0.5 * ((x - c) / 0.015) ** 2) for c in centers]
                 + [np.exp(-3 * x) + 0.05, (1 - x) * 0.5 + 0.05], axis=1)
    W = np.zeros((6, 4))
    for a in range(4):
        W[a, a] = 1.0
        W[4, a], W[5, a] = 0.3 + 0.1 * a, 0.4 - 0.05 * a
    W /= W.sum(0, keepdims=True)
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:side, 0:side] / side
    H = np.empty((4, side * side))
    H[:3] = rng.dirichlet(np.ones(3), size=side * side).T
    disk = (((xx - 0.6) ** 2 + (yy - 0.4) ** 2) < 0.2 ** 2).reshape(-1)
    H[3] = 0.5 * disk
    H[:3] *= 1.0 - H[3]
    lam = G @ W @ H
    X = rng.poisson(lam / lam.sum(0, keepdims=True) * counts).astype(np.float64)
    line = np.flatnonzero(np.abs(x - centers[3]) <= 0.03)
    return G, W, H, X, line


def _fit_truth(G, W, H, X, k):
    from espm_b200 import SmoothNMF
    scale = X.sum(0).mean() / (G @ W @ H).sum(0).mean()
    est = SmoothNMF(n_components=k, G=G, max_iter=400, tol=0, no_stop_criterion=True, verbose=0, simplex_W=False)
    _quiet(est.fit_transform, X, W=W[:, :k] * scale, H=H[:k].copy() + 1e-3)
    return est


def test_planted_missing_phase():
    """Observed on a B200: with 3 phases fitted the leading value is 5.07x the replicate's, its map correlates 0.948
    with the missing phase and its spectrum peaks at channel 119, inside that phase's line (115-124); with 4 phases
    fitted it is 1.009x the replicate's."""
    G, W, H, X, line = _planted()
    rng = np.random.default_rng(7)
    est3 = _fit_truth(G, W, H, X, 3)
    rc = est3.residual_components(X, rank=2, random_state=0)
    rep = est3.residual_components(rng.poisson(est3.G_ @ est3.W_ @ est3.H_).astype(np.float64), rank=2, random_state=0)
    ratio3 = rc.singular_values[0] / rep.singular_values[0]
    corr = np.corrcoef(rc.maps[0], H[3])[0, 1]
    peak = int(np.argmax(rc.spectra[:, 0]))
    est4 = _fit_truth(G, W, H, X, 4)
    rc4 = est4.residual_components(X, rank=2, random_state=0)
    rep4 = est4.residual_components(rng.poisson(est4.G_ @ est4.W_ @ est4.H_).astype(np.float64), rank=2,
                                    random_state=0)
    ratio4 = rc4.singular_values[0] / rep4.singular_values[0]
    print("planted: ratio3 %.3f corr %.3f peak %d (line %d-%d) ratio4 %.3f"
          % (ratio3, corr, peak, line[0], line[-1], ratio4))
    assert ratio3 >= 3.0
    assert corr >= 0.8
    assert peak in line
    assert abs(ratio4 - 1.0) <= 0.15


# ---------------------------------------------------------------------------------------------------- full size
@pytest.mark.parametrize("storage", ["dense", "uint8"])
def test_c3_against_chunked_torch(storage):
    """512 x 512 px x 2048 channels, k = 4, fp32 arithmetic: the subspace iteration of the device products against the
    same iteration from the same start with a chunked fp64 torch R."""
    import torch
    from espm_b200 import synth
    from espm_b200.host import RESID_OVERSAMPLE, residual_components
    nx = ny = 512
    n, k, seed, ls, rank, n_iter = 2048, 4, 93, 1e-14, 4, 3
    prob = synth.make_problem(nx, ny, n, k, 12, seed=seed)
    dev = torch.device("cuda", 0)
    G = prob["G_full"].astype(np.float32)
    X = synth.poisson_X_torch(prob, 0, nx * ny, seed, dev, torch.float32)
    GWt = prob["G_full"] @ prob["W_true"]
    W = (prob["W_true"] / GWt.sum(0) * prob["dens"] * prob["counts"]).astype(np.float32)
    H = prob["H_true"].astype(np.float32)
    Q0 = np.random.RandomState(3).standard_normal((n, rank + RESID_OVERSAMPLE))
    eng = _engine(X, G, W, H, ls, storage)
    try:
        dev_s = residual_components(eng.residual_left, lambda P: eng.residual_right(P).cpu().numpy(),
                                    lambda P: (P @ P.T).cpu().numpy(), Q0, rank, n_iter)[0]
    finally:
        eng.close()
    g = torch.as_tensor(np.maximum(G.astype(np.float64) @ W.astype(np.float64), ls), device=dev)
    Hc = torch.as_tensor(np.maximum(H.astype(np.float64), ls), device=dev)
    CH = 16384

    def chunks():
        for a in range(0, nx * ny, CH):
            y = g @ Hc[:, a:a + CH]
            yield a, (X[:, a:a + CH].double() - y) / torch.sqrt(y)

    def left(Q):
        Qd = torch.as_tensor(Q, device=dev)
        return torch.cat([(R.T @ Qd).T for _, R in chunks()], dim=1)

    def right(P):
        out = torch.zeros(n, P.shape[0], dtype=torch.float64, device=dev)
        for a, R in chunks():
            out += R @ P[:, a:a + CH].T
        return out.cpu().numpy()
    ref_s = residual_components(left, right, lambda P: (P @ P.T).cpu().numpy(), Q0, rank, n_iter)[0]
    del X
    assert np.max(np.abs(dev_s - ref_s) / ref_s) <= 1e-4, (dev_s, ref_s)


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
        from espm_b200.dist import make_shard
        from espm_b200.engine import FitEngine
        est, X = _fit(mu=0.05)                               # the fit is sharded as well
        s = est.residual_components(X, rank=3)               # unseeded: rank 0's start is broadcast
        s0 = est.residual_components(X, rank=3, random_state=np.random.RandomState(0))
        Q = np.random.default_rng(1).standard_normal((X.shape[0], 7))
        eng = FitEngine.for_statistics(X, est.G_, est.W_, est.H_, log_shift=est.log_shift, shard=make_shard())
        left_local = eng.residual_left(Q).cpu().numpy()
        eng.close()
        keep = espm_b200.config.distributed
        espm_b200.config.distributed = False
        try:
            u = est.residual_components(X, rank=3, random_state=np.random.RandomState(0))
            eng = FitEngine.for_statistics(X, est.G_, est.W_, est.H_, log_shift=est.log_shift)
            left_whole = eng.residual_left(Q).cpu().numpy()
            eng.close()
        finally:
            espm_b200.config.distributed = keep
        res = dict(left_local=left_local, left_whole=left_whole)
        for f in s._fields:
            res["s_" + f], res["u_" + f], res["s0_" + f] = getattr(s, f), getattr(u, f), getattr(s0, f)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False], ids=["peer-memory", "nccl"])
def test_sharded_residual_components(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer), nprocs=2, join=True)
    res = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    from espm_b200 import ResidualComponents
    for f in ResidualComponents._fields:
        assert np.array_equal(res[0]["s_" + f], res[1]["s_" + f]), f      # unseeded, identical on every rank
        assert np.array_equal(res[0]["s0_" + f], res[1]["s0_" + f]), f
    a, b = res[0]["s0_singular_values"], res[0]["u_singular_values"]
    assert np.max(np.abs(a - b) / b) <= 1e-12
    for f in ("spectra", "maps"):
        assert np.max(np.abs(res[0]["s0_" + f] - res[0]["u_" + f])) <= 1e-9, f
    # a pixel's left product does not depend on the sharding
    whole = res[0]["left_whole"]
    p0 = res[0]["left_local"].shape[1]
    assert np.array_equal(np.concatenate([res[0]["left_local"], res[1]["left_local"]], axis=1), whole)
    assert p0 < whole.shape[1]
