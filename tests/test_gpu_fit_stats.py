"""SmoothNMF.goodness_of_fit on the device (espm_fit_stats) against a NumPy fp64 evaluation of its definitions:

    y = max(G W, ls) @ max(H, ls),  kl = y - x + x ln(x / y) (0 ln 0 := 0),  chi2 = (x - y)^2 / y,

summed over channels (per pixel) and over pixels (per channel), with x and y themselves.  "Scale" of an entry is the sum
of x + y that entry covers."""
import contextlib
import io
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, M = 160, 6
SHAPE, NEW_SHAPE = (13, 11), (12, 14)
FIELDS = ("counts", "model", "kl", "chi2")


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


def _fit(k=3, identity_G=False, dtype=np.float64, hspy_comp=False, counts=20.0, **kw):
    """(fitted estimator, X (n, p) it was fitted on)."""
    from espm_b200 import SmoothNMF
    G = _G()
    X = _image(1, SHAPE, G, k, counts).astype(dtype)
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


def _oracle(X, GW, H, ls):
    X = np.asarray(X, dtype=np.float64)
    Y = np.maximum(np.asarray(GW, np.float64), ls) @ np.maximum(np.asarray(H, np.float64), ls)
    with np.errstate(divide="ignore", invalid="ignore"):
        xl = np.where(X > 0, X * np.log(X / Y), 0.0)
    terms = (X, Y, Y - X + xl, (X - Y) ** 2 / Y)
    ref = {}
    for f, t in zip(FIELDS, terms):
        ref["pixel_" + f], ref["channel_" + f] = t.sum(0), t.sum(1)
    ref["pixel_scale"], ref["channel_scale"] = (X + Y).sum(0), (X + Y).sum(1)
    ref["Y"] = Y
    return ref


def _check(stats, ref, tol):
    for side in ("pixel", "channel"):
        for f in FIELDS:
            got, want = getattr(stats, side + "_" + f), ref[side + "_" + f]
            assert got.dtype == np.float64 and got.shape == want.shape, (side, f)
            err = np.max(np.abs(got - want) / ref[side + "_scale"])
            assert err <= tol, "%s_%s: %.3e > %.1e" % (side, f, err, tol)


CASES = {
    "simplex_H_lap_mu": dict(simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE),
    "identity_G": dict(identity_G=True),
    "k5": dict(k=5),
    "k8": dict(k=8, simplex_H=True),
    "normalize": dict(normalize=True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_fp64_matches_oracle(case):
    est, X = _fit(**CASES[case])
    stats = _quiet(est.goodness_of_fit, X)
    _check(stats, _oracle(X, _GW(est), est.H_, est.log_shift), 1e-12)
    assert np.all(np.isfinite(stats.pixel_chi2))


def test_hspy_comp_layout_gives_identical_arrays():
    est, X = _fit(simplex_H=True, mu=0.05)
    est_h, X_h = _fit(simplex_H=True, mu=0.05, hspy_comp=True)
    a = est.goodness_of_fit(X)
    b = est_h.goodness_of_fit(X_h.T)
    assert np.array_equal(est.H_, est_h.H_)
    for f in a._fields:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


def test_fp32_matches_oracle_on_rounded_inputs():
    est, X = _fit(dtype=np.float32, simplex_H=True)
    assert est.W_.dtype == np.float32
    stats = est.goodness_of_fit(X)
    GW = (est.G_.astype(np.float32) @ est.W_.astype(np.float32)) if not est._identity_G else est.W_
    _check(stats, _oracle(X, GW, est.H_.astype(np.float32), est.log_shift), 2e-5)


def _recording_storage(monkeypatch):
    """Records the X storage of every engine goodness_of_fit builds."""
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
    est, X = _fit(dtype=np.float32, simplex_H=True)
    seen = _recording_storage(monkeypatch)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = "dense"
        dense = est.goodness_of_fit(X)
        espm_b200.config.x_storage = storage
        compact = est.goodness_of_fit(X)
    finally:
        espm_b200.config.x_storage = keep
    assert seen == ["dense", storage]
    for f in dense._fields:
        d, c = getattr(dense, f), getattr(compact, f)
        assert np.allclose(c, d, rtol=1e-6, atol=0), f


# (X storage, arithmetic) pairs of the kernel instances: f64 / f64 (16-channel stages), f32 / f32, uint8 / f32,
# uint16 / f32, f32 / f64
PAIRS = {"f64": (np.float64, np.float64, "dense"), "f32": (np.float32, np.float32, "dense"),
         "uint8": (np.float32, np.float32, "uint8"), "uint16": (np.float32, np.float32, "uint16"),
         "f32_storage_f64_arith": (np.float32, np.float64, "dense")}


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("n", [150, 161])
def test_padded_channels_never_count(pair, n):
    """n not a multiple of 32 (nor of 16): the pad channels of the last stage hold x = 0 and y > 0 and must reach no sum;
    p = 143 also leaves pad pixels in the last tile."""
    import espm_b200
    from espm_b200 import _lib as L
    from espm_b200.engine import FitEngine
    xdt, cdt, storage = PAIRS[pair]
    k = 5
    G = _G(n=n)
    X = _image(7, SHAPE, G, k, counts=30.0)
    rng = np.random.default_rng(8)
    W = rng.uniform(0.05, 1.0, size=(M, k))
    W[:, 2] = 0.0                                            # a column of G W below log_shift
    H = rng.uniform(0.0, 1.0, size=(k, X.shape[1]))
    H[1, ::4] = 0.0
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X.astype(xdt), G.astype(cdt), W.astype(cdt), H.astype(cdt), log_shift=1e-14)
        assert eng.x_storage == storage
        assert eng.c_code == (L.F64 if cdt == np.float64 else L.F32)
        assert eng.st.n_pad > n
        pix, chan = (t.cpu().numpy() for t in eng.fit_statistics())
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    assert pix.shape == (4, X.shape[1]) and chan.shape == (4, n)
    assert np.all(np.isfinite(pix)) and np.all(np.isfinite(chan))
    GW = G.astype(cdt) @ W.astype(cdt)
    ref = _oracle(X.astype(xdt), GW, H.astype(cdt), 1e-14)
    stats = type("S", (), {})()
    for i, f in enumerate(FIELDS):
        setattr(stats, "pixel_" + f, pix[i])
        setattr(stats, "channel_" + f, chan[i])
    _check(stats, ref, 1e-12 if cdt == np.float64 else 2e-5)


def test_clamps_of_zero_H_and_zero_G_column():
    est, X = _fit(k=4)
    W = est.W_.copy()
    W[:, 1] = 0.0                                      # a column of G W below log_shift
    est.W_ = W
    H = est.H_.copy()
    H[2, ::3] = 0.0                                    # exact zeros in H
    stats = est.goodness_of_fit(X, H=H)
    ref = _oracle(X, _GW(est), H, est.log_shift)
    _check(stats, ref, 1e-12)
    assert np.all(np.isfinite(stats.pixel_chi2)) and np.all(np.isfinite(stats.channel_chi2))


def test_identities():
    est, X = _fit(simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE, counts=400.0)
    assert np.all(X.sum(0) > 0) and np.all(X.sum(1) > 0)       # no zero line for remove_zeros_lines to patch
    s = est.goodness_of_fit(X)
    for f in FIELDS:
        a, b = getattr(s, "pixel_" + f).sum(), getattr(s, "channel_" + f).sum()
        assert abs(a - b) <= 1e-12 * abs(a), f
    assert np.array_equal(s.pixel_counts, X.sum(0))                # integer counts: exact
    ls = est.log_shift
    chan_model = np.maximum(_GW(est), ls) @ np.maximum(est.H_, ls).sum(1)
    assert np.max(np.abs(s.channel_model - chan_model) / chan_model) < 1e-12
    # the KL part of the fit's loss on the same (W, H): sum kl = n p KL_div_loss + sum_{x=0} ls ln y
    Y = np.maximum(_GW(est), ls) @ np.maximum(est.H_, ls)
    zero_term = ls * np.log(Y[X == 0]).sum()
    lhs = s.pixel_kl.sum() - zero_term
    rhs = X.size * est.detailed_loss_[0]
    assert abs(lhs - rhs) <= 1e-10 * abs(rhs)


def test_new_image_with_transformed_maps():
    est, _ = _fit(hspy_comp=True, simplex_H=True, lambda_L=2.0, mu=0.05, shape_2d=SHAPE)
    XB = _image(2, NEW_SHAPE, _G(), 3)
    H = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE).T
    stats = est.goodness_of_fit(XB.T, H=H)
    assert stats.pixel_kl.shape == (XB.shape[1],)
    _check(stats, _oracle(XB, _GW(est), H, est.log_shift), 1e-12)


def test_no_side_effects_and_deterministic():
    est, X = _fit(simplex_H=True, mu=0.05)
    _ = est.X_                                           # materialise the lazy attribute too
    before = {k: v for k, v in est.__dict__.items()}
    copies = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in before.items()}
    out = io.StringIO()
    with contextlib.redirect_stdout(out):
        a = est.goodness_of_fit(X)
        b = est.goodness_of_fit(X)
    assert out.getvalue() == ""
    assert set(est.__dict__) == set(before)
    for k, v in est.__dict__.items():
        assert v is before[k], k
        if isinstance(v, np.ndarray):
            assert np.array_equal(v, copies[k]), k
    assert est.const_KL_ == copies["const_KL_"]
    for f in a._fields:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f


def test_invalid_data_raises_fit_errors():
    est, X = _fit()
    for bad, msg in ((np.nan, "NaN"), (np.inf, "infinity"), (-1.0, "Negative")):
        Xb = X.copy()
        Xb[3, 7] = bad
        with pytest.raises(ValueError, match=msg):
            est.goodness_of_fit(Xb)


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
    GWt = prob["G_full"] @ prob["W_true"]                 # model = the Poisson mean of X
    W = (prob["W_true"] / GWt.sum(0) * prob["dens"] * prob["counts"]).astype(np.float32)
    H = prob["H_true"].astype(np.float32)
    keep = espm_b200.config.x_storage
    try:
        espm_b200.config.x_storage = storage
        eng = FitEngine.for_statistics(X, G, W, H, log_shift=ls)
        assert eng.x_storage == storage
        pix, chan = (t.cpu().numpy() for t in eng.fit_statistics())
        eng.close()
    finally:
        espm_b200.config.x_storage = keep
    Xh = X.cpu().numpy()
    del X, eng
    GWc = np.maximum((G @ W).astype(np.float64), ls)
    Hc = np.maximum(H.astype(np.float64), ls)
    chan_ref = np.zeros((4, n))
    pix_sums = np.zeros(4)
    scale_chan = np.zeros(n)
    rng = np.random.default_rng(7)
    sample = np.sort(rng.choice(nx * ny, 4096, replace=False))
    pix_ref = np.zeros((4, sample.size))
    pix_scale = np.zeros(sample.size)
    for a in range(0, nx * ny, 16384):
        b = a + 16384
        x = Xh[:, a:b].astype(np.float64)
        y = GWc @ Hc[:, a:b]
        with np.errstate(divide="ignore", invalid="ignore"):
            xl = np.where(x > 0, x * np.log(x / y), 0.0)
        terms = (x, y, y - x + xl, (x - y) ** 2 / y)
        sel = sample[(sample >= a) & (sample < b)] - a
        pos = np.searchsorted(sample, sel + a)
        for i, t in enumerate(terms):
            chan_ref[i] += t.sum(1)
            pix_ref[i, pos] = t[:, sel].sum(0)
        scale_chan += (x + y).sum(1)
        pix_scale[pos] = (x + y)[:, sel].sum(0)
        pix_sums += [t.sum() for t in terms]
    for i in range(4):
        assert abs(pix[i].sum() - pix_sums[i]) <= 1e-5 * abs(pix_sums[i]), FIELDS[i]
        assert abs(chan[i].sum() - pix_sums[i]) <= 1e-5 * abs(pix_sums[i]), FIELDS[i]
        assert np.max(np.abs(chan[i] - chan_ref[i]) / np.abs(chan_ref[i])) <= 1e-5, FIELDS[i]
        assert np.max(np.abs(pix[i, sample] - pix_ref[i]) / pix_scale) <= 2e-5, FIELDS[i]


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
        s = est.goodness_of_fit(X)
        keep = espm_b200.config.distributed
        espm_b200.config.distributed = False
        u = est.goodness_of_fit(X)
        espm_b200.config.distributed = keep
        res = {}
        for f in s._fields:
            res["s_" + f], res["u_" + f] = getattr(s, f), getattr(u, f)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False], ids=["peer-memory", "nccl"])
def test_sharded_goodness_of_fit(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer), nprocs=2, join=True)
    res = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    from espm_b200 import FitStatistics
    for f in FitStatistics._fields:
        assert np.array_equal(res[0]["s_" + f], res[1]["s_" + f]), f
        s, u = res[0]["s_" + f], res[0]["u_" + f]
        if f.startswith("pixel"):
            assert np.array_equal(s, u), f
        else:
            assert np.max(np.abs(s - u) / np.abs(u)) <= 1e-12, f
