"""SmoothNMF.transform on the device: the H-only loop (ESPM_FLAG_H_ONLY) against the oracle's fixed-W fit, its stop tests,
the device initial H, the launch chain, the benchmark size and pixel-sharded runs.

A model is fitted on one seeded image and applied to another with a different number of pixels.  The reference call
``transform`` stands for is ``oracle.fit(X, G_, W_, H0, fixed_W=W_, simplex_W=True, normalize=False, ...)``."""
import contextlib
import io
import os
import re
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N, M, K = 160, 6, 3
FIT_SHAPE, NEW_SHAPE = (13, 11), (12, 14)
ITERS = 12


def _G(seed=5):
    rng = np.random.default_rng(seed)
    x = np.linspace(0, 1, N)
    G = np.zeros((N, M))
    for j in range(M - 2):
        c, s = rng.uniform(0.05, 0.95), rng.uniform(0.01, 0.04)
        G[:, j] = np.exp(-0.5 * ((x - c) / s) ** 2)
    G[:, M - 2] = np.exp(-3 * x) + 0.05
    G[:, M - 1] = (1 - x) * 0.5 + 0.05
    return G


def _image(seed, shape, G, counts=20.0):
    rng = np.random.default_rng(seed)
    p = shape[0] * shape[1]
    Wt = np.random.default_rng(11).uniform(size=(G.shape[1], K))
    Ht = rng.uniform(size=(K, p)) ** 2
    Ht /= Ht.sum(0, keepdims=True)
    lam = G @ Wt @ Ht
    return rng.poisson(lam / lam.sum(0, keepdims=True) * counts).astype(np.float64)


def _H0(seed, p):
    H0 = np.random.default_rng(seed).uniform(0.05, 1.0, size=(K, p))
    return H0 / H0.sum(0, keepdims=True)


def _quiet(fn, *a, **kw):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **kw)


def _fitted(identity_G=False, dtype=np.float64, **kw):
    """(estimator fitted on the first image, G of the problem, the second image as (n, p'))."""
    from espm_b200 import SmoothNMF
    G = _G()
    XA = _image(1, FIT_SHAPE, G)
    XB = _image(2, NEW_SHAPE, G)
    if identity_G:
        G = None
    pA = FIT_SHAPE[0] * FIT_SHAPE[1]
    m = N if identity_G else M
    W0 = np.random.default_rng(3).uniform(0.05, 1.0, size=(m, K))
    kw.setdefault("shape_2d", FIT_SHAPE)
    est = SmoothNMF(n_components=K, G=None if G is None else G.astype(dtype), hspy_comp=True, max_iter=15, tol=0,
                    no_stop_criterion=True, verbose=0, **kw)
    _quiet(est.fit_transform, XA.T.astype(dtype), W=W0.astype(dtype), H=_H0(4, pA).astype(dtype))
    est.set_params(max_iter=ITERS)
    return est, XB.astype(dtype)


def _oracle(est, XB, H0, shape_2d, **over):
    from oracle import smooth_nmf_oracle as orc
    kw = dict(lambda_L=est.lambda_L, mu=est.mu, epsilon_reg=est.epsilon_reg, simplex_H=est.simplex_H, simplex_W=True,
              tol=est.tol, max_iter=est.max_iter, shape_2d=shape_2d, normalize=False, log_shift=est.log_shift,
              dicotomy_tol=est.dicotomy_tol, no_stop_criterion=est.no_stop_criterion, fixed_W=est.W_, algo=est.algo)
    kw.update(over)
    W = est.W_.astype(np.float64)
    return orc.fit(XB.astype(np.float64), est.G_.astype(np.float64), W, H0.astype(np.float64),
                   **dict(kw, fixed_W=W))


def _err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def _fitted_state(est):
    return {k: v for k, v in vars(est).items() if k.endswith("_") and not k.startswith("_")}


def _same_state(after, refs, values):
    """Every fitted attribute is still the same object (not rebound) holding the same values (not mutated)."""
    assert after.keys() == refs.keys()
    for k in after:
        assert after[k] is refs[k], k
        va, vb = after[k], values[k]
        if isinstance(va, np.ndarray):
            assert np.array_equal(va, vb), k
        elif isinstance(va, list):
            assert len(va) == len(vb) and all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(va, vb)), k


CASES = {
    "simplex_H_lap_mu": dict(kw=dict(simplex_H=True, simplex_W=False, lambda_L=2.0, mu=0.05), shape=NEW_SHAPE),
    "hq_lap_identity_L": dict(kw=dict(simplex_H=True, simplex_W=False, lambda_L=0.8, algo="l2_surrogate",
                                      shape_2d=None), shape=None),
    "free": dict(kw=dict(simplex_H=False, simplex_W=False, mu=0.05), shape=None),
    "identity_G": dict(kw=dict(simplex_W=True, lambda_L=0.5), shape=NEW_SHAPE, identity_G=True),
    "normalize": dict(kw=dict(simplex_H=True, simplex_W=False, normalize=True, mu=0.02), shape=None),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_trajectory_matches_oracle_fp64(case):
    c = CASES[case]
    est, XB = _fitted(identity_G=c.get("identity_G", False), **c["kw"])
    H0 = _H0(6, XB.shape[1])
    H = _quiet(est.transform, XB.T, H=H0, shape_2d=c["shape"]).T
    ref = _oracle(est, XB, H0, c["shape"])
    assert ref["n_iter"] == ITERS
    assert H.dtype == np.float64 and H.shape == H0.shape
    assert _err(H, ref["H"]) < 1e-9, case


def test_trajectory_matches_oracle_fp32():
    est, XB = _fitted(dtype=np.float32, **CASES["simplex_H_lap_mu"]["kw"])
    H0 = _H0(6, XB.shape[1]).astype(np.float32)
    H = _quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE).T
    assert H.dtype == np.float32
    ref = _oracle(est, XB, H0, NEW_SHAPE)       # fp64 oracle on the fp32-rounded inputs
    assert _err(H, ref["H"]) < 1e-4


def test_count_storage_matches_dense():
    from espm_b200 import config
    est, XB = _fitted(dtype=np.float32, **CASES["simplex_H_lap_mu"]["kw"])
    H0 = _H0(6, XB.shape[1]).astype(np.float32)
    keep = config.x_storage
    try:
        out = {}
        for mode in ("auto", "dense"):
            config.x_storage = mode
            out[mode] = _quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE)
    finally:
        config.x_storage = keep
    assert _err(out["auto"], out["dense"]) < 1e-6


_EXIT = {"rel": "exits because of relative change rel_A", "loss": "exits because of relative change <",
         "increase": "exit because of negative decrease", "nan": "exit because of the presence of NaN",
         "max_iter": "exits because max_iteration was reached"}


def test_stop_tests_match_oracle():
    est, XB = _fitted(**CASES["simplex_H_lap_mu"]["kw"])
    est.set_params(tol=1e-4, no_stop_criterion=False, verbose=1, max_iter=200)
    H0 = _H0(6, XB.shape[1])
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        H = est.transform(XB.T, H=H0, shape_2d=NEW_SHAPE).T
    out = buf.getvalue()
    ref = _oracle(est, XB, H0, NEW_SHAPE)
    assert ref["reason"] != "max_iter"
    exits = [ln for ln in out.splitlines() if ln.startswith("exit")]
    assert len(exits) == 1 and exits[0].startswith(_EXIT[ref["reason"]]), out
    n_iter = int(re.search(r"Stopped after (\d+) iterations", out).group(1))
    assert n_iter == ref["n_iter"]
    assert _err(H, ref["H"]) < 1e-9


@pytest.mark.parametrize("dtype, tol", [(np.float64, 1e-10), (np.float32, 1e-5)])
def test_default_initial_h_matches_host(dtype, tol):
    from espm_b200.engine import FitEngine
    from espm_b200.host import initialize_factors, remove_zeros_lines
    from espm_b200.init_device import initial_H_device
    est, XB = _fitted(dtype=dtype, **CASES["simplex_H_lap_mu"]["kw"])
    X_ = remove_zeros_lines(XB, est.log_shift)
    _, _, H_host = initialize_factors(X_, est.G_, est.W_, None, K, None, None, True, True, est.log_shift)
    eng = FitEngine(XB, est.G_, est.W_, np.ones((K, XB.shape[1]), dtype=dtype), h_only=True, simplex_H=True,
                    ingest=dict(eps=est.log_shift, normalize=None))
    H_dev = initial_H_device(eng, est.G_, est.W_, True, est.log_shift).cpu().numpy()
    assert _err(H_dev, H_host) < tol
    if dtype == np.float64:
        # the full default call is the oracle run from that initial H
        H = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE).T
        assert _err(H, _oracle(est, XB, H_dev, NEW_SHAPE)["H"]) < 1e-9


def test_fitted_state_is_unchanged():
    import copy
    est, XB = _fitted(**CASES["simplex_H_lap_mu"]["kw"])
    refs = _fitted_state(est)
    values = copy.deepcopy(refs)
    H0 = _H0(6, XB.shape[1])
    first = _quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE)
    _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE)
    _same_state(_fitted_state(est), refs, values)
    assert "components_" in refs and "W_" in refs and "losses_" in refs
    # a second call gives the same result: nothing of the first one was left behind
    assert np.array_equal(_quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE), first)


def test_fixed_p_prime_negative_entries_use_ingest_message():
    est, XB = _fitted(**CASES["simplex_H_lap_mu"]["kw"])
    Xbad = XB.copy()
    Xbad[3, 7] = -1.0
    with pytest.raises(ValueError, match="Negative values in data"):
        _quiet(est.transform, Xbad.T, shape_2d=NEW_SHAPE)
    Xbad[3, 7] = np.nan
    with pytest.raises(ValueError, match="NaN"):
        _quiet(est.transform, Xbad.T, shape_2d=NEW_SHAPE)


@pytest.mark.parametrize("simplex_H, per_iter", [(True, 5), (False, 4)])
def test_launch_chain(simplex_H, per_iter):
    import torch
    from espm_b200.engine import FitEngine
    G = _G()
    XB = _image(2, NEW_SHAPE, G)
    W = np.random.default_rng(3).uniform(0.05, 1.0, size=(M, K))
    eng = FitEngine(XB, G, W, _H0(6, XB.shape[1]), h_only=True, simplex_H=simplex_H, lambda_L=1.0, shape_2d=NEW_SHAPE,
                    ingest=dict(eps=1e-14, normalize=None))
    assert eng.fast_loop
    eng.evaluate(0)
    torch.cuda.synchronize()
    n0 = eng.n_launches
    iters = 6
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.run_iterations(1, iters)
        torch.cuda.synchronize()
    assert eng.n_launches - n0 == per_iter * iters
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert not [nm for nm in names if "w_pass" in nm or "w_finish" in nm or "w_reduce" in nm]
    assert sum("h_pass" in nm for nm in names) == iters
    recs = eng.read_records(1, iters + 1)
    from espm_b200 import _lib as L
    assert np.all(recs[:, L.S_REL_W] == 0.0)
    # the Python loop launches the same chain
    n1 = eng.n_launches
    eng.advance(iters + 1)
    eng.evaluate(iters + 1)
    assert eng.n_launches - n1 == per_iter


def test_benchmark_size_matches_fixed_w_fit():
    """C3 (512 x 512 px, 2048 channels, k = 4, fp32, Laplacian + mu, simplex_H): transform == the engine's fixed_W fit."""
    import torch
    from espm_b200 import SmoothNMF, _lib as L, synth
    from espm_b200.engine import FitEngine
    nx, ny, n, k = 512, 512, 2048, 4
    prob = synth.make_problem(nx, ny, n, k, 25, seed=93)
    dev = torch.device("cuda", torch.cuda.current_device())
    XA = synth.poisson_X_torch(prob, 0, nx * ny, 93, dev, torch.float32).cpu().numpy()
    G = prob["G_full"].astype(np.float32)
    W0, H0 = synth.init_factors(G.shape[1], k, nx * ny, 93, dtype=np.float32)
    kw = dict(simplex_H=True, simplex_W=False, lambda_L=2.0, mu=0.05)
    est = SmoothNMF(n_components=k, G=G, shape_2d=(nx, ny), hspy_comp=True, max_iter=3, tol=0, no_stop_criterion=True,
                    verbose=0, **kw)
    _quiet(est.fit_transform, XA.T, W=W0, H=H0)
    del XA
    XB = synth.poisson_X_torch(prob, 0, nx * ny, 94, dev, torch.float32).cpu().numpy()
    iters = 10
    est.set_params(max_iter=iters)
    H = _quiet(est.transform, XB.T, H=H0).T
    common = dict(shape_2d=(nx, ny), lambda_L=2.0, mu=0.05, simplex_H=True, ingest=dict(eps=est.log_shift, normalize=None))

    def run(eng):
        eng.evaluate(0)
        eng.run_iterations(1, iters)
        return eng.get_H(), eng.read_records(0, iters + 1)
    H_fix, rec_fix = run(FitEngine(XB, est.G_, est.W_, H0, fixed_W=est.W_, simplex_W=True, **common))
    H_only, rec_only = run(FitEngine(XB, est.G_, est.W_, H0, h_only=True, **common))
    assert _err(H, H_fix) < 1e-6
    assert _err(H_only, H_fix) < 1e-6
    assert np.array_equal(rec_only[1:, L.S_BISECT_ITS_H], rec_fix[1:, L.S_BISECT_ITS_H])


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
        est, XB = _fitted(**CASES["simplex_H_lap_mu"]["kw"])          # the fit is sharded as well
        H0 = _H0(6, XB.shape[1])
        res = {"H": _quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE),
               "H_default": _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE)}
        if rank == 0:
            keep = espm_b200.config.distributed
            espm_b200.config.distributed = False
            res["H1"] = _quiet(est.transform, XB.T, H=H0, shape_2d=NEW_SHAPE)
            res["H1_default"] = _quiet(est.transform, XB.T, shape_2d=NEW_SHAPE)
            espm_b200.config.distributed = keep
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("peer", [True, False], ids=["peer-memory", "nccl"])
def test_sharded_transform(tmp_path, peer):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer), nprocs=2, join=True)
    res = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    for key in ("H", "H_default"):
        assert np.array_equal(res[0][key], res[1][key]), key
        assert _err(res[0][key], res[0]["H1" + key[1:]]) < 1e-9, key
