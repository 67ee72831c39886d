"""Time SmoothNMF.phase_uncertainty (espm_phase_info) at the C3 size on one GPU.

    python scripts/phase_uncertainty_timing.py [--out profiles/phase_uncertainty_timing_c3.json] [--host-baseline]

C3: 512 x 512 pixels x 2048 channels, k = 4 and k = 8, G from espm_b200.synth, seeded Poisson X whose mean is the model.
For each k and X stored dense f32, dense f64 and uint8:
  - espm_phase_info device time: CUDA events around 50 launches after 5 warm-up launches (the H tiles, the streaming
    kernel and the fold of its CTA slots); the image is 2.1 / 4.3 / 0.5 GB, far above the 126 MB L2;
  - espm_w_pass timed the same way on the same engine, in the same run (its Ht is the engine's initial one: the W pass
    does the same work whatever H holds);
  - n p sizeof(X) over the information time, against the device-to-device copy bandwidth measured in the same run;
  - at k = 4, wall time of ``est.phase_uncertainty`` on a pinned host array (upload, ingest checks, the kernels,
    read-back, the host algebra), and the host algebra (``host.phase_covariance``) alone, with the real G and with
    G = None and simplex_W over the 2048 channels.
With --host-baseline also the host NumPy route once at k = 4: A_c in fp64, chunked over pixels, then the same algebra.
The GPU name and power limit are read with nvidia-smi in the same run.
"""
import argparse
import contextlib
import ctypes
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NX, NY, N, N_EL, SEED, LS = 512, 512, 2048, 25, 93, 1e-14
KS = (4, 8)
WARM, REPS = 5, 50


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"nvidia_smi": line, "torch_name": torch.cuda.get_device_name()}


def copy_bandwidth_gbs(nbytes=4 << 30, reps=10):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    t = e0.elapsed_time(e1) / 1e3
    del a, b
    return 2.0 * nbytes * reps / t / 1e9


def launch_ms(fn):
    for _ in range(WARM):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / REPS


def problem(k):
    from espm_b200 import synth
    prob = synth.make_problem(NX, NY, N, k, N_EL, seed=SEED)
    G = prob["G_full"]
    GWt = G @ prob["W_true"]
    W = prob["W_true"] / GWt.sum(0) * prob["dens"] * prob["counts"]      # G W H = the Poisson mean of X
    X = synth.poisson_X_torch(prob, 0, NX * NY, SEED, torch.device("cuda", 0), torch.float32)
    return G, W, prob["H_true"], X


def time_storage(name, G, W, H, X):
    import espm_b200
    from espm_b200 import _lib as L
    from espm_b200.engine import FitEngine
    dt = np.float64 if name == "f64" else np.float32
    Xs = X.double() if name == "f64" else X
    espm_b200.config.x_storage = "uint8" if name == "uint8" else "dense"
    eng = FitEngine.for_statistics(Xs, G.astype(dt), W.astype(dt), H.astype(dt), log_shift=LS)
    assert eng.x_storage == ("uint8" if name == "uint8" else "dense")
    st, lib = eng.st, eng.lib
    k = eng.k
    nbytes = ctypes.c_int64(0)
    L.check(lib.espm_phase_info_scratch(ctypes.byref(st), ctypes.byref(nbytes)))
    scratch = torch.empty(max(nbytes.value // 8, 1), dtype=torch.float64, device="cuda")
    out = torch.empty(k * (k + 1) // 2, eng.n, dtype=torch.float64, device="cuda")
    stream = eng.stream
    info_ms = launch_ms(lambda: L.check(lib.espm_phase_info(ctypes.byref(st), out.data_ptr(), scratch.data_ptr(),
                                                            stream)))
    first = out.clone()
    w_ms = launch_ms(lambda: L.check(lib.espm_w_pass(ctypes.byref(st), stream)))
    L.check(lib.espm_phase_info(ctypes.byref(st), out.data_ptr(), scratch.data_ptr(), stream))
    torch.cuda.synchronize()
    x_bytes = N * NX * NY * {"f32": 4, "f64": 8, "uint8": 1}[name]
    res = {"x_storage": eng.x_storage, "x_bytes": x_bytes, "scratch_bytes": nbytes.value, "phase_info_ms": info_ms,
           "w_pass_ms": w_ms, "phase_info_over_w_pass": info_ms / w_ms, "phase_info_x_gbs": x_bytes / info_ms / 1e6,
           "bit_identical_repeat": bool(torch.equal(first, out)), "A_diag0_sum": float(out[0].sum().item())}
    eng.close()
    del eng, out, first, Xs, scratch
    espm_b200.config.x_storage = "auto"
    torch.cuda.empty_cache()
    return res


def fitted(G, W, H):
    from espm_b200 import SmoothNMF
    with contextlib.redirect_stdout(io.StringIO()):
        est = SmoothNMF(n_components=H.shape[0], G=G, simplex_H=False, simplex_W=True)
    est.G_, est.W_, est.H_, est._identity_G = G.astype(np.float32), W.astype(np.float32), H.astype(np.float32), False
    est.physics_model_ = None
    return est


def host_algebra_s(est, A):
    """host.phase_covariance alone: real G, and G = None with simplex_W over the channels (the (n, k, k) block path)."""
    from espm_b200.host import phase_covariance
    m, k = est.W_.shape
    n = est.G_.shape[0]
    t0 = time.perf_counter()
    phase_covariance(A, est.G_, np.ones((m, k), bool), np.arange(m))
    t1 = time.perf_counter()
    phase_covariance(A, None, np.ones((n, k), bool), np.arange(n))
    t2 = time.perf_counter()
    return {"real_G_s": t1 - t0, "identity_G_simplex_s": t2 - t1}


def host_route(est, Xh, chunk=16384):
    """What a user does without phase_uncertainty: A_c in NumPy fp64, chunked over pixels, then the same algebra."""
    from espm_b200.host import phase_covariance
    t0 = time.perf_counter()
    g = np.maximum((est.G_ @ est.W_).astype(np.float64), LS)
    Hc = np.maximum(est.H_.astype(np.float64), LS)
    k, p = Hc.shape
    iu = np.triu_indices(k)
    A = np.zeros((g.shape[0], iu[0].size))
    for a in range(0, p, chunk):
        h = Hc[:, a:a + chunk]
        w = Xh[:, a:a + chunk].astype(np.float64) / (g @ h) ** 2
        A += w @ (h[iu[0]] * h[iu[1]]).T
    m = est.W_.shape[0]
    phase_covariance(np.ascontiguousarray(A.T), est.G_, np.ones((m, k), bool), np.arange(m))
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "phase_uncertainty_timing_c3.json"))
    ap.add_argument("--host-baseline", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("phase_uncertainty_timing.py needs a GPU")
    torch.cuda.set_device(0)
    from espm_b200 import build
    build.build()
    res = {"config": "C3 512x512 px x 2048 channels, k=4 and k=8, simplex_W", "gpu": gpu_info(),
           "warmup_launches": WARM, "timed_launches": REPS}
    res["copy_gbs"] = copy_bandwidth_gbs()
    for k in KS:
        G, W, H, X = problem(k)
        res["k%d" % k] = {name: time_storage(name, G, W, H, X) for name in ("f32", "f64", "uint8")}
        for v in res["k%d" % k].values():
            v["phase_info_x_over_copy_bw"] = v["phase_info_x_gbs"] / res["copy_gbs"]
        if k != KS[0]:
            del X
            torch.cuda.empty_cache()
            continue
        Xh = torch.empty(X.shape, dtype=torch.float32, pin_memory=True)
        Xh.copy_(X)
        del X
        torch.cuda.empty_cache()
        est = fitted(G, W, H)
        Xn = Xh.numpy()
        walls = []
        for _ in range(4):
            t0 = time.perf_counter()
            u = est.phase_uncertainty(Xn)
            walls.append(time.perf_counter() - t0)
        res["phase_uncertainty_pinned_f32_s"] = {"first": walls[0], "min_of_next_3": min(walls[1:])}
        res["phase_uncertainty_x_storage"] = "auto (uint8 for this image)"
        res["phase_uncertainty_median_std"] = float(np.nanmedian(u.std))
        eng, _, _ = est._statistics_engine(Xn, None)
        A = eng.phase_information().cpu().numpy()
        eng.close()
        res["host_algebra"] = host_algebra_s(est, A)
        if args.host_baseline:
            res["host_route_s"] = host_route(est, Xn)
        del Xh, Xn, u
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
