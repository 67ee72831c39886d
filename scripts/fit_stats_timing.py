"""Time SmoothNMF.goodness_of_fit (espm_fit_stats) at the C3 size on one GPU.

    python scripts/fit_stats_timing.py [--out profiles/fit_stats_timing_c3.json] [--host-baseline]

C3: 512 x 512 pixels x 2048 channels, k = 4, G from espm_b200.synth, seeded Poisson X whose mean is the model.
For X stored dense f32, dense f64 and uint8:
  - espm_fit_stats device time: CUDA events around 50 launches after 5 warm-up launches (the streaming kernel and the
    fold of its CTA slots); the image is 2.1 / 4.3 / 0.5 GB, far above the 126 MB L2;
  - espm_h_pass timed the same way on the same engine, in the same run;
  - n p sizeof(X) over the fit-statistics time, against the device-to-device copy bandwidth measured in the same run;
  - wall time of ``est.goodness_of_fit`` on a pinned host array (upload, ingest checks, the kernel, read-back).
With --host-baseline also the host NumPy route once: G W H as ``inverse_transform`` builds it, then the statistics in
NumPy fp64, chunked over pixels.  The GPU name and power limit are read with nvidia-smi in the same run.
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

NX, NY, N, K, N_EL, SEED, LS = 512, 512, 2048, 4, 25, 93, 1e-14
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


def problem():
    from espm_b200 import synth
    prob = synth.make_problem(NX, NY, N, K, N_EL, seed=SEED)
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
    nbytes = ctypes.c_int64(0)
    L.check(lib.espm_fit_stats_scratch(ctypes.byref(st), ctypes.byref(nbytes)))
    scratch = torch.empty(nbytes.value // 8, dtype=torch.float64, device="cuda")
    pix = torch.empty(4, eng.p_loc, dtype=torch.float64, device="cuda")
    chan = torch.empty(4, eng.n, dtype=torch.float64, device="cuda")
    stream = eng.stream
    stats_ms = launch_ms(lambda: L.check(lib.espm_fit_stats(ctypes.byref(st), pix.data_ptr(), chan.data_ptr(),
                                                            scratch.data_ptr(), stream)))
    first = pix.clone()
    h_ms = launch_ms(lambda: L.check(lib.espm_h_pass(ctypes.byref(st), stream)))
    L.check(lib.espm_fit_stats(ctypes.byref(st), pix.data_ptr(), chan.data_ptr(), scratch.data_ptr(), stream))
    torch.cuda.synchronize()
    x_bytes = N * NX * NY * {"f32": 4, "f64": 8, "uint8": 1}[name]
    out = {"x_storage": eng.x_storage, "x_bytes": x_bytes, "fit_stats_ms": stats_ms, "h_pass_ms": h_ms,
           "fit_stats_over_h_pass": stats_ms / h_ms, "fit_stats_x_gbs": x_bytes / stats_ms / 1e6,
           "scratch_bytes": int(nbytes.value), "bit_identical_repeat": bool(torch.equal(first, pix)),
           "kl_total": float(pix[2].sum().item())}
    eng.close()
    del eng, scratch, pix, chan, Xs
    espm_b200.config.x_storage = "auto"
    torch.cuda.empty_cache()
    return out


def fitted(G, W, H):
    from espm_b200 import SmoothNMF
    with contextlib.redirect_stdout(io.StringIO()):
        est = SmoothNMF(n_components=K, G=G)
    est.G_, est.W_, est.H_, est._identity_G = G.astype(np.float32), W.astype(np.float32), H.astype(np.float32), False
    return est


def host_route(est, Xh, chunk=16384):
    """What a user does without goodness_of_fit: the dense model of inverse_transform, then NumPy."""
    t0 = time.perf_counter()
    Y = est.inverse_transform(est.W_.astype(np.float64))                 # G W H, n x p fp64
    np.maximum(Y, LS, out=Y)
    pix, chan = np.zeros((4, Xh.shape[1])), np.zeros((4, Xh.shape[0]))
    for a in range(0, Xh.shape[1], chunk):
        x, y = Xh[:, a:a + chunk].astype(np.float64), Y[:, a:a + chunk]
        with np.errstate(divide="ignore", invalid="ignore"):
            xl = np.where(x > 0, x * np.log(x / y), 0.0)
        for i, t in enumerate((x, y, y - x + xl, (x - y) ** 2 / y)):
            pix[i, a:a + chunk] = t.sum(0)
            chan[i] += t.sum(1)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fit_stats_timing_c3.json"))
    ap.add_argument("--host-baseline", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fit_stats_timing.py needs a GPU")
    torch.cuda.set_device(0)
    from espm_b200 import build
    build.build()
    res = {"config": "C3 512x512 px x 2048 channels, k=4", "gpu": gpu_info(), "warmup_launches": WARM,
           "timed_launches": REPS}
    res["copy_gbs"] = copy_bandwidth_gbs()
    G, W, H, X = problem()
    res["storage"] = {name: time_storage(name, G, W, H, X) for name in ("f32", "f64", "uint8")}
    for v in res["storage"].values():
        v["fit_stats_x_over_copy_bw"] = v["fit_stats_x_gbs"] / res["copy_gbs"]
    Xh = torch.empty(X.shape, dtype=torch.float32, pin_memory=True)
    Xh.copy_(X)
    del X
    torch.cuda.empty_cache()
    est = fitted(G, W, H)
    Xn = Xh.numpy()
    walls = []
    for _ in range(4):
        t0 = time.perf_counter()
        stats = est.goodness_of_fit(Xn)
        walls.append(time.perf_counter() - t0)
    res["goodness_of_fit_pinned_f32_s"] = {"first": walls[0], "min_of_next_3": min(walls[1:])}
    res["goodness_of_fit_x_storage"] = "auto (uint8 for this image)"
    res["goodness_of_fit_kl_total"] = float(stats.pixel_kl.sum())
    if args.host_baseline:
        res["host_route_s"] = host_route(est, Xn)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
