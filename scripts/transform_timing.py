"""Time SmoothNMF.transform (the H-only loop, ESPM_FLAG_H_ONLY) against the fit loop at the C3 size on one GPU.

    python scripts/transform_timing.py --out DIR [--iters 200]

C3: 512 x 512 pixels x 2048 channels, k = 4, 25 elements (espm_b200.synth), simplex_H + Laplacian + mu like bench.py,
X stored dense.  For fp32 and fp64:
  - ms / iteration of the fit loop and of the H-only loop: CUDA events around one espm_run_iterations call of
    ``--iters`` iterations (after 10 warm-up iterations); the images are 2.1 / 4.3 GB, far above the 126 MB L2;
  - the bytes of X each loop streams per iteration (2 n p sizeof(X) for the fit, n p sizeof(X) for the H-only loop)
    over that time, against the device-to-device copy bandwidth measured in the same run;
  - wall time of ``est.transform`` (``--iters`` iterations, no_stop_criterion, default initial H) on a pinned host array:
    upload, ingest, device initial H, the loop and the read-back.
Writes transform_timing.json (with the GPU name and power limit) to DIR.
"""
import argparse
import contextlib
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

NX, NY, N, K, N_EL = 512, 512, 2048, 4, 25
KW = dict(simplex_H=True, simplex_W=False, lambda_L=2.0, mu=0.05)


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


def loop_ms(eng, iters, warm=10):
    eng.evaluate(0)
    eng.run_iterations(1, warm)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.run_iterations(1 + warm, iters)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for transform_timing.json")
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("transform_timing.py needs a CUDA device")
    from espm_b200 import SmoothNMF, build, config, synth
    from espm_b200.engine import FitEngine
    build.build()
    config.x_storage = "dense"
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda", torch.cuda.current_device())
    out = {"gpu": gpu_info(), "shape": dict(nx=NX, ny=NY, n=N, k=K), "iters": args.iters, "x_storage": "dense",
           "copy_bandwidth_gbs": copy_bandwidth_gbs()}
    prob = synth.make_problem(NX, NY, N, K, N_EL, seed=93)
    p = NX * NY
    for name, np_dt, t_dt in (("fp32", np.float32, torch.float32), ("fp64", np.float64, torch.float64)):
        G = prob["G_full"].astype(np_dt)
        W0, H0 = synth.init_factors(G.shape[1], K, p, 93, dtype=np_dt)
        XA = synth.poisson_X_torch(prob, 0, p, 93, dev, t_dt)
        est = SmoothNMF(n_components=K, G=G, shape_2d=(NX, NY), hspy_comp=True, max_iter=20, tol=0,
                        no_stop_criterion=True, verbose=0, **KW)
        with contextlib.redirect_stdout(io.StringIO()):
            est.fit_transform(XA.cpu().numpy().T, W=W0, H=H0)
        common = dict(shape_2d=(NX, NY), max_records=args.iters + 20, ingest=dict(eps=est.log_shift, normalize=None),
                      **KW)
        fit_ms = loop_ms(FitEngine(XA, G, W0, H0, **common), args.iters)
        del XA
        torch.cuda.empty_cache()
        XB = synth.poisson_X_torch(prob, 0, p, 94, dev, t_dt)
        eng = FitEngine(XB, est.G_, est.W_, H0, h_only=True, **common)
        h_ms = loop_ms(eng, args.iters)
        itemsize = np.dtype(np_dt).itemsize
        xbytes = N * p * itemsize
        del eng
        # transform on a pinned host array (the rows of X are pixels: (p, n))
        Xpin = torch.empty((p, N), dtype=t_dt, pin_memory=True)
        Xpin.copy_(XB.t())
        del XB
        torch.cuda.empty_cache()
        est.set_params(max_iter=args.iters)
        Xh = Xpin.numpy()
        with contextlib.redirect_stdout(io.StringIO()):
            est.transform(Xh[:1024 * 16], shape_2d=(32, 512))     # warm-up: module loads, allocator
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            Ht = est.transform(Xh)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        assert Ht.shape == (p, K) and np.all(np.isfinite(Ht))
        out[name] = {
            "fit_ms_per_iter": fit_ms, "transform_ms_per_iter": h_ms, "ratio": h_ms / fit_ms,
            "fit_x_gbs": 2 * xbytes / (fit_ms / 1e3) / 1e9, "transform_x_gbs": xbytes / (h_ms / 1e3) / 1e9,
            "fit_share_of_copy_bw": 2 * xbytes / (fit_ms / 1e3) / 1e9 / out["copy_bandwidth_gbs"],
            "transform_share_of_copy_bw": xbytes / (h_ms / 1e3) / 1e9 / out["copy_bandwidth_gbs"],
            "transform_wall_s": wall, "transform_wall_iters": args.iters,
        }
        print(name, json.dumps(out[name]))
        del Xpin, Xh
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "transform_timing.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
