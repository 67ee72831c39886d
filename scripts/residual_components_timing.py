"""Time SmoothNMF.residual_components (espm_resid_left / espm_resid_right) at the C3 size on one GPU.

    python scripts/residual_components_timing.py [--out profiles/residual_components_timing_c3.json]

C3: 512 x 512 pixels x 2048 channels, k = 4, G from espm_b200.synth, seeded Poisson X whose mean is the model; rank = 4,
so r = 14 columns (one launch of 16 per product).  For X stored dense f32, dense f64 and uint8:
  - espm_resid_left and espm_resid_right device time: CUDA events around 30 calls after 3 warm-up calls (the image is
    2.1 / 4.3 / 0.5 GB, far above the 126 MB L2);
  - espm_h_pass and espm_w_pass timed the same way on the same engine, in the same run;
  - n p sizeof(X) over each time, against the device-to-device copy bandwidth measured in the same run.
Then the wall time of ``est.residual_components(X, rank=4)`` (n_iter = 7: 15 products) on a pinned host f32 array, and
the same subspace iteration with the products computed by torch in fp64 on the device, chunked over pixels (the
reference of tests/test_gpu_residual_components.py).  The GPU name and power limit are read with nvidia-smi in the same
run.
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
RANK, N_ITER = 4, 7
WARM, REPS = 3, 30


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
    st, lib, stream = eng.st, eng.lib, eng.stream
    r = RANK + 10
    Q = torch.linalg.qr(torch.randn(N, r, dtype=torch.float64, device="cuda", generator=torch.Generator(
        "cuda").manual_seed(1)))[0].contiguous()
    P = torch.randn(r, eng.p_loc, dtype=torch.float64, device="cuda").contiguous()
    outs = {}
    for side, query in (("left", lib.espm_resid_left_scratch), ("right", lib.espm_resid_right_scratch)):
        nbytes = ctypes.c_int64(0)
        L.check(query(ctypes.byref(st), r, ctypes.byref(nbytes)))
        outs[side] = (torch.empty(max(nbytes.value // 8, 1), dtype=torch.float64, device="cuda"), nbytes.value)
    out_l = torch.empty(r, eng.p_loc, dtype=torch.float64, device="cuda")
    out_r = torch.empty(N, r, dtype=torch.float64, device="cuda")
    left_ms = launch_ms(lambda: L.check(lib.espm_resid_left(ctypes.byref(st), Q.data_ptr(), r, out_l.data_ptr(),
                                                            outs["left"][0].data_ptr(), stream)))
    first_l = out_l.clone()
    right_ms = launch_ms(lambda: L.check(lib.espm_resid_right(ctypes.byref(st), P.data_ptr(), r, out_r.data_ptr(),
                                                              outs["right"][0].data_ptr(), stream)))
    first_r = out_r.clone()
    h_ms = launch_ms(lambda: L.check(lib.espm_h_pass(ctypes.byref(st), stream)))
    w_ms = launch_ms(lambda: L.check(lib.espm_w_pass(ctypes.byref(st), stream)))
    L.check(lib.espm_resid_left(ctypes.byref(st), Q.data_ptr(), r, out_l.data_ptr(), outs["left"][0].data_ptr(), stream))
    L.check(lib.espm_resid_right(ctypes.byref(st), P.data_ptr(), r, out_r.data_ptr(), outs["right"][0].data_ptr(),
                                 stream))
    torch.cuda.synchronize()
    x_bytes = N * NX * NY * {"f32": 4, "f64": 8, "uint8": 1}[name]
    res = {"x_storage": eng.x_storage, "x_bytes": x_bytes, "r": r,
           "left_scratch_bytes": outs["left"][1], "right_scratch_bytes": outs["right"][1],
           "resid_left_ms": left_ms, "resid_right_ms": right_ms, "h_pass_ms": h_ms, "w_pass_ms": w_ms,
           "left_over_h_pass": left_ms / h_ms, "right_over_w_pass": right_ms / w_ms,
           "left_x_gbs": x_bytes / left_ms / 1e6, "right_x_gbs": x_bytes / right_ms / 1e6,
           "h_pass_x_gbs": x_bytes / h_ms / 1e6, "w_pass_x_gbs": x_bytes / w_ms / 1e6,
           "bit_identical_repeat": bool(torch.equal(first_l, out_l) and torch.equal(first_r, out_r))}
    eng.close()
    del eng, Xs, outs, out_l, out_r, first_l, first_r
    espm_b200.config.x_storage = "auto"
    torch.cuda.empty_cache()
    return res


def fitted(G, W, H):
    from espm_b200 import SmoothNMF
    with contextlib.redirect_stdout(io.StringIO()):
        est = SmoothNMF(n_components=H.shape[0], G=G)
    est.G_, est.W_, est.H_, est._identity_G = G.astype(np.float32), W.astype(np.float32), H.astype(np.float32), False
    est.physics_model_ = None
    return est


def torch_route(est, Xd, chunk=16384):
    """The same subspace iteration with torch fp64 products on the device (X already resident), from the same start."""
    from sklearn.utils import check_random_state
    from espm_b200.host import RESID_OVERSAMPLE, residual_components
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = Xd.device
    g = torch.as_tensor(np.maximum(est.G_.astype(np.float64) @ est.W_.astype(np.float64), LS), device=dev)
    Hc = torch.as_tensor(np.maximum(est.H_.astype(np.float64), LS), device=dev)
    p = Hc.shape[1]

    def chunks():
        for a in range(0, p, chunk):
            y = g @ Hc[:, a:a + chunk]
            yield a, (Xd[:, a:a + chunk].double() - y) / torch.sqrt(y)

    def left(Q):
        Qd = torch.as_tensor(Q, device=dev)
        return torch.cat([(R.T @ Qd).T for _, R in chunks()], dim=1)

    def right(P):
        out = torch.zeros(N, P.shape[0], dtype=torch.float64, device=dev)
        for a, R in chunks():
            out += R @ P[:, a:a + chunk].T
        return out.cpu().numpy()
    Q0 = check_random_state(0).standard_normal((N, RANK + RESID_OVERSAMPLE))
    s = residual_components(left, right, lambda P: (P @ P.T).cpu().numpy(), Q0, RANK, N_ITER)[0]
    torch.cuda.synchronize()
    return time.perf_counter() - t0, s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "residual_components_timing_c3.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("residual_components_timing.py needs a GPU")
    torch.cuda.set_device(0)
    from espm_b200 import build
    build.build()
    res = {"config": "C3 512x512 px x 2048 channels, k=4, rank=4 (r=14), n_iter=7", "gpu": gpu_info(),
           "warmup_calls": WARM, "timed_calls": REPS}
    res["copy_gbs"] = copy_bandwidth_gbs()
    G, W, H, X = problem()
    res["products"] = {name: time_storage(name, G, W, H, X) for name in ("f32", "f64", "uint8")}
    for v in res["products"].values():
        for side in ("left", "right", "h_pass", "w_pass"):
            v[side + "_x_over_copy_bw"] = v[side + "_x_gbs"] / res["copy_gbs"]
    est = fitted(G, W, H)
    t_ref, s_ref = torch_route(est, X)
    res["torch_fp64_route_s"] = t_ref
    Xh = torch.empty(X.shape, dtype=torch.float32, pin_memory=True)
    Xh.copy_(X)
    del X
    torch.cuda.empty_cache()
    Xn = Xh.numpy()
    walls = []
    for _ in range(4):
        t0 = time.perf_counter()
        rc = est.residual_components(Xn, rank=RANK, n_iter=N_ITER, random_state=0)
        walls.append(time.perf_counter() - t0)
    res["residual_components_pinned_f32_s"] = {"first": walls[0], "min_of_next_3": min(walls[1:])}
    res["residual_components_x_storage"] = "auto (uint8 for this image)"
    res["singular_values"] = rc.singular_values.tolist()
    res["torch_fp64_singular_values"] = s_ref.tolist()
    res["max_rel_diff_vs_torch_fp64"] = float(np.max(np.abs(rc.singular_values - s_ref) / s_ref))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
