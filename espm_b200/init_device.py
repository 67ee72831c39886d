"""NNDSVD initialisation of the fit on the device (SURVEY.md section 8 row a11, "next" rank 3).

``initialize_algorithms`` (espm/estimators/updates.py:160-223) calls scikit-learn's ``_initialize_nmf`` when neither
W nor H is given: a randomized SVD of X (``sklearn.utils.extmath._randomized_svd``: Gaussian test matrix, 7 (or 4)
power iterations normalised by LU, a QR, the SVD of the small projected matrix, ``svd_flip``) followed by the NNDSVD
sign split (Boutsidis & Gallopoulos 2008).  On the host that is 16 products with the full X (2 x 15 GFLOP each at
C3) and dominates ``fit_transform(X)`` by two orders of magnitude once the loop itself runs on the GPU.

Here the 16 products run on the device against the tile-major ``Xt`` the engine already holds (batched GEMMs over
the tiles through ``torch.matmul``; this is once-per-fit setup, not the per-iteration path), the tall LU / QR
factorisations run through ``torch.linalg`` on the device, and everything that is small (the (k+10) x n SVD, the LU of
the n x (k+10) matrix, the sign logic and the NNDSVD split on k vectors) stays on the host with the same SciPy calls
scikit-learn makes, so the random stream (``random_state.normal(size=(n, k+10))`` and the later draws of
``nndsvdar``) and every branch are the reference's.  The result agrees with ``_initialize_nmf`` to rounding (the
subspace iteration is contractive); ``tests/test_gpu_init.py`` checks it against scikit-learn on the same inputs.
"""
import numpy as np
import torch
from scipy import linalg

from . import _lib as L

_EPS = 1e-6   # sklearn/decomposition/_nmf.py: _initialize_nmf(..., eps=1e-6)


def _norm(x):
    """sklearn.decomposition._nmf.norm: sqrt(squared_norm(x))."""
    x = np.ravel(x)
    return np.sqrt(np.dot(x, x))


class _DeviceX:
    """Products with the processed data matrix X_ (n x p) held as tile-major Xt [tile][n_pad][128].

    Pixel-sharded fits (``eng.shard``): every rank holds the columns [j0, j1) of X_.  ``xt_times`` multiplies the local
    slab and all-gathers the rows (the tall p x r panels are 15 MB at C3: every rank then factorises the SAME full
    panel, so the algorithm and its pivoting are exactly the unsharded ones); ``x_times`` multiplies the local rows
    of its argument and all-reduces the n x r result."""

    def __init__(self, eng):
        st = eng.st
        self.n, self.p_loc, self.n_pad, self.n_tiles = eng.n, eng.p_loc, st.n_pad, st.n_tiles
        self.p, self.j0 = eng.p, eng.j0
        self.shard = eng.shard
        self.dtype = torch.float64 if eng.c_code == L.F64 else torch.float32
        if eng.x_code == L.U8:          # compact count storage: a dense copy for the 16 GEMMs of the initialisation
            self.T3 = eng.Xt.view(st.n_tiles, st.n_pad, L.TILE_PX).to(self.dtype)
        elif eng.x_code == L.U16:
            t = eng.Xt.view(torch.int16).view(st.n_tiles, st.n_pad, L.TILE_PX).to(self.dtype)
            self.T3 = torch.where(t < 0, t + 65536.0, t)
        else:
            self.T3 = eng.Xt.view(st.n_tiles, st.n_pad, L.TILE_PX)
        self.device = eng.Xt.device
        if self.shard is not None:
            import torch.distributed as dist
            self._dist = dist
            sizes = [None] * self.shard.world
            dist.all_gather_object(sizes, (int(self.j0), int(self.p_loc)), group=self.shard.group)
            self.bounds = sizes                          # (j0, p_loc) of every rank
            self.p_max = max(b[1] for b in sizes)

    def mean(self):
        # pad channels and pad pixels of Xt are zero
        tot = self.T3.sum(dtype=torch.float64).reshape(1)
        if self.shard is not None:
            self.shard.allreduce_sum(tot)
        return float(tot.item()) / (float(self.n) * float(self.p))

    def _gather_rows(self, Y_loc):
        """(p_loc x r) row blocks of every rank -> the full (p x r) matrix, on every rank."""
        if self.shard is None:
            return Y_loc
        r = Y_loc.shape[1]
        pad = torch.zeros(self.p_max, r, dtype=Y_loc.dtype, device=Y_loc.device)
        pad[:self.p_loc] = Y_loc
        parts = [torch.empty_like(pad) for _ in range(self.shard.world)]
        self._dist.all_gather(parts, pad, group=self.shard.group)
        out = torch.empty(self.p, r, dtype=Y_loc.dtype, device=Y_loc.device)
        for (j0, pl), part in zip(self.bounds, parts):
            out[j0:j0 + pl] = part[:pl]
        return out

    def xt_times(self, Qn):
        """X^T @ Qn for Qn (n x r) -> (p x r) (all pixels, on every rank)."""
        r = Qn.shape[1]
        Qp = torch.zeros(self.n_pad, r, dtype=self.dtype, device=self.device)
        Qp[:self.n] = Qn
        Y = torch.matmul(self.T3.transpose(1, 2), Qp)          # [tiles, 128, r]
        return self._gather_rows(Y.reshape(self.n_tiles * L.TILE_PX, r)[:self.p_loc])

    def x_times(self, Qp):
        """X @ Qp for Qp (p x r) -> (n x r); tiles are folded in chunks to bound the temporary."""
        r = Qp.shape[1]
        P3 = torch.zeros(self.n_tiles * L.TILE_PX, r, dtype=self.dtype, device=self.device)
        P3[:self.p_loc] = Qp[self.j0:self.j0 + self.p_loc] if self.shard is not None else Qp
        P3 = P3.view(self.n_tiles, L.TILE_PX, r)
        out = torch.zeros(self.n_pad, r, dtype=self.dtype, device=self.device)
        step = 256
        for t0 in range(0, self.n_tiles, step):
            out += torch.matmul(self.T3[t0:t0 + step], P3[t0:t0 + step]).sum(0)
        if self.shard is not None:
            self.shard.allreduce_sum(out)
        return out[:self.n]


def _lu_permute_l_device(Y):
    """scipy.linalg.lu(Y, permute_l=True)[0] for a tall device matrix: P @ L with unit lower-trapezoidal L."""
    p, r = Y.shape
    LU, piv = torch.linalg.lu_factor(Y)
    Lm = torch.tril(LU, diagonal=-1)
    idx = torch.arange(r, device=Y.device)
    Lm[idx, idx] = 1
    perm = np.arange(p)
    for i, pv in enumerate(piv.cpu().numpy().astype(np.int64) - 1):     # LAPACK row interchanges, in order
        perm[i], perm[pv] = perm[pv], perm[i]
    out = torch.empty_like(Lm)
    out[torch.as_tensor(perm, device=Y.device)] = Lm                   # row perm[j] of Y is row j of L U
    return out


def randomized_svd_device(eng, n_components, random_state, n_oversamples=10):
    """``_randomized_svd(X_, n_components, random_state=...)`` for n < p (the transposed branch of scikit-learn):
    returns (U (n x k), S (k), V (k x p)) as host arrays in X's dtype."""
    from sklearn.utils import check_random_state
    X = _DeviceX(eng)
    n, p = X.n, X.p
    if not n < p:
        raise ValueError("device NNDSVD expects fewer channels than pixels")
    rs = check_random_state(random_state)
    r = n_components + n_oversamples
    n_iter = 7 if n_components < 0.1 * min(n, p) else 4
    np_dtype = np.float32 if X.dtype == torch.float32 else np.float64
    # M = X^T (p x n); A = M; Q = normal(size=(A.shape[1], r)) = (n x r)
    Qn_host = rs.normal(size=(n, r)).astype(np_dtype, copy=False)
    Qn = torch.as_tensor(Qn_host, device=X.device)
    # cuSOLVER for the tall factorisations (torch's heuristic picks the MAGMA batched path for them: 3x slower at
    # 262144 x 14 and noisy); measured at C3: X^T Q 0.7 ms, LU 5.2 ms, X Q 1.2 ms, QR 3.1 ms
    prev = torch.backends.cuda.preferred_linalg_library()
    torch.backends.cuda.preferred_linalg_library("cusolver")
    try:
        for _ in range(n_iter):                                 # extmath.py: power iterations, LU normalised
            Qp = _lu_permute_l_device(X.xt_times(Qn))           # lu(A @ Q): p x r
            Yn = X.x_times(Qp).cpu().numpy()                    # A^T @ Q: n x r (small: host, SciPy like the reference)
            Qn = torch.as_tensor(linalg.lu(Yn, permute_l=True, check_finite=False)[0].astype(np_dtype, copy=False),
                                 device=X.device)
        Qp, _ = torch.linalg.qr(X.xt_times(Qn), mode="reduced")     # orthonormal basis of range(A): p x r
    finally:
        torch.backends.cuda.preferred_linalg_library(prev)
    B = X.x_times(Qp).t().cpu().numpy()                         # B = Q^T M = (X Q)^T: r x n
    Uhat, s, Vt = linalg.svd(B, full_matrices=False, lapack_driver="gesdd")
    # U = Q @ Uhat (p x r); only the first k columns are returned
    U_k = torch.matmul(Qp, torch.as_tensor(np.ascontiguousarray(Uhat[:, :n_components]).astype(np_dtype, copy=False),
                                           device=X.device)).cpu().numpy()
    # svd_flip(U, Vt, u_based_decision=False): signs from the largest |entry| of every row of Vt
    idx = np.argmax(np.abs(Vt), axis=1)
    signs = np.sign(Vt[np.arange(Vt.shape[0]), idx])
    Vt = Vt * signs[:, None]
    U_k = U_k * signs[None, :n_components]
    # transposed back: (Vt[:k].T, s[:k], U[:, :k].T)
    return Vt[:n_components].T.copy(), s[:n_components].copy(), U_k.T.copy(), X.mean()


def initialize_nmf_device(eng, n_components, init=None, random_state=None):
    """``sklearn.decomposition._nmf._initialize_nmf(X_, n_components, init, random_state)`` with the SVD on the
    device.  Returns (W (n x k), H (k x p)) host arrays (the D and H of updates.py:179)."""
    from sklearn.utils import check_random_state
    n, p = eng.n, eng.p
    if init is not None and init != "random" and n_components > min(n, p):
        raise ValueError("init = '{}' can only be used when n_components <= min(n_samples, n_features)".format(init))
    if init is None:
        init = "nndsvda" if n_components <= min(n, p) else "random"
    np_dtype = np.float64 if eng.c_code == L.F64 else np.float32
    if init == "random":
        avg = np_dtype(np.sqrt(_DeviceX(eng).mean() / n_components))
        rng = check_random_state(random_state)
        H = avg * rng.standard_normal(size=(n_components, p)).astype(np_dtype, copy=False)
        W = avg * rng.standard_normal(size=(n, n_components)).astype(np_dtype, copy=False)
        np.abs(H, out=H)
        np.abs(W, out=W)
        return W, H
    if init not in ("nndsvd", "nndsvda", "nndsvdar"):
        raise ValueError("Invalid init parameter: got %r instead of one of %r"
                         % (init, (None, "random", "nndsvd", "nndsvda", "nndsvdar")))
    U, S, V, x_mean = randomized_svd_device(eng, n_components, random_state)
    W = np.zeros_like(U)
    H = np.zeros_like(V)
    W[:, 0] = np.sqrt(S[0]) * np.abs(U[:, 0])
    H[0, :] = np.sqrt(S[0]) * np.abs(V[0, :])
    for j in range(1, n_components):
        x, y = U[:, j], V[j, :]
        x_p, y_p = np.maximum(x, 0), np.maximum(y, 0)
        x_n, y_n = np.abs(np.minimum(x, 0)), np.abs(np.minimum(y, 0))
        x_p_nrm, y_p_nrm = _norm(x_p), _norm(y_p)
        x_n_nrm, y_n_nrm = _norm(x_n), _norm(y_n)
        m_p, m_n = x_p_nrm * y_p_nrm, x_n_nrm * y_n_nrm
        if m_p > m_n:
            u, v, sigma = x_p / x_p_nrm, y_p / y_p_nrm, m_p
        else:
            u, v, sigma = x_n / x_n_nrm, y_n / y_n_nrm, m_n
        lbd = np.sqrt(S[j] * sigma)
        W[:, j] = lbd * u
        H[j, :] = lbd * v
    W[W < _EPS] = 0
    H[H < _EPS] = 0
    if init == "nndsvda":
        avg = np_dtype(x_mean)
        W[W == 0] = avg
        H[H == 0] = avg
    elif init == "nndsvdar":
        rng = check_random_state(random_state)
        avg = x_mean
        W[W == 0] = abs(avg * rng.standard_normal(size=len(W[W == 0])) / 100)
        H[H == 0] = abs(avg * rng.standard_normal(size=len(H[H == 0])) / 100)
    return W, H


def initial_H_device(eng, G, W, simplex_H, log_shift):
    """The H of ``initialize_factors(X_, G, W, None, ...)`` (updates.py:207-211, 220-221) with the product against X on
    the device: H0 = |lstsq(G W, X_)|, column-normalised when ``simplex_H``, clamped to ``log_shift``.

    The pseudo-inverse of G W (k x n, the minimum-norm least-squares solution with lstsq's rank cut-off) comes from the
    host; pinv(G W) X_ is one product with the tile-major Xt the engine holds (``_DeviceX.xt_times``, any storage type),
    and the abs / normalise / clamp run on the k x p device result.  No host copy of X is made.  Returns a (k, p)
    device tensor in the arithmetic type of the engine (all pixels, on every rank of a sharded engine)."""
    X = _DeviceX(eng)
    D = np.asarray(G, dtype=np.float64) @ np.asarray(W, dtype=np.float64)
    pinv = np.linalg.lstsq(D, np.eye(D.shape[0]), rcond=None)[0]           # k x n, lstsq(D, .) for any right side
    H = X.xt_times(torch.as_tensor(pinv.T.astype(_np_of(X.dtype)), device=X.device)).t().abs()   # (X_^T pinv^T)^T
    if simplex_H:
        H = H / H.sum(0, keepdim=True)
    return H.clamp_min(log_shift).contiguous()


def _np_of(dtype):
    return np.float64 if dtype == torch.float64 else np.float32
