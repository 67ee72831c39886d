"""Host-side pieces of the fit that run once per fit on k x p / m x k data (NumPy).

They are part of the reference's prologue / epilogue (SURVEY.md section 8a rows a2, a11, a15): the
zero-line repair and normalisation of X, the initial factors, and the final column rescale.  None of
them is on the per-iteration path.
"""
import numpy as np


def is_physical_model(G):
    """Duck-typed ``isinstance(G, espm.models.base.PhysicalModel)`` (base.py:269): the three callbacks
    the loop uses are NMF_update / NMF_simplex / NMF_initialize_W (models/base.py:217-264)."""
    return (G is not None and not isinstance(G, np.ndarray)
            and all(hasattr(G, a) for a in ("NMF_update", "NMF_simplex", "NMF_initialize_W")))


def remove_zeros_lines(X, epsilon):
    """All-zero rows / columns of X are set to epsilon; negatives are rejected (base.py:519-528)."""
    if not np.all(X >= 0):
        raise ValueError("Negative values in data")
    out = X.copy()
    zero_cols = np.flatnonzero(X.sum(axis=0) == 0)
    zero_rows = np.flatnonzero(X.sum(axis=1) == 0)
    if zero_cols.size:
        out[:, zero_cols] = epsilon
    if zero_rows.size:
        out[zero_rows, :] = epsilon
    return out


def normalization_factor(X, nc):
    """base.py:16-18."""
    return nc / (np.mean(X) * X.shape[0])


def rescaled_DH(D, H):
    """Column rescale so that the columns of H sum to ~1 (utils.py:79-96)."""
    from scipy.optimize import nnls
    ones = np.ones((H.shape[1],))
    s = np.linalg.lstsq(H.T, ones, rcond=None)[0]
    if (s <= 0).any():
        s = np.maximum(nnls(H.T, ones)[0], 1e-10)
    return D @ np.diag(1 / s), np.diag(s) @ H


def initialize_factors(X, G, W, H, n_components, init, random_state, simplex_H, simplex_W, log_shift,
                       physics_model=None, nmf_init=None):
    """Initial (G, W, H) following updates.py:160-223.

    Missing factors come from scikit-learn's NMF initialisation plus least squares; user-supplied
    ones are only clamped to ``log_shift`` (updates.py:220-221).  Returns ``G`` as a dense array even
    when it is the identity (the ``G_`` attribute of the reference, updates.py:166).
    """
    identity = G is None
    if identity:
        G_dense = np.diag(np.ones(X.shape[0]).astype(X.dtype))
    else:
        G_dense = np.asarray(G)
    if W is None:
        if H is None:
            if nmf_init is not None:     # NNDSVD with the SVD on the device (init_device.py); X may be None then
                D, H = nmf_init(n_components, init, random_state)
            else:
                from sklearn.decomposition._nmf import _initialize_nmf
                D, H = _initialize_nmf(X, n_components=n_components, init=init, random_state=random_state)
            if simplex_H:
                H = np.nan_to_num(H, nan=1.0 / H.shape[0])
                scale = np.sum(H, axis=0, keepdims=True)
                H = H / scale
                D = D * np.mean(scale)
        else:
            D = np.abs(np.linalg.lstsq(H.T, X.T, rcond=None)[0].T)
        if identity:
            W = D
        elif physics_model is not None:
            W = physics_model.NMF_initialize_W(D)
            if simplex_W:
                idx = physics_model.NMF_simplex()
                W = np.nan_to_num(W, nan=1.0 / W.shape[0])
                W[idx, :] = W[idx, :] / np.sum(W[idx, :], axis=0, keepdims=True)
        else:
            W = np.abs(np.linalg.lstsq(G_dense, D, rcond=None)[0])
            if simplex_W:
                W = np.nan_to_num(W, nan=1.0 / W.shape[0])
                W = W / np.sum(W, axis=0, keepdims=True)
    elif H is None:
        D = G_dense @ W
        H = np.abs(np.linalg.lstsq(D, X, rcond=None)[0])
        if simplex_H:
            H = H / np.sum(H, axis=0, keepdims=True)
    W = np.maximum(W, log_shift)
    H = np.maximum(H, log_shift)
    return G_dense, W, H


# ---- ground-truth tracking (base.py:335-347; measures.py:10-50, 125-153, 166-207, 256-285, 579-627) -------------
def _unique_min(matrix):
    """measures.py:166-207: assignment with distinct rows that minimises the sum (brute force over permutations)."""
    from itertools import permutations
    n = matrix.shape[0]
    perms = list(permutations(range(n), n))
    sums = []
    for perm in perms:
        acc = 0
        for i in range(n):
            acc += matrix[perm[i], i]
        sums.append(acc)
    best = perms[sums.index(min(sums))]
    return [matrix[best[i], i] for i in range(n)], best


def find_min_angle(true_vectors, algo_vectors):
    """measures.py:125-153 with unique=True: spectral angles (degrees) of the best one-to-one match."""
    v1 = true_vectors / np.sqrt(np.sum(true_vectors ** 2, axis=1, keepdims=True))
    v2 = algo_vectors / np.sqrt(np.sum(algo_vectors ** 2, axis=1, keepdims=True))
    ang = np.arccos(np.clip(v1 @ v2.T, -1.0, 1.0)) * 180 / np.pi
    return _unique_min(ang)[0]


def find_min_MSE(true_maps, algo_maps):
    """measures.py:256-285 with unique=True on the squared distances of measures.py:579-627."""
    xx = (true_maps * true_maps).sum(axis=1)
    yy = (algo_maps * algo_maps).sum(axis=1)
    xy = np.dot(true_maps, algo_maps.T)
    d = abs(np.kron(np.ones((algo_maps.shape[0], 1)), xx).T + np.kron(np.ones((true_maps.shape[0], 1)), yy) - 2 * xy)
    return _unique_min(d / true_maps.shape[1])[0]


# ---- SmoothNMF.phase_uncertainty: covariance of W from the per-channel information the device computes ------------
PIVOT_REL = 1e-12      # a Cholesky pivot <= PIVOT_REL max diag marks the information singular (as hinfo.cuh)


def _cholesky(F):
    """Lower Cholesky factor of F, or None when F is singular: an all-zero diagonal, a failed factorisation or a pivot
    L_ii^2 <= PIVOT_REL max_i F_ii."""
    dmax = float(np.max(np.diag(F))) if F.size else 0.0
    if not dmax > 0.0:
        return None
    try:
        L = np.linalg.cholesky(F)
    except np.linalg.LinAlgError:
        return None
    return L if np.min(np.diag(L)) ** 2 > PIVOT_REL * dmax else None


def _inverse(F):
    from scipy.linalg import cho_solve
    L = _cholesky(F)
    return None if L is None else cho_solve((L, True), np.eye(F.shape[0]))


def unpack_triangles(packed, k):
    """(k(k+1)/2, n) packed upper triangles, row by row -> (n, k, k) symmetric matrices."""
    iu = np.triu_indices(k)
    out = np.empty((packed.shape[1], k, k))
    out[:, iu[0], iu[1]] = packed.T
    out[:, iu[1], iu[0]] = packed.T
    return out


def phase_covariance(A_packed, G, free, simplex_rows):
    """Constrained Cramer-Rao bound of the phases W (m x k) from the per-channel information of the device.

    A_packed : (k(k+1)/2, n) A_c[a, b] = sum_j x_cj h_aj h_bj / y_cj^2, packed upper triangles row by row.
    G : (n, m) or None for the identity (m = n).
    free : (m, k) bool, the entries of W the fit updates.
    simplex_rows : None, or the rows S of W whose column sums the fit holds: one constraint sum_{e in S} W_ea = const per
        column a over its free entries (dropped when it has none).

    The information of vec(W), index (e, a), is F[(e,a),(f,b)] = sum_c G_ce G_cf A_c[a, b]; on the free entries
    C = F^-1 - F^-1 A^T (A F^-1 A^T)^-1 A F^-1 for the constraint matrix A.  Returns (std, covariance, information,
    spectrum_std), float64:
      real G: std (m, k), covariance and information (m, k, m, k), spectrum_std (n, k) with
              spectrum_std[c, a]^2 = sum_{e,f} G_ce G_cf C[(e,a),(f,a)]; a singular F makes std, covariance and
              spectrum_std all NaN;
      G None: F is block diagonal (blocks A_c), and only the blocks are returned: std (n, k), covariance and information
              (n, k, k), spectrum_std = std.  With B_c = A_c^-1 on the free phases of channel c and M = sum_{c in S} B_c,
              the block of C is B_c - B_c M^-1 B_c (no dense nk x nk matrix is formed).  A channel with singular A_c is
              NaN and is left out of M, as a fixed entry is.
    Fixed entries have std 0 and zero covariance rows."""
    nt, n = A_packed.shape
    k = int(round((np.sqrt(8 * nt + 1) - 1) / 2))
    A = unpack_triangles(np.asarray(A_packed, dtype=np.float64), k)
    free = np.asarray(free, dtype=bool)
    if G is None:
        return _block_covariance(A, free, simplex_rows)
    G = np.asarray(G, dtype=np.float64)
    m = G.shape[1]
    GG = (G[:, :, None] * G[:, None, :]).reshape(n, m * m)
    F = (GG.T @ A.reshape(n, k * k)).reshape(m, m, k, k).transpose(0, 2, 1, 3).reshape(m * k, m * k)
    phi = np.flatnonzero(free.reshape(-1))
    C = np.zeros((m * k, m * k))
    if phi.size:
        Fi = _inverse(F[np.ix_(phi, phi)])
        if Fi is None:
            nan = np.full((m, k), np.nan)
            return nan, np.full((m, k, m, k), np.nan), F.reshape(m, k, m, k), np.full((n, k), np.nan)
        if simplex_rows is not None:
            in_S = np.zeros(m, dtype=bool)
            in_S[np.asarray(simplex_rows, dtype=np.int64)] = True
            rows = [(in_S[:, None] & free & (np.arange(k) == a)[None, :]).reshape(-1)[phi] for a in range(k)]
            Acon = np.array([r for r in rows if r.any()], dtype=np.float64).reshape(-1, phi.size)
            if Acon.shape[0]:
                B = Fi @ Acon.T
                Fi = Fi - B @ np.linalg.solve(Acon @ B, B.T)
        C[np.ix_(phi, phi)] = 0.5 * (Fi + Fi.T)
    C = C.reshape(m, k, m, k)
    std = np.sqrt(np.maximum(np.einsum("eaea->ea", C), 0.0))
    spec = np.stack([((G @ C[:, a, :, a]) * G).sum(1) for a in range(k)], axis=1)
    return std, C, F.reshape(m, k, m, k), np.sqrt(np.maximum(spec, 0.0))


def _block_covariance(A, free, simplex_rows):
    n, k, _ = A.shape
    B = np.zeros((n, k, k))
    ok = np.ones(n, dtype=bool)
    for c in range(n):
        idx = np.flatnonzero(free[c])
        if idx.size:
            Bi = _inverse(A[c][np.ix_(idx, idx)])
            if Bi is None:
                ok[c] = False
            else:
                B[c][np.ix_(idx, idx)] = Bi
    C = B.copy()
    if simplex_rows is not None:
        in_S = np.zeros(n, dtype=bool)
        in_S[np.asarray(simplex_rows, dtype=np.int64)] = True
        sel = in_S & ok
        M = B[sel].sum(0)
        act = np.flatnonzero(np.diag(M) > 0)            # columns with a free entry
        if act.size:
            Ba = B[sel][:, :, act]                       # (s, k, r)
            C[sel] -= Ba @ np.linalg.solve(M[np.ix_(act, act)], np.swapaxes(Ba, 1, 2))
            C[sel] = 0.5 * (C[sel] + np.swapaxes(C[sel], 1, 2))
    C[~ok] = np.nan
    std = np.sqrt(np.maximum(np.diagonal(C, axis1=1, axis2=2), 0.0))
    std[~ok] = np.nan
    return std, C, A, std.copy()


RESID_OVERSAMPLE = 10   # extra columns of the residual subspace iteration (scikit-learn's randomized_svd default)


def residual_components(left, right, gram, Q0, rank, n_iter):
    """Leading ``rank`` singular triplets of the residual R (n x p) by randomized subspace iteration on the channel side,
    in fp64, with R reached only through three callables:

        left(Q)  this rank's P = (R^T Q)^T, (r, p_loc), for an orthonormal Q (n, r) (one pass over X)
        right(P) R P^T summed over the ranks in rank order, (n, r) host array (one pass over X)
        gram(P)  P P^T summed over the ranks in rank order, (r, r) host array

    Q0 (n, r) is the Gaussian start, identical on every rank.  Q = qr(Q0); n_iter times Q = qr(R R^T Q); then
    P = (R^T Q)^T, M = P P^T = U diag(s^2) U^T, spectra = Q U and maps = (P^T U / s)^T.  Every tall factorisation is on
    the n side (n x r QR); no p x r panel is gathered.  Forming M squares the condition: component i loses about
    eps (s_1 / s_i)^2 of relative accuracy, harmless in fp64 for the leading components returned.  Sign: the entry of
    largest magnitude of every spectrum is positive.

    Returns (s (rank,), spectra (n, rank), V (r, rank), P): this rank's maps are V^T P."""
    Q = np.linalg.qr(np.asarray(Q0, dtype=np.float64))[0]
    for _ in range(n_iter):
        Q = np.linalg.qr(right(left(Q)))[0]
    P = left(Q)
    w, U = np.linalg.eigh(gram(P))
    order = np.argsort(w, kind="stable")[::-1][:rank]
    s = np.sqrt(np.maximum(w[order], 0.0))
    U = U[:, order]
    spectra = Q @ U
    lead = spectra[np.argmax(np.abs(spectra), axis=0), np.arange(rank)]
    sign = np.where(lead < 0, -1.0, 1.0)
    spectra *= sign
    V = U * (sign / np.where(s > 0, s, np.inf))
    return s, spectra, V, P
