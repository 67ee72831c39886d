"""Device-side state of one SmoothNMF fit and the kernel sequencing of one iteration.

The arithmetic lives in libespm_b200.so (hand-written sm_100a CUDA, see csrc/); this module only
allocates device buffers through torch, fills the ``espm_state`` struct the C ABI takes, launches the
kernels in order on torch's current stream and rotates the W / H / GW buffers between iterations.

One iteration of the reference (base.py:316-324) maps to two phases here:

  phase A ``evaluate(slot)``   h_pass -> h_finish (its last CTA writes the scalar record)
        streams X once with (GW_cur, H_cur): ratio sums for the next H update AND every loss term of
        the current iterate (KL, log-reg, Laplacian), rel_H, written to the scalar record ``slot``.
  phase B ``advance(slot)``    [h_apply] -> w_pass -> w_reduce -> w_finish, then buffer rotation
        H_next from the lock-step bisection, streams X once more with (GW_cur, H_next), W_next,
        GW_next; rel_W goes to record ``slot`` (the record of the iterate being produced).

So X is read exactly twice per iteration (SURVEY.md section 8d); the loss of iterate t rides the H pass
of iteration t+1.  With ``h_only`` (W fixed, ``SmoothNMF.transform``) phase B is [h_apply] -> h_stats and X is read
once per iteration.
"""
import ctypes

import numpy as np
import torch

from . import _lib as L


def _round_up(a, b):
    return (a + b - 1) // b * b


def _np_dtype(code):
    return np.float64 if code == L.F64 else np.float32


def _torch_dtype(code):
    return torch.float64 if code == L.F64 else torch.float32


_X_ITEMSIZE = {L.F32: 4, L.F64: 8, L.U8: 1, L.U16: 2}
RESID_RB = 16     # columns per launch of the residual products (RESID_RB of csrc/resid.cuh)


def _resid_blocks(r):
    return -(-r // RESID_RB)


def _code_of(dtype):
    if isinstance(dtype, torch.dtype):
        dtype = {torch.float32: np.float32, torch.float64: np.float64}.get(dtype, None)
        if dtype is None:
            raise TypeError("espm_b200 supports float32 and float64 data")
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return L.F64
    if dtype == np.float32:
        return L.F32
    raise TypeError("espm_b200 supports float32 and float64 data, got %s" % dtype)


class FitEngine:
    """Owns the device buffers of one fit on ONE GPU (one pixel shard when running on several)."""

    def __init__(self, X, G, W0, H0, *, shape_2d=None, lambda_L=0.0, mu=0, epsilon_reg=1.0,
                 log_shift=1e-14, dicotomy_tol=1e-5, dicotomy_tol_w=1e-5, tol=1e-4, sigma=8.0,
                 simplex_H=False, simplex_W=True, simplex_rows=None, fixed_H=None, fixed_W=None,
                 x_scale=1.0, max_records=512, device=None, shard=None, c_dtype=None, clamp_init=True,
                 x_local=False, ingest=None, algo="log_surrogate", l2=False, l2_h=False, linesearch=False,
                 gamma_pg=None, h_only=False):
        """
        X : (n, p) array-like view (any strides; C order or the transposed hyperspy layout are
            uploaded without a host copy).  G : (n, m) array or None (identity).  W0 : (m, k), H0 : (k, p).
        shard : None, or (rank, world, comm) for pixel-sharded multi-GPU runs (see dist.py).
        ingest : None (X is used as given, times ``x_scale``), or dict(eps=..., normalize=None | n_components):
            the prologue of the reference's fit runs on the device instead of the host -- NaN / inf /
            negative checks, remove_zeros_lines (base.py:519-528), normalize (base.py:264-267) and
            const_KL_ (base.py:200-201).  Results: ``self.const_KL``, ``self.norm_factor``,
            ``self.n_zero_rows`` / ``self.n_zero_cols``.  With ``check_only=True`` only the checks run: X is held as
            given (``for_statistics``).
        h_only : W0 is held fixed and only H is iterated (``SmoothNMF.transform``, ESPM_FLAG_H_ONLY): ``advance`` runs
            [h_apply] -> h_stats and rotates the H buffers only, so an iteration streams X once (the H pass).  Only
            the multiplicative H steps (``log_surrogate`` / ``l2_surrogate``) with the KL loss.
        """
        self.lib = L.load()
        self.clamp_init = clamp_init
        self.clamped = False
        if not torch.cuda.is_available():
            raise L.EspmError("espm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        torch.cuda.set_device(self.device)
        self.shard = shard
        n, p = X.shape
        if x_local:
            p = H0.shape[1]          # X is already this rank's pixel slab (n, p_loc); H0 is global
        self.x_local = x_local
        self.profile = None          # set to {} to record CUDA events around kernel launches
        self.profile_names = ("h_pass", "w_pass")
        self.n_launches = 0          # kernels launched through the C ABI (bench.py reports the count)
        k = W0.shape[1]
        self.n, self.p, self.k = n, p, k
        self.identity_G = G is None
        self.m = n if G is None else G.shape[1]
        if W0.shape != (self.m, k) or H0.shape != (k, p):
            raise ValueError("inconsistent shapes: X %s G %s W %s H %s" % (
                X.shape, None if G is None else G.shape, W0.shape, H0.shape))
        x_code = _code_of(X.dtype)
        if c_dtype is None:
            # NumPy promotion of the reference: any float64 operand makes the update float64
            parts = [np.dtype(_np_dtype(x_code)), np.dtype(W0.dtype), np.dtype(H0.dtype)]
            if G is not None:
                parts.append(np.dtype(G.dtype))
            c_dtype = np.result_type(*parts)
        c_code = _code_of(c_dtype)
        if x_code == L.F64:
            c_code = L.F64
        self.x_code, self.c_code = x_code, c_code
        self.cdt = _torch_dtype(c_code)
        self.cnp = _np_dtype(c_code)

        # ---- pixel shard (contiguous image rows, SURVEY.md section 8e) ----
        if shape_2d is not None:
            nx, ny = int(shape_2d[0]), int(shape_2d[1])
            if nx * ny != p:
                raise ValueError("shape_2d %s does not match p=%d" % (shape_2d, p))
        else:
            nx, ny = 0, 0
        self.nx, self.ny = nx, ny
        if shard is None:
            self.rank, self.world = 0, 1
            j0, j1, row0 = 0, p, 0
        else:
            from .dist import shard_bounds
            self.rank, self.world = shard.rank, shard.world
            j0, j1, row0 = shard_bounds(p, nx, ny, self.rank, self.world)
        self.j0, self.j1, self.row0 = j0, j1, row0
        p_loc = j1 - j0
        self.p_loc = p_loc

        # ---- H2D copy of this rank's slab, then the storage type of Xt (it decides the launch plan) ----
        self.src_code = x_code                       # dtype of the uploaded raw X
        self._stage_x(X)
        x_code = self._choose_storage(x_code, c_code, x_scale, ingest)
        self.x_code = x_code

        st = L.EspmState()
        self.st = st
        st.n, st.m, st.k = n, self.m, k
        st.p_loc, st.p_total = p_loc, p
        st.nx, st.ny, st.row0 = nx, ny, row0
        st.x_dtype, st.c_dtype = x_code, c_code
        st.maxit = L.MAXIT_DICHOTOMY
        flags = 0
        if simplex_H:
            flags |= L.FLAG_SIMPLEX_H
        if simplex_W:
            flags |= L.FLAG_SIMPLEX_W
        if self.identity_G:
            flags |= L.FLAG_G_IDENTITY
        if algo == "l2_surrogate":
            flags |= L.FLAG_HQ                   # quadratic-surrogate H step (updates.py:263-301)
        elif algo == "bmd":
            flags |= L.FLAG_BMD                  # use_bregman branches (updates.py:40-48, 120-125)
        elif algo == "projected_gradient":
            flags |= L.FLAG_PG                   # proj_grad_step_h / _w (updates.py:347-391)
        elif algo != "log_surrogate":
            raise ValueError("Unknown algorithm")                      # smooth_nmf.py:374
        if l2:
            flags |= L.FLAG_L2                   # Frobenius loss + W step (base.py:197-198, updates.py:29-36)
        if l2_h:
            flags |= L.FLAG_L2_H                 # Frobenius H step / gradient (updates.py:109-118, 330-332)
        if flags & (L.FLAG_BMD | L.FLAG_PG | L.FLAG_L2):
            flags &= ~L.FLAG_SIMPLEX_W           # those W branches have no simplex projection (updates.py:29-48)
        self.h_only = bool(h_only)
        if self.h_only:
            if flags & (L.FLAG_BMD | L.FLAG_PG | L.FLAG_L2 | L.FLAG_L2_H) or linesearch or fixed_W is not None:
                raise ValueError("h_only supports the log_surrogate / l2_surrogate H steps with the KL loss, "
                                 "without linesearch or fixed_W")
            flags |= L.FLAG_H_ONLY
        self.pg_ls = False
        if linesearch:
            if flags & L.FLAG_PG:
                self.pg_ls = True                # quadratic-surrogate line search (smooth_nmf.py:383-401, 438-447)
            else:
                flags |= L.FLAG_LINESEARCH
        self.algo = algo
        self.gamma_pg = gamma_pg
        mu_arr = np.zeros(L.MAX_K)
        if np.isscalar(mu):
            mu_arr[:k] = float(mu)
        else:
            mu_v = np.asarray(mu, dtype=np.float64).reshape(-1)
            if mu_v.shape[0] != k:
                raise ValueError("mu must be a scalar or a vector of length n_components")
            mu_arr[:k] = mu_v
        if np.any(mu_arr != 0):
            flags |= L.FLAG_MU
        if lambda_L != 0:
            flags |= L.FLAG_LAPLACIAN
        for i in range(L.MAX_K):
            st.mu[i] = mu_arr[i]
        st.lambda_L, st.sigma, st.eps_reg = float(lambda_L), float(sigma), float(epsilon_reg)
        st.log_shift, st.dicotomy_tol, st.dicotomy_tol_w, st.tol = (
            float(log_shift), float(dicotomy_tol), float(dicotomy_tol_w), float(tol))
        from . import config as _config
        if not getattr(_config, "speculate_h", True):
            flags |= L.FLAG_NO_HSPEC
        st.flags = flags
        L.check(self.lib.espm_plan(ctypes.byref(st)))

        dev, cdt = self.device, self.cdt
        kp, n_pad, p_pad = st.kp, st.n_pad, st.p_pad
        halo = _round_up(ny, 32) if ny > 0 else 0
        ldh = _round_up(halo + p_pad + halo, 32)
        st.halo, st.ldh = halo, ldh
        self.halo, self.ldh = halo, ldh

        def zeros(*shape, dtype=cdt):
            return torch.zeros(*shape, dtype=dtype, device=dev)

        # ---- state buffers (rotated by pointer) ----
        # H pad pixels hold 1 so that padded pixels give y > 0 (their X is 0: they contribute nothing)
        self.peer = shard is not None and getattr(shard, "use_peer", False)
        self._seq_s = self._seq_m = 0
        if self.peer:
            self.Hbuf = shard.setup_peer(self)       # H lives in CUDA-IPC memory the neighbours can write
            if self.Hbuf is None:                    # collective: some rank cannot map a peer -> NCCL exchange
                from .dist import Shard
                self.shard = shard = Shard(group=shard.group)
                self.peer = False
            else:
                self._seq_s, self._seq_m = shard.seq  # the flag words persist across fits: keep counting
        self.inbox = None
        if not self.peer:
            self.Hbuf = [torch.ones(k, ldh, dtype=cdt, device=dev) for _ in range(3)]
        self.Wbuf = [zeros(self.m, k) for _ in range(2)]
        self.GWbuf = [zeros(n_pad, kp) for _ in range(2)]
        self.GWcbuf = [zeros(n_pad, kp) for _ in range(2)]
        self.gwstats = [zeros(2 * kp) for _ in range(2)]
        self.hstats = [zeros(3 * kp, dtype=torch.float64) for _ in range(2)]
        self.ih = [0, 1, 2]      # indices of (prev, cur, next) H buffers
        self.iw = [0, 1]         # (cur, next) for W / GW / gwstats
        self.ihs = [0, 1]        # (cur, next) for hstats
        self.have_prev = False
        # ---- scratch ----
        self.numraw = zeros(st.h_nsplit, kp, p_pad)
        self.num = zeros(kp, p_pad)
        self.den = zeros(kp, p_pad)
        self.s_part = zeros(st.w_nr, n_pad, kp)
        self.s_sum = zeros(n_pad, kp)
        self.w_num = zeros(self.m, k)
        self.w_den = zeros(self.m, k)
        self.xlogy_part = zeros(max(st.h_grid, 1), dtype=torch.float64)
        self.px_part = zeros(st.px_blocks, 3 + 3 * kp, dtype=torch.float64)
        self.mask = torch.zeros(4 * max(self.world, 1), dtype=torch.int32, device=dev)
        self.bisect_dec = torch.zeros(5 * p_pad if simplex_H else 1, dtype=torch.int32, device=dev)
        st.bisect_dec = self.bisect_dec.data_ptr()
        self.bisect_anchor = torch.zeros(2 * p_pad if simplex_H else 2, dtype=torch.float64, device=dev)
        st.bisect_anchor = self.bisect_anchor.data_ptr()
        # ---- alternative update rules ----
        self.gram = zeros(2, kp * kp, dtype=torch.float64)
        st.gram_gw, st.gram_h = self.gram[0].data_ptr(), self.gram[1].data_ptr()
        self.sigma_dev = None
        if st.flags & L.FLAG_LINESEARCH:
            self.sigma_dev = torch.full((1,), float(sigma), dtype=torch.float64, device=dev)
            self.ls_part = zeros(st.px_blocks + 3, 4 + kp, dtype=torch.float64)
            st.sigma_dev, st.ls_part = self.sigma_dev.data_ptr(), self.ls_part.data_ptr()
        if self.pg_ls:
            self.ls_part = zeros(st.px_blocks + 3, 4 + kp, dtype=torch.float64)
            st.ls_part = self.ls_part.data_ptr()
        if shard is not None and (self.pg_ls or (st.flags & L.FLAG_LINESEARCH)):
            st.flags |= L.FLAG_LS_PARTIAL        # the sums of the line search are combined over the ranks on the host
        self._eval_slot = 0
        self._pg_w_pending = None
        self._w_after_eval = None
        if gamma_pg is not None:
            st.gamma_h, st.gamma_w = float(gamma_pg[0]), float(gamma_pg[1])
        self.dev_flags = torch.zeros(8, dtype=torch.int32, device=dev)
        self.coop_part = zeros(L.COOP_BLOCKS * (2 * L.MAX_K + 4), dtype=torch.float64)
        self.max_records = int(max_records)
        # The scalar records live in PINNED HOST memory that the kernels write directly (unified addressing: the host
        # pointer is valid on the device): a record needs no D2H copy and no stream synchronisation -- its last word is
        # a stamp the host can poll (wait_record), so the loop with stop tests runs one iteration ahead of the host.
        self.records = torch.zeros(self.max_records, L.NSCALARS, dtype=torch.float64).pin_memory()
        self.rec_np = self.records.numpy()
        self._stamp = 0
        self._stamps = {}
        if self.peer:
            # sharded: every rank's share of a record lands in every host's inbox (dist._RecordInbox)
            self.inbox = shard.setup_inbox(self, self.max_records)
            if self.inbox is not None:
                self._stamp = self.inbox.stamp
        st.numraw, st.num, st.den = self.numraw.data_ptr(), self.num.data_ptr(), self.den.data_ptr()
        st.s_part, st.s_sum = self.s_part.data_ptr(), self.s_sum.data_ptr()
        # tile-major copy of H_next read by the W pass; pad pixels stay 1 (y > 0), pad rows are never read
        self.Ht = torch.ones(st.n_tiles * kp * L.TILE_PX, dtype=cdt, device=dev)
        st.Ht = self.Ht.data_ptr()
        st.w_num, st.w_den = self.w_num.data_ptr(), self.w_den.data_ptr()
        st.xlogy_part, st.px_part = self.xlogy_part.data_ptr(), self.px_part.data_ptr()
        st.bisect_mask, st.dev_flags = self.mask.data_ptr(), self.dev_flags.data_ptr()
        st.coop_part = self.coop_part.data_ptr()
        if shard is None or self.peer:
            st.flags |= L.FLAG_FUSED_WREDUCE      # w_finish folds the W-pass partials itself

        # ---- constant inputs ----
        self.fixed_H = None
        if fixed_H is not None:
            fh = torch.full((k, ldh), -1.0, dtype=cdt, device=dev)
            fh[:, halo:halo + p_loc] = torch.as_tensor(np.ascontiguousarray(fixed_H[:, j0:j1]), dtype=cdt).to(dev)
            self.fixed_H = fh
            st.fixed_H = fh.data_ptr() + halo * fh.element_size()
            st.flags |= L.FLAG_FIXED_H
            if np.any((fixed_H >= 0) & (fixed_H < log_shift)):
                st.flags |= L.FLAG_LOSS_DUAL      # H may drop below log_shift: loss clamps, update does not
        self.fixed_W = None
        if fixed_W is not None:
            self.fixed_W = torch.as_tensor(np.ascontiguousarray(fixed_W), dtype=cdt).to(dev)
            st.fixed_W = self.fixed_W.data_ptr()
            st.flags |= L.FLAG_FIXED_W
        self.simplex_rows = None
        if simplex_rows is not None:
            rows = np.asarray(simplex_rows, dtype=np.int32).reshape(-1)
            self.simplex_rows = torch.as_tensor(rows).to(dev)
            st.simplex_rows = self.simplex_rows.data_ptr()
            st.n_simplex_rows = int(rows.shape[0])
            st.flags |= L.FLAG_SIMPLEX_ROWS
        self.G = self.Gt = self.colsum_G = None
        self._bind()
        self.const_KL = None
        self.norm_factor = None
        self.n_zero_rows = self.n_zero_cols = 0
        self._retile_x(x_scale, ingest)
        self.x_colsum = self.x_rowsum = None
        if st.flags & L.FLAG_BMD:
            self.compute_x_sums()
        self.set_G(G, prepare=False)
        self._init_WH(W0, H0)

    @classmethod
    def for_statistics(cls, X, G, W, H, *, log_shift, shard=None):
        """Engine for ``fit_statistics`` of the model (G, W, H) against X: X goes through the NaN / inf / negative checks
        of the fit's ingest but is otherwise held as given (no remove_zeros_lines patch, no scale; uint8 / uint16 storage
        as ``config.x_storage`` decides), and W, H are not clamped (the kernel clamps G W and H itself)."""
        return cls(X, G, W, H, log_shift=log_shift, simplex_W=False, clamp_init=False, max_records=2, shard=shard,
                   ingest=dict(eps=log_shift, normalize=None, check_only=True))

    def fit_statistics(self):
        """Per-pixel and per-channel sums of x, y, kl and chi2 of (W_cur, H_cur) against X (espm_fit_stats): this rank's
        (4, p_loc) pixel block and (4, n) channel block, device float64 tensors."""
        st, dev = self.st, self.device
        scratch = self._scratch(self.lib.espm_fit_stats_scratch)
        pix = torch.empty(4, self.p_loc, dtype=torch.float64, device=dev)
        chan = torch.empty(4, self.n, dtype=torch.float64, device=dev)
        L.check(self.lib.espm_fit_stats(ctypes.byref(st), pix.data_ptr(), chan.data_ptr(), scratch.data_ptr(),
                                        self.stream))
        self.n_launches += 2                                 # the streaming kernel and the fold of its CTA slots
        return pix, chan

    def abundance_information(self, simplex):
        """Poisson information F_j and covariance C_j of H_cur's columns given W_cur (espm_abundance_info): this rank's
        (k + k(k+1), p_loc) device float64 tensor of the k std rows, then C and F as packed upper triangles, row by row.
        ``simplex`` projects C onto sum_a h_aj = 1."""
        k = self.k
        out = torch.empty(k + k * (k + 1), self.p_loc, dtype=torch.float64, device=self.device)
        L.check(self.lib.espm_abundance_info(ctypes.byref(self.st), 1 if simplex else 0, out.data_ptr(), self.stream))
        self.n_launches += 2                                 # the streaming kernel and the per-pixel inversion
        return out

    def phase_information(self):
        """Poisson information of the phases per channel given H_cur (espm_phase_info): this rank's (k(k+1)/2, n) device
        float64 tensor of A_c[a, b] = sum_j x_cj h_aj h_bj / y_cj^2 as packed upper triangles, row by row."""
        st, dev = self.st, self.device
        scratch = self._scratch(self.lib.espm_phase_info_scratch)
        out = torch.empty(self.k * (self.k + 1) // 2, self.n, dtype=torch.float64, device=dev)
        L.check(self.lib.espm_phase_info(ctypes.byref(st), out.data_ptr(), scratch.data_ptr(), self.stream))
        self.n_launches += 3                                 # the H tiles, the streaming kernel and the fold of its slots
        return out

    def residual_left(self, Q):
        """R^T Q of the Pearson residual R = (x - y) / sqrt(y) of (W_cur, H_cur) (espm_resid_left): Q is (n, r), host or
        device; returns this rank's (r, p_loc) device float64 tensor."""
        Q = torch.as_tensor(Q, dtype=torch.float64, device=self.device).contiguous()
        r = Q.shape[1]
        assert Q.shape == (self.n, r) and r >= 1
        scratch = self._scratch(self.lib.espm_resid_left_scratch, r)
        out = torch.empty(r, self.p_loc, dtype=torch.float64, device=self.device)
        L.check(self.lib.espm_resid_left(ctypes.byref(self.st), Q.data_ptr(), r, out.data_ptr(), scratch.data_ptr(),
                                         self.stream))
        self.n_launches += 2 * _resid_blocks(r)              # per block of columns: the [g | Q] rows, the streaming kernel
        return out

    def residual_right(self, P):
        """R P^T of the Pearson residual of (W_cur, H_cur) (espm_resid_right): P is this rank's (r, p_loc), host or
        device; returns this rank's (n, r) device float64 tensor."""
        P = torch.as_tensor(P, dtype=torch.float64, device=self.device).contiguous()
        r = P.shape[0]
        assert P.shape == (r, self.p_loc) and r >= 1
        scratch = self._scratch(self.lib.espm_resid_right_scratch, r)
        out = torch.empty(self.n, r, dtype=torch.float64, device=self.device)
        L.check(self.lib.espm_resid_right(ctypes.byref(self.st), P.data_ptr(), r, out.data_ptr(), scratch.data_ptr(),
                                          self.stream))
        self.n_launches += 3 * _resid_blocks(r)              # per block: the [h; P] tiles, the streaming kernel, the fold
        return out

    # ------------------------------------------------------------------ helpers
    def _scratch(self, query, *args):
        """Device scratch of at least the bytes that ``query`` (an espm_*_scratch entry point) reports, and >= 8."""
        nbytes = ctypes.c_int64(0)
        L.check(query(ctypes.byref(self.st), *args, ctypes.byref(nbytes)))
        return torch.empty(max(nbytes.value // 8, 1), dtype=torch.float64, device=self.device)

    @property
    def stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _hptr(self, i):
        t = self.Hbuf[i]
        return t.data_ptr() + self.halo * t.element_size()

    def _bind(self):
        """Write the rotating buffer pointers into the C struct."""
        st = self.st
        hp, hc, hn = self.ih
        wc, wn = self.iw
        sc, sn = self.ihs
        st.H_prev, st.H_cur, st.H_next = self._hptr(hp), self._hptr(hc), self._hptr(hn)
        st.W_cur, st.W_next = self.Wbuf[wc].data_ptr(), self.Wbuf[wn].data_ptr()
        st.GW_cur, st.GW_next = self.GWbuf[wc].data_ptr(), self.GWbuf[wn].data_ptr()
        st.GWc_cur, st.GWc_next = self.GWcbuf[wc].data_ptr(), self.GWcbuf[wn].data_ptr()
        st.gwstats_cur, st.gwstats_next = self.gwstats[wc].data_ptr(), self.gwstats[wn].data_ptr()
        st.hstats_cur, st.hstats_next = self.hstats[sc].data_ptr(), self.hstats[sn].data_ptr()
        if self.have_prev:
            st.flags |= L.FLAG_HAVE_HPREV
        else:
            st.flags &= ~L.FLAG_HAVE_HPREV
        if self.peer:
            st.nb_prev_halo, st.nb_prev_ldh, st.nb_next_halo, st.nb_next_ldh = self.shard.halo_targets(self, hn)

    def _set_record(self, slot):
        if not 0 <= slot < self.max_records:
            raise IndexError("scalar record slot %d out of range" % slot)
        self.st.scalars = self.records.data_ptr() + slot * L.NSCALARS * 8
        self.st.rec_slot = slot

    def _stamp_next(self, slot):
        """The coming espm_h_finish completes record ``slot``: give it a fresh stamp."""
        self._stamp += 1
        self.st.rec_stamp = float(self._stamp)
        self._stamps[slot] = self._stamp

    def _call(self, fn, name=None):
        """Launch one C-ABI entry point on the current stream.  With ``self.profile`` set to a dict,
        calls whose name is in ``self.profile_names`` (or every named call when that is None) are
        bracketed by CUDA events."""
        self.n_launches += 1
        if self.profile is None or name is None or (self.profile_names is not None
                                                    and name not in self.profile_names):
            L.check(fn(ctypes.byref(self.st), self.stream))
            return
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(fn(ctypes.byref(self.st), self.stream))
        e1.record()
        self.profile.setdefault(name, []).append((e0, e1))

    # ------------------------------------------------------------------ uploads
    def _stage_x(self, X):
        """H2D copy of this rank's pixel slab (base.py:262 copies X on the host; here the only touch of the host
        buffer is this DMA).  Leaves ``self._xraw = (device tensor, channel stride, pixel stride)``."""
        if isinstance(X, np.ndarray) and not X.flags.writeable:
            # read-only inputs (memmaps, sklearn's checks) are only ever read; silence torch's notice
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", UserWarning)
                X = torch.from_numpy(X)
        xdt = _torch_dtype(self.src_code)
        j0, j1 = self.j0, self.j1
        if self.x_local:
            if X.shape[1] != j1 - j0:
                raise ValueError("x_local: X has %d pixels, this rank owns %d" % (X.shape[1], j1 - j0))
            j0, j1 = 0, X.shape[1]
        if isinstance(X, torch.Tensor):
            Xv = X
            if Xv.stride(1) == 1 or Xv.stride(0) != 1:
                slab = Xv[:, j0:j1]
                if not slab.is_contiguous():
                    slab = slab.contiguous()
                d = slab.to(self.device, non_blocking=True)
                sc, sp = d.stride(0), 1
            else:
                slab = Xv.t()[j0:j1, :]
                d = slab.to(self.device, non_blocking=True)
                sc, sp = 1, d.stride(0)
        else:
            Xv = np.asarray(X)
            if Xv.T.flags.c_contiguous and not Xv.flags.c_contiguous:
                slab = Xv.T[j0:j1, :]                      # hyperspy layout (p, n): channels contiguous
                d = torch.from_numpy(slab).to(self.device)
                sc, sp = 1, self.n
            else:
                slab = Xv[:, j0:j1]
                if slab.flags.c_contiguous:
                    d = torch.from_numpy(slab).to(self.device)
                elif slab.strides[1] == slab.itemsize and slab.strides[0] >= slab.shape[1] * slab.itemsize:
                    # this rank's columns of a C-ordered image: strided rows, copied without a host-side pass
                    d = torch.empty(slab.shape, dtype=xdt, device=self.device)
                    L.check(self.lib.espm_upload_2d(
                        ctypes.c_void_p(d.data_ptr()), slab.shape[1] * slab.itemsize, ctypes.c_void_p(slab.ctypes.data),
                        slab.strides[0], slab.shape[1] * slab.itemsize, slab.shape[0], self.stream))
                else:
                    d = torch.from_numpy(np.ascontiguousarray(slab)).to(self.device)
                sc, sp = slab.shape[1], 1
        self._xraw = (d, sc, sp)

    def _choose_storage(self, src_code, c_code, scale, ingest):
        """Storage type of Xt.  EDXS spectrum images are Poisson counts (datasets/base.py:68): non-negative integers,
        ~3/4 of them zero.  When the arithmetic is fp32 and the uploaded slab holds only integers below 256 / 65536
        that need no patching (no all-zero channel or pixel for remove_zeros_lines, no ``normalize``, no scale), Xt
        keeps them as uint8 / uint16 and the X passes stream 4x / 2x fewer bytes (SURVEY.md section 8f-4).  One
        device pass over the uploaded slab decides; pixel-sharded fits take the widest type any rank needs."""
        from . import config
        mode = getattr(config, "x_storage", "auto")
        if mode not in ("auto", "dense", "uint8", "uint16"):
            raise ValueError("espm_b200.config.x_storage must be 'auto', 'dense', 'uint8' or 'uint16'")
        self.x_storage_reason = "dense storage requested" if mode == "dense" else None
        if (mode == "dense" or c_code != L.F32 or src_code not in (L.F32, L.F64) or float(scale) != 1.0
                or (ingest is not None and ingest.get("normalize") is not None)):
            if self.x_storage_reason is None:
                self.x_storage_reason = "fp64 arithmetic, scaling or normalisation"
            want = 2
        else:
            d, sc, sp = self._xraw
            dev = self.device
            out4 = torch.zeros(4, dtype=torch.int32, device=dev)
            row_nz = torch.zeros(self.n, dtype=torch.int32, device=dev)
            col_nz = torch.zeros(self.p_loc, dtype=torch.int32, device=dev)
            L.check(self.lib.espm_x_prescan(ctypes.c_void_p(d.data_ptr()), src_code, self.n, self.p_loc, sc, sp, 0,
                                            ctypes.c_void_p(out4.data_ptr()), ctypes.c_void_p(row_nz.data_ptr()),
                                            ctypes.c_void_p(col_nz.data_ptr()), self.stream))
            if self.shard is not None:
                self.shard.allreduce_max_int(row_nz)       # a channel is an all-zero line only if it is on every rank
            info = torch.cat([out4[:2], row_nz.sum().reshape(1).to(torch.int32),
                              col_nz.sum().reshape(1).to(torch.int32)]).cpu().numpy()
            flags = int(info[0]) & 0xffffffff
            vmax = float(np.array([info[1]], dtype=np.int32).view(np.float32)[0])
            patched = (ingest is not None and not ingest.get("check_only")
                       and (int(info[2]) < self.n or int(info[3]) < self.p_loc))
            if flags & (L.X_NAN | L.X_INF | L.X_NEGATIVE | L.X_FRACTION) or patched:
                want = 2                                   # (errors are raised by the ingest pass, with its messages)
                self.x_storage_reason = "non-integer / negative entries or all-zero lines"
            elif vmax <= 255.0 and mode in ("auto", "uint8"):
                want = 0
            elif vmax <= 65535.0:
                want = 1
            else:
                want = 2
                self.x_storage_reason = "entries above 65535"
        if self.shard is not None:
            want = int(self.shard.allreduce_max_scalar(torch.tensor(float(want), dtype=torch.float64)))
        self.x_storage = ("uint8", "uint16", "dense")[want]
        return (L.U8, L.U16, src_code)[want]

    def _retile_x(self, scale, ingest=None):
        """Re-tiling of the staged slab into the tile-major layout (base.py:262) + the device prologue."""
        st = self.st
        d, sc, sp = self._xraw
        self.Xt = torch.empty(st.n_tiles * st.n_pad * L.TILE_PX * _X_ITEMSIZE[self.x_code], dtype=torch.uint8,
                              device=self.device)
        if self.x_code in (L.F32, L.F64):
            self.Xt = self.Xt.view(_torch_dtype(self.x_code))
        st.Xt = self.Xt.data_ptr()
        src = ctypes.c_void_p(d.data_ptr())
        if ingest is None:
            L.check(self.lib.espm_retile_x(ctypes.byref(st), src, self.src_code, sc, sp, 0, float(scale), None,
                                           self.stream))
            torch.cuda.current_stream(self.device).synchronize()
        else:
            self._ingest(src, sc, sp, float(ingest.get("eps", st.log_shift)), ingest.get("normalize"),
                         bool(ingest.get("check_only")))
        self._xraw = None

    def _ingest(self, src, sc, sp, eps, normalize_nc, ingest_only_checks=False):
        """Device-side prologue of the fit (see ``ingest`` in __init__)."""
        st, dev = self.st, self.device
        i32 = torch.int32
        row_nz = torch.zeros(st.n_pad, dtype=i32, device=dev)
        col_nz = torch.zeros(st.p_pad, dtype=i32, device=dev)
        xflags = torch.zeros(1, dtype=i32, device=dev)
        sum_part = torch.zeros(st.n_tiles * (st.n_pad // 32), dtype=torch.float64, device=dev)
        io = L.EspmIngest(row_nz.data_ptr(), col_nz.data_ptr(), xflags.data_ptr(), sum_part.data_ptr())
        L.check(self.lib.espm_retile_x(ctypes.byref(st), src, self.src_code, sc, sp, 0, 1.0, ctypes.byref(io),
                                       self.stream))
        scal = torch.zeros(2, dtype=torch.float64, device=dev)
        L.check(self.lib.espm_reduce_sum(sum_part.data_ptr(), sum_part.numel(), scal.data_ptr(), self.stream))
        n, p_loc, p = self.n, self.p_loc, self.p
        info = torch.stack([xflags[0].to(torch.float64), scal[0],
                            (p_loc - col_nz[:p_loc].sum()).to(torch.float64)])
        if self.shard is not None:
            info, row_nz = self.shard.combine_ingest(info, row_nz)
        info = info.cpu().numpy()                                  # one small D2H (synchronises)
        flags = int(info[0])
        if flags & L.X_NAN:
            raise ValueError("Input X contains NaN.")
        if flags & L.X_INF:
            raise ValueError("Input X contains infinity or a value too large for dtype('%s')."
                             % np.dtype(_np_dtype(self.src_code)).name)
        if flags & L.X_NEGATIVE:
            raise ValueError("Negative values in data")            # base.py:528
        if ingest_only_checks:
            return
        total = float(info[1])
        zc = int(round(info[2]))
        zr = int(n - int(row_nz[:n].sum().item()))
        self.n_zero_rows, self.n_zero_cols = zr, zc
        scale = 1.0
        if normalize_nc is not None:                               # base.py:16-18 on the repaired X
            patched = total + eps * (zr * p + zc * n - zr * zc)
            self.norm_factor = normalize_nc / ((patched / (n * p)) * n)
            scale = self.norm_factor
        if zr or zc or scale != 1.0:
            row_zero = (1 - row_nz) if zr else None
            col_zero = (1 - col_nz) if zc else None
            L.check(self.lib.espm_xt_fixup(
                ctypes.byref(st), ctypes.c_void_p(row_zero.data_ptr() if zr else None),
                ctypes.c_void_p(col_zero.data_ptr() if zc else None), eps, scale, self.stream))
        part = torch.zeros(st.n_tiles, dtype=torch.float64, device=dev)
        L.check(self.lib.espm_xt_const(ctypes.byref(st), ctypes.c_void_p(part.data_ptr()), self.stream))
        L.check(self.lib.espm_reduce_sum(part.data_ptr(), part.numel(), scal[1:].data_ptr(), self.stream))
        c = scal[1:2].clone()
        if self.shard is not None:
            self.shard.allreduce_sum(c)
        self.const_KL = float(c.item())

    def compute_x_sums(self):
        """Per-pixel and per-channel sums of the (repaired, normalised) X: sigmaR of the Bregman steps
        (updates.py:43-45, 121) and the ingredients of the Lipschitz bounds (updates.py:393-413)."""
        st = self.st
        self.x_colsum = torch.zeros(st.p_pad, dtype=self.cdt, device=self.device)
        part = torch.zeros(st.n_tiles, st.n_pad, dtype=torch.float64, device=self.device)
        L.check(self.lib.espm_x_sums(ctypes.byref(st), ctypes.c_void_p(self.x_colsum.data_ptr()),
                                     ctypes.c_void_p(part.data_ptr()), self.stream))
        rows = part.sum(0)
        if self.shard is not None:
            self.shard.allreduce_sum(rows)
        self.x_rowsum = rows.to(self.cdt)
        self.x_total = float(rows[:self.n].sum().item())
        st.x_colsum, st.x_rowsum, st.x_total = self.x_colsum.data_ptr(), self.x_rowsum.data_ptr(), self.x_total
        return self.x_colsum, self.x_rowsum

    def set_gamma_pg(self, gamma_h, gamma_w):
        self.st.gamma_h, self.st.gamma_w = float(gamma_h), float(gamma_w)

    def set_G(self, G, prepare=True):
        """(Re)load G (base.py:269-274, 388-389).  ``prepare`` also recomputes GW for W_cur."""
        st = self.st
        if G is None:
            if not self.identity_G:
                raise ValueError("G cannot switch to identity mid-fit")
            st.G = st.Gt = st.colsum_G = 0
        else:
            Gn = np.ascontiguousarray(np.asarray(G), dtype=self.cnp)
            if Gn.shape != (self.n, self.m):
                raise ValueError("G has shape %s, expected %s" % (Gn.shape, (self.n, self.m)))
            self.G = torch.from_numpy(Gn).to(self.device)
            self.Gt = self.G.t().contiguous()
            if self.colsum_G is None:
                self.colsum_G = torch.zeros(self.m, dtype=self.cdt, device=self.device)
            st.G, st.Gt, st.colsum_G = self.G.data_ptr(), self.Gt.data_ptr(), self.colsum_G.data_ptr()
            if st.flags & L.FLAG_L2:
                self.GG = (self.Gt @ self.G).contiguous()      # G^T G (updates.py:30), m x m, once per G
                st.GG = self.GG.data_ptr()
            L.check(self.lib.espm_colsum_g(ctypes.byref(st), ctypes.c_void_p(self.colsum_G.data_ptr()), self.stream))
        if prepare:
            # GW for the CURRENT W under the new G: write into the `next` slot, then swap GW only
            wc, wn = self.iw
            self.Wbuf[wn].copy_(self.Wbuf[wc])
            self._set_record(self.max_records - 1)
            self._call(self.lib.espm_gw_prepare)
            self.iw = [wn, wc]
            self._bind()

    def _init_WH(self, W0, H0):
        """updates.py:220-221: clamp the initial factors to log_shift; then GW and the H statistics."""
        ls = self.st.log_shift
        wc, wn = self.iw
        W = torch.as_tensor(np.ascontiguousarray(W0), dtype=self.cdt).to(self.device)
        if isinstance(H0, torch.Tensor):         # e.g. the initial H computed on the device (init_device.py)
            Hs = H0[:, self.j0:self.j1].to(self.device, self.cdt)
        else:
            Hs = torch.as_tensor(np.ascontiguousarray(H0[:, self.j0:self.j1]), dtype=self.cdt).to(self.device)
        if self.clamp_init:
            W, Hs = W.clamp_min(ls), Hs.clamp_min(ls)
        self.Wbuf[wn].copy_(W)
        hp, hc, hn = self.ih
        self.Hbuf[hn][:, self.halo:self.halo + self.p_loc] = Hs
        self._bind()
        self._set_record(self.max_records - 1)
        self._call(self.lib.espm_gw_prepare)
        self._call(self.lib.espm_h_stats)
        self._sync_hstats()
        self._exchange_halo(self.ih[2])
        # rotate: next -> cur
        self.iw = [wn, wc]
        self.ih = [hp, hn, hc]
        self.ihs = [self.ihs[1], self.ihs[0]]
        self.have_prev = False
        self._bind()

    # ------------------------------------------------------------------ multi-GPU hooks (dist.py)
    def close(self):
        """Release peer memory (collective when sharded through peer memory); the engine is unusable after."""
        if self.peer and self.shard is not None:
            self.Hbuf = None
            if self.inbox is not None:
                self.inbox.stamp = self._stamp
            self.shard.close(self._seq_s, self._seq_m)
            self.peer = False

    def _sync_hstats(self):
        if self.shard is not None:
            self.shard.allreduce_hstats(self.hstats[self.ihs[1]], self.st.kp)

    def _exchange_halo(self, ibuf):
        if self.shard is not None and self.ny > 0:
            self.shard.exchange_halo(self.Hbuf[ibuf], self.halo, self.p_loc, self.ny)

    # ------------------------------------------------------------------ the two phases
    def evaluate(self, slot):
        """Phase A on (W_cur, H_cur): fills scalar record ``slot`` (loss parts, rel_H, flags)."""
        self._set_record(slot)
        self._stamp_next(slot)
        self._eval_slot = slot
        self._seq_m += 1
        self.st.seq_m = self._seq_m                          # mask exchange of this evaluation (peer mode)
        if self.st.flags & L.FLAG_L2_H:
            L.check(self.lib.espm_gram(ctypes.byref(self.st), 0, self.stream))   # (G W)^T (G W), updates.py:115
        self._call(self.lib.espm_h_pass, "h_pass")
        self._call(self.lib.espm_h_finish, "h_finish")      # its last CTA also writes the scalar record
        if self._w_after_eval is not None:
            W, self._w_after_eval = self._w_after_eval, None
            self._load_W(W)

    def set_W_after_eval(self, W):
        """H-only mode: the reference clamps W0 to log_shift (updates.py:220-221) but its fixed_W overwrites W with the
        UNCLAMPED matrix in the first update (updates.py:75-76).  The evaluation of iterate 0 uses the clamped W given at
        construction; ``W`` (unclamped) replaces it right after that evaluation is enqueued."""
        self._w_after_eval = W

    def _load_W(self, W):
        """W_cur <- W as given (no clamp), GW / gwstats recomputed; stream-ordered after what is already enqueued."""
        wc, wn = self.iw
        self.Wbuf[wn].copy_(torch.as_tensor(np.ascontiguousarray(W), dtype=self.cdt).to(self.device))
        self._set_record(self.max_records - 1)
        self._call(self.lib.espm_gw_prepare)
        self.iw = [wn, wc]
        self._bind()

    def advance(self, slot):
        """Phase B: (W_cur, H_cur) -> (W_next, H_next), rotate.  rel_W etc. go to record ``slot``."""
        st = self.st
        self._set_record(slot)
        if self.h_only:
            return self._advance_h(st)
        if st.flags & L.FLAG_SIMPLEX_H:
            if self.shard is not None and not self.peer:
                self.shard.gather_masks(self.mask)
            self._call(self.lib.espm_h_apply, "h_apply")
        if not self.peer:
            self._exchange_halo(self.ih[2])
        if self.pg_ls:
            self._pg_ls_h()
            self._set_record(slot)
        if st.flags & L.FLAG_LINESEARCH:
            self._call(self.lib.espm_linesearch, "linesearch")   # smooth_nmf.py:376-382, gamma_ stays on the device
            if self.shard is not None:
                self._ls_decide(slot)
        if st.flags & L.FLAG_L2:
            L.check(self.lib.espm_gram(ctypes.byref(st), 1, self.stream))        # H' H'^T, updates.py:31
            if self.shard is not None:
                self.shard.allreduce_sum(self.gram[1])                           # k x k sums over the pixel shards
        self._seq_s += 1
        st.seq_s = self._seq_s                               # S exchange of this update (peer mode)
        self._call(self.lib.espm_w_pass, "w_pass")
        if self.shard is not None and not self.peer:
            self._call(self.lib.espm_w_reduce, "w_reduce")
            self.shard.allreduce_sum(self.s_sum)
            self._sync_hstats()
        self._call(self.lib.espm_w_finish, "w_finish")
        if self.pg_ls:
            self._pg_ls_w_stage()
        hp, hc, hn = self.ih
        self.ih = [hc, hn, hp]
        self.iw = [self.iw[1], self.iw[0]]
        self.ihs = [self.ihs[1], self.ihs[0]]
        self.have_prev = True
        self._bind()

    def _advance_h(self, st):
        """Phase B with W fixed: H_cur -> H_next and its row statistics, then only the H buffers rotate (rel_W of the
        record stays 0).  Sharded: the masks / halos as in ``advance`` and the H' statistics combined over the ranks."""
        if st.flags & L.FLAG_SIMPLEX_H:
            if self.shard is not None and not self.peer:
                self.shard.gather_masks(self.mask)
            self._call(self.lib.espm_h_apply, "h_apply")
        if not self.peer:
            self._exchange_halo(self.ih[2])
        self._call(self.lib.espm_h_stats, "h_stats")
        self.n_launches += 1                                 # espm_h_stats is two kernels
        self._sync_hstats()
        hp, hc, hn = self.ih
        self.ih = [hc, hn, hp]
        self.ihs = [self.ihs[1], self.ihs[0]]
        self.have_prev = True
        self._bind()

    # ------------------------------------------------------------------ the loop in native code
    @property
    def fast_loop(self):
        """Can ``run_iterations`` be used?  Not when an iteration needs host work between its launches (for the H-only
        mode on a pixel shard: the H' statistics of the ranks are combined on the host)."""
        st = self.st
        return (not (st.flags & (L.FLAG_L2 | L.FLAG_L2_H | L.FLAG_LINESEARCH)) and not self.pg_ls
                and (self.shard is None or (self.peer and not self.h_only)) and self.profile is None)

    def run_iterations(self, first, n, events=None):
        """``for it in range(first, first + n): advance(it); evaluate(it)`` issued by ONE call into the library
        (espm_run_iterations): the Python binding costs ~10 us per launch, more than the kernels of a small pixel shard
        take.  ``events``: optional list of n entries, each None or a 4-tuple of recorded-once torch.cuda.Event (w_pass
        start / end, h_pass start / end) the native loop records around the two X passes of that iteration.  (An event
        between two kernels costs their programmatic-dependent-launch overlap, ~4 us per event: sample, don't record
        every iteration.)"""
        if n <= 0:
            return
        if first < 0 or first + n > self.max_records:
            raise IndexError("scalar record slots %d..%d out of range" % (first, first + n - 1))
        lp = L.EspmLoop()
        sz = self.Hbuf[0].element_size()
        for i in range(3):
            lp.H[i] = self._hptr(i)
            if self.peer:
                pp, _, npn, _ = self.shard.halo_targets(self, i)
                lp.nb_prev_halo[i], lp.nb_next_halo[i] = pp, npn
        for i in range(2):
            lp.W[i], lp.GW[i], lp.GWc[i] = self.Wbuf[i].data_ptr(), self.GWbuf[i].data_ptr(), self.GWcbuf[i].data_ptr()
            lp.gwstats[i], lp.hstats[i] = self.gwstats[i].data_ptr(), self.hstats[i].data_ptr()
        lp.records = self.records.data_ptr()
        ev_arr = None
        if events is not None:
            ev_arr = (ctypes.c_void_p * (4 * n))(*[(None if tup is None or tup[i] is None else tup[i].cuda_event)
                                                   for tup in events for i in range(4)])
            lp.ev = ctypes.cast(ev_arr, ctypes.c_void_p)
        for i in range(3):
            lp.ih[i] = self.ih[i]
        for i in range(2):
            lp.iw[i], lp.ihs[i] = self.iw[i], self.ihs[i]
        lp.have_prev = 1 if self.have_prev else 0
        lp.seq_s, lp.seq_m, lp.stamp = self._seq_s, self._seq_m, float(self._stamp)
        L.check(self.lib.espm_run_iterations(ctypes.byref(self.st), ctypes.byref(lp), first, n, self.stream))
        self.ih, self.iw, self.ihs = list(lp.ih), list(lp.iw), list(lp.ihs)
        self.have_prev = bool(lp.have_prev)
        self._seq_s, self._seq_m = int(lp.seq_s), int(lp.seq_m)
        for i in range(n):
            self._stamps[first + i] = self._stamp + 1 + i
        self._stamp = int(lp.stamp)
        self._eval_slot = first + n - 1
        self.n_launches += int(lp.launches)
        del sz

    # ------------------------------------------------------------------ single steps (operator API)
    def step_h_only(self):
        """One H update from (W_cur, H_cur): returns (H_next local, scalar record)."""
        self.evaluate(0)
        if self.st.flags & L.FLAG_SIMPLEX_H:
            if self.shard is not None:
                self.shard.gather_masks(self.mask)
            self._call(self.lib.espm_h_apply)
        rec = self.read_records(0, 1)[0]
        Hn = self.Hbuf[self.ih[2]][:, self.halo:self.halo + self.p_loc].cpu().numpy()
        return Hn, rec

    def step_w_only(self):
        """One W update from (W_cur, H_cur) (the H given by the caller plays the role of H')."""
        st = self.st
        st.H_next = st.H_cur
        self._call(self.lib.espm_h_stats)      # rebuilds Ht from H_next (= H_cur); hstats go to the `next` slot
        st.hstats_next = st.hstats_cur
        self._set_record(0)
        if st.flags & L.FLAG_L2:
            L.check(self.lib.espm_gram(ctypes.byref(st), 1, self.stream))
        self._call(self.lib.espm_w_pass)
        if self.shard is not None:
            self._call(self.lib.espm_w_reduce)
            self.shard.allreduce_sum(self.s_sum)
        self._call(self.lib.espm_w_finish)
        rec = self.read_records(0, 1)[0]
        rec[L.S_DEV_FLAGS] = float(int(self.dev_flags[0].item()) & 0xffffffff)
        Wn = self.Wbuf[self.iw[1]].cpu().numpy()
        self._bind()
        return Wn, rec

    def rollback(self):
        """Undo the last ``advance`` (used when a stop test fires one step late): the previous
        iterate's buffers are intact because every kernel writes only the `next` set."""
        hp, hc, hn = self.ih
        self.ih = [hn, hp, hc]
        if not self.h_only:                  # H-only: W / GW never rotate
            self.iw = [self.iw[1], self.iw[0]]
        self.ihs = [self.ihs[1], self.ihs[0]]
        self.have_prev = False
        self._bind()

    # ------------------------------------------------------------------ read-back
    def read_records(self, lo, hi):
        """Scalar records [lo, hi) -> float64 array (hi-lo, NSCALARS), after everything enqueued so far has run."""
        torch.cuda.current_stream(self.device).synchronize()
        if self.inbox is not None:
            return np.stack([self._fold_record(slot, 10.0) for slot in range(lo, hi)])
        rec = self.rec_np[lo:hi].copy()
        if self.shard is not None:
            rec = self.shard.combine_records(rec)
        return rec

    def _fold_record(self, slot, timeout):
        """Sharded fit: record ``slot`` with the per-shard fields folded over the ranks' shares in this host's inbox
        (sums in rank order, max, OR: identical on every rank).  Waits for the stamps of the evaluation that completes
        the slot -- the local one and every rank's share -- without touching the stream."""
        import time
        row = self.rec_np[slot]
        want = self._stamps.get(slot)
        if want is None:                       # never evaluated (e.g. a W-only step): nothing to fold
            return row.copy()
        want = float(want)
        views = self.inbox.views                   # views[r][r, slot]: rank r's share, in rank r's inbox

        def ready():
            return row[L.S_STAMP] == want and all(views[r][r, slot, 7] == want for r in range(len(views)))
        t0 = time.perf_counter()
        while not ready():
            if time.perf_counter() - t0 > timeout:
                torch.cuda.current_stream(self.device).synchronize()
                if not ready():
                    raise L.EspmError("scalar record %d was never completed by every rank (stamps %r / %r, expected %r)"
                                      % (slot, row[L.S_STAMP], [float(views[r][r, slot, 7]) for r in range(len(views))],
                                         want))
        shares = np.stack([views[r][r, slot, :] for r in range(len(views))])
        out = row.copy()
        sh = shares.copy()
        for col, s in ((0, L.S_XLOGY), (1, L.S_LOGREG), (2, L.S_LAPL)):
            acc = 0.0
            for r in range(sh.shape[0]):
                acc += float(sh[r, col])
            out[s] = acc
        out[L.S_REL_H] = float(sh[:, 3].max())
        flags = 0
        for v in sh[:, 4]:
            flags |= int(v)
        out[L.S_DEV_FLAGS] = float(flags)
        return out

    def wait_record(self, slot, timeout=2.0):
        """Record ``slot`` as soon as the espm_h_finish that completes it has stamped it -- WITHOUT synchronising the
        stream, so kernels enqueued after that evaluation keep running while the host looks at the scalars."""
        if self.inbox is not None:
            return self._fold_record(slot, timeout)
        if self.shard is not None:
            return self.read_records(slot, slot + 1)[0]
        want = float(self._stamps[slot])
        row = self.rec_np[slot]
        import time
        t0 = time.perf_counter()
        while row[L.S_STAMP] != want:
            if time.perf_counter() - t0 > timeout:
                torch.cuda.current_stream(self.device).synchronize()     # surfaces a kernel fault, if that is the reason
                if row[L.S_STAMP] != want:
                    raise L.EspmError("scalar record %d was never completed (stamp %r, expected %r)"
                                      % (slot, row[L.S_STAMP], want))
        return row.copy()

    def loss_parts(self, rec, const_KL, numel):
        """(kl, log_reg, lapl) of base.py:203-205 + smooth_nmf.py:461-469 from one scalar record."""
        kl = (rec[L.S_SUMY] - rec[L.S_XLOGY] + const_KL) / numel
        reg = rec[L.S_LOGREG] / numel
        lap = 0.5 * self.st.lambda_L * rec[L.S_LAPL] / numel
        return kl, reg, lap

    def get_W(self):
        return self.Wbuf[self.iw[0]].cpu().numpy()

    def get_H_local(self):
        return self.Hbuf[self.ih[1]][:, self.halo:self.halo + self.p_loc].cpu().numpy()

    def get_H(self):
        if self.shard is not None:
            from .dist import shard_bounds
            sizes = []
            for r in range(self.world):
                a, b, _ = shard_bounds(self.p, self.nx, self.ny, r, self.world)
                sizes.append(b - a)
            Hd = self.Hbuf[self.ih[1]][:, self.halo:self.halo + self.p_loc]
            if Hd.is_cuda:
                return self.shard.gather_H_device(Hd, sizes)
            return self.shard.gather_H(self.get_H_local(), self.p)
        return self.get_H_local()

    def get_GW(self):
        return self.GWbuf[self.iw[0]][:self.n, :self.k].cpu().numpy()

    def set_WH(self, W, H):
        """Overwrite the current iterate (e.g. after rescaled_DH) and refresh the derived buffers."""
        self._init_WH(W, H)

    # ------------------------------------------------------------------ ground-truth tracking (base.py:301-347)
    def enable_truth(self, true_D, true_H):
        """Keep X_true = true_D @ true_H on the device in the same tile-major layout as X, so that
        ``loss(W, H, X=true_DH)`` (base.py:345) is one more H pass."""
        st = self.st
        D = torch.as_tensor(np.ascontiguousarray(true_D), dtype=self.cdt).to(self.device)
        Ht = torch.as_tensor(np.ascontiguousarray(true_H[:, self.j0:self.j1]), dtype=self.cdt).to(self.device)
        # X_true is not integer-valued: dense storage in the arithmetic type, whatever the storage of X
        self.truth_code = self.c_code
        xdt = _torch_dtype(self.truth_code)
        dense = (D @ Ht).to(xdt)                 # once per fit (setup, not the per-iteration path)
        self.Xt_true = torch.empty(st.n_tiles * st.n_pad * L.TILE_PX, dtype=xdt, device=self.device)
        keep = (st.Xt, st.x_dtype)
        st.Xt, st.x_dtype = self.Xt_true.data_ptr(), self.truth_code
        L.check(self.lib.espm_retile_x(ctypes.byref(st), ctypes.c_void_p(dense.data_ptr()), self.truth_code,
                                       dense.stride(0), 1, 0, 1.0, None, self.stream))
        torch.cuda.current_stream(self.device).synchronize()
        st.Xt, st.x_dtype = keep
        del dense
        self.H_tmp = torch.ones(self.k, self.ldh, dtype=self.cdt, device=self.device)
        self.hstats_tmp = torch.zeros(3 * st.kp, dtype=torch.float64, device=self.device)

    def _eval_only(self, slot, xt_ptr=None, h_ptr=None, hstats_ptr=None):
        """Loss terms of (W_cur, H) against X into scalar record ``slot`` without touching the iteration state
        (the ``self.loss(W, H, X=...)`` calls of the reference): h_pass + h_finish with ESPM_FLAG_EVAL_ONLY."""
        st = self.st
        keep = (st.Xt, st.H_cur, st.hstats_cur, st.flags, st.x_dtype)
        if xt_ptr is not None:
            st.Xt = xt_ptr
            st.x_dtype = self.truth_code         # the truth image is stored dense (enable_truth)
        if h_ptr is not None:
            st.H_cur, st.hstats_cur = h_ptr, hstats_ptr
        st.flags = (st.flags & ~L.FLAG_HAVE_HPREV) | L.FLAG_EVAL_ONLY
        self._set_record(slot)
        self._stamp_next(slot)
        if st.flags & L.FLAG_L2_H:
            L.check(self.lib.espm_gram(ctypes.byref(st), 0, self.stream))
        self._call(self.lib.espm_h_pass)
        self._call(self.lib.espm_h_finish)
        st.Xt, st.H_cur, st.hstats_cur, st.flags, st.x_dtype = keep
        self._bind()

    def truth_loss(self, slot, H_t=None):
        """Scalar record ``slot`` <- loss terms of (W_cur, H_t or H_cur) against X_true (base.py:345)."""
        st = self.st
        h_ptr = hs_ptr = None
        if H_t is not None:
            self.H_tmp[:, self.halo:self.halo + self.p_loc] = torch.as_tensor(
                np.ascontiguousarray(H_t[:, self.j0:self.j1]), dtype=self.cdt).to(self.device)
            h_ptr = self.H_tmp.data_ptr() + self.halo * self.H_tmp.element_size()
            hs_ptr = self.hstats_tmp.data_ptr()
            keep = (st.H_next, st.hstats_next)
            st.H_next, st.hstats_next = h_ptr, hs_ptr
            self._call(self.lib.espm_h_stats)                  # row statistics of H_t (sum Y of the loss)
            st.H_next, st.hstats_next = keep
            if self.shard is not None:         # global statistics and the neighbours' rows of H_t (Laplacian term)
                self.shard.allreduce_hstats(self.hstats_tmp, st.kp)
                if self.ny > 0:
                    self.shard.exchange_halo(self.H_tmp, self.halo, self.p_loc, self.ny)
        self._eval_only(slot, xt_ptr=self.Xt_true.data_ptr(), h_ptr=h_ptr, hstats_ptr=hs_ptr)

    # ------------------------------------------------------------------ projected-gradient line search
    def _unaveraged(self, rec):
        """loss(W, H, average=False) (smooth_nmf.py:457-475) from a scalar record."""
        kl = 0.5 * rec[L.S_XLOGY] if self.st.flags & L.FLAG_L2 else rec[L.S_SUMY] - rec[L.S_XLOGY] + self.const_KL
        return kl + rec[L.S_LOGREG] + 0.5 * self.st.lambda_L * rec[L.S_LAPL]

    def _ls_totals(self):
        """Pixel-sharded line search: this rank's sums left by espm_linesearch (ESPM_FLAG_LS_PARTIAL), combined over the
        ranks -- sums for the first 4 + kp values, maxima for the kp row maxima of H'."""
        st = self.st
        nv = 4 + st.kp
        tot = self.ls_part.view(-1)[st.px_blocks * nv: st.px_blocks * nv + nv + st.kp].clone()
        self.shard.allreduce_sum(tot[:nv])
        self.shard.allreduce_max_int(tot[nv:])
        return tot.cpu().numpy(), nv

    def _ls_decide(self, slot):
        """smooth_nmf.py:376-382 for a sharded fit: d = diff_surrogate(H_old, H_new) from the global sums, then
        gamma_ /= 1.05 if d > 0 else gamma_ *= 1.5 (what the kernel does itself on one GPU)."""
        st = self.st
        t, nv = self._ls_totals()
        sigma = float(self.sigma_dev.item())
        if st.flags & L.FLAG_HQ:
            t3 = t[3]
        else:
            t3 = sum(t[nv + kk] * t[4 + kk] for kk in range(st.k))
        d = 0.5 * (2.0 * t[1] - t[0] + sigma * t3) - 0.5 * t[2]
        g = sigma / 1.05 if d > 0.0 else sigma * 1.5
        self.sigma_dev.fill_(g)
        self.rec_np[slot, L.S_GAMMA], self.rec_np[slot, L.S_LS_D] = g, d

    def _pg_ls_h(self):
        """smooth_nmf.py:383-401 for (H_cur -> H_next): d = f(Ht) + <H - Ht, grad f(Ht)> + gamma |H - Ht|^2 - f(H)."""
        st = self.st
        a1, a2 = self.max_records - 5, self.max_records - 6
        rec0 = self.read_records(self._eval_slot, self._eval_slot + 1)[0]
        self._set_record(a1)
        self._call(self.lib.espm_linesearch)                   # sums of the quadratic surrogate (den = gradH(Ht))
        self._call(self.lib.espm_h_stats)                      # row statistics of H_next for sum Y
        self._sync_hstats()                                    # (global ones when the pixels are sharded)
        self._eval_only(a2, h_ptr=st.H_next, hstats_ptr=st.hstats_next)
        r1 = self.read_records(a1, a1 + 1)[0]
        r2 = self.read_records(a2, a2 + 1)[0]
        if self.shard is not None:             # the two sums of the quadratic surrogate over all ranks
            t, _ = self._ls_totals()
            r1[L.S_LS_D], r1[L.S_GAMMA] = t[0], t[1]
        f_xt, f_x = self._unaveraged(rec0), self._unaveraged(r2)
        d = f_xt + r1[L.S_LS_D] + st.gamma_h * r1[L.S_GAMMA] - f_x
        st.gamma_h = st.gamma_h / 1.05 if d > 0 else st.gamma_h * 1.5
        self._pg_f_x = f_x

    def _pg_ls_w_stage(self):
        """After the W step: keep what smooth_nmf.py:438-447 needs until loss(W', H') is known."""
        Wold = self.Wbuf[self.iw[0]].double()
        Wn = self.Wbuf[self.iw[1]].double()
        grad = self.w_den.double()
        dW = Wn - Wold
        self._pg_w_pending = (self._pg_f_x, float((dW * grad).sum().item()), float((dW * dW).sum().item()))

    def pg_ls_w_update(self, rec):
        """gamma_[1] update once the record of the new iterate (f(W', H')) has been read."""
        if self._pg_w_pending is None:
            return
        f_xt, s1, s2 = self._pg_w_pending
        self._pg_w_pending = None
        st = self.st
        d = f_xt + s1 + st.gamma_w * s2 - self._unaveraged(rec)
        st.gamma_w = st.gamma_w / 1.05 if d > 0 else st.gamma_w * 1.5

    def enable_clamp(self):
        """Switch to the reference's NaN fallback (updates.py:129-131, 54-56: GWH = max(GWH, log_shift)) and to
        the separately clamped GW of the loss (measures.py:493); clears the sticky device error word."""
        self.st.flags |= L.FLAG_CLAMP_Y | L.FLAG_LOSS_DUAL
        self.clamped = True
        self.dev_flags[0] = 0

    def gw_flags_init(self):
        """ESPM_DEV_GW_* bits of the initial G W (one small D2H)."""
        torch.cuda.current_stream(self.device).synchronize()
        return int(self.rec_np[self.max_records - 1][L.S_GW_FLAGS])

    def set_flag(self, flag, on=True):
        if on:
            self.st.flags |= flag
        else:
            self.st.flags &= ~flag
