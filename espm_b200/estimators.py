"""``SmoothNMF`` -- drop-in for ``espm.estimators.SmoothNMF`` whose fit loop runs on a B200.

Same constructor arguments, ``fit`` / ``fit_transform`` / ``inverse_transform`` / ``loss`` /
``get_losses``, fitted attributes and printed messages as the reference
(espm/estimators/smooth_nmf.py:84-113, base.py:126-152, 209-517).  The host code below only validates,
initialises and runs the stop tests; every pass over X happens in the CUDA kernels behind
``espm_b200.engine.FitEngine``.  There is no CPU fallback: without a CUDA device ``fit`` raises.

On the device: every ``algo`` of the reference (``"log_surrogate"``, ``"l2_surrogate"``, ``"bmd"``,
``"projected_gradient"``), the KL and (``l2=True``) Frobenius losses, ``simplex_H`` / ``simplex_W``, ``mu`` (scalar or
per phase), ``lambda_L`` with ``shape_2d`` (5-point Laplacian) or without (identity), ``fixed_H`` / ``fixed_W``,
``normalize``, ``linesearch``, ground-truth tracking (``true_D`` / ``true_H``), ``G`` as ``None`` / ndarray / physical
model, ``hspy_comp``; the NNDSVD initialisation of a call without ``W`` and ``H`` runs its randomized SVD on the device
too (``init_device.py``).  With ``hspy_comp=True``, ``transform`` estimates the maps of another spectrum image with the
fitted phases held fixed (only the H half of an iteration runs).  ``goodness_of_fit`` maps where a fitted model
explains the data and where it does not (per-pixel and per-channel KL and chi-square sums, one pass over X), and
``abundance_uncertainty`` how precise the maps are (per-pixel standard errors and covariances from the Poisson
information, one pass over X), and ``phase_uncertainty`` how precise the phases are (standard errors and covariances of
``W_`` and error bands of the phase spectra, from the per-channel Poisson information, one pass over X), and
``residual_components`` what the model misses (the leading singular triplets of its Pearson residual, by a randomized
SVD whose products stream X on the device).  Pixel-sharded fits (one process per GPU) support every
algorithm, loss and option, including ``linesearch`` and ground-truth tracking.
"""
import sys
import time
from collections import namedtuple

import numpy as np
from sklearn.base import BaseEstimator, TransformerMixin
from sklearn.utils._available_if import available_if
from sklearn.utils.validation import check_array, check_is_fitted, validate_data

from . import _lib as L
from . import config
from .conf import dicotomy_tol as _DICOTOMY_TOL
from .conf import log_shift as _LOG_SHIFT
from .conf import sigmaL as _SIGMA_L
from .host import (find_min_angle, find_min_MSE, initialize_factors, is_physical_model, normalization_factor,
                   remove_zeros_lines, rescaled_DH)


FitStatistics = namedtuple("FitStatistics", ["pixel_counts", "pixel_model", "pixel_kl", "pixel_chi2",
                                             "channel_counts", "channel_model", "channel_kl", "channel_chi2"])
FitStatistics.__doc__ = """Goodness of fit of a SmoothNMF model (``SmoothNMF.goodness_of_fit``), float64 arrays.

With x the data, y = sum_k max(GW, log_shift) max(H, log_shift) the model (the Y of the KL loss),
kl = y - x + x ln(x / y) (0 ln 0 := 0) and chi2 = (x - y)^2 / y:
``pixel_*`` (p,) are the sums over channels of x, y, kl, chi2 for every pixel (pixel order of the X passed in),
``channel_*`` (n,) the sums over pixels for every channel."""

AbundanceUncertainty = namedtuple("AbundanceUncertainty", ["std", "covariance", "information"])
AbundanceUncertainty.__doc__ = """Precision of the abundance maps of a SmoothNMF model (``SmoothNMF.abundance_uncertainty``), float64
arrays: ``std`` (k, p) the standard error of every entry of H, ``covariance`` (p, k, k) the covariance of every pixel's
column of H and ``information`` (p, k, k) its Poisson information matrix (both symmetric).  NaN ``std`` and
``covariance`` mark a pixel whose information is singular."""

PhaseUncertainty = namedtuple("PhaseUncertainty", ["std", "covariance", "information", "spectrum_std"])
PhaseUncertainty.__doc__ = """Precision of the phases of a SmoothNMF model (``SmoothNMF.phase_uncertainty``), float64 arrays.
With a real G (n x m): ``std`` (m, k) the standard error of every entry of W, ``covariance`` and ``information`` (m, k,
m, k) the covariance and Poisson information of vec(W).  With G = None (m = n): ``std`` (n, k) and the diagonal blocks
only, ``covariance`` and ``information`` (n, k, k), one per channel.  ``spectrum_std`` (n, k) is the standard error of
the phase spectra G W (``components_``).  NaN marks singular information: all of std, covariance and spectrum_std with a
real G, the channel's entries with G = None."""

ResidualComponents = namedtuple("ResidualComponents", ["singular_values", "spectra", "maps"])
ResidualComponents.__doc__ = """Leading singular triplets of the Pearson residual (x - y) / sqrt(y) of a SmoothNMF model
(``SmoothNMF.residual_components``), float64 arrays: ``singular_values`` (rank,) descending, ``spectra`` (n, rank) with
orthonormal columns (the channel side; the entry of largest magnitude of each column is positive) and ``maps`` (rank, p)
with orthonormal rows (the pixel side, pixel order of the X passed in)."""


class SmoothNMF(TransformerMixin, BaseEstimator):
    """NMF ``X ~ G W H`` with KL loss, simplex constraints, Laplacian and log regularisation."""

    loss_names_ = ["KL_div_loss", "log_reg_loss", "Lapl_reg_loss", "gamma"]
    const_KL_ = None

    def __init__(self, lambda_L=0.0, linesearch=False, mu=0, epsilon_reg=1, algo="log_surrogate",
                 dicotomy_tol=_DICOTOMY_TOL, gamma=None, n_components=2, init=None, tol=1e-4, max_iter=200,
                 random_state=None, verbose=1, debug=False, l2=False, G=None, shape_2d=None, normalize=False,
                 log_shift=_LOG_SHIFT, eval_print=10, true_D=None, true_H=None, fixed_H=None, fixed_W=None,
                 hspy_comp=False, no_stop_criterion=False, simplex_H=False, simplex_W=True):
        self.n_components = n_components
        self.init = init
        self.tol = tol
        self.max_iter = max_iter
        self.random_state = random_state
        self.verbose = verbose
        self.log_shift = log_shift
        self.debug = debug
        self.l2 = l2
        self.G = G
        self.shape_2d = shape_2d
        self.eval_print = eval_print
        self.true_D = true_D
        self.true_H = true_H
        self.fixed_H = fixed_H
        self.fixed_W = fixed_W
        self.hspy_comp = hspy_comp
        self.normalize = normalize
        self.no_stop_criterion = no_stop_criterion
        self.simplex_H = simplex_H
        self.simplex_W = simplex_W
        self.lambda_L = lambda_L
        self.linesearch = linesearch
        self.mu = mu
        self.epsilon_reg = epsilon_reg
        self.dicotomy_tol = dicotomy_tol
        self.algo = algo
        self.gamma = gamma
        self.check_params()

    # ------------------------------------------------------------------ sklearn plumbing
    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.input_tags.positive_only = True
        return tags

    def _more_tags(self):
        return {"requires_positive_X": True}

    # (parameter, accepted types, replacement, subject of the two printed lines, wording of the requirement, shown value)
    _TYPE_RULES = (
        ("lambda_L", (int, float), 0.0, "The regularization parameter lambda_L", "a float or int", "0.0"),
        ("linesearch", bool, False, "The linesearch parameter", "a boolean", "False"),
        ("mu", (int, float, np.ndarray), 0, "The regularization parameter mu", "a float, int or np.ndarray", "0"),
        ("epsilon_reg", (int, float), 1, "The regularization parameter epsilon_reg", "a float or int", "1"),
        ("algo", str, "log_surrogate", "The algorithm", "a string", "'log_surrogate'"),
        ("simplex_H", bool, False, "The simplex_H parameter", "a boolean", "False"),
        ("simplex_W", bool, True, "The simplex_W parameter", "a boolean", "True"),
        ("dicotomy_tol", (int, float), 1e-3, "The dicotomy_tol parameter", "a float or int", "1e-3"),
        ("gamma", (int, float, list, type(None)), None, "The gamma parameter", "a float, int, or list", "None"),
        ("verbose", (bool, int), 1, "The verbose parameter", "a boolean or int", "1"),
        ("debug", bool, False, "The debug parameter", "a boolean", "False"),
        ("l2", bool, False, "The l2 parameter", "a boolean", "False"),
        ("n_components", int, 2, "The n_components parameter", "an int", "2"),
    )

    def check_params(self):
        """Soft validation: bad values are reported on stdout and reset, never raised; the two printed lines per
        correction are the reference's (smooth_nmf.py:145-237), types first, then values, then the combinations."""
        def correct(name, value, subject, requirement, shown):
            print("%s %s" % (subject, requirement))
            print("%s is set to %s" % (subject, shown))
            setattr(self, name, value)

        for name, types, value, subject, wording, shown in self._TYPE_RULES:
            if not isinstance(getattr(self, name), types):
                # the reference words the type complaint about `algo` differently from its reset line
                lead = "The algorithm parameter" if name == "algo" else subject
                print("%s must be %s" % (lead, wording))
                print("%s is set to %s" % (subject, shown))
                setattr(self, name, value)
        if self.algo not in ("l2_surrogate", "log_surrogate", "projected_gradient", "bmd"):
            correct("algo", "log_surrogate", "The algorithm",
                    "must be 'l2_surrogate', 'log_surrogate', 'bmd' or 'projected_gradient'", "'log_surrogate'")
        if not (self.lambda_L >= 0):
            correct("lambda_L", 0, "The regularization parameter lambda_L", "must be non-negative", "0")
        if not (self.epsilon_reg > 0.0):
            correct("epsilon_reg", 1.0, "The regularization parameter epsilon_reg", "must be positive", "1")
        if not np.all(np.array(self.mu) >= 0):
            correct("mu", 0, "The regularization parameter mu", "must be non-negative", "0")
        if self.simplex_H and self.simplex_W:
            print("The simplex constraint must be applied to either W or H or none of them")
            print("The simplex constraint is applied to W and not to H")
            self.simplex_W = True
            self.simplex_H = False
        if self.linesearch:
            if self.l2:
                correct("l2", False, "The l2 parameter", "must be False when using linesearch", "False")
            if not (self.lambda_L > 0):
                print("The regularization parameter lambda_L must be non-zero when using linesearch")
                print("The regularization parameter lambda_L is set to 1")
                self.lambda_L = 1
        if self.algo != "l2_surrogate" and self.l2:
            correct("l2", False, "The l2 parameter", "must be False when using the algorithm " + self.algo, "False")

    def _require_supported(self):
        if self.algo == "projected_gradient":
            if self.simplex_W:                                          # updates.py:365-366
                raise NotImplementedError(
                    "Simplex constraint not implemented for W using the projected gradient method")


    # ------------------------------------------------------------------ X_ (lazy)
    def _host_X(self, Xv):
        """The reference's processed data matrix (base.py:262-267) computed on the host."""
        from sklearn.utils import assert_all_finite
        assert_all_finite(Xv, input_name="X")
        Xh = remove_zeros_lines(Xv, self.log_shift)
        if self.normalize:
            Xh = normalization_factor(Xh, self.n_components) * Xh
        return Xh

    def __getattr__(self, name):
        # ``X_`` is a fitted attribute of the reference (a repaired / normalised COPY of the input).  The
        # device never needs that copy, so it is only built if somebody asks for it.
        if name == "X_" and "_X_in" in self.__dict__:
            Xv = self.__dict__["_X_in"]
            fix = self.__dict__.get("_x_fix")
            if fix is None or fix[0]:
                Xh = remove_zeros_lines(Xv, self.log_shift)
            else:
                Xh = Xv
            if fix is not None and fix[1] is not None:
                Xh = fix[1] * Xh
            elif fix is None and self.normalize:
                Xh = normalization_factor(Xh, self.n_components) * Xh
            self.__dict__["X_"] = Xh
            return Xh
        raise AttributeError("%r object has no attribute %r" % (type(self).__name__, name))

    # ------------------------------------------------------------------ loss
    def _loss_from_record(self, rec, gamma=None):
        """base.py:197-205 + smooth_nmf.py:461-473 from one scalar record of the device."""
        numel = self.GWH_numel_
        if self.l2:                      # 0.5 * Frobenius_loss: the H pass accumulated sum (G W H - X)^2
            kl = 0.5 * rec[L.S_XLOGY] / numel
        else:
            kl = (rec[L.S_SUMY] - rec[L.S_XLOGY] + self.const_KL_) / numel
        reg = rec[L.S_LOGREG] / numel
        lap = 0.5 * self.lambda_L * rec[L.S_LAPL] / numel
        if gamma is None:
            gamma = self.gamma_[0] if isinstance(self.gamma_, list) else self.gamma_
        self.detailed_loss_ = [kl, reg, lap, gamma]
        return kl + reg + lap

    def __getstate__(self):
        state = super().__getstate__()
        state.pop("_engine", None)      # device buffers / ctypes handles never travel with a pickle
        return state

    def loss(self, W, H, average=True, X=None):
        """Regularised loss of (W, H) (smooth_nmf.py:457-475, base.py:167-207), evaluated on the device."""
        from .ops import full_loss
        check_is_fitted(self, "G_")
        Xe = self.X_ if X is None else X
        if self.const_KL_ is None and not self.l2:
            # base.py:200-201: computed once (mixing X and self.X_ exactly like the reference), then reused for
            # every later call, whatever X that call is given
            self.const_KL_ = float(np.sum(Xe * np.log(np.maximum(self.X_, self.log_shift))) - np.sum(Xe))
        # clamp=False: G W and H are clamped inside the KL term only (measures.py:493-495), not in the
        # regularisers (smooth_nmf.py:461-466)
        val, det = full_loss(Xe, self.G_ if not self._identity_G else None, W, H, mu=self.mu,
                             epsilon_reg=self.epsilon_reg, lambda_L=self.lambda_L, shape_2d=self.shape_2d,
                             log_shift=self.log_shift, const=0.0 if self.l2 else self.const_KL_, average=average,
                             l2=bool(self.l2), clamp=False)
        self.GWH_numel_ = Xe.shape[0] * H.shape[1]
        self.detailed_loss_ = det + [self.gamma_ if not isinstance(self.gamma_, list) else self.gamma_[0]]
        return val

    # ------------------------------------------------------------------ fit
    def fit_transform(self, X, y=None, W=None, H=None):
        """Learn the model on a B200 and return ``G W`` (or ``H.T`` with ``hspy_comp``), base.py:209-420."""
        from .engine import FitEngine
        self._require_supported()
        self.gamma_ = None                                             # smooth_nmf.py:280
        self.__dict__.pop("X_", None)
        # base.py:243-247.  NaN / inf are rejected by the device pass over X (FitEngine ingest) with
        # sklearn's messages instead of a host pass here.
        if self.hspy_comp:
            Xv = validate_data(self, X.T, dtype=[np.float64, np.float32], ensure_all_finite=False)
        else:
            Xv = validate_data(self, X, dtype=[np.float64, np.float32], ensure_all_finite=False)
            f = sys._getframe(1)                                       # base.py:249-259
            if f is not None and f.f_code.co_name == "fit":
                f = f.f_back
            if f is not None and f.f_code.co_name == "decomposition" and "hyperspy" in f.f_code.co_filename:
                print("Are you calling the function decomposition from Hyperspy?\n"
                      "If so, please set the compatibility argument 'hspy_comp' to True.\n\n"
                      "If this argument is not set correctly, the function will not work properly!!!")
        self._X_in = Xv          # X_ (base.py:262-267) is materialised on first access, see __getattr__
        self._x_fix = None
        self.const_KL_ = None
        if is_physical_model(self.G):                                  # base.py:269-274
            self.physics_model_ = self.G
            G = self.physics_model_.NMF_update()
        else:
            self.physics_model_ = None
            G = self.G
        self._identity_G = G is None
        n, p = Xv.shape
        from . import config
        distributed = False
        if config.distributed:
            import torch.distributed as dist
            distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        # initial factors (updates.py:160-223).  Given factors are only clamped; one missing factor needs a least-squares
        # solve against the data on the host; when BOTH are missing (the reference's default call) the NNDSVD of
        # scikit-learn runs its randomized SVD on the device against the X the engine holds (init_device.py), so the
        # engine is created first, with placeholders, and receives the real factors afterwards.
        device_init = (W is None and H is None and config.device_init
                       and self.n_components + 10 <= n < p)      # tall factorisations of init_device.py
        if device_init:
            c_np = np.result_type(Xv.dtype, *([] if G is None else [np.asarray(G).dtype]))
            m_cols = n if G is None else np.asarray(G).shape[1]
            G_full = np.diag(np.ones(n).astype(Xv.dtype)) if G is None else np.asarray(G)
            W0 = np.ones((m_cols, self.n_components), dtype=c_np)
            H0 = np.ones((self.n_components, p), dtype=c_np)
        else:
            X_init = Xv if (W is not None and H is not None) else self._host_X(Xv)
            G_full, W0, H0 = initialize_factors(X_init, G, W, H, self.n_components, self.init, self.random_state,
                                                self.simplex_H, self.simplex_W, self.log_shift, self.physics_model_)
            del X_init
        self.GWH_numel_ = n * p
        pg = self.algo == "projected_gradient"
        if self.algo == "bmd" and G_full.shape[0] != G_full.shape[1]:
            # the reference's Bregman W step compares G with eye(n) (updates.py:42) and cannot broadcast otherwise
            raise ValueError("operands could not be broadcast together with shapes (%d,%d) (%d,%d) "
                             % (G_full.shape + (G_full.shape[0], G_full.shape[0])))
        bmd_identity = self.algo == "bmd" and (self._identity_G or np.allclose(G_full, np.eye(G_full.shape[0])))
        if self.gamma is not None:                                     # smooth_nmf.py:290-306
            self.gamma_ = list(self.gamma) if isinstance(self.gamma, list) else self.gamma
        elif not pg:
            self.gamma_ = _SIGMA_L
        simplex_rows = None
        if self.physics_model_ is not None and self.simplex_W:
            simplex_rows = self.physics_model_.NMF_simplex()           # updates.py:62-65
        if self.lambda_L != 0 and self.shape_2d is not None:
            from .ops import check_shape_2d
            check_shape_2d(self.shape_2d, p)
        max_iter = int(self.max_iter)
        shard = None
        if distributed:
            from .dist import make_shard
            shard = make_shard()
        G_dev = None if (self._identity_G or bmd_identity) else G
        eng = FitEngine(Xv, G_dev, W0, H0,
                        shape_2d=self.shape_2d, lambda_L=self.lambda_L, mu=self.mu, epsilon_reg=self.epsilon_reg,
                        log_shift=self.log_shift, dicotomy_tol=self.dicotomy_tol, dicotomy_tol_w=_DICOTOMY_TOL,
                        tol=self.tol, sigma=_SIGMA_L if pg else float(self.gamma_), simplex_H=self.simplex_H,
                        simplex_W=self.simplex_W, simplex_rows=simplex_rows, fixed_H=self.fixed_H,
                        fixed_W=None if pg else self.fixed_W,     # smooth_nmf.py:430-437 passes no fixed_W
                        max_records=max(max_iter, 1) + 8, shard=shard, algo=self.algo, l2=bool(self.l2),
                        linesearch=bool(self.linesearch), gamma_pg=self.gamma_ if pg and self.gamma is not None else None,
                        clamp_init=True,
                        ingest=dict(eps=self.log_shift, normalize=self.n_components if self.normalize else None))
        self._engine = eng
        self.x_storage_ = eng.x_storage      # "dense" | "uint8" | "uint16": how X is held on the device (config.x_storage)
        if device_init:
            from .init_device import initialize_nmf_device
            _, W0, H0 = initialize_factors(
                Xv, G, None, None, self.n_components, self.init, self.random_state, self.simplex_H, self.simplex_W,
                self.log_shift, self.physics_model_,
                nmf_init=lambda k_, init_, rs_: initialize_nmf_device(eng, k_, init_, rs_))
            eng.set_WH(W0, H0)
        if pg and self.gamma is None:
            # estimate_Lipschitz_bound_h / _w (updates.py:393-413) with W = H = log_shift everywhere: they reduce to
            # max_j colsum(X)_j / (k ls^2) + 2 lambda_L + mu eps   and   max_c rowsum(X)_c / (k ls^2 rowsum(G)_c^2)
            cs, rs = eng.compute_x_sums()
            k_, ls_ = self.n_components, self.log_shift
            cmax = cs[:eng.p_loc].max().to("cpu", dtype=__import__("torch").float64)
            if shard is not None:
                cmax = shard.allreduce_max_scalar(cmax)
            rsG = np.ones(n) if self._identity_G else np.asarray(G_full, dtype=np.float64).sum(1)
            with np.errstate(divide="ignore", invalid="ignore"):
                gamma_W = float(np.max(rs[:n].cpu().numpy().astype(np.float64) / (k_ * ls_ ** 2 * rsG ** 2)))
            gamma_H = float(cmax) / (k_ * ls_ ** 2) + 2 * self.lambda_L + self.mu * self.epsilon_reg
            self.gamma_ = [gamma_H, gamma_W]
            eng.set_gamma_pg(float(np.max(gamma_H)), gamma_W)
        gwf = eng.gw_flags_init()
        if gwf & L.DEV_GW_ZERO_ROW:        # x / 0 would appear in the first pass: updates.py:129-131, 54-56
            eng.enable_clamp()
        elif gwf & L.DEV_GW_BELOW_LS:      # measures.py:493: the loss clamps G W, the updates do not
            eng.set_flag(L.FLAG_LOSS_DUAL)
        self._init_WH = (W0, H0)
        # device-side prologue results: const_KL_ (base.py:200-201), norm_factor_ (base.py:264-267)
        self.const_KL_ = eng.const_KL
        if self.normalize:
            self.norm_factor_ = eng.norm_factor
        self._x_fix = (eng.n_zero_rows > 0 or eng.n_zero_cols > 0, self.norm_factor_ if self.normalize else None)
        self.G_ = G_full
        # base.py:287-291.  The kernels apply the Laplacian as a stencil; L_ is the reference's matrix all the same
        # (assembled on first use: `est.L_ @ x`, `.toarray()`, `.shape` work like on the scipy.sparse original)
        from .ops import GridLaplacian
        self.L_ = GridLaplacian(*self.shape_2d) if self.shape_2d is not None else GridLaplacian(None, identity=p)

        algo_start = time.time()
        self.n_iter_ = 0
        self.losses_, self.rel_, self.detailed_losses_ = [], [], []
        self._track = False
        if self.true_D is not None and self.true_H is not None:        # base.py:301-308
            if self.true_D.shape[1] == self.n_components and self.true_H.shape[0] == self.n_components:
                self.angles_, self.mse_, self.true_losses_ = [], [], []
                eng.enable_truth(self.true_D, self.true_H)
                self._track = True
            else:
                print("The chosen number of components does not match the number of components of the provided "
                      "truth. The ground truth will be ignored.")
        batch = (self.no_stop_criterion and self.physics_model_ is None and not self._track and not eng.pg_ls
                 and not (self.verbose > 0 and self.eval_print > 0))
        try:
            if batch:
                self._run_batch(eng, max_iter)
            else:
                self._run_checked(eng, max_iter, algo_start)
        except KeyboardInterrupt:                                      # base.py:393-394
            pass

        self.W_ = eng.get_W()
        self.H_ = eng.get_H()
        if not self.simplex_H and not self.simplex_W:                  # base.py:399-400
            self.W_, self.H_ = rescaled_DH(self.W_, self.H_)
            eng.set_WH(self.W_, self.H_)
            eng.evaluate(eng.max_records - 2)
            self._final_rec = eng.read_records(eng.max_records - 2, eng.max_records - 1)[0]
        algo_time = time.time() - algo_start
        print(f"Stopped after {self.n_iter_} iterations in {algo_time // 60} minutes "
              f"and {np.round(algo_time) % 60} seconds.")
        self.reconstruction_err_ = self._loss_from_record(self._final_rec)   # base.py:407
        self._check_flags(self._final_rec)
        if self.normalize:                                             # base.py:409-410
            self.W_ = self.W_ / self.norm_factor_
        GW = self.G_ @ self.W_ if not self._identity_G else self.W_.copy()
        self.n_components_ = self.H_.shape[0]
        eng.close()
        self._engine = None            # release the device copy of X
        self._init_WH = None
        register_with_espm()
        if self.hspy_comp:                                             # base.py:415-420
            self.components_ = GW.T
            return self.H_.T
        self.components_ = self.H_
        return GW

    # ---- loop variants -----------------------------------------------------------------------
    def _append(self, rec):
        if self.linesearch and self.algo != "projected_gradient":
            self.gamma_ = float(rec[L.S_GAMMA])        # gamma_ after this iteration's update (smooth_nmf.py:378-382)
        elif self.linesearch:
            eng = self._engine
            eng.pg_ls_w_update(rec)                    # smooth_nmf.py:438-447 needs loss(W', H') = this record
            self.gamma_ = [eng.st.gamma_h, eng.st.gamma_w]
        loss = self._loss_from_record(rec)
        self.losses_.append(loss)
        self.detailed_losses_.append(self.detailed_loss_)
        self.rel_.append([rec[L.S_REL_W], rec[L.S_REL_H]])
        return loss

    def _check_flags(self, rec):
        flags = int(rec[L.S_DEV_FLAGS])
        if flags & L.DEV_PEER_TIMEOUT:
            raise RuntimeError("espm_b200: a peer rank did not answer within the exchange time-out; "
                               "the sharded fit is invalid")
        if flags & L.DEV_NONFINITE:
            raise FloatingPointError("espm_b200: non-finite values in the H update (zero row in G W?)")
        if flags & (L.DEV_BRACKET | L.DEV_NEGATIVE):
            raise AssertionError("espm_b200: simplex bisection preconditions violated "
                                 "(dicotomy.py:17-19,141-144), device flags=%#x" % flags)

    def _run_batch(self, eng, max_iter):
        """no_stop_criterion and nothing to print: enqueue every iteration, read the scalars once."""
        eng.evaluate(0)
        if eng.fast_loop:
            eng.run_iterations(1, max_iter)          # one call: the launches of every iteration are issued natively
        else:
            for it in range(1, max_iter + 1):
                eng.advance(it)
                eng.evaluate(it)
        recs = eng.read_records(0, max_iter + 1)
        if not eng.clamped and any(int(r[L.S_DEV_FLAGS]) & L.DEV_NONFINITE for r in recs):
            # x / 0 appeared mid-fit (a row of G W became zero): the reference then clamps GWH
            # (updates.py:129-131, 54-56).  Restart from the initial factors with the clamped kernels.
            eng.enable_clamp()
            eng.set_WH(*self._init_WH)
            return self._run_batch(eng, max_iter)
        self._eval_init = self._loss_from_record(recs[0])
        for it in range(1, max_iter + 1):
            self._append(recs[it])
        self.n_iter_ = max_iter
        self._final_rec = recs[max_iter]
        print("exits because max_iteration was reached")

    def _run_checked(self, eng, max_iter, algo_start):
        """The reference's while-loop with its ordered stop tests (base.py:313-393).

        The device runs ONE ITERATION AHEAD of the host: the scalar record of iterate t is written by the kernels into
        pinned host memory and stamped (engine.wait_record), so the host enqueues iteration t+1 before it looks at
        record t and the stream never drains between iterations.  When a stop test fires at t the speculative
        iteration is undone (engine.rollback: every kernel writes only the `next` buffer set).  Anything that feeds
        host results back into the next iteration -- physical-model G refresh, ground-truth tracking, the projected-
        gradient line search -- or changes device state that rollback cannot restore (the gamma_ line search) runs
        without speculation, as before."""
        eng.evaluate(0)
        rec = eng.wait_record(0)
        if int(rec[L.S_DEV_FLAGS]) & L.DEV_NONFINITE and not eng.clamped:
            eng.enable_clamp()
            eng.evaluate(0)
            rec = eng.wait_record(0)
        self._check_flags(rec)
        eval_init = self._loss_from_record(rec)                        # base.py:295
        self._eval_init = eval_init
        self._final_rec = rec
        eval_before = np.inf
        speculate = self.physics_model_ is None and not self._track and not self.linesearch and not eng.pg_ls
        ahead = False                      # is iteration n_iter_ + 1 already enqueued?
        native = eng.fast_loop and not self._track

        def step(i):
            if native:
                eng.run_iterations(i, 1)
            else:
                eng.advance(i)
                if self._track:
                    self._track_truth(eng)
                eng.evaluate(i)

        while True:
            it = self.n_iter_ + 1
            if not ahead:
                step(it)
            ahead = speculate and it < max_iter
            if ahead:                      # iteration it + 1, before the host has seen record `it`
                step(it + 1)
            rec = eng.wait_record(it)
            if int(rec[L.S_DEV_FLAGS]) & L.DEV_NONFINITE and not eng.clamped:
                # x / 0 in this iteration: redo it like the reference's NaN fallback (updates.py:129-131, 54-56) -- the
                # W pass of advance(it) when the ratio sums of W were hit, then the H pass of evaluate(it)
                if ahead:
                    eng.rollback()
                    ahead = False
                rel_w = rec[L.S_REL_W]
                eng.enable_clamp()
                if int(rec[L.S_DEV_FLAGS]) & L.DEV_NONFINITE_W:
                    # back to iterate it - 1; its H update has to be rebuilt as well (the trace / ratio sums on the
                    # device belong to a later evaluation by now), then the whole step is repeated with the clamp
                    eng.rollback()
                    eng.evaluate(eng.max_records - 7)
                    eng.advance(it)
                    rel_w = None
                eng.evaluate(it)
                rec = eng.wait_record(it)
                if rel_w is not None:
                    rec[L.S_REL_W] = rel_w
            gwf = int(rec[L.S_GW_FLAGS])
            if gwf & L.DEV_GW_BELOW_LS and not (eng.st.flags & L.FLAG_LOSS_DUAL):
                # an entry of G W fell below log_shift during the fit: from here on the loss clamps it separately
                # (measures.py:493) while the updates do not
                if ahead:
                    eng.rollback()
                    ahead = False
                eng.set_flag(L.FLAG_LOSS_DUAL)
                eng.evaluate(it)
                rel_w = rec[L.S_REL_W]
                rec = eng.wait_record(it)
                rec[L.S_REL_W] = rel_w
            self._check_flags(rec)
            eval_after = self._append(rec)                             # base.py:320-351
            self.n_iter_ = it
            self._final_rec = rec
            rel_W, rel_H = rec[L.S_REL_W], rec[L.S_REL_H]
            stop = False
            if self.n_iter_ >= max_iter:                               # base.py:354-378
                print("exits because max_iteration was reached")
                stop = True
            elif not self.no_stop_criterion:
                if max(rel_H, rel_W) < self.tol:
                    print("exits because of relative change rel_A {} and rel_P {} < tol ".format(rel_H, rel_W))
                    stop = True
                elif abs((eval_before - eval_after) / eval_init) < self.tol:
                    print("exits because of relative change < tol: {}".format((eval_before - eval_after) / eval_init))
                    stop = True
                elif np.isnan(eval_after):
                    print("exit because of the presence of NaN")
                    stop = True
                elif (eval_before - eval_after) < 0:
                    print("exit because of negative decrease {}: {}, {}".format(
                        (eval_before - eval_after), eval_before, eval_after))
                    stop = True
            if stop:
                if ahead:
                    eng.rollback()         # the iterate of the stop test is the result; drop the speculative one
                break
            if self.verbose > 0 and np.mod(self.n_iter_, self.eval_print) == 0:
                print(f"It {self.n_iter_} / {max_iter}: loss {eval_after:3e},  "
                      f"{self.n_iter_ / (time.time() - algo_start + _LOG_SHIFT):0.3f} it/s")
            if self.physics_model_ is not None and self.n_iter_ % 3 == 0:   # base.py:388-392
                self.G_ = self.physics_model_.NMF_update(eng.get_W())
                eng.set_G(self.G_)
                slot = eng.max_records - 3
                eng.evaluate(slot)
                rec2 = eng.read_records(slot, slot + 1)[0]
                eval_before = self._loss_from_record(rec2)
                self._final_rec = rec2
            else:
                eval_before = eval_after

    def _track_truth(self, eng):
        """base.py:335-347: angles / MSE against the ground truth and the loss on true_D @ true_H."""
        W, H = eng.get_W(), eng.get_H()
        rescale = not (self.simplex_H or self.simplex_W)
        if rescale:
            W, H = rescaled_DH(W, H)
        GW = self.G_ @ W if not self._identity_G else W
        self.angles_.append(find_min_angle(self.true_D.T, GW.T))
        self.mse_.append(find_min_MSE(self.true_H, H))
        slot = eng.max_records - 4
        eng.truth_loss(slot, H if rescale else None)
        rec = eng.read_records(slot, slot + 1)[0]
        keep = self.__dict__.get("detailed_loss_")
        self.true_losses_.append(self._loss_from_record(rec))
        self.detailed_loss_ = keep

    def fit(self, X, y=None, **params):
        """Learn the model (base.py:422-441)."""
        self.fit_transform(X, **params)
        return self

    def goodness_of_fit(self, X, H=None):
        """Where the fitted model explains X and where it does not: per-pixel and per-channel sums of the counts, the
        model, the KL divergence and Pearson's chi-square, computed on the device in one pass over X.

        X : the data, laid out as for ``fit_transform`` ((n, p), or (p, n) with ``hspy_comp=True``), with the n channels
            of the fitted ``G_``.  Used as given: zero lines are not patched and nothing is normalised; NaN, inf and
            negative entries raise the errors of ``fit``.
        H : (k, p) maps in the internal orientation, e.g. ``est.transform(X_b).T`` for a new image; by default the
            fitted ``H_`` (X must then have the fitted pixel count).

        The model is ``G_ W_ H`` with the fitted ``W_`` (already on the scale of the raw data when ``normalize=True``) and
        ``G_`` as fitted.  ``algo``, ``l2`` and the regularisers play no part.  Returns a ``FitStatistics``; the residual
        sum spectrum is ``channel_counts - channel_model``.  Leaves every fitted attribute unchanged.  In a pixel-sharded
        run every rank passes the whole X and gets the whole, identical, result."""
        eng, shard, p = self._statistics_engine(X, H)
        try:
            pix, chan = eng.fit_statistics()
            if shard is None:
                pix, chan = pix.cpu().numpy(), chan.cpu().numpy()
            else:
                chan = self._sum_ranks(shard, chan)
                pix = self._gather_pixels(eng, shard, p, pix)
        finally:
            eng.close()
        return FitStatistics(*pix, *chan)

    def abundance_uncertainty(self, X, H=None):
        """Standard errors and covariances of the abundance maps, per pixel, from the Poisson information of X given the
        fitted phases, computed on the device in one pass over X.

        With g = max(G_ W_, log_shift), h = max(H, log_shift) and y = g h (the clamped model of the KL loss), pixel j's
        information is F_j[a, b] = sum_c x_cj g_ca g_cb / y_cj^2, the Hessian of the KL loss in the column H[:, j].  Its
        covariance is C_j = F_j^-1, and with ``simplex_H=True`` the covariance under sum_a h_aj = 1,
        C_j = F_j^-1 - (F_j^-1 1)(F_j^-1 1)^T / (1^T F_j^-1 1) (so C_j 1 = 0); ``std`` is sqrt(diag C_j).

        This is the Poisson (likelihood, Cramer-Rao) bound given the fitted phases G_ W_, which are treated as exact.  It is
        not a posterior of the regularised objective: ``lambda_L``, ``mu`` and ``epsilon_reg`` play no part, nor do
        ``algo`` and ``l2``.  Where a phase sits on the ``log_shift`` bound the bound treats that phase as free.

        X : the data, laid out as for ``fit_transform`` ((n, p), or (p, n) with ``hspy_comp=True``), with the n channels
            of the fitted ``G_``.  Used as given: zero lines are not patched and nothing is normalised; NaN, inf and
            negative entries raise the errors of ``fit``.
        H : (k, p) maps in the internal orientation, e.g. ``est.transform(X_b).T`` for a new image; by default the
            fitted ``H_`` (X must then have the fitted pixel count).

        Returns an ``AbundanceUncertainty`` of float64 arrays: ``std`` (k, p), ``covariance`` and ``information``
        (p, k, k).  A pixel whose F_j is singular (a Cholesky pivot <= 1e-12 max_a F_j[a, a], e.g. a pixel without
        counts) gets NaN ``std`` and ``covariance``; its ``information`` is returned all the same.  Nothing is printed and
        no fitted attribute changes.  In a pixel-sharded run every rank passes the whole X and gets the whole, identical,
        result."""
        eng, shard, p = self._statistics_engine(X, H)
        try:
            out = eng.abundance_information(bool(self.simplex_H))
            out = out.cpu().numpy() if shard is None else self._gather_pixels(eng, shard, p, out)
        finally:
            eng.close()
        k = eng.k
        iu = np.triu_indices(k)
        cov = np.empty((p, k, k))
        info = np.empty((p, k, k))
        nt = iu[0].size
        for full, rows in ((cov, out[k:k + nt]), (info, out[k + nt:])):
            full[:, iu[0], iu[1]] = rows.T
            full[:, iu[1], iu[0]] = rows.T
        return AbundanceUncertainty(np.ascontiguousarray(out[:k]), cov, info)

    def phase_uncertainty(self, X, H=None):
        """Standard errors and covariances of the phases W_ from the Poisson information of X given the maps, with the
        per-channel sums computed on the device in one pass over X and the small algebra on the host in fp64.

        With g = max(G_ W_, log_shift), h = max(H, log_shift) and y = g h (the clamped model of the KL loss), channel c
        contributes A_c[a, b] = sum_j x_cj h_aj h_bj / y_cj^2, and the information of vec(W), index (e, a), is
        F[(e,a),(f,b)] = sum_c G_ce G_cf A_c[a, b] (with G = None, G is the identity and F is block diagonal with blocks
        A_c).  The covariance is the constrained Cramer-Rao bound on the free entries phi = {(e, a): fixed_W is None or
        fixed_W[e, a] < 0}: with ``simplex_W`` one constraint sum_{e in S} W_ea = const per column a over its free
        entries, S = ``physics_model_.NMF_simplex()`` for a physical model and every row otherwise, and with constraint
        matrix A, C = F^-1 - F^-1 A^T (A F^-1 A^T)^-1 A F^-1.  ``std`` is sqrt(diag C) and ``spectrum_std[c, a]`` =
        sqrt(sum_{e,f} G_ce G_cf C[(e,a),(f,a)]), the error band of the phase spectra G W (``components_``).  Fixed
        entries have std 0 and zero covariance.

        This is the Poisson (likelihood) bound with the maps H held fixed and treated as exact.  It is not a posterior of
        the regularised objective: ``lambda_L``, ``mu``, ``epsilon_reg``, ``algo`` and ``l2`` play no part.

        X : the data, laid out as for ``fit_transform``, with the n channels of the fitted ``G_``.  Used as given; NaN,
            inf and negative entries raise the errors of ``fit``.
        H : (k, p) maps in the internal orientation, e.g. ``est.transform(X_b).T`` for a new image; by default the
            fitted ``H_``.

        Returns a ``PhaseUncertainty``.  With a real G, ``std`` is (m, k) and ``covariance`` and ``information`` the full
        (m, k, m, k) matrices; with G = None, ``std`` is (n, k) and ``covariance`` and ``information`` are the (n, k, k)
        diagonal blocks (the full nk x nk matrix would take gigabytes); with ``simplex_W`` a block is B_c - B_c M^-1 B_c,
        B_c = A_c^-1 on the free phases and M = sum_c B_c.  ``spectrum_std`` is (n, k).  Singular information (a
        Cholesky pivot <= 1e-12 of the largest diagonal entry) is NaN: with a real G all of std, covariance and
        spectrum_std; with G = None only that channel (e.g. one without counts), which is then left out of M, as a fixed
        entry is.  ``information`` is always returned.  Nothing is printed and no fitted attribute changes.  In a
        pixel-sharded run every rank passes the whole X and gets the whole, identical, result."""
        from .host import phase_covariance
        eng, shard, _ = self._statistics_engine(X, H)
        try:
            A = eng.phase_information()
            A = A.cpu().numpy() if shard is None else self._sum_ranks(shard, A)
        finally:
            eng.close()
        m, k = self.W_.shape
        # the projected gradient fit passes no fixed_W to its updates (smooth_nmf.py:430-437)
        fixed = None if self.algo == "projected_gradient" else self.fixed_W
        free = np.ones((m, k), dtype=bool) if fixed is None else np.asarray(fixed) < 0
        rows = None
        if self.simplex_W:
            rows = np.arange(m) if self.physics_model_ is None else np.asarray(self.physics_model_.NMF_simplex())
        return PhaseUncertainty(*phase_covariance(A, None if self._identity_G else self.G_, free, rows))

    def residual_components(self, X, rank=4, H=None, n_iter=7, random_state=None):
        """What the fitted model misses: the leading singular values and vectors of its Pearson residual, by a randomized
        SVD whose passes over X run on the device.

        With g = max(G_ W_, log_shift), h = max(H, log_shift) and y = g h (the clamped model of the KL loss, as in
        ``goodness_of_fit``), the residual is R[c, j] = (x_cj - y_cj) / sqrt(y_cj), an (n, p) matrix whose squared
        Frobenius norm is the total Pearson chi-square of ``goodness_of_fit``.  Where the model is right its entries have
        unit variance; structure the model lacks (a missing phase, an element line, a detector artefact) shows up as a
        component with a large singular value, a spectrum with the lines and a map with the shape of what is missing.

        The values are descriptive: there is no built-in significance threshold.  For low-count data the Pearson entries
        are far from Gaussian, so the Marchenko-Pastur edge sqrt(n) + sqrt(p) is not a reliable noise level.  Compare
        instead with the same call on a Poisson replicate of the fitted model, e.g.
        ``est.residual_components(rng.poisson(est.G_ @ est.W_ @ H), rank)``: components that stand well above the
        replicate's are structure the model misses.

        Algorithm: randomized subspace iteration on the channel side with r = rank + 10 columns (``host.
        residual_components``); each of the 2 n_iter + 1 products R^T Q / R P^T is one pass over X per 16 columns.

        X : the data, laid out as for ``fit_transform``, with the n channels of the fitted ``G_``.  Used as given; NaN,
            inf and negative entries raise the errors of ``fit``.
        rank : number of components, an integer with 1 <= rank <= min(n, p) - 10.
        H : (k, p) maps in the internal orientation, e.g. ``est.transform(X_b).T`` for a new image; by default the
            fitted ``H_``.
        n_iter : power iterations (>= 0).  Each sharpens the separation of the components by another factor
            (s_i / s_(r+1))^2; with n_iter = 0 the result is R projected on the random start only (values below the
            true ones).
        random_state : seed of the Gaussian start (scikit-learn's ``check_random_state``).

        Returns a ``ResidualComponents``: ``singular_values`` (rank,) descending, ``spectra`` (n, rank) with orthonormal
        columns and ``maps`` (rank, p) with orthonormal rows (reshape a row with ``shape_2d``); in every component the
        entry of ``spectra[:, i]`` of largest magnitude is positive.  Nothing is printed and no fitted attribute changes.
        In a pixel-sharded run every rank passes the whole X and gets the whole, identical, result."""
        import torch
        from sklearn.utils import check_random_state
        from .host import RESID_OVERSAMPLE, residual_components
        check_is_fitted(self, "G_")
        if isinstance(rank, (bool, np.bool_)) or not isinstance(rank, (int, np.integer)):
            raise ValueError("rank must be an integer, got %r" % (rank,))
        if isinstance(n_iter, (bool, np.bool_)) or not isinstance(n_iter, (int, np.integer)) or n_iter < 0:
            raise ValueError("n_iter must be an integer >= 0, got %r" % (n_iter,))
        shape = np.shape(X)
        if len(shape) == 2:
            n, p = shape[::-1] if self.hspy_comp else shape
            if not 1 <= rank <= min(n, p) - RESID_OVERSAMPLE:
                raise ValueError("rank must be between 1 and min(n, p) - %d = %d, got %d"
                                 % (RESID_OVERSAMPLE, min(n, p) - RESID_OVERSAMPLE, rank))
        elif rank < 1:
            raise ValueError("rank must be >= 1, got %d" % rank)
        rng = check_random_state(random_state)
        rank, n_iter = int(rank), int(n_iter)
        r = rank + RESID_OVERSAMPLE
        Q0 = rng.standard_normal((self.G_.shape[0], r))
        eng, shard, p = self._statistics_engine(X, H)
        try:
            if shard is not None:                            # the start of rank 0, so that an unseeded call agrees too
                import torch.distributed as dist
                t = torch.as_tensor(Q0, device=eng.device)
                dist.broadcast(t, src=shard._peer(0), group=shard.group)
                Q0 = t.cpu().numpy()

            def right(P):
                Y = eng.residual_right(P)
                return Y.cpu().numpy() if shard is None else self._sum_ranks(shard, Y)

            def gram(P):
                Ph = P.cpu().numpy()
                M = Ph @ Ph.T
                return M if shard is None else self._sum_ranks(shard, torch.as_tensor(M, device=eng.device))

            s, spectra, V, P = residual_components(eng.residual_left, right, gram, Q0, rank, n_iter)
            maps = V.T @ P.cpu().numpy()
            if shard is not None:
                maps = self._gather_pixels(eng, shard, p, torch.as_tensor(maps, device=eng.device))
        finally:
            eng.close()
        return ResidualComponents(s, spectra, np.ascontiguousarray(maps))

    def _statistics_engine(self, X, H):
        """Checks the arguments of goodness_of_fit / abundance_uncertainty / phase_uncertainty (before any device work)
        and builds the FitEngine of the fitted model against X: (engine, shard or None, pixel count)."""
        from .engine import FitEngine
        check_is_fitted(self, "G_")
        Xa = check_array(X, dtype=[np.float64, np.float32], ensure_all_finite=False)
        Xv = Xa.T if self.hspy_comp else Xa                       # (n, p): channels x pixels
        n, p = Xv.shape
        if n != self.G_.shape[0]:
            raise ValueError("X has %d channels, but this SmoothNMF was fitted with %d" % (n, self.G_.shape[0]))
        k = self.W_.shape[1]
        if H is None:
            if p != self.H_.shape[1]:
                raise ValueError("X has %d pixels but the fitted H_ has %d: pass the maps of this image as H"
                                 % (p, self.H_.shape[1]))
            H = self.H_
        elif np.shape(H) != (k, p):
            raise ValueError("H has shape %s, expected %s" % (np.shape(H), (k, p)))
        shard = None
        if config.distributed:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
                from .dist import make_shard
                shard = make_shard()
        eng = FitEngine.for_statistics(Xv, None if self._identity_G else self.G_, self.W_, np.asarray(H),
                                       log_shift=self.log_shift, shard=shard)
        return eng, shard, p

    @staticmethod
    def _sum_ranks(shard, block):
        """The host array of the sum over ranks of every rank's device block, added in rank order so that every rank gets
        the same bits."""
        import torch
        import torch.distributed as dist
        parts = [torch.empty_like(block) for _ in range(shard.world)]
        dist.all_gather(parts, block, group=shard.group)
        for r in range(1, shard.world):
            parts[0] += parts[r]
        return parts[0].cpu().numpy()

    @staticmethod
    def _gather_pixels(eng, shard, p, block):
        """The (rows, p) host array of every rank's (rows, p_loc) device block, in rank order, identical on all ranks."""
        from .dist import shard_bounds
        sizes = [b - a for a, b, _ in (shard_bounds(p, eng.nx, eng.ny, r, shard.world) for r in range(shard.world))]
        return shard.gather_H_device(block, sizes)

    def inverse_transform(self, W):
        """G W H (base.py:461-477)."""
        check_is_fitted(self)
        return self.G_ @ W @ self.H_

    def get_losses(self):
        """Structured array of the loss history (base.py:479-517); with ``true_D`` / ``true_H`` also the angles,
        the mean squared errors and the loss against the ground truth of every iteration."""
        names = ["full_loss"] + self.loss_names_ + ["rel_W", "rel_H"]
        truth = self.true_D is not None and self.true_H is not None
        if truth:
            names += ["ang_p%d" % i for i in range(self.n_components)]
            names += ["mse_p%d" % i for i in range(self.n_components)] + ["true_KL_loss"]
        dt = np.dtype([(name, "float64") for name in names])
        rows = []
        for i in range(len(self.losses_)):
            row = (self.losses_[i],) + tuple(self.detailed_losses_[i]) + tuple(self.rel_[i])
            if truth:
                row += tuple(self.angles_[i]) + tuple(self.mse_[i]) + (self.true_losses_[i],)
            rows.append(row)
        return np.array(rows, dtype=dt)


def _transform_available(est):
    return bool(est.hspy_comp)


def _transform(self, X, H=None, shape_2d=None):
    """Abundance maps of a new spectrum image with the fitted phases held fixed (``hspy_comp=True`` only).

    X : (p', n) array, one row per pixel (p' may differ from the fitted image), the n channels of the fitted ``G_``.
    H : optional (k, p') initial H (internal orientation, as in ``fit_transform``).  By default
        H0 = |lstsq(G_ W_, X)| (simplex-normalised with ``simplex_H``, clamped to ``log_shift``), computed on the device.
    shape_2d : image shape of X for the Laplacian (``lambda_L != 0``); by default the fitted ``shape_2d`` when it
        matches p', the identity Laplacian when the model has no ``shape_2d``.

    Returns H'^T, (p', k): the H of
    ``SmoothNMF(<same params>, G=G_, fixed_W=W_, normalize=False).fit_transform(X, W=W_, H=H)`` without its final
    rescale.  W_ and G_ are used as fitted (a physical model is not refreshed, X is not normalised, ``fixed_H`` is
    ignored); ``max_iter``, ``tol``, ``no_stop_criterion``, ``verbose`` and ``eval_print`` govern the loop, whose stop
    tests and printed exits are those of the fit (with rel_W = 0).  Each iteration streams X once (the H pass).  The
    fitted attributes are left unchanged."""
    import copy
    import torch
    from .engine import FitEngine
    from .init_device import initial_H_device
    check_is_fitted(self, "G_")
    for name, bad in (("algo=%r" % self.algo, self.algo in ("bmd", "projected_gradient")),
                      ("l2=True", bool(self.l2)), ("linesearch=True", bool(self.linesearch))):
        if bad:
            raise NotImplementedError("SmoothNMF.transform does not support %s" % name)
    Xv = check_array(X, dtype=[np.float64, np.float32], ensure_all_finite=False).T     # (n, p'): channels x pixels
    n, p = Xv.shape
    if n != self.G_.shape[0]:
        raise ValueError("X has %d features (channels), but this SmoothNMF was fitted with %d" % (n, self.G_.shape[0]))
    k = self.W_.shape[1]
    if H is not None and np.shape(H) != (k, p):
        raise ValueError("H has shape %s, expected %s" % (np.shape(H), (k, p)))
    shape = None
    if self.lambda_L != 0:                                   # base.py:280-291
        from .ops import check_shape_2d
        if shape_2d is not None:
            shape = shape_2d
        elif self.shape_2d is not None and int(np.prod(self.shape_2d)) == p:
            shape = self.shape_2d
        elif self.shape_2d is not None:
            shape = self.shape_2d                            # check_shape_2d raises its ValueError
        if shape is not None:
            shape = check_shape_2d(shape, p)
    W = self.W_
    distributed = False
    if config.distributed:
        import torch.distributed as dist
        distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    shard = None
    if distributed:
        from .dist import make_shard
        shard = make_shard()
    max_iter = int(self.max_iter)
    gamma = self.gamma if self.gamma is not None else _SIGMA_L
    H_init = np.ones((k, p), dtype=np.result_type(W.dtype, Xv.dtype)) if H is None else np.asarray(H)
    eng = FitEngine(Xv, None if self._identity_G else self.G_, W, H_init,
                    shape_2d=shape, lambda_L=self.lambda_L, mu=self.mu, epsilon_reg=self.epsilon_reg,
                    log_shift=self.log_shift, dicotomy_tol=self.dicotomy_tol, dicotomy_tol_w=_DICOTOMY_TOL,
                    tol=self.tol, sigma=float(gamma), simplex_H=self.simplex_H, simplex_W=True,
                    max_records=max(max_iter, 1) + 8, shard=shard, algo=self.algo, clamp_init=True, h_only=True,
                    ingest=dict(eps=self.log_shift, normalize=None))
    try:
        if H is None:
            H_init = initial_H_device(eng, self.G_, W, self.simplex_H, self.log_shift)
            eng.set_WH(W, H_init)
        if np.any(W < self.log_shift):
            # the first H update uses W clamped to log_shift, every later one fixed_W itself (updates.py:75-76, 220-221)
            eng.set_W_after_eval(W)
            GW = W if self._identity_G else self.G_ @ W
            if np.any(GW < self.log_shift):
                eng.set_flag(L.FLAG_LOSS_DUAL)
        gwf = eng.gw_flags_init()
        if gwf & L.DEV_GW_ZERO_ROW:
            eng.enable_clamp()
        elif gwf & L.DEV_GW_BELOW_LS:
            eng.set_flag(L.FLAG_LOSS_DUAL)
        # the loop helpers record their results on the estimator they run on: give them a copy
        run = copy.copy(self)
        run.physics_model_ = None
        run._track = False
        run._engine = eng
        run.gamma_ = gamma
        run.const_KL_ = eng.const_KL
        run.GWH_numel_ = n * p
        run._init_WH = (W, H_init)
        run.n_iter_ = 0
        run.losses_, run.rel_, run.detailed_losses_ = [], [], []
        algo_start = time.time()
        batch = self.no_stop_criterion and not (self.verbose > 0 and self.eval_print > 0)
        try:
            if batch:
                run._run_batch(eng, max_iter)
            else:
                run._run_checked(eng, max_iter, algo_start)
        except KeyboardInterrupt:
            pass
        Hn = eng.get_H()
        algo_time = time.time() - algo_start
        print(f"Stopped after {run.n_iter_} iterations in {algo_time // 60} minutes "
              f"and {np.round(algo_time) % 60} seconds.")
        run._check_flags(run._final_rec)
    finally:
        eng.close()
    return Hn.T


# ``transform`` exists only with ``hspy_comp=True`` (rows of X are pixels there, as scikit-learn expects).  It is attached
# after the class body: TransformerMixin wraps a ``transform`` defined in the class body for ``set_output``, and that
# wrapper would make it visible on every instance.
SmoothNMF.transform = available_if(_transform_available)(_transform)


def register_with_espm():
    """``isinstance(est, espm.estimators.NMFEstimator)`` is how the reference's hyperspy signal class recognises a
    fitted espm estimator (eds_spim.py:607, 639).  NMFEstimator is an ABC (base.py:20), so the drop-in registers as
    a virtual subclass -- only when espm is already imported: importing it here would pull in hyperspy / exspy."""
    mod = sys.modules.get("espm.estimators")
    base = getattr(mod, "NMFEstimator", None)
    if base is None or not hasattr(base, "register"):
        return False
    if not issubclass(SmoothNMF, base):
        base.register(SmoothNMF)
    return True


register_with_espm()
