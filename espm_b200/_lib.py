"""ctypes binding of libespm_b200.so (the C ABI declared in include/espm_b200.h).

The product path has NO CPU fallback: importing this module never builds anything silently and
``load()`` raises if the CUDA library is missing or cannot be loaded.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(HERE, "lib", "libespm_b200.so")

F32, F64, U8, U16 = 0, 1, 2, 3
TILE_PX = 128
MAX_K = 16
NSCALARS = 24
MAXIT_DICHOTOMY = 100
MAX_RANKS = 16
PF_SFLAG, PF_MFLAG, PF_MASK, PF_TFLAG, PF_WORDS = 0, 16, 32, 128, 640

# espm_state.flags
FLAG_SIMPLEX_H = 1 << 0
FLAG_SIMPLEX_W = 1 << 1
FLAG_G_IDENTITY = 1 << 2
FLAG_CLAMP_Y = 1 << 3
FLAG_LOSS_DUAL = 1 << 4
FLAG_FIXED_H = 1 << 5
FLAG_FIXED_W = 1 << 6
FLAG_MU = 1 << 7
FLAG_LAPLACIAN = 1 << 8
FLAG_HAVE_HPREV = 1 << 9
FLAG_SIMPLEX_ROWS = 1 << 10
FLAG_HQ = 1 << 11
FLAG_FUSED_WREDUCE = 1 << 12
FLAG_PEER = 1 << 13
FLAG_BMD = 1 << 14
FLAG_PG = 1 << 15
FLAG_L2 = 1 << 16
FLAG_L2_H = 1 << 17
FLAG_LINESEARCH = 1 << 18
FLAG_EVAL_ONLY = 1 << 19
FLAG_LS_PARTIAL = 1 << 20
FLAG_NO_HSPEC = 1 << 21
FLAG_TIMING = 1 << 22
FLAG_H_ONLY = 1 << 23
COOP_BLOCKS = 32

# device error word
DEV_NONFINITE = 1 << 0
DEV_BRACKET = 1 << 1
DEV_NEGATIVE = 1 << 2
DEV_GW_BELOW_LS = 1 << 3
DEV_GW_ZERO_ROW = 1 << 4
DEV_PEER_TIMEOUT = 1 << 5
DEV_NONFINITE_W = 1 << 6

# scalar record slots
S_XLOGY, S_SUMY, S_LOGREG, S_LAPL, S_REL_H, S_REL_W, S_BISECT_ITS_H, S_BISECT_ITS_W, S_DEV_FLAGS, \
    S_MEAN_H, S_MEAN_W, S_GW_FLAGS, S_GAMMA, S_LS_D = range(14)
S_T0 = 14
S_STAMP = 23

_i32, _u32, _i64, _f64, _vp = ctypes.c_int32, ctypes.c_uint32, ctypes.c_int64, ctypes.c_double, ctypes.c_void_p


class EspmState(ctypes.Structure):
    """Mirror of ``struct espm_state`` (include/espm_b200.h) -- keep the field order identical."""
    _fields_ = [
        ("n", _i32), ("n_pad", _i32), ("m", _i32), ("k", _i32), ("kp", _i32),
        ("p_loc", _i32), ("p_pad", _i32), ("n_tiles", _i32), ("nx", _i32), ("ny", _i32),
        ("row0", _i32), ("halo", _i32), ("ldh", _i32), ("x_dtype", _i32), ("c_dtype", _i32),
        ("flags", _u32), ("n_simplex_rows", _i32), ("maxit", _i32),
        ("n_sms", _i32), ("h_grid", _i32), ("h_nsplit", _i32), ("w_upc", _i32), ("w_nr", _i32),
        ("px_blocks", _i32), ("h_depth", _i32), ("w_depth", _i32), ("cs", _i32),
        ("h_smem", _i32), ("w_smem", _i32), ("w_grid", _i32),
        ("p_total", _i64),
        ("lambda_L", _f64), ("sigma", _f64), ("eps_reg", _f64), ("log_shift", _f64),
        ("dicotomy_tol", _f64), ("dicotomy_tol_w", _f64), ("tol", _f64),
        ("mu", _f64 * MAX_K),
        ("Xt", _vp), ("G", _vp), ("Gt", _vp), ("colsum_G", _vp),
        ("W_cur", _vp), ("W_next", _vp),
        ("GW_cur", _vp), ("GWc_cur", _vp), ("GW_next", _vp), ("GWc_next", _vp),
        ("gwstats_cur", _vp), ("gwstats_next", _vp),
        ("H_prev", _vp), ("H_cur", _vp), ("H_next", _vp),
        ("hstats_cur", _vp), ("hstats_next", _vp),
        ("fixed_H", _vp), ("fixed_W", _vp), ("simplex_rows", _vp),
        ("numraw", _vp), ("num", _vp), ("den", _vp),
        ("s_part", _vp), ("s_sum", _vp), ("Ht", _vp), ("w_num", _vp), ("w_den", _vp),
        ("xlogy_part", _vp), ("px_part", _vp), ("bisect_mask", _vp), ("dev_flags", _vp), ("scalars", _vp), ("coop_part", _vp),
        ("rank", _i32), ("world", _i32), ("seq_s", _u32), ("seq_m", _u32), ("nb_prev_ldh", _i32), ("nb_next_ldh", _i32),
        ("xchg_stride", _i64), ("xchg_slot", _i64), ("xchg_hs_off", _i64), ("nb_prev_halo", _vp), ("nb_next_halo", _vp),
        ("peer_xchg", _vp * MAX_RANKS), ("peer_flags", _vp * MAX_RANKS),
        ("bisect_dec", _vp), ("bisect_anchor", _vp),
        ("gamma_h", _f64), ("gamma_w", _f64), ("x_total", _f64),
        ("x_colsum", _vp), ("x_rowsum", _vp), ("GG", _vp), ("gram_gw", _vp), ("gram_h", _vp), ("sigma_dev", _vp),
        ("ls_part", _vp), ("rec_stamp", _f64),
        ("peer_rec", _vp * MAX_RANKS), ("rec_slot", _i32), ("rec_cap", _i32),
    ]


class EspmLoop(ctypes.Structure):
    """Mirror of ``struct espm_loop`` (espm_run_iterations)."""
    _fields_ = [
        ("H", _vp * 3), ("W", _vp * 2), ("GW", _vp * 2), ("GWc", _vp * 2), ("gwstats", _vp * 2), ("hstats", _vp * 2),
        ("nb_prev_halo", _vp * 3), ("nb_next_halo", _vp * 3), ("records", _vp), ("ev", _vp),
        ("ih", _i32 * 3), ("iw", _i32 * 2), ("ihs", _i32 * 2), ("have_prev", _i32),
        ("seq_s", _u32), ("seq_m", _u32), ("stamp", _f64), ("launches", _i64),
    ]


class EspmIngest(ctypes.Structure):
    """Mirror of ``struct espm_ingest``."""
    _fields_ = [("row_nz", _vp), ("col_nz", _vp), ("flags", _vp), ("sum_part", _vp)]


X_NAN, X_INF, X_NEGATIVE, X_FRACTION = 1, 2, 4, 8


class EspmError(RuntimeError):
    pass


_EXPORTS = {
    # name: (restype, argtypes)
    "espm_last_error": (ctypes.c_char_p, []),
    "espm_version": (ctypes.c_int, []),
    "espm_state_layout": (ctypes.c_int, [ctypes.POINTER(_i64)]),
    "espm_device_count": (ctypes.c_int, []),
    "espm_plan": (ctypes.c_int, [ctypes.POINTER(EspmState)]),
    "espm_plan_info": (ctypes.c_int, [ctypes.POINTER(EspmState), ctypes.POINTER(_i32)]),
    "espm_upload_2d": (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "espm_x_prescan": (ctypes.c_int, [_vp, _i32, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "espm_retile_x": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _i32, _i64, _i64, _i64, _f64,
                                     ctypes.POINTER(EspmIngest), _vp]),
    "espm_xt_fixup": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp, _f64, _f64, _vp]),
    "espm_xt_const": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp]),
    "espm_reduce_sum": (ctypes.c_int, [_vp, _i64, _vp, _vp]),
    "espm_log2_table": (ctypes.c_int, [_vp, _i64, _vp, _vp]),
    "espm_gw_prepare": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_colsum_g": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp]),
    "espm_h_stats": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_h_pass": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_fit_stats_scratch": (ctypes.c_int, [ctypes.POINTER(EspmState), ctypes.POINTER(_i64)]),
    "espm_fit_stats": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp, _vp, _vp]),
    "espm_abundance_info": (ctypes.c_int, [ctypes.POINTER(EspmState), ctypes.c_int, _vp, _vp]),
    "espm_phase_info_scratch": (ctypes.c_int, [ctypes.POINTER(EspmState), ctypes.POINTER(_i64)]),
    "espm_phase_info": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp, _vp]),
    "espm_resid_left_scratch": (ctypes.c_int, [ctypes.POINTER(EspmState), _i32, ctypes.POINTER(_i64)]),
    "espm_resid_left": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _i32, _vp, _vp, _vp]),
    "espm_resid_right_scratch": (ctypes.c_int, [ctypes.POINTER(EspmState), _i32, ctypes.POINTER(_i64)]),
    "espm_resid_right": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _i32, _vp, _vp, _vp]),
    "espm_h_finish": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_h_apply": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_w_pass": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_w_reduce": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_w_finish": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_run_iterations": (ctypes.c_int, [ctypes.POINTER(EspmState), ctypes.POINTER(EspmLoop), _i32, _i32, _vp]),
    "espm_peer_alloc": (ctypes.c_int, [_i64, ctypes.POINTER(_vp)]),
    "espm_peer_export": (ctypes.c_int, [_vp, ctypes.c_char_p]),
    "espm_peer_open": (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(_vp)]),
    "espm_peer_close": (ctypes.c_int, [_vp]),
    "espm_peer_free": (ctypes.c_int, [_vp]),
    "espm_host_register": (ctypes.c_int, [_vp, _i64, ctypes.POINTER(_vp)]),
    "espm_host_unregister": (ctypes.c_int, [_vp]),
    "espm_dichotomy_simplex": (ctypes.c_int, [_i32, _i32, _i64, _vp, _vp, _f64, _f64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "espm_gram": (ctypes.c_int, [ctypes.POINTER(EspmState), _i32, _vp]),
    "espm_x_sums": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp, _vp, _vp]),
    "espm_linesearch": (ctypes.c_int, [ctypes.POINTER(EspmState), _vp]),
    "espm_dichotomy_simplex_pg": (ctypes.c_int, [_i32, _i32, _i64, _vp, _f64, _f64, _i32, _vp, _vp, _vp, _vp, _vp]),
    "espm_dichotomy_simplex_acc": (ctypes.c_int, [_i32, _i32, _i64, _f64, _vp, _vp, _f64, _f64, _i32, _vp, _vp, _vp,
                                                  _vp, _vp]),
}

_lib = None


def exported_symbols():
    """Names every entry point include/espm_b200.h declares (used by the CPU symbol test)."""
    return sorted(_EXPORTS)


def load():
    """Load libespm_b200.so.  Raises EspmError if it is missing -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise EspmError(
            "espm_b200: %s is missing. Build it with `python -m espm_b200.build` (needs nvcc); "
            "there is no CPU fallback." % LIBPATH)
    lib = ctypes.CDLL(LIBPATH)
    for name, (restype, argtypes) in _EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc < 0:
        msg = load().espm_last_error()
        raise EspmError("espm_b200 error %d: %s" % (rc, msg.decode() if msg else "?"))
    return rc
