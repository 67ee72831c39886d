/*
 * espm_b200.h -- C ABI of the B200-native SmoothNMF fit loop (libespm_b200.so).
 *
 * This is the drop-in boundary for ONE path of adriente/espm v1.1.3: the SmoothNMF fit loop
 * (espm/estimators/base.py:209-420, smooth_nmf.py:284-475, updates.py:6-156, dicotomy.py:4-173,
 * measures.py:456-577, utils.py:39-76).  The reference has no FFI of its own (it is pure Python);
 * the entry points below are what a ctypes binding inside espm.estimators would call -- see
 * INTEGRATION.md for that binding.  Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *   - every entry point returns 0 on success, a negative espm_status otherwise;
 *     espm_last_error() returns a thread-local human-readable message.
 *   - all device pointers are allocated by the caller (the Python host uses torch for that);
 *     `stream` is a cudaStream_t passed as void*.  Launches are asynchronous on that stream.
 *   - X: n energy channels x p pixels, G: n x m, W: m x k, H: k x p, GW = G.W: n x k  (base.py:58-63).
 *   - "x dtype" is the storage type of X, "c dtype" the arithmetic type (ESPM_F32 / ESPM_F64).
 *
 * Device layouts (all chosen for streaming from HBM3e, see DESIGN.md section 3)
 *   Xt   tile-major copy of X: Xt[tile][channel 0..n_pad)[pixel 0..128), zero padded.
 *        pixel j of the local shard lives in tile j/128, lane j%128.  One (tile, 16 KiB channel
 *        chunk) is contiguous, so a stage of the pipeline is ONE cp.async.bulk (TMA) copy.
 *   GW   [n_pad][kp] row-major (c dtype); pad rows are (1,0,..,0) so that padded channels give y>0.
 *   H    k rows of `ldh` elements; the pointer addresses local pixel 0, and `halo` elements before
 *        and after the p_loc owned pixels hold the neighbouring ranks' image rows (Laplacian stencil).
 */
#ifndef ESPM_B200_H
#define ESPM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ESPM_F32 0
#define ESPM_F64 1
/* compact storage of count data (x dtype only): X holds non-negative integers (Poisson counts, datasets/base.py:68)
 * below 256 / 65536; the kernels convert on the fly and compute in fp32.  4x / 2x fewer bytes per pass. */
#define ESPM_U8  2
#define ESPM_U16 3

#define ESPM_TILE_PX 128          /* pixels per tile of Xt */
#define ESPM_STAGE_BYTES 16384    /* bytes of X per pipeline stage (one bulk copy) for f32 / f64 storage; a stage is
                                   * always 32 (f64: 16) channels x 128 pixels, i.e. 8 / 4 KiB for uint16 / uint8 */
#define ESPM_MAX_K 16             /* largest supported n_components */
#define ESPM_COOP_BLOCKS 32        /* CTAs of the cooperative w_finish kernel */
#define ESPM_MAX_RANKS 16          /* largest number of pixel shards (GPUs of one NVLink domain) */
/* layout of a rank's peer flag block (uint32 words), see ESPM_FLAG_PEER */
#define ESPM_PF_SFLAG 0            /* [r]: rank r published its S / H' statistics with this sequence number */
#define ESPM_PF_MFLAG 16           /* [r]: rank r pushed its bisection trace mask with this sequence number */
#define ESPM_PF_MASK  32           /* [4*r .. 4*r+3]: rank r's 128-bit trace mask */
#define ESPM_PF_TFLAG 128          /* [32*r + c]: CTA c of rank r's espm_w_finish pushed its part of G^T S_r / the H' statistics */
#define ESPM_PF_WORDS 640
#define ESPM_NSCALARS 24          /* doubles per slot of the per-iteration scalar record */
#define ESPM_MAXIT_DICHOTOMY 100  /* espm/conf.py:59 */

typedef enum espm_status {
    ESPM_OK = 0,
    ESPM_ERR_CUDA = -1,        /* a CUDA runtime call failed (message has the CUDA error string) */
    ESPM_ERR_BAD_ARG = -2,     /* inconsistent sizes / unsupported k / null pointer */
    ESPM_ERR_NO_DEVICE = -3,   /* no sm_100 device: the product path has NO CPU fallback */
    ESPM_ERR_UNSUPPORTED = -4
} espm_status;

/* flag bits of espm_state.flags */
#define ESPM_FLAG_SIMPLEX_H   (1u << 0)  /* updates.py:143-144 */
#define ESPM_FLAG_SIMPLEX_W   (1u << 1)  /* updates.py:61-68 */
#define ESPM_FLAG_G_IDENTITY  (1u << 2)  /* G=None: G is the identity, m == n (updates.py:163-166) */
#define ESPM_FLAG_CLAMP_Y     (1u << 3)  /* GWH = max(GWH, log_shift) fallback (updates.py:129-131, 54-56) */
#define ESPM_FLAG_LOSS_DUAL   (1u << 4)  /* loss needs max(GW,ls).max(H,ls) != GW.H (measures.py:493-497) */
#define ESPM_FLAG_FIXED_H     (1u << 5)  /* updates.py:154-155 */
#define ESPM_FLAG_FIXED_W     (1u << 6)  /* updates.py:75-76 */
#define ESPM_FLAG_MU          (1u << 7)  /* log regulariser active (updates.py:134-137) */
#define ESPM_FLAG_LAPLACIAN   (1u << 8)  /* lambda_L != 0 (updates.py:93-96, 138-141) */
#define ESPM_FLAG_HAVE_HPREV  (1u << 9)  /* H_prev is valid: h_finish also emits rel_H of the current iterate */
#define ESPM_FLAG_SIMPLEX_ROWS (1u << 10) /* simplex_W restricted to simplex_rows (updates.py:62-65) */
#define ESPM_FLAG_HQ          (1u << 11) /* algo="l2_surrogate": quadratic surrogate H step (updates.py:263-301):
                                          * ratio = x / (GWH + log_shift), b = colsum(GW) + lambda (HL - sigma H),
                                          * H' = (-(b+nu) + sqrt((b+nu)^2 + 4 a c)) / 2a with a = lambda sigma */
#define ESPM_FLAG_FUSED_WREDUCE (1u << 12) /* espm_w_finish also does the work of espm_w_reduce (single-GPU fits) */
#define ESPM_FLAG_PEER        (1u << 13) /* pixel-sharded fit exchanging through peer memory (NVLink), see below */
#define ESPM_FLAG_BMD         (1u << 14) /* algo="bmd": the use_bregman branches (updates.py:40-48, 120-125) */
#define ESPM_FLAG_PG          (1u << 15) /* algo="projected_gradient": proj_grad_step_h / _w (updates.py:347-391) */
#define ESPM_FLAG_L2          (1u << 16) /* l2=True: 0.5 Frobenius loss (base.py:197-198, measures.py:350-385) and the
                                          * Frobenius W step / W gradient (updates.py:29-36, 307-308) */
#define ESPM_FLAG_L2_H        (1u << 17) /* Frobenius H step / H gradient (updates.py:109-118, 330-332); only reachable
                                          * through the operator-level API, like in the reference */
#define ESPM_FLAG_EVAL_ONLY   (1u << 19) /* espm_h_finish only evaluates the loss terms of (W_cur, H_cur): no update, no
                                          * bisection, H_next / Ht untouched (loss(W, H, X=...) calls of the reference) */
#define ESPM_FLAG_LS_PARTIAL  (1u << 20) /* pixel-sharded fit: espm_linesearch only leaves this rank's sums (4 + kp values,
                                          * then the kp row maxima of H') in row `px_blocks` of ls_part; the caller
                                          * combines the ranks and takes the gamma_ decision */
#define ESPM_FLAG_NO_HSPEC    (1u << 21) /* espm_h_finish does not apply the previous lock-step count speculatively: espm_h_apply
                                         * always replays (tests / diagnostics; the results are identical either way) */
#define ESPM_FLAG_TIMING      (1u << 22) /* diagnostics: the small kernels leave %globaltimer stamps (ns, as doubles) in
                                         * ESPM_S_T0 .. ESPM_S_T0 + 8 of the record they work on (scripts/timeline.py) */
#define ESPM_FLAG_LINESEARCH  (1u << 18) /* smooth_nmf.py:376-386: gamma_ adapts from diff_surrogate; see sigma_dev */
#define ESPM_FLAG_H_ONLY      (1u << 23) /* W is held fixed (fit_transform with fixed_W = W, base.py:316-324 with
                                          * updates.py:75-76 overwriting W every iteration): espm_run_iterations only
                                          * runs the H half of an iteration, [h_apply] -> h_stats -> h_pass -> h_finish;
                                          * W / GW / GWc / gwstats keep the `cur` set espm_gw_prepare wrote, and the
                                          * rel_W of every record stays 0 (SmoothNMF.transform) */

/* bits of the device-side error word (espm_state.dev_flags[0]) */
#define ESPM_DEV_NONFINITE    (1u << 0)  /* non-finite ratio sums (x/0): caller must redo with CLAMP_Y */
#define ESPM_DEV_BRACKET      (1u << 1)  /* bisection bracket precondition failed (dicotomy.py:141-144) */
#define ESPM_DEV_NEGATIVE     (1u << 2)  /* negative num/denum (updates.py:148-149, dicotomy.py:17-19) */
#define ESPM_DEV_GW_BELOW_LS  (1u << 3)  /* some GW entry < log_shift: loss needs ESPM_FLAG_LOSS_DUAL */
#define ESPM_DEV_GW_ZERO_ROW  (1u << 4)  /* some row of GW is all zero: updates need ESPM_FLAG_CLAMP_Y */
#define ESPM_DEV_NONFINITE_W  (1u << 6)  /* (with ESPM_DEV_NONFINITE) the non-finite sums came from the W pass (updates.py:53-56) */
#define ESPM_DEV_PEER_TIMEOUT (1u << 5)  /* a peer rank did not signal within ~1 s: results of this fit are invalid */

/* layout of one scalar record (doubles), written by espm_h_finish / espm_w_finish */
enum {
    ESPM_S_XLOGY = 0,     /* sum max(X,ls)*log(Y) of the iterate fed to the H pass (measures.py:503) */
    ESPM_S_SUMY = 1,      /* sum Y = colsum(max(GW,ls)) . rowsum(max(H,ls)) (measures.py:502) */
    ESPM_S_LOGREG = 2,    /* sum mu_k log(H+eps) (measures.py:548) */
    ESPM_S_LAPL = 3,      /* sum H*(HL) (measures.py:577) */
    ESPM_S_REL_H = 4,     /* base.py:324 for (H_cur, H_prev) */
    ESPM_S_REL_W = 5,     /* base.py:323, written by espm_w_finish for (W_next, W_cur) */
    ESPM_S_BISECT_ITS_H = 6, /* lock-step iteration count of the H bisection (dicotomy.py:152-171) */
    ESPM_S_BISECT_ITS_W = 7,
    ESPM_S_DEV_FLAGS = 8, /* copy of the device error word */
    ESPM_S_MEAN_H = 9,
    ESPM_S_MEAN_W = 10,
    ESPM_S_GW_FLAGS = 11, /* ESPM_DEV_GW_* bits of the GW produced for the NEXT H pass */
    ESPM_S_GAMMA = 12,    /* line search: gamma_ after this iteration's update (smooth_nmf.py:378-382) */
    ESPM_S_LS_D = 13,     /* line search: diff_surrogate(H_old, H_new) (surrogates.py:116-149) */
    ESPM_S_T0 = 14,       /* .. 22: ESPM_FLAG_TIMING stamps -- h_apply start / after the mask wait, w_finish start / rows
                           * pushed / flags seen / end, h_finish start / end */
    ESPM_S_STAMP = 23     /* espm_state.rec_stamp of the espm_h_finish that completed this record: written LAST, after a
                           * system-scope fence, so a host that sees the stamp in (pinned, device-mapped) memory sees
                           * the whole record without synchronising the stream */
};

/*
 * One fit's device state.  Plain data; the Python host mirrors it with ctypes.Structure and rotates
 * the W/H/GW buffer pointers between iterations.  All pointers are device pointers unless noted.
 */
typedef struct espm_state {
    /* ---- sizes ---- */
    int32_t n;          /* energy channels */
    int32_t n_pad;      /* n rounded up to a whole number of pipeline stages */
    int32_t m;          /* columns of G (== n when G is the identity) */
    int32_t k;          /* phases (n_components) */
    int32_t kp;         /* k padded to an instantiated kernel width (2,3,4,5,6,8,12,16) */
    int32_t p_loc;      /* pixels owned by this rank */
    int32_t p_pad;      /* n_tiles * 128: row stride of numraw / num / den */
    int32_t n_tiles;    /* ceil(p_loc / 128) */
    int32_t nx;         /* global image height (rows); 0 when shape_2d is None */
    int32_t ny;         /* image width; 0 when shape_2d is None (identity Laplacian, base.py:289-291) */
    int32_t row0;       /* first global image row owned by this rank */
    int32_t halo;       /* elements available before/after the owned pixels in every H row (>= ny) */
    int32_t ldh;        /* row stride of the H buffers, in elements */
    int32_t x_dtype;    /* ESPM_F32 / ESPM_F64 / ESPM_U8 / ESPM_U16: storage of Xt */
    int32_t c_dtype;    /* ESPM_F32 / ESPM_F64: arithmetic, and storage of every other array */
    uint32_t flags;     /* ESPM_FLAG_* */
    int32_t n_simplex_rows;
    int32_t maxit;      /* maxit_dichotomy (conf.py:59) */
    /* ---- launch plan (filled by espm_plan) ---- */
    int32_t n_sms;
    int32_t h_grid;     /* CTAs of the H pass */
    int32_t h_nsplit;   /* channel splits of a tile in the H pass (partial ratio sums are added in h_finish) */
    int32_t w_upc;      /* W pass: (channel block, pixel tile) work units per CTA */
    int32_t w_nr;       /* W pass: partial-sum slots per channel block (max CTAs touching one block) */
    int32_t px_blocks;  /* CTAs of the per-pixel kernels (h_finish / h_apply) */
    int32_t h_depth;    /* pipeline stages of the H pass */
    int32_t w_depth;    /* pipeline stages of the W pass */
    int32_t cs;         /* channels per pipeline stage = channels per W-pass channel block */
    int32_t h_smem;     /* dynamic shared memory bytes of the H pass */
    int32_t w_smem;     /* dynamic shared memory bytes of the W pass */
    int32_t w_grid;     /* CTAs of the W pass */
    int64_t p_total;    /* pixels of the whole image (all ranks), for mean(H) in rel_H (base.py:324) */
    /* ---- hyper-parameters ---- */
    double lambda_L;    /* smooth_nmf.py:58 */
    double sigma;       /* gamma_ = sigmaL (smooth_nmf.py:293-294) */
    double eps_reg;     /* epsilon_reg */
    double log_shift;
    double dicotomy_tol;
    double dicotomy_tol_w; /* the W bisection uses the module constant (updates.py:64,67) */
    double tol;         /* for rel_W / rel_H (base.py:323-324) */
    double mu[ESPM_MAX_K];
    /* ---- data ---- */
    const void* Xt;         /* tile-major X (x dtype) */
    const void* G;          /* n x m row-major (c dtype) or NULL when identity */
    const void* Gt;         /* m x n row-major (G transposed) or NULL when identity */
    const void* colsum_G;   /* m (c dtype) */
    const void* W_cur;      /* m x k row-major */
    void* W_next;
    const void* GW_cur;     /* n_pad x kp */
    const void* GWc_cur;    /* max(GW, ls), n_pad x kp (written by every espm_gw_prepare; read by the X passes only with
                             * ESPM_FLAG_LOSS_DUAL, always by espm_fit_stats,
                             * espm_abundance_info, espm_phase_info and the espm_resid_* products) */
    void* GW_next;
    void* GWc_next;
    void* gwstats_cur;      /* 2*kp (c dtype): colsum(GW), colsum(max(GW,ls)) over the n real rows */
    void* gwstats_next;
    const void* H_prev;     /* k x ldh */
    const void* H_cur;
    void* H_next;
    void* hstats_cur;       /* 3*kp doubles: rowsum(H), rowsum(max(H,ls)), rowmax(H)  (global) */
    void* hstats_next;
    const void* fixed_H;    /* k x ldh (negative = free) or NULL */
    const void* fixed_W;    /* m x k or NULL */
    const int32_t* simplex_rows; /* n_simplex_rows row indices of W or NULL */
    /* ---- scratch ---- */
    void* numraw;           /* h_nsplit x kp x p_loc */
    void* num;              /* kp x p_loc */
    void* den;              /* kp x p_loc */
    void* s_part;           /* w_nr x n_pad x kp */
    void* s_sum;            /* n_pad x kp: sum over tile ranges; all-reduced across ranks by the host */
    void* Ht;               /* tile-major copy of H_next for the W pass: [n_tiles][kp][128] (pad pixels > 0) */
    void* w_num;            /* m x k scratch */
    void* w_den;            /* m x k scratch */
    double* xlogy_part;     /* h_grid */
    double* px_part;        /* px_blocks x (4 + 3*kp) partials of the per-pixel kernels */
    uint32_t* bisect_mask;  /* 4 words: bit j set <=> max|f_j| > tol somewhere (lock-step trace) */
    uint32_t* dev_flags;    /* 8 words: [0] sticky ESPM_DEV_* error bits, [1] ESPM_DEV_GW_* of GW_next,
                             * [2] h_finish completion ticket, [3] grid-barrier counter of w_finish (start at 0),
                             * [4] w_finish completion ticket, [5] w_finish "pushed" ticket (peer exchange),
                             * [6] lock-step count + 1 of the last espm_h_apply (the next espm_h_finish applies it
                             * speculatively; 0: none), [7] the count + 1 the last espm_h_finish applied (0: none) */
    double* scalars;        /* ESPM_NSCALARS doubles: the record being filled.  Only ever WRITTEN by the kernels: it may
                             * live in pinned host memory (the host then polls ESPM_S_STAMP instead of synchronising) */
    double* coop_part;      /* ESPM_COOP_BLOCKS x (2*ESPM_MAX_K + 4) doubles: per-CTA partials of w_finish */
    /* ---- ESPM_FLAG_PEER: exchange between the pixel shards through CUDA-IPC peer memory over NVLink ----
     * No host-launched collective sits on the per-iteration path: the kernels signal and wait on flag words
     * (system-scope release/acquire) and move the few KiB that cross ranks with plain peer loads / stores.
     *   - espm_w_finish PUSHES this rank's G^T S (m x k values; S itself, n x k, when G is the identity or the update
     *     rule is not the plain KL one) and H' statistics into slot [rank] of every rank's receive buffer (remote
     *     stores), raises its S flag on every rank, waits for all flags and folds the slots of its own (local) buffer
     *     in rank order (identical everywhere, no remote load on the path);
     *   - the H update pushes its first / last image row into the neighbours' halo columns (Laplacian);
     *   - espm_h_finish pushes the 128-bit bisection trace mask to every rank, espm_h_apply waits for all. */
    int32_t rank;           /* this shard */
    int32_t world;          /* number of shards (<= ESPM_MAX_RANKS) */
    uint32_t seq_s;         /* sequence number of the coming S exchange (strictly increasing, > 0) */
    uint32_t seq_m;         /* sequence number of the mask exchange (set before espm_h_finish, kept for espm_h_apply) */
    int32_t nb_prev_ldh;    /* row stride (elements) of the previous rank's H buffers */
    int32_t nb_next_ldh;
    int64_t xchg_stride;    /* bytes between the two parities of a receive buffer (= world * xchg_slot, aligned) */
    int64_t xchg_slot;      /* bytes of one source rank's slot {S [n_pad][kp], statistics} inside a parity */
    int64_t xchg_hs_off;    /* byte offset of the 3*kp statistics doubles inside one slot */
    void* nb_prev_halo;     /* in the previous rank's H_next: where my FIRST image row goes (row kk at + kk*ldh) or NULL */
    void* nb_next_halo;     /* in the next rank's H_next: where my LAST image row goes, or NULL */
    void* peer_xchg[ESPM_MAX_RANKS];       /* every rank's receive buffer: 2 parities x world slots x {S, statistics} */
    uint32_t* peer_flags[ESPM_MAX_RANKS];  /* every rank's flag block (ESPM_PF_WORDS words, zero at start) */
    /* ---- recorded bisection (simplex_H): espm_h_finish writes, espm_h_apply reads ----
     * [5][p_pad] words per pixel: words 0..3 = bit j set <=> iteration j of dicotomy.py:152-168 moved the
     * upper end (b = new); word 4 = number of iterations the trace evaluated | 1<<8 if the bracket became
     * stationary.  The replay of the it* global iterations follows these bits instead of re-evaluating f. */
    uint32_t* bisect_dec;
    /* [2][p_pad] doubles per pixel (KL simplex only): the root nu* of the pixel's simplex function found by
     * espm_h_finish and the distance |x - nu*| beyond which the sign of f(x) is certain (+inf: no anchor); lets
     * espm_h_apply decide the replayed iterations the trace has not seen without evaluating f. */
    double* bisect_anchor;
    /* ---- alternative update rules (algo = "bmd" / "projected_gradient", l2 = True, linesearch) ---- */
    double gamma_h;         /* projected gradient: step 1/gamma_h of proj_grad_step_h (updates.py:378) */
    double gamma_w;         /* projected gradient: step 1/gamma_w of proj_grad_step_w (updates.py:357) */
    double x_total;         /* sum(X): sigmaR of the Bregman W step when G is not the identity (updates.py:45) */
    const void* x_colsum;   /* p_pad (c dtype): per-pixel sums of X, sigmaR of the Bregman H step (updates.py:121) */
    const void* x_rowsum;   /* n_pad (c dtype): per-channel sums of X, sigmaR of the Bregman W step for G = identity */
    const void* GG;         /* m x m (c dtype): G^T G of the Frobenius W step (updates.py:30); NULL when G = identity */
    double* gram_gw;        /* kp*kp doubles: (G W_cur)^T (G W_cur), see espm_gram (updates.py:115) */
    double* gram_h;         /* kp*kp doubles: H_next H_next^T over ALL pixels, see espm_gram (updates.py:31) */
    double* sigma_dev;      /* line search: device-resident gamma_ read by espm_h_finish / espm_h_apply and updated by
                             * espm_linesearch; NULL: the kernels use `sigma` */
    double* ls_part;        /* px_blocks x (4 + kp) partial sums of espm_linesearch */
    double rec_stamp;       /* value espm_h_finish leaves in ESPM_S_STAMP of the record it completes (> 0, increasing) */
    /* ---- ESPM_FLAG_PEER: record inboxes.  peer_rec[r] = rank r's inbox (pinned host memory of r's process, mapped into
     * this one with espm_host_register): [world][rec_cap][8] doubles.  espm_h_finish stores this rank's share
     * {sum X log Y, log-reg, Laplacian, rel_H, device flags, -, -, stamp} of record `rec_slot` into [rank][rec_slot] of
     * its OWN inbox (peer_rec[rank]; the other entries are not dereferenced) under the same system fence as the record;
     * every host has every inbox mapped and folds the shares.  rec_cap == 0: no inboxes (the caller gathers the
     * records itself). */
    double* peer_rec[ESPM_MAX_RANKS];
    int32_t rec_slot;
    int32_t rec_cap;
} espm_state;

/* library / device */
const char* espm_last_error(void);
int espm_version(void);
/* ABI self-check for bindings: out8 = {sizeof(espm_state), offsetof p_total, lambda_L, mu, Xt, H_prev,
 * numraw, scalars}. */
int espm_state_layout(int64_t* out8);
/* number of usable CUDA devices; ESPM_ERR_NO_DEVICE if none (there is no CPU fallback). */
int espm_device_count(void);
/* fills n_pad, kp, n_tiles and the launch plan of `st` for the current device. */
int espm_plan(espm_state* st);
/* bytes of dynamic shared memory / CTAs per SM the H and W pass kernels will use (diagnostics). */
int espm_plan_info(const espm_state* st, int32_t* info8);

/*
 * X ingest: what the reference does to X on the host before the loop (base.py:243-267, 519-528, 200-201)
 * as device passes, so that a fit touches the host copy of X exactly once (the H2D copy).
 *
 * espm_retile_x: re-tile a device copy of X into Xt (replaces the host-side copy of base.py:262).
 *   src: device pointer, element (c, j) at src[c*stride_c + j*stride_p] (so both the (n,p) layout of
 *   base.py:246-247 and the transposed hyperspy layout of base.py:243-244 are accepted in place).
 *   j0: first source pixel of this rank's shard.  `scale` multiplies every entry.
 *   stats (may be NULL): what remove_zeros_lines / validate_data / normalize need to know about the RAW
 *   values -- the caller zero-fills the arrays first:
 *     row_nz[n_pad], col_nz[p_pad]  set to 1 where a channel / pixel has a non-zero entry (base.py:522-526)
 *     flags[1]                      ESPM_X_* bits (NaN / inf -> sklearn's check, negative -> base.py:528)
 *     sum_part[n_tiles * n_pad/32]  block sums of the finite raw values (mean(X), base.py:16-18)
 * espm_xt_fixup: Xt <- (row_zero[c] or col_zero[j] ? eps : Xt) * scale on the real entries (base.py:525-526,
 *   267); either array may be NULL.
 * espm_xt_const: part_out[tile] = sum X log max(X, log_shift) - sum X over the tile (const_KL_, base.py:200-201).
 * espm_reduce_sum: out[0] = sum of n doubles with a fixed summation tree.
 */
#define ESPM_X_NAN       (1u << 0)
#define ESPM_X_INF       (1u << 1)
#define ESPM_X_NEGATIVE  (1u << 2)
#define ESPM_X_FRACTION  (1u << 3)   /* espm_x_prescan: some entry is not an integer */
typedef struct espm_ingest {
    int32_t* row_nz;
    int32_t* col_nz;
    uint32_t* flags;
    double* sum_part;
} espm_ingest;
/* Strided host -> device copy (cudaMemcpy2DAsync): `height` rows of `width_bytes`, source rows `spitch_bytes` apart.
 * Lets a rank upload its pixel slab X[:, j0:j1] of a C-ordered host image without a host-side copy. */
int espm_upload_2d(void* dst, int64_t dpitch_bytes, const void* src_host, int64_t spitch_bytes, int64_t width_bytes,
                   int64_t height, void* stream);
/* Pre-scan of the uploaded raw X (before espm_plan: the storage type decides the layout): which compact storage would
 * hold it exactly, and whether remove_zeros_lines (base.py:519-528) would have to patch it.
 *   src, src_dtype (ESPM_F32 / ESPM_F64), strides, j0 as in espm_retile_x; n channels, p_loc pixels.
 *   out4 (device, zero-filled by the caller): [0] ESPM_X_* bits, [1] float bits of the largest finite entry
 *   row_nz[n], col_nz[p_loc] (device, zero-filled): set to 1 where a channel / pixel has a non-zero entry. */
int espm_x_prescan(const void* src, int32_t src_dtype, int32_t n, int64_t p_loc, int64_t stride_c, int64_t stride_p,
                   int64_t j0, uint32_t* out4, int32_t* row_nz, int32_t* col_nz, void* stream);
int espm_retile_x(const espm_state* st, const void* src, int32_t src_dtype, int64_t stride_c,
                  int64_t stride_p, int64_t j0, double scale, const espm_ingest* stats, void* stream);
int espm_xt_fixup(const espm_state* st, const int32_t* row_zero, const int32_t* col_zero, double eps,
                  double scale, void* stream);
int espm_xt_const(const espm_state* st, double* part_out, void* stream);
int espm_reduce_sum(const double* in, int64_t n, double* out, void* stream);
/* Diagnostic: out[i] = log2(y[i]) evaluated by the table-driven routine the fp64 H pass uses for the
 * max(X, ls) * log(Y) term of KLdiv_loss (measures.py:497-503); y, out: n device doubles. */
int espm_log2_table(const double* y, int64_t n, double* out, void* stream);

/* GW_next = G.W_next (+pad rows), gwstats_next, ESPM_DEV_GW_* flags.  base.py:189, updates.py:107. */
int espm_gw_prepare(const espm_state* st, void* stream);
/* colsum_G[m] = sum_c G[c][m]  (updates.py:60). */
int espm_colsum_g(const espm_state* st, void* colsum_out, void* stream);
/* hstats_next = {rowsum, rowsum(max(.,ls)), rowmax} of H_next over the local pixels (updates.py:139);
 * also rebuilds Ht from H_next (used when H_next was written by the host rather than by a kernel). */
int espm_h_stats(const espm_state* st, void* stream);

/*
 * H pass (updates.py:127-128 + measures.py:497-503): streams Xt once.
 *   numraw[s][k][j] = sum_{c in split s} GW[c][k] * X[c][j] / (GW.H)[c][j]
 *   xlogy_part[cta] = partial of sum max(X,ls)*log(Y) for (GW_cur, H_cur)
 */
int espm_h_pass(const espm_state* st, void* stream);
/*
 * Goodness of fit of (GW_cur, H_cur) against Xt over this rank's pixels (SmoothNMF.goodness_of_fit), one pass over Xt:
 *   y = sum_k max(GW, ls) max(H, ls),  kl = y - x + x ln(x / y) (x ln x := 0 at x == 0),  chi2 = (x - y)^2 / y
 *   pixel_out   [4][p_loc] doubles: per pixel sum over the n channels of x, y, kl, chi2
 *   channel_out [4][n]     doubles: per channel sum over this rank's pixels, folded in a fixed order
 *   scratch: espm_fit_stats_scratch() bytes of device memory owned by the caller.
 * Reads Xt, GWc_cur (= max(GW_cur, ls), written with GW_cur by espm_gw_prepare), H_cur (k x ldh) and log_shift; writes
 * no record and no device flag.  Deterministic: two calls give identical bits.
 */
int espm_fit_stats_scratch(const espm_state* st, int64_t* bytes_out);
int espm_fit_stats(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, void* stream);
/*
 * Poisson information and covariance of the abundance maps H_cur given (GW_cur) over this rank's pixels
 * (SmoothNMF.abundance_uncertainty), one pass over Xt:
 *   y_cj     = sum_a g_ca h_aj,   g = max(GW, ls), h = max(H, ls)            (the clamped Y of the KL loss)
 *   F_j[a,b] = sum_c x_cj g_ca g_cb / y_cj^2                                  (Hessian of the KL loss in H[:, j])
 *   C_j      = F_j^-1                                                         simplex == 0
 *   C_j      = F_j^-1 - (F_j^-1 1)(F_j^-1 1)^T / (1^T F_j^-1 1)              simplex != 0 (sum_a h_aj = 1; C_j 1 = 0)
 *   std_aj   = sqrt(C_j[a,a])
 * out: [k + 2 k (k + 1) / 2][p_loc] doubles: the k std rows, then C, then F, each symmetric matrix as its packed upper
 * triangle row by row ((0,0), (0,1), ..., (0,k-1), (1,1), ...).  A pixel whose F_j meets a Cholesky pivot
 * <= 1e-12 max_a F_j[a,a] (or is zero: no counts) gets NaN std and C; its F is written all the same.
 * Reads Xt, GWc_cur, H_cur (k x ldh) and log_shift; writes no record and no device flag.  No atomics, fixed summation
 * order: two calls give identical bits, and a pixel shard gives the bits of the whole image.  Two launches.
 */
int espm_abundance_info(const espm_state* st, int simplex, double* out, void* stream);
/*
 * Poisson information of the phases, per channel, over this rank's pixels (SmoothNMF.phase_uncertainty), one pass over
 * Xt in W-pass order:
 *   y_cj      = sum_a g_ca h_aj,   g = max(GW, ls), h = max(H, ls)           (the clamped Y of the KL loss)
 *   A_c[a,b]  = sum_j x_cj h_aj h_bj / y_cj^2
 * The information of vec(W) is F[(e,a),(f,b)] = sum_c G_ce G_cf A_c[a,b].
 * out: [k (k + 1) / 2][n] doubles, A_c as its packed upper triangle row by row ((0,0), (0,1), ..., (1,1), ...).
 * scratch: espm_phase_info_scratch bytes (a tile-major copy of max(H, ls) and the per-CTA channel sums).
 * Reads Xt, GWc_cur, H_cur (k x ldh) and log_shift; writes no record and no device flag.  No atomics, fixed summation
 * order: two calls give identical bits.  Three launches.
 */
int espm_phase_info_scratch(const espm_state* st, int64_t* bytes_out);
int espm_phase_info(const espm_state* st, double* out, void* scratch, void* stream);
/*
 * Products of the Pearson residual of (GW_cur, H_cur) with a block of vectors, over this rank's pixels
 * (SmoothNMF.residual_components), one pass over Xt per 16 columns:
 *   y_cj = sum_a g_ca h_aj,   g = max(GW, ls), h = max(H, ls)       (the clamped Y of the KL loss)
 *   R_cj = (x_cj - y_cj) / sqrt(y_cj)
 *   espm_resid_left:  out [r][p_loc] = R^T Q, Q [n][r] (row-major device doubles); H pass order
 *   espm_resid_right: out [n][r]     = R P^T, P [r][p_loc] (row-major device doubles); W pass order
 * scratch: espm_resid_left_scratch / espm_resid_right_scratch bytes for the same r (the left product's [g | Q] rows;
 * the right product's tile-major [h; P] blocks and per-CTA channel sums).
 * Reads Xt, GWc_cur, H_cur (k x ldh) and log_shift; writes no record and no device flag.  No atomics, fixed summation
 * order: two calls give identical bits, and a pixel's left product does not depend on the grid or on the sharding.
 */
int espm_resid_left_scratch(const espm_state* st, int r, int64_t* bytes_out);
int espm_resid_left(const espm_state* st, const double* Q, int r, double* out, void* scratch, void* stream);
int espm_resid_right_scratch(const espm_state* st, int r, int64_t* bytes_out);
int espm_resid_right(const espm_state* st, const double* P, int r, double* out, void* scratch, void* stream);
/*
 * Per-pixel assembly (updates.py:132-142): num, den with the log and Laplacian surrogates, the loss
 * regularisers of the CURRENT iterate (measures.py:548,577), rel_H (base.py:324), and either
 *   simplex_H: the bisection bracket and the lock-step trace mask (dicotomy.py:29-49, 138-171), or
 *   otherwise: H_next = max(num/den, ls) (+fixed_H) directly (updates.py:152-155).
 * Its last CTA reduces the H-side partials into st->scalars (loss parts of the current iterate, rel_H, flags).
 */
int espm_h_finish(const espm_state* st, void* stream);
/* Replays exactly it* bisection iterations (first clear bit of bisect_mask) and writes H_next (and Ht). */
int espm_h_apply(const espm_state* st, void* stream);

/* W pass (updates.py:38-59, re-associated as G^T (R H^T)): streams Xt once with H_next.
 *   s_part[s][c][k] = sum_{j in the tiles CTA (first_cta(c/cs)+s) owns} X[c][j]/(GW.H_next)[c][j] * H_next[k][j] */
int espm_w_pass(const espm_state* st, void* stream);
/* s_sum = sum over the slots of each channel block of s_part (fixed order => deterministic). */
int espm_w_reduce(const espm_state* st, void* stream);
/* W_next (updates.py:59-76, incl. simplex_W bisection and fixed_W), rel_W, then GW_next / gwstats_next for
 * the next H pass; with ESPM_FLAG_FUSED_WREDUCE also s_sum and hstats_next (espm_w_reduce).  One
 * cooperative kernel of ESPM_COOP_BLOCKS CTAs. */
int espm_w_finish(const espm_state* st, void* stream);

/*
 * The iteration loop in native code.  One SmoothNMF iteration is five launches (espm_h_apply, espm_w_pass,
 * espm_w_finish, then espm_h_pass, espm_h_finish for the new iterate) plus the rotation of the `prev / cur / next`
 * buffer sets; issued one by one through a Python binding that costs more host time than the kernels take on a
 * small pixel shard.  espm_run_iterations does the launches and the rotation for `n_iters` iterations in one call:
 *   for it = first_slot .. first_slot + n_iters - 1:
 *       advance:  record `it` <- rel_W ...; [h_apply]; w_pass; w_finish; rotate          (base.py:316-318)
 *       evaluate: h_pass; h_finish -> record `it` completed and stamped                   (base.py:320-324)
 * `st` is left bound to the last iterate, `lp` carries the buffer sets and the counters (in / out).  Only for fits
 * whose iteration needs nothing from the host in between (no NCCL exchange, no Gram matrices, no line search).
 * With ESPM_FLAG_H_ONLY (W fixed) an iteration is
 *       advance:  [h_apply]; h_stats (2 launches); rotate H / hstats only                    (base.py:316-317)
 *       evaluate: h_pass; h_finish -> record `it` completed and stamped, rel_W left at 0
 * i.e. 5 launches with simplex_H, 4 without, and seq_s is not advanced (there is no S exchange).  Not with
 * ESPM_FLAG_PEER: a pixel-sharded H-only loop runs from the host, which combines the ranks' H' statistics after h_stats.
 */
typedef struct espm_loop {
    void* H[3];              /* the three H buffers (pointers to local pixel 0) */
    void* W[2];
    void* GW[2];
    void* GWc[2];
    void* gwstats[2];
    void* hstats[2];
    void* nb_prev_halo[3];   /* ESPM_FLAG_PEER: halo targets in the neighbours' copy of H buffer i, or NULL */
    void* nb_next_halo[3];
    double* records;         /* base of the scalar records (ESPM_NSCALARS doubles per slot) */
    void* const* ev;         /* optional: 4 cudaEvent_t per iteration, recorded before / after h_pass and w_pass
                              * ({w0, w1, h0, h1}); NULL: none */
    int32_t ih[3];           /* indices of the (prev, cur, next) H buffers            in / out */
    int32_t iw[2];           /* (cur, next) of W / GW / GWc / gwstats                 in / out */
    int32_t ihs[2];          /* (cur, next) of hstats                                 in / out */
    int32_t have_prev;       /* H_prev is valid                                       in / out */
    uint32_t seq_s, seq_m;   /* exchange sequence numbers                             in / out */
    double stamp;            /* last record stamp handed out                          in / out */
    int64_t launches;        /* kernels launched by the call                          out */
} espm_loop;
int espm_run_iterations(espm_state* st, espm_loop* lp, int32_t first_slot, int32_t n_iters, void* stream);

/* Peer memory for ESPM_FLAG_PEER: cudaMalloc'ed (zero-filled) regions that other processes of the same
 * box map through CUDA IPC.  handle64 is the 64-byte cudaIpcMemHandle_t. */
int espm_peer_alloc(int64_t bytes, void** ptr_out);
int espm_peer_export(void* ptr, unsigned char* handle64);
int espm_peer_open(const unsigned char* handle64, void** ptr_out);
int espm_peer_close(void* ptr);
int espm_peer_free(void* ptr);
/* Page-lock `bytes` of host memory at `ptr` (e.g. a POSIX shared-memory mapping every process of the box has opened) and
 * map it into the device address space; *dev_ptr_out is the address kernels use.  espm_host_unregister undoes it. */
int espm_host_register(void* ptr, int64_t bytes, void** dev_ptr_out);
int espm_host_unregister(void* ptr);

/* Standalone operator used by the unit-level API: nu = dichotomy_simplex(num, den) (dicotomy.py:4-55).
 * num/den: k x p (c dtype, row stride p), nu_out: p.  its_out (device int32) receives it*. */
int espm_dichotomy_simplex(int32_t c_dtype, int32_t k, int64_t p, const void* num, const void* den,
                           double log_shift, double tol, int32_t maxit, void* nu_out,
                           uint32_t* mask4, uint32_t* dev_flags, int32_t* its_out, void* stream);

/* Gram matrices of the Frobenius branches: which = 0: gram_gw = GW_cur^T GW_cur (over the n real channels);
 * which = 1: gram_h = H_next H_next^T over this rank's pixels (the caller sums the ranks). */
int espm_gram(const espm_state* st, int32_t which, void* stream);
/* Sums of X for the Bregman branches (from Xt, once per fit): colsum_out[p_pad] (c dtype, per pixel),
 * rowsum_part[n_tiles][n_pad] doubles (per tile partials of the per-channel sums; the caller folds them). */
int espm_x_sums(const espm_state* st, void* colsum_out, double* rowsum_part, void* stream);
/* Line search on the Laplacian surrogate (smooth_nmf.py:376-382, surrogates.py:116-149) for (H_cur, H_next):
 * d = diff_surrogate(H_cur, H_next, L, sigmaL = *sigma_dev, algo); *sigma_dev /= 1.05 if d > 0 else *= 1.5.
 * Writes ESPM_S_GAMMA / ESPM_S_LS_D of st->scalars.  Run after espm_h_apply / espm_h_finish. */
int espm_linesearch(const espm_state* st, void* stream);
/* With ESPM_FLAG_PG the same entry point produces the two sums of the quadratic surrogate of the projected-gradient
 * line search (surrogates.py:153-171, smooth_nmf.py:383-401) for (H_cur, H_next) and the gradient left in `den` by
 * espm_h_finish: ESPM_S_LS_D = sum (H_next - H_cur) * grad, ESPM_S_GAMMA = sum (H_next - H_cur)^2. */
/* nu = dichotomy_simplex_projected_gradient(a) (dicotomy.py:83-108); a: k x p (c dtype, row stride p). */
int espm_dichotomy_simplex_pg(int32_t c_dtype, int32_t k, int64_t p, const void* a, double log_shift, double tol,
                              int32_t maxit, void* nu_out, uint32_t* mask4, uint32_t* dev_flags,
                              int32_t* its_out, void* stream);

/* nu = dichotomy_simplex_acc(a, b, minus_c) (dicotomy.py:57-81), the bisection of the quadratic-surrogate
 * H step (updates.py:286-289).  a > 0 scalar; b, minus_c: k x p.  Evaluated in fp64 whatever c_dtype. */
int espm_dichotomy_simplex_acc(int32_t c_dtype, int32_t k, int64_t p, double a, const void* b,
                               const void* minus_c, double log_shift, double tol, int32_t maxit,
                               void* nu_out, uint32_t* mask4, uint32_t* dev_flags, int32_t* its_out,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ESPM_B200_H */
