// C ABI of libespm_b200.so (see include/espm_b200.h): argument checking, launch planning and kernel
// dispatch.  No device memory is owned here; the host passes every buffer.
#include <cstdlib>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>

#include "ingest_decl.h"
#include "small_inst.cuh"
#include "xpass_inst.cuh"

namespace espm {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static int pad_k(int k) {
    static const int widths[] = {2, 3, 4, 5, 6, 8, 12, 16};
    for (int w : widths)
        if (k <= w) return w;
    return -1;
}

static const StreamPair* const stream_pairs[] = {&stream_f32f32, &stream_f32f64, &stream_f64f64, &stream_u8f32,
                                                  &stream_u16f32};

// the launchers of the state's (storage, compute) pair; null, with the error set, for a pair without kernels
static const StreamPair* stream_pair(const espm_state* st) {
    for (const StreamPair* row : stream_pairs)
        if (row->x_dtype == st->x_dtype && row->c_dtype == st->c_dtype) return row;
    set_error("unsupported dtype pair x=%d c=%d (f64 storage requires f64 arithmetic, uint8 / uint16 storage fp32)",
              st->x_dtype, st->c_dtype);
    return nullptr;
}

// the Frobenius branches never divide by G W H and their loss does not clamp (measures.py:350-385)
static bool is_safe(const espm_state* st) {
    return !(st->flags & (ESPM_FLAG_L2 | ESPM_FLAG_L2_H)) && (st->flags & (ESPM_FLAG_CLAMP_Y | ESPM_FLAG_LOSS_DUAL)) != 0;
}
static int h_mode(const espm_state* st) {
    if (st->flags & ESPM_FLAG_L2_H) return XMODE_FROB;
    return (st->flags & ESPM_FLAG_L2) ? XMODE_KL_FROB : XMODE_KL;
}
static int w_mode(const espm_state* st) { return (st->flags & ESPM_FLAG_L2) ? XMODE_FROB : XMODE_KL; }

static int check_state(const espm_state* st) {
    if (!st) {
        set_error("null state");
        return ESPM_ERR_BAD_ARG;
    }
    if (!stream_pair(st)) return ESPM_ERR_UNSUPPORTED;
    if (st->k < 1 || st->k > ESPM_MAX_K) {
        set_error("n_components=%d is outside the supported range 1..%d", st->k, ESPM_MAX_K);
        return ESPM_ERR_UNSUPPORTED;
    }
    if (st->n < 1 || st->p_loc < 1 || st->m < 1) {
        set_error("empty problem n=%d p_loc=%d m=%d", st->n, st->p_loc, st->m);
        return ESPM_ERR_BAD_ARG;
    }
    if (st->flags & ESPM_FLAG_PEER) {
        if (st->world < 1 || st->world > ESPM_MAX_RANKS || st->rank < 0 || st->rank >= st->world) {
            set_error("peer exchange: bad rank %d / world %d", st->rank, st->world);
            return ESPM_ERR_BAD_ARG;
        }
        if (!(st->flags & ESPM_FLAG_FUSED_WREDUCE)) {
            set_error("ESPM_FLAG_PEER requires ESPM_FLAG_FUSED_WREDUCE");
            return ESPM_ERR_BAD_ARG;
        }
    }
    return ESPM_OK;
}

static XPassArgs make_args(const espm_state* st, bool w_pass) {
    XPassArgs a;
    memset(&a, 0, sizeof(a));
    a.Xt = st->Xt;
    a.GW = st->GW_cur;
    a.GWc = st->GWc_cur;
    a.H = st->H_cur;
    a.Ht = st->Ht;
    a.numraw = st->numraw;
    a.xlogy_part = st->xlogy_part;
    a.bisect_mask = st->bisect_mask;
    a.s_part = st->s_part;
    a.n_pad = st->n_pad;
    a.k = st->k;
    a.n_tiles = st->n_tiles;
    a.ldh = st->ldh;
    a.p_pad = st->p_pad;
    a.nstages_tile = st->n_pad / st->cs;
    a.nsplit = st->h_nsplit;
    a.w_upc = st->w_upc;
    a.depth = w_pass ? st->w_depth : st->h_depth;
    // the quadratic-surrogate H step divides by GWH + log_shift and has no NaN fallback (updates.py:280)
    a.clamp_y = ((st->flags & ESPM_FLAG_CLAMP_Y) && (w_pass || !(st->flags & ESPM_FLAG_HQ))) ? 1 : 0;
    a.dual = (st->flags & ESPM_FLAG_LOSS_DUAL) ? 1 : 0;
    a.log_shift = st->log_shift;
    a.y_shift = (!w_pass && (st->flags & ESPM_FLAG_HQ)) ? st->log_shift : 0.0;
    a.n = st->n;
    a.p_loc = st->p_loc;
    return a;
}

}  // namespace espm

using namespace espm;

extern "C" {

const char* espm_last_error(void) { return g_err; }

int espm_version(void) { return 100; }

int espm_state_layout(int64_t* out8) {
    if (!out8) return ESPM_ERR_BAD_ARG;
    out8[0] = (int64_t)sizeof(espm_state);
    out8[1] = (int64_t)offsetof(espm_state, p_total);
    out8[2] = (int64_t)offsetof(espm_state, lambda_L);
    out8[3] = (int64_t)offsetof(espm_state, mu);
    out8[4] = (int64_t)offsetof(espm_state, Xt);
    out8[5] = (int64_t)offsetof(espm_state, H_prev);
    out8[6] = (int64_t)offsetof(espm_state, numraw);
    out8[7] = (int64_t)offsetof(espm_state, scalars);
    return ESPM_OK;
}

int espm_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error("no CUDA device available (%s); espm_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return ESPM_ERR_NO_DEVICE;
    }
    return n;
}

int espm_plan(espm_state* st) {
    if (!st) {
        set_error("null state");
        return ESPM_ERR_BAD_ARG;
    }
    st->kp = pad_k(st->k);
    int rc = check_state(st);
    if (rc) return rc;
    int dev = 0;
    ESPM_CUDA_CHECK(cudaGetDevice(&dev));
    // cudaGetDeviceProperties takes milliseconds (it queries everything); a fit plans once, but a fit of 20 iterations
    // is only 15 ms of kernels -- keep the properties of every device after the first query
    static cudaDeviceProp props[64];
    static bool have[64] = {false};
    if (dev < 0 || dev >= 64) {
        set_error("device index %d out of range", dev);
        return ESPM_ERR_BAD_ARG;
    }
    if (!have[dev]) {
        ESPM_CUDA_CHECK(cudaGetDeviceProperties(&props[dev], dev));
        have[dev] = true;
    }
    const cudaDeviceProp& prop = props[dev];
    if (prop.major < 10) {
        set_error("device %s is sm_%d%d; espm_b200 is built for sm_100a only", prop.name, prop.major, prop.minor);
        return ESPM_ERR_NO_DEVICE;
    }
    st->n_sms = prop.multiProcessorCount;
    st->n_tiles = (st->p_loc + TILE_PX - 1) / TILE_PX;
    st->p_pad = st->n_tiles * TILE_PX;
    st->px_blocks = (st->p_loc + PX_THREADS - 1) / PX_THREADS;
    if (st->maxit <= 0 || st->maxit > 127) st->maxit = ESPM_MAXIT_DICHOTOMY;

    // The plan is made for the SAFE variant's shared-memory footprint so that switching on the
    // clamp / dual-loss fallbacks mid-fit never needs a re-plan.
    const StreamPair* row = stream_pair(st);
    XPassSizes z;
    rc = row->xpass_sizes(st->kp, 1, &z);
    if (rc) return rc;
    st->cs = z.cs;
    st->n_pad = (st->n + 31) / 32 * 32;   // whole stages for every storage type (CS is 32 or 16)
    const int NS = st->n_pad / z.cs;
    const SmemLimits lim{(int)prop.sharedMemPerMultiprocessor, (int)prop.sharedMemPerBlockOptin};   // 228, 227 KiB on B200

    // ---- H pass ----
    const int depth = ring_depth(lim, z.h_occ, z.fixed, z.h_tail, z.h_stride, 8, "H pass", st->kp);
    if (depth < 0) return depth;
    st->h_depth = depth;
    st->h_smem = z.fixed + depth * z.h_stride + z.h_tail;
    int occ = 0;
    {
        XPassLaunch l{XPASS_H, st->kp, 1, 1, st->h_smem, XMODE_KL};
        rc = row->xpass(l, nullptr, &occ, 0);
        if (rc) return rc;
        if (occ < 1) {
            set_error("H pass kernel does not fit on an SM (smem=%d)", st->h_smem);
            return ESPM_ERR_UNSUPPORTED;
        }
    }
    const int cap_h = st->n_sms * occ;
    {
        // channel splits: smallest split count whose static schedule keeps >= 95 % of the CTAs busy
        static const int cand[] = {1, 2, 3, 4, 6, 8, 12, 16};
        int best = 1;
        double best_eff = -1.0;
        for (int s : cand) {
            if (s > NS) break;
            const long long items = (long long)st->n_tiles * s;
            const long long grid = items < cap_h ? items : cap_h;
            const long long rounds = (items + grid - 1) / grid;
            // small problems: also reward filling the machine
            const double eff = (double)items / (double)(rounds * cap_h);
            if (eff > best_eff + 1e-9) {
                best_eff = eff;
                best = s;
            }
            if (eff >= 0.95) break;
        }
        st->h_nsplit = best;
        const long long items = (long long)st->n_tiles * best;
        st->h_grid = (int)(items < cap_h ? items : cap_h);
    }

    // ---- W pass: contiguous ranges of (channel block, tile) units, one per CTA ----
    {
        // Measured on B200 (C3 f32, profiles/r01f_summary.md): the W pass is FASTER with a shallow ring -- 6 stages
        // 0.347 ms, 5: 0.340, 4: 0.323, 3: 0.316, 2: 0.344.  Consecutive units of a CTA are 1 MiB apart in Xt (same
        // channel block, next tile), so every stage in flight opens another DRAM page; three stages per CTA keep the
        // HBM queues short enough for the 592 concurrent streams.
        const int wdepth = ring_depth(lim, z.w_occ, z.fixed, z.w_tail, z.w_stride, 3, "W pass", st->kp);
        if (wdepth < 0) return wdepth;
        st->w_depth = wdepth;
        st->w_smem = z.fixed + wdepth * z.w_stride + z.w_tail;
        int wocc = 0;
        XPassLaunch l{XPASS_W, st->kp, 1, 1, st->w_smem, XMODE_KL};
        rc = row->xpass(l, nullptr, &wocc, 0);
        if (rc) return rc;
        if (wocc < 1) {
            set_error("W pass kernel does not fit on an SM (smem=%d)", st->w_smem);
            return ESPM_ERR_UNSUPPORTED;
        }
        plan_w_units(NS, st->n_tiles, (long long)st->n_sms * wocc, &st->w_upc, &st->w_grid, &st->w_nr);
    }
    return ESPM_OK;
}

int espm_plan_info(const espm_state* st, int32_t* info8) {
    if (!st || !info8) return ESPM_ERR_BAD_ARG;
    const StreamPair* row = stream_pair(st);
    if (!row) return ESPM_ERR_UNSUPPORTED;
    XPassSizes z;
    int rc = row->xpass_sizes(st->kp, 1, &z);
    if (rc) return rc;
    info8[0] = z.h_stride;
    info8[1] = z.w_stride;
    info8[2] = z.cs;
    info8[3] = z.halves;
    info8[4] = st->h_smem;
    info8[5] = st->w_smem;
    info8[6] = st->h_grid;
    info8[7] = st->w_grid;
    return ESPM_OK;
}

int espm_upload_2d(void* dst, int64_t dpitch_bytes, const void* src_host, int64_t spitch_bytes, int64_t width_bytes,
                   int64_t height, void* stream) {
    if (!dst || !src_host || width_bytes <= 0 || height <= 0 || dpitch_bytes < width_bytes || spitch_bytes < width_bytes) {
        set_error("espm_upload_2d: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    ESPM_CUDA_CHECK(cudaMemcpy2DAsync(dst, (size_t)dpitch_bytes, src_host, (size_t)spitch_bytes, (size_t)width_bytes,
                                      (size_t)height, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return ESPM_OK;
}

int espm_x_prescan(const void* src, int32_t src_dtype, int32_t n, int64_t p_loc, int64_t stride_c, int64_t stride_p,
                   int64_t j0, uint32_t* out4, int32_t* row_nz, int32_t* col_nz, void* stream) {
    if (!src || !out4 || !row_nz || !col_nz || n < 1 || p_loc < 1 || (src_dtype != ESPM_F32 && src_dtype != ESPM_F64)) {
        set_error("espm_x_prescan: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    return prescan_launch(src, src_dtype, n, (long long)p_loc, stride_c, stride_p, j0, out4, row_nz, col_nz,
                          (cudaStream_t)stream);
}

int espm_retile_x(const espm_state* st, const void* src, int32_t src_dtype, int64_t stride_c, int64_t stride_p,
                  int64_t j0, double scale, const espm_ingest* stats, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    IngestOut io{nullptr, nullptr, nullptr, nullptr};
    if (stats) {
        if (!stats->row_nz || !stats->col_nz || !stats->flags || !stats->sum_part) {
            set_error("espm_retile_x: incomplete espm_ingest");
            return ESPM_ERR_BAD_ARG;
        }
        io = IngestOut{stats->row_nz, stats->col_nz, stats->flags, stats->sum_part};
    }
    return retile_launch(st, src, src_dtype, stride_c, stride_p, j0, scale, io, (cudaStream_t)stream);
}

int espm_xt_fixup(const espm_state* st, const int32_t* row_zero, const int32_t* col_zero, double eps, double scale,
                  void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    return xt_fixup_launch(st, row_zero, col_zero, eps, scale, (cudaStream_t)stream);
}

int espm_xt_const(const espm_state* st, double* part_out, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!part_out) {
        set_error("espm_xt_const: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return xt_const_launch(st, part_out, (cudaStream_t)stream);
}

int espm_log2_table(const double* y, int64_t n, double* out, void* stream) {
    if (!y || !out || n < 0) {
        set_error("espm_log2_table: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    return log2_table_launch(y, (long long)n, out, (cudaStream_t)stream);
}

int espm_reduce_sum(const double* in, int64_t n, double* out, void* stream) {
    if (!in || !out || n < 0) {
        set_error("espm_reduce_sum: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    return reduce_sum_launch(in, (long long)n, out, (cudaStream_t)stream);
}

static int small(int op, const espm_state* st, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    return st->c_dtype == ESPM_F64 ? small_launch_f64(op, st, (cudaStream_t)stream)
                                   : small_launch_f32(op, st, (cudaStream_t)stream);
}

int espm_gw_prepare(const espm_state* st, void* stream) { return small(OP_GW_PREPARE, st, stream); }
int espm_h_stats(const espm_state* st, void* stream) { return small(OP_H_STATS, st, stream); }
int espm_h_finish(const espm_state* st, void* stream) { return small(OP_H_FINISH, st, stream); }
int espm_h_apply(const espm_state* st, void* stream) { return small(OP_H_APPLY, st, stream); }
int espm_w_reduce(const espm_state* st, void* stream) { return small(OP_W_REDUCE, st, stream); }
int espm_w_finish(const espm_state* st, void* stream) { return small(OP_W_FINISH, st, stream); }

int espm_linesearch(const espm_state* st, void* stream) {
    if (st && (!st->ls_part || (!st->sigma_dev && !(st->flags & ESPM_FLAG_PG)))) {
        set_error("espm_linesearch needs ls_part (and sigma_dev for the surrogate algorithms)");
        return ESPM_ERR_BAD_ARG;
    }
    return small(OP_LINESEARCH, st, stream);
}

int espm_gram(const espm_state* st, int32_t which, void* stream) {
    if (st && !(which == 0 ? st->gram_gw : st->gram_h)) {
        set_error("espm_gram: output buffer is null");
        return ESPM_ERR_BAD_ARG;
    }
    return small(which == 0 ? OP_GRAM_GW : OP_GRAM_H, st, stream);
}

int espm_x_sums(const espm_state* st, void* colsum_out, double* rowsum_part, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!colsum_out || !rowsum_part) {
        set_error("espm_x_sums: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return x_sums_launch(st, colsum_out, rowsum_part, (cudaStream_t)stream);
}

int espm_colsum_g(const espm_state* st, void* colsum_out, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!st->Gt) {
        set_error("colsum_g needs Gt");
        return ESPM_ERR_BAD_ARG;
    }
    return st->c_dtype == ESPM_F64 ? colsum_launch_f64(st, colsum_out, (cudaStream_t)stream)
                                   : colsum_launch_f32(st, colsum_out, (cudaStream_t)stream);
}

int espm_h_pass(const espm_state* st, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    // (the kernel also clears the trace mask of the coming h_finish)
    XPassArgs a = make_args(st, false);
    XPassLaunch l{XPASS_H, st->kp, is_safe(st) ? 1 : 0, st->h_grid, st->h_smem, h_mode(st)};
    return stream_pair(st)->xpass(l, &a, nullptr, (cudaStream_t)stream);
}

int espm_fit_stats_scratch(const espm_state* st, int64_t* bytes_out) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!bytes_out) {
        set_error("espm_fit_stats_scratch: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->fit_stats(st, nullptr, nullptr, nullptr, bytes_out, nullptr);
}

int espm_fit_stats(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!pixel_out || !channel_out || !scratch || !st->Xt || !st->GWc_cur || !st->H_cur) {
        set_error("espm_fit_stats: null output, scratch or input buffer");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->fit_stats(st, pixel_out, channel_out, scratch, nullptr, (cudaStream_t)stream);
}

int espm_abundance_info(const espm_state* st, int simplex, double* out, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!out || !st->Xt || !st->GWc_cur || !st->H_cur) {
        set_error("espm_abundance_info: null output or input buffer");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->h_info(st, simplex ? 1 : 0, out, (cudaStream_t)stream);
}

int espm_phase_info_scratch(const espm_state* st, int64_t* bytes_out) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!bytes_out) {
        set_error("espm_phase_info_scratch: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->w_info(st, nullptr, nullptr, bytes_out, nullptr);
}

int espm_phase_info(const espm_state* st, double* out, void* scratch, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!out || !scratch || !st->Xt || !st->GWc_cur || !st->H_cur) {
        set_error("espm_phase_info: null output, scratch or input buffer");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->w_info(st, out, scratch, nullptr, (cudaStream_t)stream);
}

static int resid_check(const espm_state* st, int r, const char* what) {
    int rc = check_state(st);
    if (rc) return rc;
    if (r < 1) {
        set_error("%s: r=%d columns, at least 1 required", what, r);
        return ESPM_ERR_BAD_ARG;
    }
    return ESPM_OK;
}

int espm_resid_left_scratch(const espm_state* st, int r, int64_t* bytes_out) {
    int rc = resid_check(st, r, "espm_resid_left_scratch");
    if (rc) return rc;
    if (!bytes_out) {
        set_error("espm_resid_left_scratch: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->resid_left(st, nullptr, r, nullptr, nullptr, bytes_out, nullptr);
}

int espm_resid_left(const espm_state* st, const double* Q, int r, double* out, void* scratch, void* stream) {
    int rc = resid_check(st, r, "espm_resid_left");
    if (rc) return rc;
    if (!Q || !out || !scratch || !st->Xt || !st->GWc_cur || !st->H_cur) {
        set_error("espm_resid_left: null input, output or scratch buffer");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->resid_left(st, Q, r, out, scratch, nullptr, (cudaStream_t)stream);
}

int espm_resid_right_scratch(const espm_state* st, int r, int64_t* bytes_out) {
    int rc = resid_check(st, r, "espm_resid_right_scratch");
    if (rc) return rc;
    if (!bytes_out) {
        set_error("espm_resid_right_scratch: null output");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->resid_right(st, nullptr, r, nullptr, nullptr, bytes_out, nullptr);
}

int espm_resid_right(const espm_state* st, const double* P, int r, double* out, void* scratch, void* stream) {
    int rc = resid_check(st, r, "espm_resid_right");
    if (rc) return rc;
    if (!P || !out || !scratch || !st->Xt || !st->GWc_cur || !st->H_cur) {
        set_error("espm_resid_right: null input, output or scratch buffer");
        return ESPM_ERR_BAD_ARG;
    }
    return stream_pair(st)->resid_right(st, P, r, out, scratch, nullptr, (cudaStream_t)stream);
}

int espm_w_pass(const espm_state* st, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    XPassArgs a = make_args(st, true);
    XPassLaunch l{XPASS_W, st->kp, is_safe(st) ? 1 : 0, st->w_grid, st->w_smem, w_mode(st)};
    return stream_pair(st)->xpass(l, &a, nullptr, (cudaStream_t)stream);
}

static void loop_bind(espm_state* st, const espm_loop* lp) {
    const int hp = lp->ih[0], hc = lp->ih[1], hn = lp->ih[2];
    const int wc = lp->iw[0], wn = lp->iw[1], sc = lp->ihs[0], sn = lp->ihs[1];
    st->H_prev = lp->H[hp];
    st->H_cur = lp->H[hc];
    st->H_next = lp->H[hn];
    st->W_cur = lp->W[wc];
    st->W_next = lp->W[wn];
    st->GW_cur = lp->GW[wc];
    st->GW_next = lp->GW[wn];
    st->GWc_cur = lp->GWc[wc];
    st->GWc_next = lp->GWc[wn];
    st->gwstats_cur = lp->gwstats[wc];
    st->gwstats_next = lp->gwstats[wn];
    st->hstats_cur = lp->hstats[sc];
    st->hstats_next = lp->hstats[sn];
    if (lp->have_prev) st->flags |= ESPM_FLAG_HAVE_HPREV;
    else st->flags &= ~ESPM_FLAG_HAVE_HPREV;
    if (st->flags & ESPM_FLAG_PEER) {
        st->nb_prev_halo = lp->nb_prev_halo[hn];
        st->nb_next_halo = lp->nb_next_halo[hn];
    }
}

int espm_run_iterations(espm_state* st, espm_loop* lp, int32_t first_slot, int32_t n_iters, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!lp || !lp->records || n_iters < 0 || first_slot < 0) {
        set_error("espm_run_iterations: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    if (st->flags & (ESPM_FLAG_L2 | ESPM_FLAG_L2_H | ESPM_FLAG_LINESEARCH | ESPM_FLAG_EVAL_ONLY)) {
        set_error("espm_run_iterations: this fit needs host work between the launches (Gram matrices / line search)");
        return ESPM_ERR_UNSUPPORTED;
    }
    const bool h_only = (st->flags & ESPM_FLAG_H_ONLY) != 0;
    if (h_only && (st->flags & ESPM_FLAG_PEER)) {
        set_error("espm_run_iterations: ESPM_FLAG_H_ONLY on a pixel shard needs the host to combine the H' statistics");
        return ESPM_ERR_UNSUPPORTED;
    }
    cudaStream_t s = (cudaStream_t)stream;
    lp->launches = 0;
    loop_bind(st, lp);
    for (int32_t it = first_slot; it < first_slot + n_iters; ++it) {
        void* const* ev = lp->ev ? lp->ev + (size_t)(it - first_slot) * 4 : nullptr;
        // ---- advance: (W_cur, H_cur) -> (W_next, H_next), rel_W etc. to record `it`
        st->scalars = lp->records + (size_t)it * ESPM_NSCALARS;
        st->rec_slot = it;
        if (st->flags & ESPM_FLAG_SIMPLEX_H) {
            if ((rc = espm_h_apply(st, stream))) return rc;
            ++lp->launches;
        }
        if (h_only) {
            // W stays: the row statistics of H' that w_finish would fold come from h_stats; only H / hstats rotate
            if ((rc = espm_h_stats(st, stream))) return rc;
            lp->launches += 2;
            const int hp = lp->ih[0], hc = lp->ih[1], hn = lp->ih[2];
            lp->ih[0] = hc;
            lp->ih[1] = hn;
            lp->ih[2] = hp;
            const int s0 = lp->ihs[0];
            lp->ihs[0] = lp->ihs[1];
            lp->ihs[1] = s0;
            lp->have_prev = 1;
            loop_bind(st, lp);
            lp->stamp += 1.0;
            st->rec_stamp = lp->stamp;
            st->seq_m = ++lp->seq_m;
            if (ev && ev[2]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[2], s));
            if ((rc = espm_h_pass(st, stream))) return rc;
            if (ev && ev[3]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[3], s));
            if ((rc = espm_h_finish(st, stream))) return rc;
            lp->launches += 2;
            continue;
        }
        st->seq_s = ++lp->seq_s;
        if (ev && ev[0]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[0], s));
        if ((rc = espm_w_pass(st, stream))) return rc;
        if (ev && ev[1]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[1], s));
        if ((rc = espm_w_finish(st, stream))) return rc;
        lp->launches += 2;
        {   // rotate: next -> cur
            const int hp = lp->ih[0], hc = lp->ih[1], hn = lp->ih[2];
            lp->ih[0] = hc;
            lp->ih[1] = hn;
            lp->ih[2] = hp;
            const int w0 = lp->iw[0];
            lp->iw[0] = lp->iw[1];
            lp->iw[1] = w0;
            const int s0 = lp->ihs[0];
            lp->ihs[0] = lp->ihs[1];
            lp->ihs[1] = s0;
            lp->have_prev = 1;
            loop_bind(st, lp);
        }
        // ---- evaluate the new iterate: completes and stamps record `it`
        lp->stamp += 1.0;
        st->rec_stamp = lp->stamp;
        st->seq_m = ++lp->seq_m;
        if (ev && ev[2]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[2], s));
        if ((rc = espm_h_pass(st, stream))) return rc;
        if (ev && ev[3]) ESPM_CUDA_CHECK(cudaEventRecord((cudaEvent_t)ev[3], s));
        if ((rc = espm_h_finish(st, stream))) return rc;
        lp->launches += 2;
    }
    return ESPM_OK;
}

int espm_peer_alloc(int64_t bytes, void** ptr_out) {
    if (!ptr_out || bytes <= 0) {
        set_error("espm_peer_alloc: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    void* p = nullptr;
    ESPM_CUDA_CHECK(cudaMalloc(&p, (size_t)bytes));
    ESPM_CUDA_CHECK(cudaMemset(p, 0, (size_t)bytes));
    ESPM_CUDA_CHECK(cudaDeviceSynchronize());
    *ptr_out = p;
    return ESPM_OK;
}

int espm_peer_export(void* ptr, unsigned char* handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!ptr || !handle64) return ESPM_ERR_BAD_ARG;
    cudaIpcMemHandle_t h;
    ESPM_CUDA_CHECK(cudaIpcGetMemHandle(&h, ptr));
    memcpy(handle64, &h, 64);
    return ESPM_OK;
}

int espm_peer_open(const unsigned char* handle64, void** ptr_out) {
    if (!handle64 || !ptr_out) return ESPM_ERR_BAD_ARG;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    void* p = nullptr;
    ESPM_CUDA_CHECK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    *ptr_out = p;
    return ESPM_OK;
}

int espm_peer_close(void* ptr) {
    if (!ptr) return ESPM_OK;
    ESPM_CUDA_CHECK(cudaIpcCloseMemHandle(ptr));
    return ESPM_OK;
}

int espm_peer_free(void* ptr) {
    if (!ptr) return ESPM_OK;
    ESPM_CUDA_CHECK(cudaFree(ptr));
    return ESPM_OK;
}

int espm_host_register(void* ptr, int64_t bytes, void** dev_ptr_out) {
    if (!ptr || bytes <= 0 || !dev_ptr_out) {
        set_error("espm_host_register: bad arguments");
        return ESPM_ERR_BAD_ARG;
    }
    ESPM_CUDA_CHECK(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
    void* d = nullptr;
    ESPM_CUDA_CHECK(cudaHostGetDevicePointer(&d, ptr, 0));
    *dev_ptr_out = d;
    return ESPM_OK;
}

int espm_host_unregister(void* ptr) {
    if (!ptr) return ESPM_OK;
    ESPM_CUDA_CHECK(cudaHostUnregister(ptr));
    return ESPM_OK;
}

static int dicho_common(int32_t c_dtype, int32_t k, int64_t p, const void* num, const void* den, double log_shift,
                        double tol, int32_t maxit, double acc_a, void* nu_out, uint32_t* mask4, uint32_t* dev_flags,
                        int32_t* its_out, void* stream) {
    const int kp = pad_k(k);
    if (kp < 0 || p < 1 || !num || !den || !nu_out || !mask4 || !dev_flags) {
        set_error("dichotomy_simplex: bad arguments (k=%d p=%lld)", k, (long long)p);
        return ESPM_ERR_BAD_ARG;
    }
    if (maxit <= 0 || maxit > 127) maxit = ESPM_MAXIT_DICHOTOMY;
    DichoArgs d{k, kp, maxit, (long long)p, num, den, log_shift, tol, acc_a, nu_out, mask4, dev_flags, its_out};
    return c_dtype == ESPM_F64 ? dicho_launch_f64(d, (cudaStream_t)stream) : dicho_launch_f32(d, (cudaStream_t)stream);
}

int espm_dichotomy_simplex(int32_t c_dtype, int32_t k, int64_t p, const void* num, const void* den, double log_shift,
                           double tol, int32_t maxit, void* nu_out, uint32_t* mask4, uint32_t* dev_flags,
                           int32_t* its_out, void* stream) {
    return dicho_common(c_dtype, k, p, num, den, log_shift, tol, maxit, 0.0, nu_out, mask4, dev_flags, its_out, stream);
}

int espm_dichotomy_simplex_pg(int32_t c_dtype, int32_t k, int64_t p, const void* a, double log_shift, double tol,
                              int32_t maxit, void* nu_out, uint32_t* mask4, uint32_t* dev_flags, int32_t* its_out,
                              void* stream) {
    return dicho_common(c_dtype, k, p, a, a, log_shift, tol, maxit, -1.0, nu_out, mask4, dev_flags, its_out, stream);
}

int espm_dichotomy_simplex_acc(int32_t c_dtype, int32_t k, int64_t p, double a, const void* b, const void* minus_c,
                               double log_shift, double tol, int32_t maxit, void* nu_out, uint32_t* mask4,
                               uint32_t* dev_flags, int32_t* its_out, void* stream) {
    if (!(a > 0.0)) {
        set_error("dichotomy_simplex_acc needs a > 0 (got %g)", a);
        return ESPM_ERR_BAD_ARG;
    }
    return dicho_common(c_dtype, k, p, minus_c, b, log_shift, tol, maxit, a, nu_out, mask4, dev_flags, its_out, stream);
}

}  // extern "C"
