// Goodness of fit of (GW, H) against X in one streaming pass (espm_fit_stats, SmoothNMF.goodness_of_fit).
//
//   y[c][j]    = sum_k max(GW[c][k], ls) * max(H[k][j], ls)          (the Y of KLdiv_loss, measures.py:493-497)
//   kl[c][j]   = y - x + x ln(x / y)        (x ln x := 0 at x == 0)
//   chi2[c][j] = (x - y)^2 / y
//
// and their sums over channels (per pixel) and over pixels (per channel), together with those of x and y.
//
// The stages come from produce_tile_stages (xpass.cuh) with the clamped GW (GWc_cur, written by espm_gw_prepare);
// a lane owns PPL pixels of the tile and walks the channels of its warp slot.  So
//   - the per-pixel sums stay in the lane across the stages of a tile (terms of one stage are added in the compute
//     type, then into fp64 accumulators), and the NSLOT warps that share a pixel are added in fp64, in slot order,
//     through shared memory once per tile;
//   - the per-channel sums cross the lanes once per (channel, stage): a reduce-scatter butterfly turns the 4 partial
//     statistics of a channel held by 32 lanes into 4 warp sums with 2 + 1 + 3 = 6 shuffles (instead of 4 x 5 for
//     four warp_sum), and one lane per statistic adds the sum, in fp64, to this CTA's private slot in `scratch` (the
//     old value is loaded one stage ahead, so the read-modify-write never waits on memory).
//     fit_stats_fold adds the slots of every CTA (and both halves of a tile row for fp64) in a fixed order.
// No atomics anywhere: two calls give bit-identical results, and the per-pixel sums do not depend on the grid (a pixel
// shard computes the same bits as the whole image).
//
// The KL statistic is accumulated as L = sum x log2(x / y) and assembled as y - x + ln2 L from the fp64 sums.  The log
// argument is x * rcp(y), clamped below at the smallest normal number so that x == 0 gives 0 * finite = 0.  fp32: one
// MUFU.RCP serves x / y and chi2, one MUFU.LG2 the log (2 MUFU per element, as in the H pass); fp64: the Newton
// reciprocal of Num<double> and the table log2 of common.cuh.
#pragma once
#include "xpass.cuh"

namespace espm {

struct FitStatsArgs {
    const void* Xt;
    const void* GWc;      // [n_pad][KP], max(GW, ls) on the real entries
    const void* H;        // [k][ldh] from local pixel 0
    double* pixel_out;    // [4][p_loc]
    double* part;         // [grid][HALVES][4][n_pad]: per-CTA channel sums of x, y, L, chi2
    int n, n_pad, k, ldh, p_loc, n_tiles, nstages_tile, depth;
    double log_shift;
};

constexpr int FIT_STATS_NSTAT = 4;
constexpr double FIT_STATS_LN2 = 0.6931471805599453094;

template <typename TX, typename TC, int KP>
struct FitStatsGeom {
    using S = XPassSmem<TX, TC, KP, false>;
    static constexpr int STRIDE = S::H_STRIDE;                      // X chunk + GW rows, as in the H pass
    static constexpr int FIXED = S::BAR_BYTES + S::MISC_BYTES;
    static constexpr int RED_BYTES = PassGeom<TX, TC>::NSLOT * FIT_STATS_NSTAT * TILE_PX * (int)sizeof(double);
    static constexpr int TAIL = RED_BYTES + (sizeof(TC) == 8 ? LOG2TAB_BYTES : 0);   // pixel epilogue + fp64 log table
};

// Reduce-scatter of NV values across the warp: afterwards v[0] of lane l is the warp sum of the value with index
// l >> (5 - log2 NV) (lanes that differ only in the lower bits hold the same sum).  A step at distance O keeps half of
// the values, sends the other half and adds what the partner sent; once one value is left the steps are a warp_sum.
template <int O, int M, typename T>
__device__ __forceinline__ void reduce_scatter_step(T* v, int lane) {
    if constexpr (O > 0) {
        if constexpr (M == 1) {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], O);
        } else {
            constexpr int HM = M / 2;
            const bool up = (lane & O) != 0;
#pragma unroll
            for (int i = 0; i < HM; ++i) {
                const T send = up ? v[i] : v[i + HM];
                const T keep = up ? v[i + HM] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, O);
            }
        }
        reduce_scatter_step<O / 2, (M > 1 ? M / 2 : 1), T>(v, lane);
    }
}

template <typename TX, typename TC, int KP>
__global__ void __launch_bounds__(XPASS_THREADS, 1) fit_stats_kernel(const FitStatsArgs a) {
    using G = PassGeom<TX, TC>;
    using F = FitStatsGeom<TX, TC, KP>;
    constexpr int PPL = G::PPL;
    constexpr int NS4 = FIT_STATS_NSTAT;
    constexpr bool FAST32 = sizeof(TC) == 4;
    static_assert(FAST32 || sizeof(TC) == 8, "compute type");
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<F::STRIDE> ring(smem, a.depth, F::FIXED);
    double* red = reinterpret_cast<double*>(smem + F::FIXED + (size_t)a.depth * F::STRIDE);   // [NSLOT][4][TILE_PX]
    [[maybe_unused]] double2* ltab_all = reinterpret_cast<double2*>(reinterpret_cast<unsigned char*>(red) + F::RED_BYTES);
    if constexpr (!FAST32) log2tab_fill(ltab_all, threadIdx.x, XPASS_THREADS);
    [[maybe_unused]] const double2* ltab = log2tab_lane(ltab_all, threadIdx.x & 31);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) ring.init();
    __syncthreads();
    const int NS = a.nstages_tile;

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            const uint64_t pol_x = l2_policy_evict_first();
            const uint64_t pol_gw = l2_policy_evict_last();
            typename Ring<F::STRIDE>::Pos pos{0, 0u};
            for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x)
                produce_tile_stages<TX, TC, KP, &FitStatsArgs::GWc>(ring, pos, pol_x, pol_gw, a, tile, 0, NS, false);
        }
        return;
    }

    const int half = warp % G::HALVES, slot = warp / G::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;
    const TC ls = (TC)a.log_shift;
    const TC* Hc = reinterpret_cast<const TC*>(a.H);
    // this lane's statistic after the reduce-scatter of 4 values, and whether it stores it
    const int rs_stat = lane >> 3;
    const bool rs_owner = (lane & 7) == 0;
    double* part = a.part + ((size_t)blockIdx.x * G::HALVES + half) * NS4 * a.n_pad + (size_t)rs_stat * a.n_pad;
    typename Ring<F::STRIDE>::Pos pos{0, 0u};
    // the owner lane's running channel sums for the coming stage, loaded one stage ahead of their use
    double nxt[G::CPW];
#pragma unroll
    for (int ci = 0; ci < G::CPW; ++ci) nxt[ci] = 0.0;

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const bool first = tile == (int)blockIdx.x;
        const int px0 = tile * TILE_PX + lane_px;
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, Hc, a.ldh, a.k, px0);
        TC pm[PPL];   // 1 for real pixels, 0 for padding (their y > 0 must not reach the channel sums)
#pragma unroll
        for (int q = 0; q < PPL; ++q) {
            pm[q] = px0 + q < a.p_loc ? TC(1) : TC(0);
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
                if (kk < a.k) h[kk][q] = Num<TC>::vmax(h[kk][q], ls);
        }
        double pacc[NS4][PPL];
#pragma unroll
        for (int s = 0; s < NS4; ++s)
#pragma unroll
            for (int q = 0; q < PPL; ++q) pacc[s][q] = 0.0;

        for (int st = 0; st < NS; ++st, ring.next(pos)) {
            ring.consumer_wait(pos);
            const unsigned char* xs = ring.stage(pos.slot);
            const unsigned char* gs = xs + G::X_BYTES;
            TC pst[NS4][PPL];   // fp32: this stage's per-pixel terms (fp64 adds them to pacc directly)
#pragma unroll
            for (int s = 0; s < NS4; ++s)
#pragma unroll
                for (int q = 0; q < PPL; ++q) pst[s][q] = TC(0);
#pragma unroll
            for (int ci = 0; ci < G::CPW; ++ci) {
                const int c = slot + ci * G::NSLOT;
                const int ch = st * G::CS + c;
                const TC cm = ch < a.n ? TC(1) : TC(0);   // pad channels: x == 0 but y > 0
                TC cs[NS4];
                if constexpr (FAST32) {
                    float2 x2[2];
                    load_x4<TX>(xs, c, lane_px, x2);
                    float gw[KP];
                    lds_gw<float, KP>(gw, gs + (size_t)c * KP * sizeof(float));
                    float2 c2[NS4];
#pragma unroll
                    for (int s = 0; s < NS4; ++s) c2[s] = make_float2(0.f, 0.f);
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const float2 hj0 = make_float2(h[0][2 * j], h[0][2 * j + 1]);
                        float2 y = __fmul2_rn(dup2(gw[0]), hj0);
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk)
                            y = __ffma2_rn(dup2(gw[kk]), make_float2(h[kk][2 * j], h[kk][2 * j + 1]), y);
                        const float2 r = make_float2(rcp_ftz(y.x), rcp_ftz(y.y));
                        const float2 xr = __fmul2_rn(x2[j], r);
                        const float2 lg = make_float2(lg2_ftz(fmaxf(xr.x, 1.17549435e-38f)),
                                                      lg2_ftz(fmaxf(xr.y, 1.17549435e-38f)));
                        const float2 xl = __fmul2_rn(x2[j], lg);
                        const float2 d = __fadd2_rn(x2[j], make_float2(-y.x, -y.y));
                        const float2 chi = __fmul2_rn(__fmul2_rn(d, r), d);
                        const float2 cm2 = dup2(cm), pm2 = make_float2(pm[2 * j], pm[2 * j + 1]);
                        // x (and so x log) is 0 on pad pixels / channels: only y and chi2 need the masks
                        float2 p0 = make_float2(pst[0][2 * j], pst[0][2 * j + 1]);
                        float2 p1 = make_float2(pst[1][2 * j], pst[1][2 * j + 1]);
                        float2 p2 = make_float2(pst[2][2 * j], pst[2][2 * j + 1]);
                        float2 p3 = make_float2(pst[3][2 * j], pst[3][2 * j + 1]);
                        p0 = __fadd2_rn(p0, x2[j]);
                        p1 = __ffma2_rn(cm2, y, p1);
                        p2 = __fadd2_rn(p2, xl);
                        p3 = __ffma2_rn(cm2, chi, p3);
                        pst[0][2 * j] = p0.x, pst[0][2 * j + 1] = p0.y;
                        pst[1][2 * j] = p1.x, pst[1][2 * j + 1] = p1.y;
                        pst[2][2 * j] = p2.x, pst[2][2 * j + 1] = p2.y;
                        pst[3][2 * j] = p3.x, pst[3][2 * j + 1] = p3.y;
                        c2[0] = __fadd2_rn(c2[0], x2[j]);
                        c2[1] = __ffma2_rn(pm2, y, c2[1]);
                        c2[2] = __fadd2_rn(c2[2], xl);
                        c2[3] = __ffma2_rn(pm2, chi, c2[3]);
                    }
#pragma unroll
                    for (int s = 0; s < NS4; ++s) cs[s] = c2[s].x + c2[s].y;
                } else {
                    TX xv[PPL];
                    TC gw[KP];
                    lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                    lds_gw<TC, KP>(gw, gs + (size_t)c * KP * sizeof(TC));
#pragma unroll
                    for (int s = 0; s < NS4; ++s) cs[s] = TC(0);
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        const TC x = (TC)xv[q];
                        TC y = gw[0] * h[0][q];
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y = fma(gw[kk], h[kk][q], y);
                        const TC r = Num<TC>::rcp(y);
                        const TC xl = x * log2_tab(max_nonneg(x * r, 2.2250738585072014e-308), ltab);
                        const TC d = x - y;
                        const TC chi = d * r * d;
                        pacc[0][q] += x;
                        pacc[1][q] = fma(cm, y, pacc[1][q]);
                        pacc[2][q] += xl;
                        pacc[3][q] = fma(cm, chi, pacc[3][q]);
                        cs[0] += x;
                        cs[1] = fma(pm[q], y, cs[1]);
                        cs[2] += xl;
                        cs[3] = fma(pm[q], chi, cs[3]);
                    }
                }
                // ---- per-channel sums of this stage: reduce-scatter, then one fp64 add per statistic ----
                reduce_scatter_step<16, NS4, TC>(cs, lane);
                if (rs_owner) {
                    part[ch] = nxt[ci] + (double)cs[0];
                    // the same channel of the next stage (of the next tile after the last stage); a slot the first
                    // tile has not reached yet holds nothing
                    const bool next_written = !first || st + 1 == NS;
                    nxt[ci] = next_written ? part[(st + 1 == NS ? 0 : st + 1) * G::CS + c] : 0.0;
                }
            }
            ring.consumer_release(pos, lane);
            if constexpr (FAST32) {
#pragma unroll
                for (int s = 0; s < NS4; ++s)
#pragma unroll
                    for (int q = 0; q < PPL; ++q) pacc[s][q] += (double)pst[s][q];
            }
        }

        // ---- per-pixel sums of this tile: the NSLOT warps that share a pixel hold different channels ----
#pragma unroll
        for (int t = 0; t < NS4; ++t)
#pragma unroll
            for (int q = 0; q < PPL; ++q) red[((size_t)slot * NS4 + t) * TILE_PX + lane_px + q] = pacc[t][q];
        named_bar_sync(1, N_CONSUMER_THREADS);
        if (threadIdx.x < TILE_PX) {
            const int j = tile * TILE_PX + threadIdx.x;
            double v[NS4];
#pragma unroll
            for (int t = 0; t < NS4; ++t) {
                v[t] = red[(size_t)t * TILE_PX + threadIdx.x];
#pragma unroll
                for (int sl = 1; sl < G::NSLOT; ++sl) v[t] += red[((size_t)sl * NS4 + t) * TILE_PX + threadIdx.x];
            }
            if (j < a.p_loc) {
                a.pixel_out[j] = v[0];
                a.pixel_out[(size_t)a.p_loc + j] = v[1];
                a.pixel_out[2 * (size_t)a.p_loc + j] = v[1] - v[0] + FIT_STATS_LN2 * v[2];
                a.pixel_out[3 * (size_t)a.p_loc + j] = v[3];
            }
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
    }
}

// channel_out[4][n] <- the CTA slots of `part` added in slot order; the KL row from the x, y and x log2(x/y) sums.
static __global__ void __launch_bounds__(256) fit_stats_fold_kernel(const double* part, int n_slots, int n, int n_pad,
                                                             double* channel_out) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    double s[FIT_STATS_NSTAT] = {0.0, 0.0, 0.0, 0.0};
    for (int b = 0; b < n_slots; ++b)
#pragma unroll
        for (int t = 0; t < FIT_STATS_NSTAT; ++t) s[t] += part[((size_t)b * FIT_STATS_NSTAT + t) * n_pad + c];
    channel_out[c] = s[0];
    channel_out[(size_t)n + c] = s[1];
    channel_out[2 * (size_t)n + c] = s[1] - s[0] + FIT_STATS_LN2 * s[2];
    channel_out[3 * (size_t)n + c] = s[3];
}

// Launch plan shared by the scratch query and the launch; one pixel tile (all its channels) per work item.
template <typename TX, typename TC, int KP>
static int fit_stats_do(const espm_state* st, double* pixel_out, double* channel_out, void* scratch,
                        int64_t* bytes_out, cudaStream_t stream) {
    using F = FitStatsGeom<TX, TC, KP>;
    using G = PassGeom<TX, TC>;
    void (*kern)(const FitStatsArgs) = fit_stats_kernel<TX, TC, KP>;
    // One CTA per SM with the deepest ring the shared memory holds (at most 8 stages, 128 KiB of X in flight per SM):
    // the kernel needs more registers than the 96 per thread of two CTAs per SM, and one CTA of 8 consumer warps has
    // 16 independent elements per lane and stage to hide the MUFU latency.
    SmemLimits lim;
    int rc = query_smem_limits(&lim);
    if (rc) return rc;
    const int depth = ring_depth(lim, 1, F::FIXED, F::TAIL, F::STRIDE, 8, "fit statistics kernel", st->kp);
    if (depth < 0) return depth;
    const int smem = F::FIXED + depth * F::STRIDE + F::TAIL;
    int occ = 0;
    if ((rc = kernel_fit(kern, smem, "fit statistics kernel", &occ))) return rc;
    const int cap = st->n_sms * occ;
    const int grid = st->n_tiles < cap ? st->n_tiles : cap;
    const int n_slots = grid * G::HALVES;
    const int64_t bytes = (int64_t)n_slots * FIT_STATS_NSTAT * st->n_pad * (int64_t)sizeof(double);
    if (bytes_out) {
        *bytes_out = bytes;
        return ESPM_OK;
    }
    FitStatsArgs a;
    a.Xt = st->Xt;
    a.GWc = st->GWc_cur;
    a.H = st->H_cur;
    a.pixel_out = pixel_out;
    a.part = reinterpret_cast<double*>(scratch);
    a.n = st->n;
    a.n_pad = st->n_pad;
    a.k = st->k;
    a.ldh = st->ldh;
    a.p_loc = st->p_loc;
    a.n_tiles = st->n_tiles;
    a.nstages_tile = st->n_pad / G::CS;
    a.depth = depth;
    a.log_shift = st->log_shift;
    fit_stats_kernel<TX, TC, KP><<<grid, XPASS_THREADS, smem, stream>>>(a);
    ESPM_CUDA_CHECK(cudaGetLastError());
    fit_stats_fold_kernel<<<(st->n + 255) / 256, 256, 0, stream>>>(a.part, n_slots, st->n, st->n_pad, channel_out);
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

template <typename TX, typename TC>
static int fit_stats_entry(const espm_state* st, double* pixel_out, double* channel_out, void* scratch,
                           int64_t* bytes_out, cudaStream_t stream) {
    ESPM_KP_SWITCH(st->kp, return fit_stats_do<TX, TC, KP>(st, pixel_out, channel_out, scratch, bytes_out, stream));
}

}  // namespace espm
