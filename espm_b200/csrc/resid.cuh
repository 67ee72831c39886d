// Products of the Pearson residual of a fitted model with a block of vectors (espm_resid_left / espm_resid_right,
// SmoothNMF.residual_components).
//
//   y[c][j] = sum_a g[c][a] h[a][j],   g = max(GW, ls), h = max(H, ls)      (the Y of KLdiv_loss, measures.py:493-497)
//   R[c][j] = (x[c][j] - y[c][j]) / sqrt(y[c][j])
//   left:   out[i][j] = sum_c R[c][j] Q[c][i]      (R^T Q, a contraction over channels, per pixel)
//   right:  out[c][i] = sum_j R[c][j] P[i][j]      (R P^T, a contraction over pixels, per channel)
//
// Q is (n, r) and P is (r, p_loc), fp64 on the device.  Each launch takes RB = RESID_RB columns of Q (rows of P); the
// entry points run the blocks of a wider r one after the other.  R is never stored: every element is rebuilt from x, g
// and h where it is used.  Per element: y (KP FMAs), one reciprocal square root (MUFU.RSQ in fp32, the library rsqrt
// in fp64), t = (x - y) rsqrt(y), and RB FMAs.
//
// resid_left_kernel   H pass order: the stages come from produce_tile_stages (xpass.cuh) instantiated at width
//                     KW = KA + RB, the operand beside the X chunk being the rows [g | Q block] that resid_rows_kernel
//                     writes to the caller's scratch (KA = KP rounded up to 16 bytes, so that both parts load with
//                     128-bit LDS; pad columns and the Q rows of pad channels are 0).  A lane owns PPL pixels of the
//                     tile (fp32 2, fp64 1) and holds their h; the sums of a stage (CPW channels) are formed in the
//                     compute type and
//                     added into fp64 per-pixel accumulators; once per tile the NSLOT warps that share a pixel are added
//                     in fp64, in slot order, through shared memory, as fit_stats_kernel does.  A pixel's result does
//                     not depend on the grid (a pixel shard computes the bits of the whole image).
// resid_right_kernel  W pass order: the stages come from produce_units (xpass.cuh) instantiated at width KW = KP + RB,
//                     the per-tile operand being the tile-major block [h; P block] that resid_tiles_kernel writes to the
//                     caller's scratch (h = ls and P = 0 on pad pixels).  Accumulators, runs and per-CTA slots follow
//                     w_info_kernel (winfo.cuh): a lane sums t P over its PPL pixels into CPW x RB accumulators (fp32:
//                     f32x2 over channel pairs); after RUN = 256 / PPL tiles (and at the end of a channel block) they
//                     are summed over the warp in fp64 into the CTA's slot, and resid_right_fold_kernel adds the slots
//                     of a channel in a fixed order.
// No atomics anywhere: two calls give identical bits.
//
// Pad channels have g = (1, 0, ...) and pad pixels h >= ls, so y > 0 everywhere and t is finite; their Q rows / P columns
// are 0, so they add nothing.
//
// fp32 accuracy.  The terms t Q and t P have mixed signs, so the bound is relative to the sum of their absolute values
// with |R[c][j]| replaced by a[c][j] = (x + y) / sqrt(y) >= |R[c][j]| (x - y cancels; the rounding of y does not):
//   |left error [i][j]|  <= E_L sum_c a[c][j] |Q[c][i]|,    |right error [c][i]| <= E_R sum_j a[c][j] |P[i][j]|.
// A term: y from KP FMAs of positive products (KP ulps, plus 2 for the fp32 rounding of g and h), MUFU.RSQ (2^-22.9),
// x - y, the product with rsqrt (2 ulps), the fp32 rounding of Q / P and the FMA (2 ulps): <= (KP + 6) 2^-24 + 2^-22.9.
// Left: a stage adds CPW <= 8 terms in series in fp32, then everything is fp64: E_L <= (KP + 14) 2^-24 + 2^-22.9 <=
// 1.93e-6 at KP = 16.  Right: a run adds m = RUN PPL = 256 terms in series: E_R <= (KP + 261) 2^-24 + 2^-22.9 <= 1.67e-5
// at KP = 16.  The fp64 remainder (warp sums, runs, slots) is below 1e-13 at any size.
#pragma once
#include <cstring>

#include "xpass.cuh"

namespace espm {

// Columns of Q (rows of P) per launch.  16 keeps every instance free of local-memory spills up to kp = 16 in every
// (storage, arithmetic) pair (profiles/residual_components_ptxas.md); a rank-4 call (r = 14) is one launch per product.
constexpr int RESID_RB = 16;

struct ResidArgs {
    const void* Xt;
    const void* GWQ;      // left: [n_pad][KA + RB] rows [g | Q block]
    const void* H;        // left: H_cur [k][ldh] from local pixel 0
    const void* GWc;      // right: [n_pad][KP], max(GW, ls) on the real entries
    const void* Ht;       // right: [n_tiles][KP + RB][TILE_PX], written by resid_tiles_kernel
    double* out;          // left: [rows][p_loc] (row stride p_loc); right: CTA slots [nr][n_pad][RB]
    int rows;             // left: columns of this block that are written (<= RB)
    int n_pad, k, ldh, p_loc, n_tiles, nstages_tile, w_upc, depth;
    double log_shift;
};

__device__ __forceinline__ float resid_rsqrt(float y) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
    return r;
}
__device__ __forceinline__ double resid_rsqrt(double y) { return rsqrt(y); }

// ------------------------------------------------------------------------------------------------
// Left product
// ------------------------------------------------------------------------------------------------
template <typename TX, typename TC, int KP, int RB>
struct ResidLeftGeom {
    static constexpr int KA = (KP * (int)sizeof(TC) + 15) / 16 * 16 / (int)sizeof(TC);   // g part of a row, padded
    static constexpr int KW = KA + RB;                                                    // row width
    using S = XPassSmem<TX, TC, KW, false>;
    static constexpr int STRIDE = S::H_STRIDE;                     // X chunk + CS rows [g | Q]
    static constexpr int CS = S::G::CS;
    static constexpr int X_BYTES = S::X_BYTES;
    // pixels per lane: fp32 a packed f32x2 pair; fp64 one (two need more than the 168 registers of one CTA per SM at
    // kp >= 4 and spill)
    static constexpr int PPL = sizeof(TC) == 4 ? 2 : 1;
    static constexpr int HALVES = TILE_PX / (32 * PPL);
    static constexpr int NSLOT = N_CONSUMER_WARPS / HALVES;
    static constexpr int CPW = CS / NSLOT;                         // channels per warp per stage
    static constexpr int FIXED = S::BAR_BYTES + S::MISC_BYTES;
    static constexpr int TAIL = NSLOT * RB * TILE_PX * (int)sizeof(double);   // per-tile slot reduction
    static_assert(CPW * NSLOT == CS && (RB * (int)sizeof(TC)) % 16 == 0, "geometry");
};

// GWQ[c][0:KA] = g row (0 past KP), GWQ[c][KA + i] = Q[c][col0 + i] for real channels and i < rows, else 0.
template <typename TC, int KP, int RB>
static __global__ void __launch_bounds__(256) resid_rows_kernel(const TC* GWc, const double* Q, int ldq, int col0,
                                                                int rows, int n, int n_pad, TC* GWQ) {
    constexpr int KA = ResidLeftGeom<float, TC, KP, RB>::KA, KW = KA + RB;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_pad * KW) return;
    const int c = (int)(idx / KW), col = (int)(idx - (long long)c * KW);
    TC v = TC(0);
    if (col < KA) {
        if (col < KP) v = GWc[(size_t)c * KP + col];
    } else if (c < n && col - KA < rows) {
        v = (TC)Q[(size_t)c * ldq + col0 + col - KA];
    }
    GWQ[idx] = v;
}

template <typename TX, typename TC, int KP, int RB>
__global__ void __launch_bounds__(XPASS_THREADS, 1) resid_left_kernel(const ResidArgs a) {
    using L = ResidLeftGeom<TX, TC, KP, RB>;
    constexpr int PPL = L::PPL, CPW = L::CPW, NSLOT = L::NSLOT, KA = L::KA, KW = L::KW;
    constexpr bool FAST32 = sizeof(TC) == 4;
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<L::STRIDE> ring(smem, a.depth, L::FIXED);
    double* red = reinterpret_cast<double*>(smem + L::FIXED + (size_t)a.depth * L::STRIDE);   // [NSLOT][RB][TILE_PX]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) ring.init();
    __syncthreads();
    const int NS = a.nstages_tile;

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            const uint64_t pol_x = l2_policy_evict_first();
            const uint64_t pol_gw = l2_policy_evict_last();
            typename Ring<L::STRIDE>::Pos pos{0, 0u};
            for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x)
                produce_tile_stages<TX, TC, KW, &ResidArgs::GWQ>(ring, pos, pol_x, pol_gw, a, tile, 0, NS, false);
        }
        return;
    }

    const int half = warp % L::HALVES, slot = warp / L::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;
    const TC ls = (TC)a.log_shift;
    const TC* Hc = reinterpret_cast<const TC*>(a.H);
    typename Ring<L::STRIDE>::Pos pos{0, 0u};

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const int px0 = tile * TILE_PX + lane_px;
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, Hc, a.ldh, a.k, px0);
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
#pragma unroll
            for (int q = 0; q < PPL; ++q)
                if (kk < a.k) h[kk][q] = Num<TC>::vmax(h[kk][q], ls);
        double acc[RB][PPL];
#pragma unroll
        for (int i = 0; i < RB; ++i)
#pragma unroll
            for (int q = 0; q < PPL; ++q) acc[i][q] = 0.0;

        for (int st = 0; st < NS; ++st, ring.next(pos)) {
            ring.consumer_wait(pos);
            const unsigned char* xs = ring.stage(pos.slot);
            const unsigned char* gs = xs + L::X_BYTES;
            if constexpr (FAST32) {
                float2 h2[KP];
#pragma unroll
                for (int kk = 0; kk < KP; ++kk) h2[kk] = make_float2(h[kk][0], h[kk][1]);
                float2 s2[RB];   // this stage's sums of the lane's pixel pair
#pragma unroll
                for (int i = 0; i < RB; ++i) s2[i] = make_float2(0.f, 0.f);
#pragma unroll
                for (int ci = 0; ci < CPW; ++ci) {
                    const int c = slot + ci * NSLOT;
                    TX xv[2];
                    lds_vec<TX, 2>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                    const unsigned char* row = gs + (size_t)c * KW * sizeof(float);
                    float g[KA];
                    lds_gw<float, KA>(g, row);
                    float2 y = __fmul2_rn(dup2(g[0]), h2[0]);
#pragma unroll
                    for (int kk = 1; kk < KP; ++kk) y = __ffma2_rn(dup2(g[kk]), h2[kk], y);
                    const float2 d = __fadd2_rn(make_float2((float)xv[0], (float)xv[1]), make_float2(-y.x, -y.y));
                    const float2 t = __fmul2_rn(d, make_float2(resid_rsqrt(y.x), resid_rsqrt(y.y)));
                    float qv[RB];
                    lds_gw<float, RB>(qv, row + KA * sizeof(float));
#pragma unroll
                    for (int i = 0; i < RB; ++i) s2[i] = __ffma2_rn(dup2(qv[i]), t, s2[i]);
                }
                ring.consumer_release(pos, lane);
#pragma unroll
                for (int i = 0; i < RB; ++i) {
                    acc[i][0] += (double)s2[i].x;
                    acc[i][1] += (double)s2[i].y;
                }
            } else {
#pragma unroll
                for (int ci = 0; ci < CPW; ++ci) {
                    const int c = slot + ci * NSLOT;
                    TX xv[PPL];
                    lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                    const unsigned char* row = gs + (size_t)c * KW * sizeof(TC);
                    TC g[KA];
                    lds_gw<TC, KA>(g, row);
                    TC t[PPL];
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        TC y = g[0] * h[0][q];
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y = fma(g[kk], h[kk][q], y);
                        t[q] = ((TC)xv[q] - y) * resid_rsqrt(y);
                    }
                    TC qv[RB];
                    lds_gw<TC, RB>(qv, row + KA * sizeof(TC));
#pragma unroll
                    for (int i = 0; i < RB; ++i)
#pragma unroll
                        for (int q = 0; q < PPL; ++q) acc[i][q] = fma((double)qv[i], (double)t[q], acc[i][q]);
                }
                ring.consumer_release(pos, lane);
            }
        }

        // ---- per-pixel sums of this tile: the NSLOT warps that share a pixel hold different channels ----
#pragma unroll
        for (int i = 0; i < RB; ++i)
#pragma unroll
            for (int q = 0; q < PPL; ++q) red[((size_t)slot * RB + i) * TILE_PX + lane_px + q] = acc[i][q];
        named_bar_sync(1, N_CONSUMER_THREADS);
        for (int idx = threadIdx.x; idx < RB * TILE_PX; idx += N_CONSUMER_THREADS) {
            const int i = idx / TILE_PX, px = idx - i * TILE_PX;
            const int j = tile * TILE_PX + px;
            double v = red[(size_t)i * TILE_PX + px];
#pragma unroll
            for (int sl = 1; sl < NSLOT; ++sl) v += red[((size_t)sl * RB + i) * TILE_PX + px];
            if (i < a.rows && j < a.p_loc) a.out[(size_t)i * a.p_loc + j] = v;
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
    }
}

// ------------------------------------------------------------------------------------------------
// Right product
// ------------------------------------------------------------------------------------------------
template <typename TX, typename TC, int KP, int RB>
struct ResidRightGeom {
    static constexpr bool FAST32 = sizeof(TC) == 4;
    static constexpr int KW = KP + RB;                               // rows of a tile block [h; P]
    static constexpr int PPL = (FAST32 && KP <= 4) ? 4 : 2;
    static constexpr int HALVES = TILE_PX / (32 * PPL);
    static constexpr int NSLOT = N_CONSUMER_WARPS / HALVES;
    static constexpr int CPW = FAST32 ? (KP <= 4 ? 4 : 2) : (KP <= 4 ? 2 : 1);
    static constexpr int CS = NSLOT * CPW;                           // channels per stage (divides n_pad, a multiple of 32)
    static constexpr int RUN = 256 / PPL;                            // tiles per fp32 run
    static constexpr int X_BYTES = CS * TILE_PX * (int)sizeof(TX);
    static constexpr int H_BYTES = KW * TILE_PX * (int)sizeof(TC);
    static constexpr int STRIDE = X_BYTES + H_BYTES;
    static constexpr int FIXED = 256 + 128;                          // barriers + misc, as XPassSmem
    static constexpr int GW_BYTES = (CS * KP * (int)sizeof(TC) + 127) / 128 * 128;
    static constexpr int ACC_BYTES = HALVES * CS * RB * (int)sizeof(double);
    static constexpr int TAIL = GW_BYTES + ACC_BYTES;
    static_assert(!FAST32 || CPW % 2 == 0, "fp32 packs channel pairs");
    static_assert(32 % CS == 0 && X_BYTES % 16 == 0 && H_BYTES % 16 == 0, "geometry");
};

// Ht[tile][0:KP][128] = max(H_cur, ls) (rows >= k are 0, pad pixels hold ls); Ht[tile][KP + i][128] = P[row0 + i][j]
// for real pixels and i < rows, else 0.
template <typename TC, int KP, int RB>
static __global__ void __launch_bounds__(256) resid_tiles_kernel(const TC* H, int ldh, int k, const double* P, int ldp,
                                                                 int row0, int rows, int p_loc, int p_pad, TC ls,
                                                                 TC* Ht) {
    constexpr int KW = KP + RB;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)KW * p_pad) return;
    const int kk = (int)(i / p_pad), j = (int)(i % p_pad);
    TC v = TC(0);
    if (kk < KP) {
        if (kk < k) v = j < p_loc ? Num<TC>::vmax(H[(size_t)kk * ldh + j], ls) : ls;
    } else if (kk - KP < rows && j < p_loc) {
        v = (TC)P[(size_t)(row0 + kk - KP) * ldp + j];
    }
    Ht[((size_t)(j / TILE_PX) * KW + kk) * TILE_PX + (j % TILE_PX)] = v;
}

template <typename TX, typename TC, int KP, int RB>
__global__ void __launch_bounds__(XPASS_THREADS, 1) resid_right_kernel(const ResidArgs a) {
    using I = ResidRightGeom<TX, TC, KP, RB>;
    constexpr int PPL = I::PPL, CPW = I::CPW, NSLOT = I::NSLOT;
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<I::STRIDE> ring(smem, a.depth, I::FIXED);
    unsigned char* tail0 = smem + I::FIXED + (size_t)a.depth * I::STRIDE;
    TC* gwbuf = reinterpret_cast<TC*>(tail0);                                      // [CS][KP]
    double* acc64 = reinterpret_cast<double*>(tail0 + I::GW_BYTES);                // [HALVES][CS][RB]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const UnitRange units(a);
    const int n_units = units.n_units;

    if (threadIdx.x == 0) ring.init();
    for (int i = threadIdx.x; i < I::HALVES * I::CS * RB; i += blockDim.x) acc64[i] = 0.0;
    __syncthreads();

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            typename Ring<I::STRIDE>::Pos pos{0, 0u};
            produce_units<TX, TC, I::KW, I::CS>(ring, pos, units, a);
        }
        return;
    }

    const int half = warp % I::HALVES, slot = warp / I::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;

    // run accumulators: fp32 (c_{2i}, c_{2i+1}) channel pairs, fp64 one channel each
    float2 acc2[I::FAST32 ? CPW / 2 : 1][I::FAST32 ? RB : 1];
    double accd[I::FAST32 ? 1 : CPW][I::FAST32 ? 1 : RB];
    auto zero = [&]() {
#pragma unroll
        for (int i = 0; i < RB; ++i) {
            if constexpr (I::FAST32) {
#pragma unroll
                for (int pi = 0; pi < CPW / 2; ++pi) acc2[pi][i] = make_float2(0.f, 0.f);
            } else {
#pragma unroll
                for (int ci = 0; ci < CPW; ++ci) accd[ci][i] = 0.0;
            }
        }
    };
    zero();

    // ends a run: warp sums in fp64 into this half's slot of the CTA
    auto end_run = [&]() {
#pragma unroll
        for (int ci = 0; ci < CPW; ++ci)
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                double v;
                if constexpr (I::FAST32) v = (double)(ci % 2 == 0 ? acc2[ci / 2][i].x : acc2[ci / 2][i].y);
                else v = accd[ci][i];
                v = warp_sum(v);
                __syncwarp();
                if (lane == 0) acc64[((size_t)half * I::CS + slot + ci * NSLOT) * RB + i] += v;
            }
        zero();
    };

    // ends the channel block `cb` of this CTA: part[slot of this CTA in cb][channels of cb][RB]
    auto flush = [&](int cb) {
        named_bar_sync(1, N_CONSUMER_THREADS);
        const int ps = blockIdx.x - w_first_cta(cb, a.n_tiles, a.w_upc);
        double* out = a.out + ((size_t)ps * a.n_pad + (size_t)cb * I::CS) * RB;
        for (int i = threadIdx.x; i < I::CS * RB; i += N_CONSUMER_THREADS) {
            double v = acc64[i];
            if constexpr (I::HALVES == 2) v += acc64[(size_t)I::CS * RB + i];
            out[i] = v;
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
        for (int i = threadIdx.x; i < I::HALVES * I::CS * RB; i += N_CONSUMER_THREADS) acc64[i] = 0.0;
    };

    auto load_gw = [&](int cb) {
        const TC* src = reinterpret_cast<const TC*>(a.GWc) + (size_t)cb * I::CS * KP;
        for (int i = threadIdx.x; i < I::CS * KP; i += N_CONSUMER_THREADS) gwbuf[i] = src[i];
        named_bar_sync(1, N_CONSUMER_THREADS);
    };

    typename Ring<I::STRIDE>::Pos pos{0, 0u};
    int cb = units.cb0, tile = units.tile0, run = 0;
    if (n_units > 0) load_gw(cb);
    for (int u = 0; u < n_units; ++u, ring.next(pos)) {
        ring.consumer_wait(pos);
        const unsigned char* xs = ring.stage(pos.slot);
        const TC* hs = reinterpret_cast<const TC*>(xs + I::X_BYTES);
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, hs, TILE_PX, a.k, lane_px);

        if constexpr (I::FAST32) {
            // t of the lane's channel pairs and pixels, then the RB rows of P one at a time
            float2 t2[CPW / 2][PPL];
#pragma unroll
            for (int pi = 0; pi < CPW / 2; ++pi) {
                const int c0 = slot + 2 * pi * NSLOT, c1 = c0 + NSLOT;
                float g0[KP], g1[KP];
                lds_gw<float, KP>(g0, gwbuf + (size_t)c0 * KP);
                lds_gw<float, KP>(g1, gwbuf + (size_t)c1 * KP);
                TX va[PPL], vb[PPL];
                lds_vec<TX, PPL>(va, xs + ((size_t)c0 * TILE_PX + lane_px) * sizeof(TX));
                lds_vec<TX, PPL>(vb, xs + ((size_t)c1 * TILE_PX + lane_px) * sizeof(TX));
#pragma unroll
                for (int q = 0; q < PPL; ++q) {
                    float2 y = __fmul2_rn(make_float2(g0[0], g1[0]), dup2(h[0][q]));
#pragma unroll
                    for (int kk = 1; kk < KP; ++kk) y = __ffma2_rn(make_float2(g0[kk], g1[kk]), dup2(h[kk][q]), y);
                    const float2 d = __fadd2_rn(make_float2((float)va[q], (float)vb[q]), make_float2(-y.x, -y.y));
                    t2[pi][q] = __fmul2_rn(d, make_float2(resid_rsqrt(y.x), resid_rsqrt(y.y)));
                }
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                float pv[PPL];
                lds_vec<float, PPL>(pv, hs + (size_t)(KP + i) * TILE_PX + lane_px);
#pragma unroll
                for (int pi = 0; pi < CPW / 2; ++pi)
#pragma unroll
                    for (int q = 0; q < PPL; ++q) acc2[pi][i] = __ffma2_rn(t2[pi][q], dup2(pv[q]), acc2[pi][i]);
            }
        } else {
            TC t[CPW][PPL];
#pragma unroll
            for (int ci = 0; ci < CPW; ++ci) {
                const int c = slot + ci * NSLOT;
                TC g[KP];
                lds_gw<TC, KP>(g, gwbuf + (size_t)c * KP);
                TX xv[PPL];
                lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
#pragma unroll
                for (int q = 0; q < PPL; ++q) {
                    TC y = g[0] * h[0][q];
#pragma unroll
                    for (int kk = 1; kk < KP; ++kk) y = fma(g[kk], h[kk][q], y);
                    t[ci][q] = ((TC)xv[q] - y) * resid_rsqrt(y);
                }
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                TC pv[PPL];
                lds_vec<TC, PPL>(pv, hs + (size_t)(KP + i) * TILE_PX + lane_px);
#pragma unroll
                for (int ci = 0; ci < CPW; ++ci)
#pragma unroll
                    for (int q = 0; q < PPL; ++q) accd[ci][i] = fma(t[ci][q], pv[q], accd[ci][i]);
            }
        }
        ring.consumer_release(pos, lane);
        const bool block_end = ++tile == a.n_tiles || u + 1 == n_units;
        if (++run == I::RUN || block_end) {
            end_run();
            run = 0;
        }
        if (block_end) {
            flush(cb);
            if (u + 1 < n_units) {
                tile = 0;
                ++cb;
                load_gw(cb);   // the barrier of flush: every warp is done with gwbuf and acc64 is zero
            }
        }
    }
}

// out[c][col0 + i] (row stride ldo) = the CTA slots of channel c, added in slot order, for i < rows.
template <int RB>
static __global__ void __launch_bounds__(256) resid_right_fold_kernel(const double* part, int n_tiles, int upc, int cs,
                                                                      int n, int n_pad, int rows, double* out, int ldo,
                                                                      int col0) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n * rows) return;
    const int c = (int)(idx / rows), i = (int)(idx - (long long)c * rows);
    const int cb = c / cs;
    const int ns = w_last_cta(cb, n_tiles, upc) - w_first_cta(cb, n_tiles, upc) + 1;
    double s = 0.0;
    for (int ps = 0; ps < ns; ++ps) s += part[((size_t)ps * n_pad + c) * RB + i];
    out[(size_t)c * ldo + col0 + i] = s;
}

// ------------------------------------------------------------------------------------------------
// Launch plans, shared by the scratch queries and the launches.  r columns run as ceil(r / RB) blocks.
// Left scratch: the [g | Q block] rows.  Right scratch: the tile blocks [h; P block], then the CTA slots.
// ------------------------------------------------------------------------------------------------
template <typename TX, typename TC, int KP>
static int resid_left_do(const espm_state* st, const double* Q, int r, double* out, void* scratch, int64_t* bytes_out,
                         cudaStream_t stream) {
    constexpr int RB = RESID_RB;
    using L = ResidLeftGeom<TX, TC, KP, RB>;
    const size_t rows_bytes = ((size_t)st->n_pad * L::KW * sizeof(TC) + 255) / 256 * 256;
    if (bytes_out) {
        *bytes_out = (int64_t)rows_bytes;
        return ESPM_OK;
    }
    void (*kern)(const ResidArgs) = resid_left_kernel<TX, TC, KP, RB>;
    SmemLimits lim;
    int rc = query_smem_limits(&lim);
    if (rc) return rc;
    // one CTA per SM (the RB x PPL fp64 accumulators do not fit the registers of two) with the deepest ring, as
    // fit_stats_kernel
    const int depth = ring_depth(lim, 1, L::FIXED, L::TAIL, L::STRIDE, 8, "residual left product", st->kp);
    if (depth < 0) return depth;
    const int smem = L::FIXED + depth * L::STRIDE + L::TAIL;
    int occ = 0;
    if ((rc = kernel_fit(kern, smem, "residual left product", &occ))) return rc;
    const int cap = st->n_sms * occ;
    const int grid = st->n_tiles < cap ? st->n_tiles : cap;
    TC* GWQ = reinterpret_cast<TC*>(scratch);
    ResidArgs a;
    memset(&a, 0, sizeof(a));
    a.Xt = st->Xt;
    a.GWQ = GWQ;
    a.H = st->H_cur;
    a.n_pad = st->n_pad;
    a.k = st->k;
    a.ldh = st->ldh;
    a.p_loc = st->p_loc;
    a.n_tiles = st->n_tiles;
    a.nstages_tile = st->n_pad / L::CS;
    a.depth = depth;
    a.log_shift = st->log_shift;
    const long long nrow = (long long)st->n_pad * L::KW;
    for (int col0 = 0; col0 < r; col0 += RB) {
        const int rows = r - col0 < RB ? r - col0 : RB;
        resid_rows_kernel<TC, KP, RB><<<(unsigned)((nrow + 255) / 256), 256, 0, stream>>>(
            reinterpret_cast<const TC*>(st->GWc_cur), Q, r, col0, rows, st->n, st->n_pad, GWQ);
        ESPM_CUDA_CHECK(cudaGetLastError());
        a.out = out + (size_t)col0 * st->p_loc;
        a.rows = rows;
        resid_left_kernel<TX, TC, KP, RB><<<grid, XPASS_THREADS, smem, stream>>>(a);
        ESPM_CUDA_CHECK(cudaGetLastError());
    }
    return ESPM_OK;
}

template <typename TX, typename TC, int KP>
static int resid_right_do(const espm_state* st, const double* P, int r, double* out, void* scratch, int64_t* bytes_out,
                          cudaStream_t stream) {
    constexpr int RB = RESID_RB;
    using I = ResidRightGeom<TX, TC, KP, RB>;
    void (*kern)(const ResidArgs) = resid_right_kernel<TX, TC, KP, RB>;
    SmemLimits lim;
    int rc = query_smem_limits(&lim);
    if (rc) return rc;
    // about 96 KiB of X in flight per SM, as w_info_kernel
    const int want = 98304 / I::X_BYTES;
    const int depth = ring_depth(lim, 1, I::FIXED, I::TAIL, I::STRIDE, want < 8 ? want : 8, "residual right product",
                                 st->kp);
    if (depth < 0) return depth;
    const int smem = I::FIXED + depth * I::STRIDE + I::TAIL;
    const int NS = st->n_pad / I::CS;
    int upc = 0, grid = 0, nr = 0;
    plan_w_units(NS, st->n_tiles, st->n_sms, &upc, &grid, &nr);
    const size_t ht_bytes = ((size_t)st->n_tiles * I::H_BYTES + 255) / 256 * 256;
    const size_t part_bytes = (size_t)nr * st->n_pad * RB * sizeof(double);
    if (bytes_out) {
        *bytes_out = (int64_t)(ht_bytes + part_bytes);
        return ESPM_OK;
    }
    int occ = 0;
    if ((rc = kernel_fit(kern, smem, "residual right product", &occ))) return rc;
    TC* Ht = reinterpret_cast<TC*>(scratch);
    ResidArgs a;
    memset(&a, 0, sizeof(a));
    a.Xt = st->Xt;
    a.GWc = st->GWc_cur;
    a.Ht = Ht;
    a.out = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(scratch) + ht_bytes);
    a.n_pad = st->n_pad;
    a.k = st->k;
    a.n_tiles = st->n_tiles;
    a.nstages_tile = NS;
    a.w_upc = upc;
    a.depth = depth;
    const long long nh = (long long)I::KW * st->n_tiles * TILE_PX;
    for (int row0 = 0; row0 < r; row0 += RB) {
        const int rows = r - row0 < RB ? r - row0 : RB;
        resid_tiles_kernel<TC, KP, RB><<<(unsigned)((nh + 255) / 256), 256, 0, stream>>>(
            reinterpret_cast<const TC*>(st->H_cur), st->ldh, st->k, P, st->p_loc, row0, rows, st->p_loc,
            st->n_tiles * TILE_PX, (TC)st->log_shift, Ht);
        ESPM_CUDA_CHECK(cudaGetLastError());
        resid_right_kernel<TX, TC, KP, RB><<<grid, XPASS_THREADS, smem, stream>>>(a);
        ESPM_CUDA_CHECK(cudaGetLastError());
        const long long nf = (long long)st->n * rows;
        resid_right_fold_kernel<RB><<<(unsigned)((nf + 255) / 256), 256, 0, stream>>>(
            a.out, st->n_tiles, upc, I::CS, st->n, st->n_pad, rows, out, r, row0);
        ESPM_CUDA_CHECK(cudaGetLastError());
    }
    return ESPM_OK;
}

template <typename TX, typename TC>
static int resid_left_entry(const espm_state* st, const double* Q, int r, double* out, void* scratch,
                            int64_t* bytes_out, cudaStream_t stream) {
    ESPM_KP_SWITCH(st->kp, return resid_left_do<TX, TC, KP>(st, Q, r, out, scratch, bytes_out, stream));
}

template <typename TX, typename TC>
static int resid_right_entry(const espm_state* st, const double* P, int r, double* out, void* scratch,
                             int64_t* bytes_out, cudaStream_t stream) {
    ESPM_KP_SWITCH(st->kp, return resid_right_do<TX, TC, KP>(st, P, r, out, scratch, bytes_out, stream));
}

}  // namespace espm
