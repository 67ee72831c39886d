// Poisson information of the phases, per channel, in one streaming pass (espm_phase_info, SmoothNMF.phase_uncertainty).
//
//   y[c][j]    = sum_a g[c][a] h[a][j],   g = max(GW, ls), h = max(H, ls)      (the Y of KLdiv_loss, measures.py:493-497)
//   A_c[a][b]  = sum_j x[c][j] h[a][j] h[b][j] / y[c][j]^2
//
// The information of vec(W) is F[(e,a),(f,b)] = sum_c G_ce G_cf A_c[a][b]; the host assembles it from A (host.py).
//
// Three launches:
//   w_info_tiles_kernel  Ht[tile][KP][128] = max(H_cur, ls) tile-major in the caller's scratch (rows >= k are 0, pad
//                        pixels hold ls, so y > 0 there and their x = 0 gives w = x r r = 0);
//   w_info_kernel        the sums, in W pass order: the stages come from produce_units (xpass.cuh); the GW rows of the
//                        channel block sit in shared memory while the block is processed;
//   w_info_fold_kernel   A[tri(a, b)][c] = sum of the CTA slots of channel c, in slot order.
//
// Work of a lane: PPL pixels of the tile (HALVES warps cover a 128-px row) x CPW channels (warp slot s owns channels
// s, s + NSLOT, ...).  Per element: y (KP FMA), one reciprocal r (MUFU.RCP in fp32, the Newton reciprocal of Num<double>
// in fp64), w = x r r, u_a = w h_a (KP multiplies) and the KP (KP + 1) / 2 FMAs u_a h_b.  The lane sums its pixels into
// CPW x NT accumulators; fp32 packs them over channel pairs (f32x2: FFMA2 on (c, c + NSLOT)), so CPW x NT registers hold
// them.  The geometry follows kp: fp32 PPL = 4, CPW = 4 up to kp = 4, PPL = 2, CPW = 2 above; fp64 PPL = 2, CPW = 2 up
// to kp = 4, 1 above.  No instance spills for kp <= 8; kp 12 and 16 do (profiles/phase_uncertainty_ptxas.md).
//
// Runs: after RUN = 256 / PPL tiles of a channel block (and at the end of the block) every accumulator is converted to
// fp64, summed over the warp (fixed butterfly) and added by lane 0 to the CTA's fp64 slot acc64[half][c][t] in shared
// memory.  When the CTA leaves a channel block it writes acc64 (halves added in order) to its slot of `part`
// (slot = CTA - first CTA of the block, as the W pass).  No atomics: two calls give identical bits.
//
// fp32 accuracy: every term x h_a h_b / y^2 is >= 0, so a run partial of m = RUN PPL = 256 terms summed in series has a
// relative error <= (m - 1) 2^-24 = 1.52e-5, plus the error of a term: y from KP positive FMAs (KP ulps), doubled by
// r^2, one MUFU.RCP.FTZ ulp, and w, u, the final product (5 ulps), i.e. (2 KP + 6) 2^-24 <= 2.2e-6 at KP = 16.  The rest
// is fp64 (the warp sum, the runs, the slots: < 1e-13 at any size), so the bound, 1.74e-5, holds at 2048 channels x 512^2
// pixels and at any larger image.
#pragma once
#include "hinfo.cuh"

namespace espm {

struct WInfoArgs {
    const void* Xt;
    const void* GWc;      // [n_pad][KP], max(GW, ls) on the real entries
    const void* Ht;       // [n_tiles][KP][TILE_PX], written by w_info_tiles_kernel
    double* part;         // [nr][n_pad][NT] CTA slots
    int n_pad, k, n_tiles, nstages_tile, w_upc, depth;
};

template <typename TX, typename TC, int KP>
struct WInfoGeom {
    static constexpr bool FAST32 = sizeof(TC) == 4;
    static constexpr int PPL = (FAST32 && KP <= 4) ? 4 : 2;
    static constexpr int HALVES = TILE_PX / (32 * PPL);
    static constexpr int NSLOT = N_CONSUMER_WARPS / HALVES;
    static constexpr int CPW = FAST32 ? (KP <= 4 ? 4 : 2) : (KP <= 4 ? 2 : 1);
    static constexpr int CS = NSLOT * CPW;                           // channels per stage (divides n_pad, a multiple of 32)
    static constexpr int NT = KP * (KP + 1) / 2;
    static constexpr int RUN = 256 / PPL;                            // tiles per fp32 run
    static constexpr int X_BYTES = CS * TILE_PX * (int)sizeof(TX);
    static constexpr int H_BYTES = KP * TILE_PX * (int)sizeof(TC);
    static constexpr int STRIDE = X_BYTES + H_BYTES;
    static constexpr int FIXED = 256 + 128;                          // barriers + misc, as XPassSmem
    static constexpr int GW_BYTES = (CS * KP * (int)sizeof(TC) + 127) / 128 * 128;
    static constexpr int ACC_BYTES = HALVES * CS * NT * (int)sizeof(double);
    static constexpr int TAIL = GW_BYTES + ACC_BYTES;
    static_assert(!FAST32 || CPW % 2 == 0, "fp32 packs channel pairs");
    static_assert(32 % CS == 0 && X_BYTES % 16 == 0 && H_BYTES % 16 == 0, "geometry");
};

template <typename TC, int KP>
static __global__ void __launch_bounds__(256) w_info_tiles_kernel(const TC* H, int ldh, int k, int p_loc, int p_pad,
                                                                  TC ls, TC* Ht) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)KP * p_pad) return;
    const int kk = (int)(i / p_pad), j = (int)(i % p_pad);
    TC v = TC(0);
    if (kk < k) v = j < p_loc ? Num<TC>::vmax(H[(size_t)kk * ldh + j], ls) : ls;
    Ht[((size_t)(j / TILE_PX) * KP + kk) * TILE_PX + (j % TILE_PX)] = v;
}

template <typename TX, typename TC, int KP>
__global__ void __launch_bounds__(XPASS_THREADS, 1) w_info_kernel(const WInfoArgs a) {
    using I = WInfoGeom<TX, TC, KP>;
    constexpr int PPL = I::PPL, CPW = I::CPW, NT = I::NT, NSLOT = I::NSLOT;
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<I::STRIDE> ring(smem, a.depth, I::FIXED);
    unsigned char* tail0 = smem + I::FIXED + (size_t)a.depth * I::STRIDE;
    TC* gwbuf = reinterpret_cast<TC*>(tail0);                                      // [CS][KP]
    double* acc64 = reinterpret_cast<double*>(tail0 + I::GW_BYTES);                // [HALVES][CS][NT]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const UnitRange units(a);
    const int n_units = units.n_units, cb0 = units.cb0, tile0 = units.tile0;

    if (threadIdx.x == 0) ring.init();
    for (int i = threadIdx.x; i < I::HALVES * I::CS * NT; i += blockDim.x) acc64[i] = 0.0;
    __syncthreads();

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            typename Ring<I::STRIDE>::Pos pos{0, 0u};
            produce_units<TX, TC, KP, I::CS>(ring, pos, units, a);
        }
        return;
    }

    const int half = warp % I::HALVES, slot = warp / I::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;

    // run accumulators: fp32 (c_{2i}, c_{2i+1}) channel pairs, fp64 one channel each
    float2 acc2[I::FAST32 ? CPW / 2 : 1][I::FAST32 ? NT : 1];
    double accd[I::FAST32 ? 1 : CPW][I::FAST32 ? 1 : NT];
    auto zero = [&]() {
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            if constexpr (I::FAST32) {
#pragma unroll
                for (int i = 0; i < CPW / 2; ++i) acc2[i][t] = make_float2(0.f, 0.f);
            } else {
#pragma unroll
                for (int i = 0; i < CPW; ++i) accd[i][t] = 0.0;
            }
        }
    };
    zero();

    // ends a run: warp sums in fp64 into this half's slot of the CTA
    auto end_run = [&]() {
#pragma unroll
        for (int ci = 0; ci < CPW; ++ci)
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                double v;
                if constexpr (I::FAST32) v = (double)(ci % 2 == 0 ? acc2[ci / 2][t].x : acc2[ci / 2][t].y);
                else v = accd[ci][t];
                v = warp_sum(v);
                __syncwarp();   // one value at a time: converting all of them first spills at kp = 8
                if (lane == 0) acc64[((size_t)half * I::CS + slot + ci * NSLOT) * NT + t] += v;
            }
        zero();
    };

    // ends the channel block `cb` of this CTA: part[slot of this CTA in cb][channels of cb][NT]
    auto flush = [&](int cb) {
        named_bar_sync(1, N_CONSUMER_THREADS);
        const int ps = blockIdx.x - w_first_cta(cb, a.n_tiles, a.w_upc);
        double* out = a.part + ((size_t)ps * a.n_pad + (size_t)cb * I::CS) * NT;
        for (int i = threadIdx.x; i < I::CS * NT; i += N_CONSUMER_THREADS) {
            double v = acc64[i];
            if constexpr (I::HALVES == 2) v += acc64[(size_t)I::CS * NT + i];
            out[i] = v;
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
        for (int i = threadIdx.x; i < I::HALVES * I::CS * NT; i += N_CONSUMER_THREADS) acc64[i] = 0.0;
    };

    auto load_gw = [&](int cb) {
        const TC* src = reinterpret_cast<const TC*>(a.GWc) + (size_t)cb * I::CS * KP;
        for (int i = threadIdx.x; i < I::CS * KP; i += N_CONSUMER_THREADS) gwbuf[i] = src[i];
        named_bar_sync(1, N_CONSUMER_THREADS);
    };

    typename Ring<I::STRIDE>::Pos pos{0, 0u};
    int cb = cb0, tile = tile0, run = 0;
    if (n_units > 0) load_gw(cb);
    for (int i = 0; i < n_units; ++i, ring.next(pos)) {
        ring.consumer_wait(pos);
        const unsigned char* xs = ring.stage(pos.slot);
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, reinterpret_cast<const TC*>(xs + I::X_BYTES), TILE_PX, a.k, lane_px);

        if constexpr (I::FAST32) {
#pragma unroll
            for (int pi = 0; pi < CPW / 2; ++pi) {
                const int c0 = slot + 2 * pi * NSLOT, c1 = c0 + NSLOT;
                float g0[KP], g1[KP];
                lds_gw<float, KP>(g0, gwbuf + (size_t)c0 * KP);
                lds_gw<float, KP>(g1, gwbuf + (size_t)c1 * KP);
                float2 xa[2], xb[2];
                if constexpr (PPL == 4) {
                    load_x4<TX>(xs, c0, lane_px, xa);
                    load_x4<TX>(xs, c1, lane_px, xb);
                } else {
                    TX va[2], vb[2];
                    lds_vec<TX, 2>(va, xs + ((size_t)c0 * TILE_PX + lane_px) * sizeof(TX));
                    lds_vec<TX, 2>(vb, xs + ((size_t)c1 * TILE_PX + lane_px) * sizeof(TX));
                    xa[0] = make_float2((float)va[0], (float)va[1]);
                    xb[0] = make_float2((float)vb[0], (float)vb[1]);
                }
#pragma unroll
                for (int q = 0; q < PPL; ++q) {
                    const float2 x = q % 2 == 0 ? make_float2(xa[q / 2].x, xb[q / 2].x) : make_float2(xa[q / 2].y, xb[q / 2].y);
                    float2 y = __fmul2_rn(make_float2(g0[0], g1[0]), dup2(h[0][q]));
#pragma unroll
                    for (int kk = 1; kk < KP; ++kk) y = __ffma2_rn(make_float2(g0[kk], g1[kk]), dup2(h[kk][q]), y);
                    const float2 r = make_float2(rcp_ftz(y.x), rcp_ftz(y.y));
                    const float2 w = __fmul2_rn(__fmul2_rn(x, r), r);   // x r first: x == 0 gives 0, not 0 inf
                    int t = 0;
#pragma unroll
                    for (int aa = 0; aa < KP; ++aa) {
                        const float2 u = __fmul2_rn(w, dup2(h[aa][q]));
#pragma unroll
                        for (int bb = aa; bb < KP; ++bb, ++t) acc2[pi][t] = __ffma2_rn(u, dup2(h[bb][q]), acc2[pi][t]);
                    }
                }
            }
        } else {
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
                    const TC r = h_info_rcp(y);
                    const TC w = ((TC)xv[q] * r) * r;
                    int t = 0;
#pragma unroll
                    for (int aa = 0; aa < KP; ++aa) {
                        const TC u = w * h[aa][q];
#pragma unroll
                        for (int bb = aa; bb < KP; ++bb, ++t) accd[ci][t] = fma(u, h[bb][q], accd[ci][t]);
                    }
                }
            }
        }
        ring.consumer_release(pos, lane);
        const bool block_end = ++tile == a.n_tiles || i + 1 == n_units;
        if (++run == I::RUN || block_end) {
            end_run();
            run = 0;
        }
        if (block_end) {
            flush(cb);
            if (i + 1 < n_units) {
                tile = 0;
                ++cb;
                load_gw(cb);   // the barrier of flush: every warp is done with gwbuf and acc64 is zero
            }
        }
    }
}

// A[tri(a, b)][c] (the k x k triangle) = the CTA slots of channel c (the KP x KP triangle), added in slot order.
template <int KP>
static __global__ void __launch_bounds__(256) w_info_fold_kernel(const double* part, int n_tiles, int upc, int cs, int n,
                                                                 int n_pad, int k, double* A) {
    constexpr int NT = KP * (KP + 1) / 2;
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    const int cb = c / cs;
    const int ns = w_last_cta(cb, n_tiles, upc) - w_first_cta(cb, n_tiles, upc) + 1;
    int t = 0;
    for (int aa = 0; aa < KP; ++aa)
        for (int bb = aa; bb < KP; ++bb, ++t) {
            if (bb >= k) continue;
            double s = 0.0;
            for (int ps = 0; ps < ns; ++ps) s += part[((size_t)ps * n_pad + c) * NT + t];
            A[(size_t)tri_index(aa, bb, k) * n + c] = s;
        }
}

// Launch plan shared by the scratch query and the launch.  Scratch: Ht, then the CTA slots.
template <typename TX, typename TC, int KP>
static int w_info_do(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t stream) {
    using I = WInfoGeom<TX, TC, KP>;
    void (*kern)(const WInfoArgs) = w_info_kernel<TX, TC, KP>;
    SmemLimits lim;
    int rc = query_smem_limits(&lim);
    if (rc) return rc;
    // about 96 KiB of X in flight per SM, the amount of the W pass's best ring (profiles/r01f_summary.md)
    const int want = 98304 / I::X_BYTES;
    const int depth = ring_depth(lim, 1, I::FIXED, I::TAIL, I::STRIDE, want < 8 ? want : 8, "phase information kernel",
                                 st->kp);
    if (depth < 0) return depth;
    const int smem = I::FIXED + depth * I::STRIDE + I::TAIL;
    const int NS = st->n_pad / I::CS;
    int upc = 0, grid = 0, nr = 0;
    plan_w_units(NS, st->n_tiles, st->n_sms, &upc, &grid, &nr);
    const size_t ht_bytes = ((size_t)st->n_tiles * I::H_BYTES + 255) / 256 * 256;
    const size_t part_bytes = (size_t)nr * st->n_pad * I::NT * sizeof(double);
    if (bytes_out) {
        *bytes_out = (int64_t)(ht_bytes + part_bytes);
        return ESPM_OK;
    }
    int occ = 0;
    if ((rc = kernel_fit(kern, smem, "phase information kernel", &occ))) return rc;
    TC* Ht = reinterpret_cast<TC*>(scratch);
    const long long nh = (long long)KP * st->n_tiles * TILE_PX;
    w_info_tiles_kernel<TC, KP><<<(unsigned)((nh + 255) / 256), 256, 0, stream>>>(
        reinterpret_cast<const TC*>(st->H_cur), st->ldh, st->k, st->p_loc, st->n_tiles * TILE_PX, (TC)st->log_shift, Ht);
    ESPM_CUDA_CHECK(cudaGetLastError());
    WInfoArgs a;
    a.Xt = st->Xt;
    a.GWc = st->GWc_cur;
    a.Ht = Ht;
    a.part = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(scratch) + ht_bytes);
    a.n_pad = st->n_pad;
    a.k = st->k;
    a.n_tiles = st->n_tiles;
    a.nstages_tile = NS;
    a.w_upc = upc;
    a.depth = depth;
    w_info_kernel<TX, TC, KP><<<grid, XPASS_THREADS, smem, stream>>>(a);
    ESPM_CUDA_CHECK(cudaGetLastError());
    w_info_fold_kernel<KP><<<(st->n + 255) / 256, 256, 0, stream>>>(a.part, st->n_tiles, upc, I::CS, st->n,
                                                                    st->n_pad, st->k, out);
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

template <typename TX, typename TC>
static int w_info_entry(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t stream) {
    ESPM_KP_SWITCH(st->kp, return w_info_do<TX, TC, KP>(st, out, scratch, bytes_out, stream));
}

}  // namespace espm
