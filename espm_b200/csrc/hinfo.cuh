// Poisson information of the abundance maps in one streaming pass (espm_abundance_info,
// SmoothNMF.abundance_uncertainty).
//
//   y[c][j]    = sum_a g[c][a] h[a][j],   g = max(GW, ls), h = max(H, ls)      (the Y of KLdiv_loss, measures.py:493-497)
//   F_j[a][b]  = sum_c x[c][j] g[c][a] g[c][b] / y[c][j]^2                     (Hessian of the KL loss in H[:, j])
//
// h_info_kernel streams Xt once in H pass order, the stages coming from produce_tile_stages (xpass.cuh) with GWc_cur; a
// lane owns PPL pixels of the tile and walks the channels of its warp slot.  Per element: y (KP FMA), one reciprocal r,
// w = x r r, u_a = w g_a (KP multiplies) and the KP (KP + 1) / 2 FMAs u_a g_b of the upper triangle.  fp32: packed
// f32x2 arithmetic, one MUFU.RCP per element (the H pass spends two); fp64: the Newton reciprocal of Num<double>, no log.
// Everything is per pixel: no cross-lane reduction in the channel loop.  Once per tile the NSLOT warps that share a pixel
// are added in fp64, in slot order, through shared memory (in rounds of RCH entries), and the tile writes its packed F
// rows [k (k + 1) / 2][p_loc] in fp64 directly: no scratch, no cross-CTA state, no atomics.  Two calls give identical
// bits, and the result of a pixel does not depend on the grid (a pixel shard computes the bits of the whole image).
//
// fp32 accuracy: every term x g_a g_b / y^2 is >= 0, so summing the m = n_pad / NSLOT terms of a lane in fp32, in
// series, bounds the relative error of the lane's partial by (m - 1) 2^-24 plus the few ulps of a term (MUFU.RCP.FTZ
// <= 1 ulp, four rounded products); the NSLOT partials are converted and added in fp64.  At n = 2048 channels and
// NSLOT = 8 that is m = 256, i.e. <= 1.6e-5 worst case (the observed error grows like sqrt(m) 2^-24, ~1e-6).  Keeping the
// lane sums in fp32 is what lets the kp <= 4 instances fit the 96 registers of two CTAs per SM (with the channels of a
// stage walked one at a time: unrolling them costs a 4-byte spill at kp = 4).
//
// Pixels per lane by kp (the accumulators are KP (KP + 1) / 2 x PPL values): fp32 4 up to kp = 5, 2 for kp 6-8, 1 for kp
// 12-16; fp64 2 up to kp = 6, 1 above.  PPL < 4 splits a 128-pixel tile row over HALVES = 4 / PPL warps, as PassGeom
// does for fp64, so NSLOT = 8 / HALVES warps share a pixel.
//
// h_info_finish_kernel (fp64, one thread per pixel): the Cholesky F = R^T R, R^-1 and C = R^-1 R^-T in place, and with
// simplex the projection C - (C 1)(C 1)^T / (1^T C 1).  A pivot <= 1e-12 max_a F[a][a] (or an all-zero F) marks the
// pixel singular: NaN in its C and std.
#pragma once
#include "xpass.cuh"

namespace espm {

struct HInfoArgs {
    const void* Xt;
    const void* GWc;      // [n_pad][KP], max(GW, ls) on the real entries
    const void* H;        // [k][ldh] from local pixel 0
    double* F;            // [k (k + 1) / 2][p_loc], packed upper triangle, row by row
    int n_pad, k, ldh, p_loc, n_tiles, nstages_tile, depth;
    double log_shift;
};

constexpr double H_INFO_PIVOT_REL = 1e-12;

// index of (a, b), a <= b, in the packed upper triangle of a k x k matrix
__host__ __device__ __forceinline__ int tri_index(int a, int b, int k) { return a * (2 * k - a - 1) / 2 + b; }

template <typename TX, typename TC, int KP>
struct HInfoGeom {
    using S = XPassSmem<TX, TC, KP, false>;
    static constexpr bool FAST32 = sizeof(TC) == 4;
    static constexpr int PPL = FAST32 ? (KP <= 5 ? 4 : KP <= 8 ? 2 : 1) : (KP <= 6 ? 2 : 1);
    static constexpr int HALVES = TILE_PX / (32 * PPL);             // warps covering one 128-px row
    static constexpr int NSLOT = N_CONSUMER_WARPS / HALVES;         // warps sharing a pixel (channel rows at once)
    static constexpr int CS = PassGeom<TX, TC>::CS;
    static constexpr int X_BYTES = PassGeom<TX, TC>::X_BYTES;
    static constexpr int CPW = CS / NSLOT;                          // channels per warp per stage
    static constexpr int NT = KP * (KP + 1) / 2;                    // entries of the upper triangle
    // CTAs per SM the kernel is compiled for: the fp32 kp <= 4 accumulators (<= 40 registers) fit two
    static constexpr int OCC = (FAST32 && KP <= 4) ? 2 : 1;
    // channels of a stage unrolled: fully at one CTA per SM; one at a time at two, where unrolling spills at kp = 4
    static constexpr int CI_UNROLL = OCC == 2 ? 1 : CPW;
    static constexpr int STRIDE = S::H_STRIDE;                      // X chunk + GW rows, as in the H pass
    static constexpr int FIXED = S::BAR_BYTES + S::MISC_BYTES;
    // tile epilogue: RCH entries per round, NSLOT x RCH x 128 partials in the compute type (<= 16 KiB)
    static constexpr int RCH_MAX = 16384 / (NSLOT * TILE_PX * (int)sizeof(TC));
    static constexpr int RCH = NT < RCH_MAX ? NT : RCH_MAX;
    static constexpr int TAIL = NSLOT * RCH * TILE_PX * (int)sizeof(TC);
    static_assert(CS % NSLOT == 0 && RCH >= 1, "geometry");
};

__device__ __forceinline__ float h_info_rcp(float y) { return rcp_ftz(y); }
__device__ __forceinline__ double h_info_rcp(double y) { return Num<double>::rcp(y); }

template <typename TX, typename TC, int KP>
__global__ void __launch_bounds__(XPASS_THREADS, (HInfoGeom<TX, TC, KP>::OCC)) h_info_kernel(const HInfoArgs a) {
    using I = HInfoGeom<TX, TC, KP>;
    constexpr int PPL = I::PPL, NT = I::NT, RCH = I::RCH;
    constexpr bool PACKED = I::FAST32 && PPL % 2 == 0;
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<I::STRIDE> ring(smem, a.depth, I::FIXED);
    TC* red = reinterpret_cast<TC*>(smem + I::FIXED + (size_t)a.depth * I::STRIDE);   // [NSLOT][RCH][TILE_PX]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) ring.init();
    __syncthreads();
    const int NS = a.nstages_tile;

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            const uint64_t pol_x = l2_policy_evict_first();
            const uint64_t pol_gw = l2_policy_evict_last();
            typename Ring<I::STRIDE>::Pos pos{0, 0u};
            for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x)
                produce_tile_stages<TX, TC, KP, &HInfoArgs::GWc>(ring, pos, pol_x, pol_gw, a, tile, 0, NS, false);
        }
        return;
    }

    const int half = warp % I::HALVES, slot = warp / I::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;
    const TC ls = (TC)a.log_shift;
    const TC* Hc = reinterpret_cast<const TC*>(a.H);
    typename Ring<I::STRIDE>::Pos pos{0, 0u};

    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, Hc, a.ldh, a.k, tile * TILE_PX + lane_px);
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < a.k)
#pragma unroll
                for (int q = 0; q < PPL; ++q) h[kk][q] = Num<TC>::vmax(h[kk][q], ls);
        TC acc[NT][PPL];   // F of this lane's pixels over its channels, entry t of the upper triangle
#pragma unroll
        for (int t = 0; t < NT; ++t)
#pragma unroll
            for (int q = 0; q < PPL; ++q) acc[t][q] = TC(0);

        for (int st = 0; st < NS; ++st, ring.next(pos)) {
            ring.consumer_wait(pos);
            const unsigned char* xs = ring.stage(pos.slot);
            const unsigned char* gs = xs + I::X_BYTES;
#pragma unroll(I::CI_UNROLL)
            for (int ci = 0; ci < I::CPW; ++ci) {
                const int c = slot + ci * I::NSLOT;
                TC gw[KP];
                lds_gw<TC, KP>(gw, gs + (size_t)c * KP * sizeof(TC));
                if constexpr (PACKED) {
                    constexpr int NP = PPL / 2;
                    float2 x2[NP];
                    if constexpr (PPL == 4) {
                        load_x4<TX>(xs, c, lane_px, x2);
                    } else {
                        TX xv[2];
                        lds_vec<TX, 2>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                        x2[0] = make_float2((float)xv[0], (float)xv[1]);
                    }
#pragma unroll
                    for (int j = 0; j < NP; ++j) {
                        float2 y = __fmul2_rn(dup2(gw[0]), make_float2(h[0][2 * j], h[0][2 * j + 1]));
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk)
                            y = __ffma2_rn(dup2(gw[kk]), make_float2(h[kk][2 * j], h[kk][2 * j + 1]), y);
                        const float2 r = make_float2(rcp_ftz(y.x), rcp_ftz(y.y));
                        const float2 w = __fmul2_rn(__fmul2_rn(x2[j], r), r);   // x r first: x == 0 gives 0, not 0 inf
                        int t = 0;
#pragma unroll
                        for (int aa = 0; aa < KP; ++aa) {
                            const float2 u = __fmul2_rn(w, dup2(gw[aa]));
#pragma unroll
                            for (int bb = aa; bb < KP; ++bb, ++t) {
                                const float2 s = __ffma2_rn(u, dup2(gw[bb]), make_float2(acc[t][2 * j], acc[t][2 * j + 1]));
                                acc[t][2 * j] = s.x, acc[t][2 * j + 1] = s.y;
                            }
                        }
                    }
                } else {
                    TX xv[PPL];
                    lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        TC y = gw[0] * h[0][q];
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y = fma(gw[kk], h[kk][q], y);
                        const TC r = h_info_rcp(y);
                        const TC w = ((TC)xv[q] * r) * r;
                        int t = 0;
#pragma unroll
                        for (int aa = 0; aa < KP; ++aa) {
                            const TC u = w * gw[aa];
#pragma unroll
                            for (int bb = aa; bb < KP; ++bb, ++t) acc[t][q] = fma(u, gw[bb], acc[t][q]);
                        }
                    }
                }
            }
            ring.consumer_release(pos, lane);
        }

        // ---- tile epilogue: add the NSLOT warps that share a pixel, in fp64 and slot order, RCH entries per round ----
        const int j0 = tile * TILE_PX;
#pragma unroll
        for (int t0 = 0; t0 < NT; t0 += RCH) {
#pragma unroll
            for (int tt = 0; tt < RCH; ++tt)
                if (t0 + tt < NT)
#pragma unroll
                    for (int q = 0; q < PPL; ++q) red[((size_t)slot * RCH + tt) * TILE_PX + lane_px + q] = acc[t0 + tt][q];
            named_bar_sync(1, N_CONSUMER_THREADS);
            for (int i = threadIdx.x; i < RCH * TILE_PX; i += N_CONSUMER_THREADS) {
                const int tt = i / TILE_PX, px = i % TILE_PX;
                const int t = t0 + tt, j = j0 + px;
                if (t >= NT || j >= a.p_loc) continue;
                int aa = 0, rest = t;   // (aa, bb) of entry t in the KP x KP triangle
                while (rest >= KP - aa) rest -= KP - aa++;
                const int bb = aa + rest;
                if (bb < a.k) {
                    double v = (double)red[(size_t)tt * TILE_PX + px];
#pragma unroll
                    for (int sl = 1; sl < I::NSLOT; ++sl) v += (double)red[((size_t)sl * RCH + tt) * TILE_PX + px];
                    a.F[(size_t)tri_index(aa, bb, a.k) * a.p_loc + j] = v;
                }
            }
            named_bar_sync(1, N_CONSUMER_THREADS);
        }
    }
}

// F [k(k+1)/2][p] -> C [k(k+1)/2][p] (packed upper triangle) and std [k][p]; see the header comment.
template <int KP>
static __global__ void __launch_bounds__(128) h_info_finish_kernel(const double* F, double* C, double* stdv, int k, int p,
                                                                    int simplex) {
    constexpr int NT = KP * (KP + 1) / 2;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    // R[t(a, b)]: F on entry, then R (F = R^T R), then R^-1, then C; entries with b >= k stay 0
    double R[NT];
    double dmax = 0.0;
    {
        int t = 0;
#pragma unroll
        for (int aa = 0; aa < KP; ++aa)
#pragma unroll
            for (int bb = aa; bb < KP; ++bb, ++t) {
                R[t] = bb < k ? F[(size_t)tri_index(aa, bb, k) * p + j] : 0.0;
                if (aa == bb) dmax = fmax(dmax, R[t]);
            }
    }
#define TI(aa, bb) ((aa) * (2 * KP - (aa) - 1) / 2 + (bb))
    const double thr = H_INFO_PIVOT_REL * dmax;
    bool ok = true;
    double rinv[KP];   // 1 / R[a][a]
    // Cholesky, row by row: R[a][a] = sqrt(F[a][a] - sum_c<a R[c][a]^2), R[a][b] = (F[a][b] - sum_c<a R[c][a] R[c][b]) / R[a][a]
#pragma unroll
    for (int aa = 0; aa < KP; ++aa) {
        rinv[aa] = 0.0;
        if (aa < k) {
            double d = R[TI(aa, aa)];
#pragma unroll
            for (int c = 0; c < aa; ++c) d = fma(-R[TI(c, aa)], R[TI(c, aa)], d);
            ok = ok && d > thr;
            const double rd = sqrt(fmax(d, 0.0));
            rinv[aa] = 1.0 / rd;
            R[TI(aa, aa)] = rd;
#pragma unroll
            for (int bb = aa + 1; bb < KP; ++bb) {
                double s = R[TI(aa, bb)];
#pragma unroll
                for (int c = 0; c < aa; ++c) s = fma(-R[TI(c, aa)], R[TI(c, bb)], s);
                R[TI(aa, bb)] = s * rinv[aa];
            }
        }
    }
    if (ok) {
        // R^-1 in place, column by column: Ri[a][b] = -(sum_{c=a}^{b-1} Ri[a][c] R[c][b]) / R[b][b]
#pragma unroll
        for (int bb = 0; bb < KP; ++bb) {
#pragma unroll
            for (int aa = 0; aa < bb; ++aa) {
                double s = 0.0;
#pragma unroll
                for (int c = aa; c < bb; ++c) s = fma(c == aa ? rinv[aa] : R[TI(aa, c)], R[TI(c, bb)], s);
                R[TI(aa, bb)] = -s * rinv[bb];
            }
        }
#pragma unroll
        for (int aa = 0; aa < KP; ++aa) R[TI(aa, aa)] = rinv[aa];
        // C = R^-1 R^-T in place, row by row: C[a][b] = sum_{c>=b} Ri[a][c] Ri[b][c]
#pragma unroll
        for (int aa = 0; aa < KP; ++aa)
#pragma unroll
            for (int bb = aa; bb < KP; ++bb) {
                double s = 0.0;
#pragma unroll
                for (int c = bb; c < KP; ++c) s = fma(R[TI(aa, c)], R[TI(bb, c)], s);
                R[TI(aa, bb)] = s;
            }
        if (simplex) {
            double v[KP], tot = 0.0;   // v = C 1, tot = 1^T C 1
#pragma unroll
            for (int aa = 0; aa < KP; ++aa) {
                v[aa] = 0.0;
#pragma unroll
                for (int bb = 0; bb < KP; ++bb) v[aa] += R[aa <= bb ? TI(aa, bb) : TI(bb, aa)];
                tot += v[aa];
            }
            const double itot = 1.0 / tot;
#pragma unroll
            for (int aa = 0; aa < KP; ++aa)
#pragma unroll
                for (int bb = aa; bb < KP; ++bb) R[TI(aa, bb)] = fma(-v[aa] * itot, v[bb], R[TI(aa, bb)]);
        }
    }
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
    for (int aa = 0; aa < KP; ++aa) {
        if (aa < k) {
            stdv[(size_t)aa * p + j] = ok ? sqrt(fmax(R[TI(aa, aa)], 0.0)) : nan;
#pragma unroll
            for (int bb = aa; bb < KP; ++bb)
                if (bb < k) C[(size_t)tri_index(aa, bb, k) * p + j] = ok ? R[TI(aa, bb)] : nan;
        }
    }
#undef TI
}

// Launch plan and launch of both kernels; out = [k std rows][k(k+1)/2 C rows][k(k+1)/2 F rows] x p_loc doubles.
template <typename TX, typename TC, int KP>
static int h_info_do(const espm_state* st, int simplex, double* out, cudaStream_t stream) {
    using I = HInfoGeom<TX, TC, KP>;
    void (*kern)(const HInfoArgs) = h_info_kernel<TX, TC, KP>;
    SmemLimits lim;
    int rc = query_smem_limits(&lim);
    if (rc) return rc;
    const int depth = ring_depth(lim, I::OCC, I::FIXED, I::TAIL, I::STRIDE, 8, "abundance information kernel", st->kp);
    if (depth < 0) return depth;
    const int smem = I::FIXED + depth * I::STRIDE + I::TAIL;
    int occ = 0;
    if ((rc = kernel_fit(kern, smem, "abundance information kernel", &occ))) return rc;
    const int cap = st->n_sms * occ;
    const int grid = st->n_tiles < cap ? st->n_tiles : cap;
    const int k = st->k, p = st->p_loc;
    const size_t nt = (size_t)k * (k + 1) / 2;
    HInfoArgs a;
    a.Xt = st->Xt;
    a.GWc = st->GWc_cur;
    a.H = st->H_cur;
    a.F = out + ((size_t)k + nt) * p;
    a.n_pad = st->n_pad;
    a.k = k;
    a.ldh = st->ldh;
    a.p_loc = p;
    a.n_tiles = st->n_tiles;
    a.nstages_tile = st->n_pad / I::CS;
    a.depth = depth;
    a.log_shift = st->log_shift;
    h_info_kernel<TX, TC, KP><<<grid, XPASS_THREADS, smem, stream>>>(a);
    ESPM_CUDA_CHECK(cudaGetLastError());
    h_info_finish_kernel<KP><<<(p + 127) / 128, 128, 0, stream>>>(a.F, out + (size_t)k * p, out, k, p, simplex);
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

template <typename TX, typename TC>
static int h_info_entry(const espm_state* st, int simplex, double* out, cudaStream_t stream) {
    ESPM_KP_SWITCH(st->kp, return h_info_do<TX, TC, KP>(st, simplex, out, stream));
}

}  // namespace espm
