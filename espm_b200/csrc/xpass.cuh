// The two kernels that stream X from HBM: the H pass and the W pass.
//
// Both are warp-specialised persistent kernels: one producer warp issues TMA bulk copies
// (cp.async.bulk, SASS UBLKCP) of 16 KiB X chunks (8 / 4 KiB for uint16 / uint8 count storage) + the matching GW rows (+ the H tile in the W pass)
// into a ring of shared-memory stages guarded by mbarriers; eight consumer warps read the stages with
// 128-bit LDS, rebuild y = GW.H in registers (never materialised), form x/y and contract it on the fly.
//
//   h_pass : numraw[k][j] = sum_c GW[c][k] * X[c][j] / y[c][j]      (updates.py:127-128)
//            + partial sums of max(X,ls)*log(y)                      (measures.py:497-503)
//   w_pass : S[c][k]      = sum_j X[c][j] / y'[c][j] * H'[k][j]      (updates.py:53-59, G^T(R H^T))
//
// The fp32 fast path (TX = TC = float, !SAFE) uses the packed f32x2 FMAs of sm_100 (FFMA2/FMUL2: two
// pixels per issue slot) and single-instruction .ftz MUFU.RCP / MUFU.LG2.
#pragma once
#include "common.cuh"

namespace espm {

struct XPassArgs {
    const void* Xt;
    const void* GW;
    const void* GWc;
    const void* H;       // H pass: H_cur [k][ldh] (points at local pixel 0)
    const void* Ht;      // W pass: tile-major copy of H_next, [tile][KP][128]
    void* numraw;        // [nsplit][KP][P_pad]
    double* xlogy_part;  // [grid]
    uint32_t* bisect_mask;  // H pass: cleared for the h_finish that follows
    void* s_part;        // [w_nr][n_pad][KP]
    int n_pad, k, n_tiles, ldh, p_pad;
    int nstages_tile;    // n_pad / CS
    int nsplit;          // H pass
    int w_upc;           // W pass: (channel block, tile) units per CTA
    int depth;           // pipeline stages
    int clamp_y, dual;   // SAFE variants only
    double log_shift;
    double y_shift;      // H pass: ratio = x / (y + y_shift); log_shift for algo="l2_surrogate" (updates.py:280), else 0
    int n, p_loc;        // real channel / pixel counts (the Frobenius loss masks the padding)
};

// MODE of the X passes (template parameter):
//   XMODE_KL      ratio sums of x / y and the KL loss terms                      (updates.py:127-128, measures.py:497-503)
//   XMODE_FROB    Frobenius branches: the "ratio" is x itself                   (updates.py:109-118, 29-36)
//                 H pass: numraw = GW^T X, partial of sum (y - x)^2; W pass: S = X H'^T
//   XMODE_KL_FROB H pass only: KL ratio sums, Frobenius loss (algo="l2_surrogate" with l2=True: the H step is
//                 updates.py:263-301, the loss is 0.5 Frobenius_loss, base.py:197-198)
constexpr int XMODE_KL = 0, XMODE_FROB = 1, XMODE_KL_FROB = 2;

template <typename TX, typename TC, int KP, bool SAFE>
struct XPassSmem {
    using G = PassGeom<TX, TC>;
    static constexpr int X_BYTES = G::X_BYTES;
    static constexpr int GW_BYTES = G::CS * KP * (int)sizeof(TC);
    static constexpr int GW_BYTES_AL = (GW_BYTES + 127) / 128 * 128;
    static constexpr int HROW_BYTES = TILE_PX * (int)sizeof(TC);
    static constexpr int H_STRIDE = X_BYTES + GW_BYTES_AL * (SAFE ? 2 : 1);   // stage of the H pass
    static constexpr int W_STRIDE = X_BYTES + KP * HROW_BYTES;                // stage of the W pass: X + H tile
    static constexpr int BAR_BYTES = 256;  // up to 16 full + 16 empty barriers
    static constexpr int MISC_BYTES = 128;
    static constexpr int RED_BYTES = G::NSLOT * KP * TILE_PX * (int)sizeof(TC);          // H pass epilogue
    static constexpr int LOGTAB_BYTES = sizeof(TC) == 8 ? LOG2TAB_BYTES : 0;             // fp64 H pass: log2_tab()
    static constexpr int HTAIL_BYTES = RED_BYTES + LOGTAB_BYTES;
    static constexpr int WACC_BYTES = G::HALVES * G::CS * KP * (int)sizeof(TC);           // W pass flush / accumulator
    static constexpr int WTAIL_BYTES = GW_BYTES_AL + WACC_BYTES;                          // + GW rows of the channel block
    // the W pass keeps CPW x KP ratio sums per lane in registers when they fit, else in shared memory
    static constexpr bool FAST32 = !SAFE && sizeof(TX) <= 4 && sizeof(TC) == 4;   // f32 / uint16 / uint8 storage
    static constexpr int ACC_WORDS = G::CPW * KP * (FAST32 ? 2 : (int)sizeof(TC) / 4);
    static constexpr bool ACC_REG = ACC_WORDS <= 64;
    // CTAs per SM the kernels are compiled for (register budget: 96 regs/thread at 2, 168 at 1)
    static constexpr int OCC_BASE = (KP * (int)sizeof(TC) <= 32) ? 2 : 1;
    static constexpr int W_REGS_EST = (ACC_REG ? ACC_WORDS : KP * (int)sizeof(TC) / 4 * (FAST32 ? 2 : 1)) +
                                      KP * G::PPL * (int)sizeof(TC) / 4 + 36;
    static constexpr int W_OCC = (OCC_BASE == 2 && W_REGS_EST <= 110) ? 2 : 1;
};

template <typename T, int N>
__device__ __forceinline__ void lds_vec(T (&dst)[N], const void* src) {
    constexpr int BYTES = N * (int)sizeof(T);
    if constexpr (BYTES == 16) {
        uint4 v = *reinterpret_cast<const uint4*>(src);
        memcpy(dst, &v, 16);
    } else if constexpr (BYTES == 8) {
        uint2 v = *reinterpret_cast<const uint2*>(src);
        memcpy(dst, &v, 8);
    } else if constexpr (BYTES == 4) {
        uint32_t v = *reinterpret_cast<const uint32_t*>(src);
        memcpy(dst, &v, 4);
    } else {
        const T* s = reinterpret_cast<const T*>(src);
#pragma unroll
        for (int i = 0; i < N; ++i) dst[i] = s[i];
    }
}

template <typename TC, int KP>
__device__ __forceinline__ void lds_gw(TC (&gw)[KP], const void* row) {
    constexpr int BYTES = KP * (int)sizeof(TC);
    if constexpr (BYTES % 16 == 0) {
        const uint4* s = reinterpret_cast<const uint4*>(row);
        uint4 tmp[BYTES / 16];
#pragma unroll
        for (int i = 0; i < BYTES / 16; ++i) tmp[i] = s[i];
        memcpy(gw, tmp, BYTES);
    } else if constexpr (BYTES % 8 == 0) {
        const uint2* s = reinterpret_cast<const uint2*>(row);
        uint2 tmp[BYTES / 8];
#pragma unroll
        for (int i = 0; i < BYTES / 8; ++i) tmp[i] = s[i];
        memcpy(gw, tmp, BYTES);
    } else {
        const TC* s = reinterpret_cast<const TC*>(row);
#pragma unroll
        for (int i = 0; i < KP; ++i) gw[i] = s[i];
    }
}

// Loads the PPL consecutive H values of KP rows for this lane's pixels (H pad pixels hold a positive
// value, pad rows are treated as 0).  `H` may be global or shared memory.
template <typename TC, int KP, int PPL>
__device__ __forceinline__ void load_h(TC (&h)[KP][PPL], const TC* H, int ldh, int k, int px0) {
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) {
        if (kk < k) {
            lds_vec<TC, PPL>(h[kk], H + (size_t)kk * ldh + px0);
        } else {
#pragma unroll
            for (int q = 0; q < PPL; ++q) h[kk][q] = TC(0);
        }
    }
}

// single-instruction MUFU forms (no denormal fix-up code around them)
__device__ __forceinline__ float rcp_ftz(float y) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
    return r;
}
__device__ __forceinline__ float lg2_ftz(float y) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y));
    return r;
}
__device__ __forceinline__ float2 dup2(float v) { return make_float2(v, v); }

// The 4 pixels of this lane in channel row `c` of a stage, as two packed pixel pairs (fp32 fast path).
//   float    one LDS.128
//   uint16   one LDS.64;  uint8  one LDS.32.  Counts become floats WITHOUT the conversion unit (I2F shares the XU pipe
//            with MUFU, the busiest pipe of the H pass): PRMT drops the integer into the mantissa of 2^23
//            (0x4B000000 | v  ==  8388608.0f + v, exact for v < 2^23) and one packed FADD removes the 2^23 again:
//            1 PRMT per element + 1 FADD2 per pair.
template <typename TX>
__device__ __forceinline__ void load_x4(const unsigned char* xs, int c, int lane_px, float2 (&x2)[2]) {
    const unsigned char* p = xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX);
    if constexpr (sizeof(TX) == 4) {
        const float4 xv = *reinterpret_cast<const float4*>(p);
        x2[0] = make_float2(xv.x, xv.y);
        x2[1] = make_float2(xv.z, xv.w);
    } else {
        constexpr uint32_t MAGIC = 0x4B000000u;
        uint32_t m[4];
        if constexpr (sizeof(TX) == 1) {
            const uint32_t w = *reinterpret_cast<const uint32_t*>(p);
            m[0] = __byte_perm(w, MAGIC, 0x7440);
            m[1] = __byte_perm(w, MAGIC, 0x7441);
            m[2] = __byte_perm(w, MAGIC, 0x7442);
            m[3] = __byte_perm(w, MAGIC, 0x7443);
        } else {
            const uint2 w = *reinterpret_cast<const uint2*>(p);
            m[0] = __byte_perm(w.x, MAGIC, 0x7410);
            m[1] = __byte_perm(w.x, MAGIC, 0x7432);
            m[2] = __byte_perm(w.y, MAGIC, 0x7410);
            m[3] = __byte_perm(w.y, MAGIC, 0x7432);
        }
        const float2 off = make_float2(-8388608.0f, -8388608.0f);
        x2[0] = __fadd2_rn(make_float2(__uint_as_float(m[0]), __uint_as_float(m[1])), off);
        x2[1] = __fadd2_rn(make_float2(__uint_as_float(m[2]), __uint_as_float(m[3])), off);
    }
}

// ------------------------------------------------------------------------------------------------
// Ring of pipeline stages: one elected producer lane fills it, the consumer warps drain it.
// ------------------------------------------------------------------------------------------------
template <int STRIDE>
struct Ring {
    uint64_t* full;
    uint64_t* empty;
    unsigned char* stages;
    int depth;
    __device__ __forceinline__ Ring(unsigned char* smem, int depth_, int head_bytes) : depth(depth_) {
        full = reinterpret_cast<uint64_t*>(smem);
        empty = full + 16;
        stages = smem + head_bytes;
    }
    __device__ __forceinline__ void init() {
        for (int i = 0; i < depth; ++i) {
            mbar_init(&full[i], 1);
            mbar_init(&empty[i], N_CONSUMER_WARPS);
        }
        mbar_fence_init();
    }
    __device__ __forceinline__ unsigned char* stage(int slot) { return stages + (size_t)slot * STRIDE; }
    // position in the ring: slot index + phase parity (no integer division in the loops)
    struct Pos {
        int slot;
        uint32_t phase;
    };
    __device__ __forceinline__ void next(Pos& p) const {
        if (++p.slot == depth) {
            p.slot = 0;
            p.phase ^= 1u;
        }
    }
    // producer: wait until the slot is free
    __device__ __forceinline__ void acquire(const Pos& p) { mbar_wait(&empty[p.slot], p.phase ^ 1u); }
    __device__ __forceinline__ void consumer_wait(const Pos& p) { mbar_wait(&full[p.slot], p.phase); }
    __device__ __forceinline__ void consumer_release(const Pos& p, int lane) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[p.slot]);
    }
};

// ------------------------------------------------------------------------------------------------
// The two producers, called by the elected producer lane.  Every kernel that streams X uses one of them.  They read
// Xt, n_pad (and Ht, n_tiles, w_upc) from the kernel's argument struct `a` where the copies are issued.  The kernel
// owns the ring position `pos`: the H pass calls produce_tile_stages once per work item and continues the ring.  X is
// copied with the evict-first L2 policy, the GW rows and H tiles, which every CTA reads, with evict-last.
//
// Tile stages (H pass order): the stages [s0, s1) of pixel tile `tile`, each the X chunk of CS channels plus the
// CS x KP rows of a.*GW behind it; with `dual` (SAFE H pass only) also the rows of a.GWc at GW_BYTES_AL.
// ------------------------------------------------------------------------------------------------
template <typename TX, typename TC, int KP, auto GW, int STRIDE, typename Args>
__device__ __forceinline__ void produce_tile_stages(Ring<STRIDE>& ring, typename Ring<STRIDE>::Pos& pos,
                                                    uint64_t pol_x, uint64_t pol_gw, const Args& a, int tile, int s0,
                                                    int s1, bool dual) {
    using S = XPassSmem<TX, TC, KP, false>;
    constexpr int CS = S::G::CS;
    for (int st = s0; st < s1; ++st, ring.next(pos)) {
        ring.acquire(pos);
        const int slot = pos.slot;
        unsigned char* sp = ring.stage(slot);
        mbar_expect_tx(&ring.full[slot], S::X_BYTES + S::GW_BYTES * (dual ? 2 : 1));
        const TX* xsrc = reinterpret_cast<const TX*>(a.Xt) + ((size_t)tile * a.n_pad + (size_t)st * CS) * TILE_PX;
        tma_bulk_g2s(sp, xsrc, S::X_BYTES, &ring.full[slot], pol_x);
        const TC* gsrc = reinterpret_cast<const TC*>(a.*GW) + (size_t)st * CS * KP;
        tma_bulk_g2s(sp + S::X_BYTES, gsrc, S::GW_BYTES, &ring.full[slot], pol_gw);
        if (dual) {
            const TC* csrc = reinterpret_cast<const TC*>(a.GWc) + (size_t)st * CS * KP;
            tma_bulk_g2s(sp + S::X_BYTES + S::GW_BYTES_AL, csrc, S::GW_BYTES, &ring.full[slot], pol_gw);
        }
    }
}

// Units (W pass order): work unit = (channel block of CS channels, pixel tile), ordered channel-block major; CTA i owns
// the contiguous range [i w_upc, (i + 1) w_upc) of the nstages_tile x n_tiles units.
struct UnitRange {
    int n_units, cb0, tile0;
    template <typename Args>
    __device__ __forceinline__ explicit UnitRange(const Args& a) {
        const long long total = (long long)a.nstages_tile * a.n_tiles;
        const long long u0 = (long long)blockIdx.x * a.w_upc;
        const long long u1 = (u0 + a.w_upc < total) ? u0 + a.w_upc : total;
        n_units = (u1 > u0) ? (int)(u1 - u0) : 0;
        cb0 = (int)(u0 / a.n_tiles);
        tile0 = (int)(u0 - (long long)cb0 * a.n_tiles);
    }
};

// One stage per unit: the X chunk of channel block cb of the tile, then the tile's KP x TILE_PX block of a.Ht.
template <typename TX, typename TC, int KP, int CS, int STRIDE, typename Args>
__device__ __forceinline__ void produce_units(Ring<STRIDE>& ring, typename Ring<STRIDE>::Pos& pos, const UnitRange& u,
                                              const Args& a) {
    constexpr int X_BYTES = CS * TILE_PX * (int)sizeof(TX);
    constexpr int H_BYTES = KP * TILE_PX * (int)sizeof(TC);
    const uint64_t pol_x = l2_policy_evict_first();
    const uint64_t pol_h = l2_policy_evict_last();
    const TC* Ht = reinterpret_cast<const TC*>(a.Ht);
    int cb = u.cb0, tile = u.tile0;
    for (int i = 0; i < u.n_units; ++i, ring.next(pos)) {
        ring.acquire(pos);
        unsigned char* sp = ring.stage(pos.slot);
        mbar_expect_tx(&ring.full[pos.slot], X_BYTES + H_BYTES);
        const TX* xsrc = reinterpret_cast<const TX*>(a.Xt) + ((size_t)tile * a.n_pad + (size_t)cb * CS) * TILE_PX;
        tma_bulk_g2s(sp, xsrc, X_BYTES, &ring.full[pos.slot], pol_x);
        tma_bulk_g2s(sp + X_BYTES, Ht + (size_t)tile * KP * TILE_PX, H_BYTES, &ring.full[pos.slot], pol_h);
        if (++tile == a.n_tiles) {
            tile = 0;
            ++cb;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// H pass
// ------------------------------------------------------------------------------------------------
template <typename TX, typename TC, int KP, bool SAFE, int MODE = XMODE_KL>
__global__ void __launch_bounds__(XPASS_THREADS, (XPassSmem<TX, TC, KP, SAFE>::OCC_BASE))
h_pass_kernel(const XPassArgs a) {
    using G = PassGeom<TX, TC>;
    using S = XPassSmem<TX, TC, KP, SAFE>;
    constexpr int PPL = G::PPL;
    constexpr bool FAST32 = MODE == XMODE_KL && S::FAST32;
    constexpr bool FAST64 = MODE == XMODE_KL && !SAFE && sizeof(TC) == 8;   // table log2, branch-free loss terms
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<S::H_STRIDE> ring(smem, a.depth, S::BAR_BYTES + S::MISC_BYTES);
    double* misc = reinterpret_cast<double*>(smem + S::BAR_BYTES);
    TC* red = reinterpret_cast<TC*>(smem + S::BAR_BYTES + S::MISC_BYTES + (size_t)a.depth * S::H_STRIDE);
    [[maybe_unused]] const double2* ltab = log2tab_lane(
        reinterpret_cast<const double2*>(reinterpret_cast<unsigned char*>(red) + S::RED_BYTES), threadIdx.x & 31);
    if constexpr (sizeof(TC) == 8 && MODE == XMODE_KL)
        log2tab_fill(reinterpret_cast<double2*>(reinterpret_cast<unsigned char*>(red) + S::RED_BYTES), threadIdx.x, XPASS_THREADS);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) ring.init();      // shared memory only: may overlap the previous kernel's tail
    pdl_wait();
    pdl_trigger();
    if (blockIdx.x == 0 && threadIdx.x < 4 && a.bisect_mask) a.bisect_mask[threadIdx.x] = 0u;
    __syncthreads();

    const int n_items = a.n_tiles * a.nsplit;
    const int NS = a.nstages_tile;

    if (warp == N_CONSUMER_WARPS) {
        // ---------------- producer warp ----------------
        if (lane == 0) {
            const uint64_t pol_x = l2_policy_evict_first();
            const uint64_t pol_gw = l2_policy_evict_last();
            const bool dual = SAFE && a.dual;   // compile-time false in the non-SAFE instances
            typename Ring<S::H_STRIDE>::Pos pos{0, 0u};
            for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
                const int tile = it / a.nsplit, split = it - tile * a.nsplit;
                const int s0 = (int)((long long)split * NS / a.nsplit), s1 = (int)((long long)(split + 1) * NS / a.nsplit);
                produce_tile_stages<TX, TC, KP, &XPassArgs::GW>(ring, pos, pol_x, pol_gw, a, tile, s0, s1, dual);
            }
        }
        return;
    }

    // ---------------- consumer warps ----------------
    const int half = warp % G::HALVES, slot = warp / G::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;  // pixel offset inside the tile
    const TC ls = (TC)a.log_shift;
    const TC* Hc = reinterpret_cast<const TC*>(a.H);
    double xl_total = 0.0;   // sum x*log2(y) over x>0
    double zl_total = 0.0;   // sum log2(y) over x==0 (weighted by log_shift at the end)
    typename Ring<S::H_STRIDE>::Pos pos{0, 0u};

    for (int it = blockIdx.x; it < n_items; it += gridDim.x) {
        const int tile = it / a.nsplit, split = it - tile * a.nsplit;
        const int s0 = (int)((long long)split * NS / a.nsplit), s1 = (int)((long long)(split + 1) * NS / a.nsplit);
        TC h[KP][PPL], num[KP][PPL];
        load_h<TC, KP, PPL>(h, Hc, a.ldh, a.k, tile * TILE_PX + lane_px);

        if constexpr (FAST32) {
            // ---- fp32 fast path: pixel pairs in packed f32x2 registers ----
            float2 h2[KP][2], num2[KP][2];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    h2[kk][j] = make_float2(h[kk][2 * j], h[kk][2 * j + 1]);
                    num2[kk][j] = make_float2(0.f, 0.f);
                }
            // y starts from y_shift (0, or log_shift for the quadratic surrogate): fma(gw, h, 0) == gw * h.
            // With a shift the loss below sees log(y + ls) instead of log(y): 1e-14 / y relative, far below
            // fp32 resolution.
            const float2 ysh = dup2((float)a.y_shift);
            for (int st = s0; st < s1; ++st, ring.next(pos)) {
                ring.consumer_wait(pos);
                const unsigned char* xs = ring.stage(pos.slot);
                const unsigned char* gs = xs + S::X_BYTES;
                float2 xl2 = make_float2(0.f, 0.f);
#pragma unroll
                for (int ci = 0; ci < G::CPW; ++ci) {
                    const int c = slot + ci * G::NSLOT;
                    float2 x2[2];
                    load_x4<TX>(xs, c, lane_px, x2);
                    float gw[KP];
                    lds_gw<float, KP>(gw, gs + (size_t)c * KP * sizeof(float));
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        float2 y = __ffma2_rn(dup2(gw[0]), h2[0][j], ysh);
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y = __ffma2_rn(dup2(gw[kk]), h2[kk][j], y);
                        const float2 r = __fmul2_rn(x2[j], make_float2(rcp_ftz(y.x), rcp_ftz(y.y)));
#pragma unroll
                        for (int kk = 0; kk < KP; ++kk) num2[kk][j] = __ffma2_rn(dup2(gw[kk]), r, num2[kk][j]);
                        // 0*log2(y) == 0 because y > 0 is guaranteed on this path; the reference's
                        // ls*log(Y) terms of zero entries are below fp32 rounding of the sum.
                        xl2 = __ffma2_rn(x2[j], make_float2(lg2_ftz(y.x), lg2_ftz(y.y)), xl2);
                    }
                }
                ring.consumer_release(pos, lane);
                xl_total += (double)(xl2.x + xl2.y);
            }
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    num[kk][2 * j] = num2[kk][j].x;
                    num[kk][2 * j + 1] = num2[kk][j].y;
                }
        } else {
            TC hc[SAFE ? KP : 1][PPL];
            const TC ysh = (TC)a.y_shift;
            const bool shifted = a.y_shift != 0.0;
            [[maybe_unused]] unsigned lrange = 0u;
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
#pragma unroll
                for (int q = 0; q < PPL; ++q) {
                    num[kk][q] = TC(0);
                    if constexpr (SAFE) hc[kk][q] = (kk < a.k) ? Num<TC>::vmax(h[kk][q], ls) : TC(0);
                }
            for (int st = s0; st < s1; ++st, ring.next(pos)) {
                ring.consumer_wait(pos);
                const unsigned char* xs = ring.stage(pos.slot);
                const unsigned char* gs = xs + S::X_BYTES;
                const unsigned char* gcs = gs + S::GW_BYTES_AL;
                TC xl = TC(0);
                float zl = 0.f;
#pragma unroll
                for (int ci = 0; ci < G::CPW; ++ci) {
                    const int c = slot + ci * G::NSLOT;
                    TX xv[PPL];
                    TC gw[KP];
                    lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                    lds_gw<TC, KP>(gw, gs + (size_t)c * KP * sizeof(TC));
                    TC y[PPL], r[PPL];
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        y[q] = gw[0] * h[0][q];
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y[q] = fma(gw[kk], h[kk][q], y[q]);
                    }
                    if constexpr (SAFE) {
                        if (a.clamp_y) {
#pragma unroll
                            for (int q = 0; q < PPL; ++q) y[q] = Num<TC>::vmax(y[q], ls);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        if constexpr (MODE == XMODE_FROB) r[q] = (TC)xv[q];
                        else r[q] = Num<TC>::ratio((TC)xv[q], shifted ? y[q] + ysh : y[q]);
                    }
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk)
#pragma unroll
                        for (int q = 0; q < PPL; ++q) num[kk][q] = fma(gw[kk], r[q], num[kk][q]);
                    // ---- loss of the current iterate: sum max(x,ls)*log(Y), Y from clamped GW, H ----
                    TC yl[PPL];
                    if constexpr (SAFE) {
                        if (a.dual) {
                            TC gwc[KP];
                            lds_gw<TC, KP>(gwc, gcs + (size_t)c * KP * sizeof(TC));
#pragma unroll
                            for (int q = 0; q < PPL; ++q) {
                                yl[q] = gwc[0] * hc[0][q];
#pragma unroll
                                for (int kk = 1; kk < KP; ++kk) yl[q] = fma(gwc[kk], hc[kk][q], yl[q]);
                            }
                        } else {
#pragma unroll
                            for (int q = 0; q < PPL; ++q) yl[q] = y[q];
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < PPL; ++q) yl[q] = y[q];
                    }
                    if constexpr (MODE != XMODE_KL) {
                        // 0.5 Frobenius_loss (measures.py:350-385) of the unclamped G W H; padding is masked out
                        const bool c_real = st * G::CS + c < a.n;
#pragma unroll
                        for (int q = 0; q < PPL; ++q) {
                            const TC d = y[q] - (TC)xv[q];
                            if (c_real && tile * TILE_PX + lane_px + q < a.p_loc) xl = fma(d, d, xl);
                        }
                    } else {
#pragma unroll
                        for (int q = 0; q < PPL; ++q) {
                            const TC x = (TC)xv[q];
                            if constexpr (FAST64) {
                                // branch-free: max(x, ls) * log2(y) for every element (measures.py:497-503 as written);
                                // X >= 0 was checked at ingest (base.py:528)
                                xl = fma(max_nonneg(x, ls), log2_tab_core(y[q], ltab, lrange), xl);
                            } else if constexpr (sizeof(TC) == 8) {
                                xl = fma(Num<TC>::vmax(x, ls), log2_tab(yl[q], ltab), xl);
                            } else if (x > TC(0)) {
                                xl = fma(Num<TC>::vmax(x, ls), Num<TC>::log2_fast(yl[q]), xl);
                            } else {
                                zl += __log2f((float)yl[q]);
                            }
                        }
                    }
                }
                if constexpr (FAST64) {
                    if (__any_sync(0xffffffffu, log2_range_bad(lrange))) {
                        // some y of this stage is zero / subnormal / negative / non-finite: redo the stage's loss terms
                        // with the library log2 (cold path)
                        xl = TC(0);
                        lrange = 0u;
#pragma unroll 1
                        for (int ci = 0; ci < G::CPW; ++ci) {
                            const int c = slot + ci * G::NSLOT;
                            TX xv[PPL];
                            TC gw[KP];
                            lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                            lds_gw<TC, KP>(gw, gs + (size_t)c * KP * sizeof(TC));
#pragma unroll
                            for (int q = 0; q < PPL; ++q) {
                                TC yq = gw[0] * h[0][q];
#pragma unroll
                                for (int kk = 1; kk < KP; ++kk) yq = fma(gw[kk], h[kk][q], yq);
                                xl = fma(Num<TC>::vmax((TC)xv[q], ls), (TC)log2((double)yq), xl);
                            }
                        }
                    }
                }
                ring.consumer_release(pos, lane);
                xl_total += (double)xl;
                zl_total += (double)zl;
            }
        }

        // ---- cross-warp reduction of the ratio sums of this item (fixed order => deterministic) ----
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
#pragma unroll
            for (int q = 0; q < PPL; ++q) red[((size_t)slot * KP + kk) * TILE_PX + lane_px + q] = num[kk][q];
        named_bar_sync(1, N_CONSUMER_THREADS);
        TC* out = reinterpret_cast<TC*>(a.numraw) + (size_t)split * KP * a.p_pad + (size_t)tile * TILE_PX;
        for (int idx = threadIdx.x; idx < KP * TILE_PX; idx += N_CONSUMER_THREADS) {
            const int kk = idx / TILE_PX, q = idx - kk * TILE_PX;
            TC s = red[(size_t)kk * TILE_PX + q];
#pragma unroll
            for (int sl = 1; sl < G::NSLOT; ++sl) s += red[((size_t)sl * KP + kk) * TILE_PX + q];
            out[(size_t)kk * a.p_pad + q] = s;
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
    }

    // ---- loss partial of this CTA ----
    // pad pixels / pad channels contribute x == 0 only; the zero-entry term is weighted by log_shift.
    double v = xl_total + a.log_shift * zl_total;
    v = warp_sum(v);
    if (lane == 0) misc[warp] = v;
    named_bar_sync(1, N_CONSUMER_THREADS);
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < N_CONSUMER_WARPS; ++w) s += misc[w];
        a.xlogy_part[blockIdx.x] = (MODE != XMODE_KL) ? s : s * 0.6931471805599453094;  // log2 -> ln
    }
}

// ------------------------------------------------------------------------------------------------
// W pass
//
// Work unit = (channel block of CS channels, pixel tile) = one pipeline stage.  Units are ordered
// channel-block major and CTA i owns the contiguous range [i*upc, (i+1)*upc).  Every consumer lane keeps
// the ratio sums of ITS channels and pixels in registers across all tiles of a channel block; the
// cross-lane reduction happens once per (CTA, channel block), when the block changes ("flush").
// Partial slot of a flush = CTA index - first CTA that touches the block, so w_reduce can add the slots
// of a block in a fixed order without zero-filling.
// ------------------------------------------------------------------------------------------------
__host__ __device__ inline int w_first_cta(int cb, int n_tiles, int upc) {
    return (int)(((long long)cb * n_tiles) / upc);
}
__host__ __device__ inline int w_last_cta(int cb, int n_tiles, int upc) {
    return (int)((((long long)cb + 1) * n_tiles - 1) / upc);
}

// ------------------------------------------------------------------------------------------------
// Host planning shared by every X-streaming kernel.
// ------------------------------------------------------------------------------------------------
struct SmemLimits {
    int per_sm, optin;   // shared memory per SM, and the opt-in maximum of one CTA
};

inline int query_smem_limits(SmemLimits* lim) {
    int dev = 0;
    ESPM_CUDA_CHECK(cudaGetDevice(&dev));
    ESPM_CUDA_CHECK(cudaDeviceGetAttribute(&lim->optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    ESPM_CUDA_CHECK(cudaDeviceGetAttribute(&lim->per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
    return ESPM_OK;
}

// Stages of `stride` bytes for a kernel compiled for `occ` CTAs per SM: the per-CTA budget is per_sm / occ less the
// 1 KiB the runtime reserves per CTA, at most the opt-in maximum; `fixed` (barriers) and `tail` (epilogue) come first.
// Returns the depth (at most max_depth), or a negative error code when fewer than two stages fit.
inline int ring_depth(const SmemLimits& lim, int occ, int fixed, int tail, int stride, int max_depth, const char* what,
                      int kp) {
    int budget = lim.per_sm / occ - 1024;
    if (budget > lim.optin) budget = lim.optin;
    int depth = (budget - fixed - tail) / stride;
    if (depth > max_depth) depth = max_depth;
    if (depth < 2) {
        set_error("shared memory budget too small for the %s (kp=%d)", what, kp);
        return ESPM_ERR_UNSUPPORTED;
    }
    return depth;
}

// Sets the kernel's dynamic shared memory to `smem` and returns its resident CTAs per SM in *occ (>= 1).
template <typename Kernel>
inline int kernel_fit(Kernel kern, int smem, const char* what, int* occ) {
    ESPM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    ESPM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, kern, XPASS_THREADS, smem));
    if (*occ < 1) {
        set_error("%s does not fit on an SM (smem=%d)", what, smem);
        return ESPM_ERR_UNSUPPORTED;
    }
    return ESPM_OK;
}

// Splits the NS x n_tiles units of the W pass order over at most `cap` CTAs: units per CTA, CTAs, and the largest
// number of CTAs that share a channel block (the partial slots per channel).
inline void plan_w_units(int NS, int n_tiles, long long cap, int* upc, int* grid, int* nr) {
    const long long total = (long long)NS * n_tiles;
    const long long u = (total + cap - 1) / cap;
    *upc = (int)u;
    *grid = (int)((total + u - 1) / u);
    *nr = 1;
    for (int cb = 0; cb < NS; ++cb) {
        const int c = w_last_cta(cb, n_tiles, *upc) - w_first_cta(cb, n_tiles, *upc) + 1;
        if (c > *nr) *nr = c;
    }
}

template <typename TX, typename TC, int KP, bool SAFE, int MODE = XMODE_KL>
__global__ void __launch_bounds__(XPASS_THREADS, (XPassSmem<TX, TC, KP, SAFE>::W_OCC))
w_pass_kernel(const XPassArgs a) {
    using G = PassGeom<TX, TC>;
    using S = XPassSmem<TX, TC, KP, SAFE>;
    constexpr int PPL = G::PPL;
    constexpr int CPW = G::CPW;
    constexpr bool FAST32 = MODE == XMODE_KL && S::FAST32;
    constexpr bool ACC_REG = S::ACC_REG;
    extern __shared__ __align__(128) unsigned char smem[];
    Ring<S::W_STRIDE> ring(smem, a.depth, S::BAR_BYTES + S::MISC_BYTES);
    // tail: GW rows of the current channel block, then [HALVES][CS][KP] flush staging (ACC_REG) or the
    // running accumulator (!ACC_REG)
    unsigned char* tail0 = smem + S::BAR_BYTES + S::MISC_BYTES + (size_t)a.depth * S::W_STRIDE;
    TC* gwbuf = reinterpret_cast<TC*>(tail0);
    TC* tail = reinterpret_cast<TC*>(tail0 + S::GW_BYTES_AL);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const UnitRange units(a);
    const int n_units = units.n_units;

    if (threadIdx.x == 0) ring.init();      // shared memory only: may overlap the previous kernel's tail
    for (int i = threadIdx.x; i < G::HALVES * G::CS * KP; i += blockDim.x) tail[i] = TC(0);
    pdl_wait();
    pdl_trigger();
    __syncthreads();

    if (warp == N_CONSUMER_WARPS) {
        if (lane == 0) {
            typename Ring<S::W_STRIDE>::Pos pos{0, 0u};
            produce_units<TX, TC, KP, G::CS>(ring, pos, units, a);
        }
        return;
    }

    const int half = warp % G::HALVES, slot = warp / G::HALVES;
    const int lane_px = half * (32 * PPL) + lane * PPL;
    const TC ls = (TC)a.log_shift;
    (void)ls;

    // per-lane accumulators: CPW channels x KP phases (x 2 pixel parities on the packed path)
    constexpr int NACC = ACC_REG ? CPW : 1;
    TC acc[FAST32 ? 1 : NACC][FAST32 ? 1 : KP];
    float2 acc2[FAST32 ? NACC : 1][FAST32 ? KP : 1];
#pragma unroll
    for (int ci = 0; ci < NACC; ++ci)
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            if constexpr (FAST32) acc2[ci][kk] = make_float2(0.f, 0.f);
            else acc[ci][kk] = TC(0);
        }

    // Ends the channel block `cb` of this CTA: s_part[slot of this CTA in cb][channels of cb][KP].
    auto flush = [&](int cb) {
        const int ps = blockIdx.x - w_first_cta(cb, a.n_tiles, a.w_upc);
        TC* out = reinterpret_cast<TC*>(a.s_part) + ((size_t)ps * a.n_pad + (size_t)cb * G::CS) * KP;
        if constexpr (ACC_REG) {
#pragma unroll
            for (int ci = 0; ci < CPW; ++ci)
#pragma unroll
                for (int kk = 0; kk < KP; ++kk) {
                    TC v;
                    if constexpr (FAST32) {
                        v = acc2[ci][kk].x + acc2[ci][kk].y;
                        acc2[ci][kk] = make_float2(0.f, 0.f);
                    } else {
                        v = acc[ci][kk];
                        acc[ci][kk] = TC(0);
                    }
                    v = warp_sum(v);
                    if (lane == 0) tail[((size_t)half * G::CS + slot + ci * G::NSLOT) * KP + kk] = v;
                }
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
        for (int i = threadIdx.x; i < G::CS * KP; i += N_CONSUMER_THREADS) {
            TC v = tail[i];
            if constexpr (G::HALVES == 2) v += tail[(size_t)G::CS * KP + i];
            out[i] = v;
        }
        named_bar_sync(1, N_CONSUMER_THREADS);
        if constexpr (!ACC_REG) {
            for (int i = threadIdx.x; i < G::HALVES * G::CS * KP; i += N_CONSUMER_THREADS) tail[i] = TC(0);
            named_bar_sync(1, N_CONSUMER_THREADS);
        }
    };

    // GW rows of a channel block: CS x KP values, kept in shared memory while the block is processed
    auto load_gw = [&](int cb) {
        const TC* src = reinterpret_cast<const TC*>(a.GW) + (size_t)cb * G::CS * KP;
        for (int i = threadIdx.x; i < G::CS * KP; i += N_CONSUMER_THREADS) gwbuf[i] = src[i];
        named_bar_sync(1, N_CONSUMER_THREADS);
    };

    typename Ring<S::W_STRIDE>::Pos pos{0, 0u};
    int cb = units.cb0, tile = units.tile0;
    if (n_units > 0) load_gw(cb);
    for (int i = 0; i < n_units; ++i, ring.next(pos)) {
        ring.consumer_wait(pos);
        const unsigned char* xs = ring.stage(pos.slot);
        const unsigned char* gs = reinterpret_cast<const unsigned char*>(gwbuf);
        const TC* hs = reinterpret_cast<const TC*>(xs + S::X_BYTES);
        TC h[KP][PPL];
        load_h<TC, KP, PPL>(h, hs, TILE_PX, a.k, lane_px);

        if constexpr (FAST32) {
            float2 h2[KP][2];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                h2[kk][0] = make_float2(h[kk][0], h[kk][1]);
                h2[kk][1] = make_float2(h[kk][2], h[kk][3]);
            }
#pragma unroll
            for (int ci = 0; ci < CPW; ++ci) {
                const int c = slot + ci * G::NSLOT;
                float2 x2[2];
                load_x4<TX>(xs, c, lane_px, x2);
                float gw[KP];
                lds_gw<float, KP>(gw, gs + (size_t)c * KP * sizeof(float));
                float2 tloc[KP];
                float2 (&t2)[KP] = ACC_REG ? acc2[ACC_REG ? ci : 0] : tloc;
                if constexpr (!ACC_REG) {
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) tloc[kk] = make_float2(0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    float2 y = __fmul2_rn(dup2(gw[0]), h2[0][j]);
#pragma unroll
                    for (int kk = 1; kk < KP; ++kk) y = __ffma2_rn(dup2(gw[kk]), h2[kk][j], y);
                    const float2 r = __fmul2_rn(x2[j], make_float2(rcp_ftz(y.x), rcp_ftz(y.y)));
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) t2[kk] = __ffma2_rn(r, h2[kk][j], t2[kk]);
                }
                if constexpr (!ACC_REG) {
                    float mine = 0.f;
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) {
                        const float sv = warp_sum(tloc[kk].x + tloc[kk].y);
                        if (lane == kk) mine = sv;
                    }
                    if (lane < KP) tail[((size_t)half * G::CS + c) * KP + lane] += mine;
                }
            }
        } else {
#pragma unroll
            for (int ci = 0; ci < CPW; ++ci) {
                const int c = slot + ci * G::NSLOT;
                TX xv[PPL];
                TC gw[KP];
                lds_vec<TX, PPL>(xv, xs + ((size_t)c * TILE_PX + lane_px) * sizeof(TX));
                lds_gw<TC, KP>(gw, gs + (size_t)c * KP * sizeof(TC));
                TC tloc[KP];
                TC (&t)[KP] = ACC_REG ? acc[ACC_REG ? ci : 0] : tloc;
                if constexpr (!ACC_REG) {
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) tloc[kk] = TC(0);
                }
#pragma unroll
                for (int q = 0; q < PPL; ++q) {
                    TC rq;
                    if constexpr (MODE == XMODE_FROB) {
                        rq = (TC)xv[q];                       // S = X H'^T (updates.py:33)
                    } else {
                        TC y = gw[0] * h[0][q];
#pragma unroll
                        for (int kk = 1; kk < KP; ++kk) y = fma(gw[kk], h[kk][q], y);
                        if constexpr (SAFE) {
                            if (a.clamp_y) y = Num<TC>::vmax(y, ls);
                        }
                        rq = Num<TC>::ratio((TC)xv[q], y);
                    }
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) t[kk] = fma(rq, h[kk][q], t[kk]);
                }
                if constexpr (!ACC_REG) {
                    TC mine = TC(0);
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) {
                        const TC sv = warp_sum(tloc[kk]);
                        if (lane == kk) mine = sv;
                    }
                    if (lane < KP) tail[((size_t)half * G::CS + c) * KP + lane] += mine;
                }
            }
        }
        ring.consumer_release(pos, lane);
        if (++tile == a.n_tiles && i + 1 < n_units) {
            flush(cb);   // ends with a barrier: every warp is done with gwbuf
            tile = 0;
            ++cb;
            load_gw(cb);
        }
    }
    if (n_units > 0) flush(cb);
}

}  // namespace espm
