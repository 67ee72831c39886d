// Kernels that only touch k x p / m x k data (L2 resident): per-pixel assembly of the H update, the
// lock-step simplex bisection (trace + replay), the W update, and the scalar reductions.
#pragma once
#include "common.cuh"

namespace espm {

constexpr int PX_THREADS = 256;

// KP consecutive values of one row (16-byte vector loads when the row size allows it)
template <typename T, int N>
__device__ __forceinline__ void lds_row(T (&dst)[N], const T* src) {
    constexpr int BYTES = N * (int)sizeof(T);
    if constexpr (BYTES % 16 == 0) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4 tmp[BYTES / 16];
#pragma unroll
        for (int i = 0; i < BYTES / 16; ++i) tmp[i] = s4[i];
        memcpy(dst, tmp, BYTES);
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) dst[i] = src[i];
    }
}
// the same through L2 only (ld.global.cg): data another GPU stored into this GPU's memory
template <typename T, int N>
__device__ __forceinline__ void ldcg_row(T (&dst)[N], const T* src) {
    constexpr int BYTES = N * (int)sizeof(T);
    if constexpr (BYTES % 16 == 0) {
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4 tmp[BYTES / 16];
#pragma unroll
        for (int i = 0; i < BYTES / 16; ++i) tmp[i] = __ldcg(s4 + i);
        memcpy(dst, tmp, BYTES);
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) dst[i] = __ldcg(src + i);
    }
}
constexpr int PX_WARPS = PX_THREADS / 32;

// ESPM_FLAG_TIMING: one thread leaves a %globaltimer stamp in the record (diagnostics only)
__device__ __forceinline__ void time_stamp(const espm_state& st, int which) {
    if (st.flags & ESPM_FLAG_TIMING) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        st.scalars[ESPM_S_T0 + which] = (double)t;
    }
}

// ------------------------------------------------------------------------------------------------
// Peer exchange primitives (ESPM_FLAG_PEER): system-scope flags in CUDA-IPC memory over NVLink.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// Threads 0..world-1 of the CTA wait until flags[r] has reached `seq` for every rank r; bounded (~1 s) so
// that a dead peer turns into ESPM_DEV_PEER_TIMEOUT instead of a hung GPU.  Ends with __syncthreads().
__device__ __forceinline__ void wait_peer_flags(const uint32_t* flags, int world, uint32_t seq, uint32_t* dev_flags) {
    if ((int)threadIdx.x < world) {
        const long long t0 = clock64();
        while ((int32_t)(ld_acquire_sys(flags + threadIdx.x) - seq) < 0) {
            if (clock64() - t0 > (1ll << 31)) {
                atomicOr(dev_flags, ESPM_DEV_PEER_TIMEOUT);
                break;
            }
            __nanosleep(64);
        }
    }
    __syncthreads();
}

// px_part row layout (doubles), sums first, maxima last:
//   [0] log-reg  [1] laplacian trace  [2 + kk] rowsum(H_next)  [2 + kp + kk] rowsum(max(H_next, ls))
//   [2 + 2kp] rel_H max   [3 + 2kp + kk] rowmax(H_next)
__host__ __device__ inline int px_part_stride(int kp) { return 3 + 3 * kp; }
__host__ __device__ inline int px_part_nsum(int kp) { return 2 + 2 * kp; }

// ------------------------------------------------------------------------------------------------
// simplex function  f(x) = sum_k max(num_k / (x + den_k), ls) - 1   (dicotomy.py:51-53)
// Sequential sum over k like the NumPy reference.  The fp64 quotient is the Newton reciprocal plus one
// residual correction (q' = q + (a - b q) r): correctly rounded like the IEEE division NumPy uses, except
// for rare double-rounding cases, at a third of the cost.  Bit-level agreement matters: when a pixel has
// no counts the root sits within a few ulps of -den and the bisection result is decided by the last bit
// of f (it then runs to maxit, dicotomy.py:169-171).
// ------------------------------------------------------------------------------------------------
template <typename TC>
__device__ __forceinline__ TC simplex_quot(TC a, TC b) {
    if constexpr (sizeof(TC) == 8) {
        const double r = Num<double>::rcp(b);
        const double q = a * r;
        const double rem = fma(-b, q, a);
        return fma(rem, r, q);
    } else {
        return a / b;
    }
}
template <typename TC, int KP>
__device__ __forceinline__ TC simplex_f(const TC (&num)[KP], const TC (&den)[KP], TC x, int k, TC ls) {
    TC s = Num<TC>::vmax(simplex_quot<TC>(num[0], x + den[0]), ls);
#pragma unroll
    for (int kk = 1; kk < KP; ++kk)
        if (kk < k) s += Num<TC>::vmax(simplex_quot<TC>(num[kk], x + den[kk]), ls);
    return s - TC(1);
}

// bracket of dicotomy.py:29-49
template <typename TC, int KP>
__device__ __forceinline__ void simplex_bracket(const TC (&num)[KP], const TC (&den)[KP], int k, TC& a, TC& b) {
    TC amax = -Num<TC>::inf(), nmax = num[0], dmin = den[0];
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
        if (kk < k) {
            if (num[kk] > TC(0)) amax = Num<TC>::vmax(amax, num[kk] / TC(2) - den[kk]);
            nmax = Num<TC>::vmax(nmax, num[kk]);
            dmin = Num<TC>::vmin(dmin, den[kk]);
        }
    a = amax;
    b = (TC)k * nmax / TC(0.5) - dmin;
}

struct Mask128 {
    uint32_t w[4];
    __device__ __forceinline__ void clear() { w[0] = w[1] = w[2] = w[3] = 0u; }
    __device__ __forceinline__ void set(int j) {
        const uint32_t bit = 1u << (j & 31);
        const int wi = j >> 5;
        w[0] |= (wi == 0) ? bit : 0u;
        w[1] |= (wi == 1) ? bit : 0u;
        w[2] |= (wi == 2) ? bit : 0u;
        w[3] |= (wi == 3) ? bit : 0u;
    }
    __device__ __forceinline__ void set_from(int j, int end) {  // bits [j, end)
        for (int i = j; i < end; ++i) set(i);
    }
    __device__ __forceinline__ void or_word(int wi, uint32_t v) {
        w[0] |= (wi == 0) ? v : 0u;
        w[1] |= (wi == 1) ? v : 0u;
        w[2] |= (wi == 2) ? v : 0u;
        w[3] |= (wi == 3) ? v : 0u;
    }
    __device__ __forceinline__ bool get(int j) const {
        const int wi = j >> 5;
        const uint32_t v = (wi == 0) ? w[0] : (wi == 1) ? w[1] : (wi == 2) ? w[2] : w[3];
        return (v >> (j & 31)) & 1u;
    }
};

// first clear bit in [0, maxit) of the global trace mask, or maxit (dicotomy.py:152,169-171)
__device__ __forceinline__ int first_clear_bit(const uint32_t* mask, int maxit) {
    for (int wv = 0; wv < 4; ++wv) {
        const uint32_t inv = ~mask[wv];
        if (inv) {
            const int j = wv * 32 + (__ffs((int)inv) - 1);
            return j < maxit ? j : maxit;
        }
    }
    return maxit;
}

// Lock-step trace of one column's bisection (dicotomy.py:138-171) for a monotone f with f(a) > 0 > f(b):
// records for every iteration j whether |f(new_j)| > tol.  Exits early when every later midpoint is
// provably within tol (f is monotone on the bracket) or when the bracket is stationary in floating
// point (then new, and the bit, never change again).
template <typename TC, typename F>
__device__ __forceinline__ void bisect_trace(TC a, TC b, F&& f, TC tol, int maxit, Mask128& bits, uint32_t& err) {
    TC fa = f(a);
    TC fb = f(b);
    // dicotomy.py:141-144 preconditions
    if (!(fa > TC(0)) || !(fb < TC(0))) err |= ESPM_DEV_BRACKET;
    TC nw = (a + b) / TC(2);
    TC fn = f(nw);
    for (int j = 0; j < maxit; ++j) {
        const bool bad = Num<TC>::vabs(fn) > tol;
        if (bad) bits.set(j);
        if (fa <= tol && -fb <= tol) break;
        if (nw == a || nw == b) {
            if (bad) bits.set_from(j + 1, maxit);
            break;
        }
        if (fa * fn <= TC(0)) {
            b = nw;
            fb = fn;
        } else {
            a = nw;
            fa = fn;
        }
        nw = (a + b) / TC(2);
        fn = f(nw);
    }
}

// Replays exactly `its` updates of dicotomy.py:152-168 and returns new.
template <typename TC, typename F>
__device__ __forceinline__ TC bisect_replay(TC a, TC b, F&& f, int its) {
    TC fa = f(a);
    TC nw = (a + b) / TC(2);
    TC fn = f(nw);
    for (int j = 0; j < its; ++j) {
        if (nw == a || nw == b) break;  // stationary: new no longer changes
        if (fa * fn <= TC(0)) {
            b = nw;
        } else {
            a = nw;
            fa = fn;
        }
        nw = (a + b) / TC(2);
        fn = f(nw);
    }
    return nw;
}

template <typename TC, int KP>
__device__ __forceinline__ void simplex_trace(const TC (&num)[KP], const TC (&den)[KP], int k, TC ls, TC tol,
                                              int maxit, Mask128& bits, uint32_t& err) {
    TC a, b;
    simplex_bracket<TC, KP>(num, den, k, a, b);
    bisect_trace<TC>(a, b, [&](TC x) { return simplex_f<TC, KP>(num, den, x, k, ls); }, tol, maxit, bits, err);
}

template <typename TC, int KP>
__device__ __forceinline__ TC simplex_replay(const TC (&num)[KP], const TC (&den)[KP], int k, TC ls, int its) {
    TC a, b;
    simplex_bracket<TC, KP>(num, den, k, a, b);
    return bisect_replay<TC>(a, b, [&](TC x) { return simplex_f<TC, KP>(num, den, x, k, ls); }, its);
}

// ------------------------------------------------------------------------------------------------
// Quadratic-surrogate simplex function (algo="l2_surrogate", dicotomy.py:57-81), always in fp64:
//   f(x) = 2a - sum_k max( sqrt((b_k + x)^2 + 4 a c_k) - x - b_k, 2 a ls )
// increasing in x; bracket (f > 0 at nu_max, f < 0 at nu_min) of dicotomy.py:74-75.  Written with
// explicit round-to-nearest operations (no FMA contraction) so that the sign decisions of the
// bisection follow NumPy's.
// ------------------------------------------------------------------------------------------------
template <int KP>
__device__ __forceinline__ double acc_f(const double (&c)[KP], const double (&b)[KP], double x, int k, double a,
                                        double ls) {
    const double four_a = 4.0 * a, floor_v = __dmul_rn(ls * 2.0, a);
    double s = 0.0;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
        if (kk < k) {
            const double t = __dadd_rn(b[kk], x);
            const double q = __dadd_rn(__dmul_rn(t, t), __dmul_rn(four_a, c[kk]));
            double g = __dsub_rn(__dsub_rn(sqrt(q), x), b[kk]);
            g = fmax(g, floor_v);
            s = (kk == 0) ? g : __dadd_rn(s, g);
        }
    return __dsub_rn(2.0 * a, s);
}
template <int KP>
__device__ __forceinline__ void acc_bracket(const double (&c)[KP], const double (&b)[KP], int k, double a,
                                            double& nu_max, double& nu_min) {
    double mx = -Num<double>::inf(), sb = 0.0;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
        if (kk < k) {
            const double v = __dadd_rn(__dadd_rn(__ddiv_rn(__dmul_rn(b[kk], b[kk]), a), 2.0 * a),
                                       __dmul_rn(2.0, __dadd_rn(b[kk], c[kk])));
            mx = fmax(mx, v);
            sb = (kk == 0) ? b[kk] : __dadd_rn(sb, b[kk]);
        }
    nu_max = __dadd_rn(__dmul_rn(__dmul_rn((double)k, mx), 1.5), 1e-3);
    nu_min = __dsub_rn(__dmul_rn(__ddiv_rn(-__dadd_rn(2.0 * a, sb), (double)k), 1.1), 1e-3);
}
template <int KP>
__device__ __forceinline__ void acc_trace(const double (&c)[KP], const double (&b)[KP], int k, double a, double ls,
                                          double tol, int maxit, Mask128& bits, uint32_t& err) {
    double lo, hi;
    acc_bracket<KP>(c, b, k, a, lo, hi);
    bisect_trace<double>(lo, hi, [&](double x) { return acc_f<KP>(c, b, x, k, a, ls); }, tol, maxit, bits, err);
}
template <int KP>
__device__ __forceinline__ double acc_replay(const double (&c)[KP], const double (&b)[KP], int k, double a, double ls,
                                             int its) {
    double lo, hi;
    acc_bracket<KP>(c, b, k, a, lo, hi);
    return bisect_replay<double>(lo, hi, [&](double x) { return acc_f<KP>(c, b, x, k, a, ls); }, its);
}
// ------------------------------------------------------------------------------------------------
// Recorded lock-step bisection of the H update (h_finish traces, h_apply replays).
//
// The reference's loop (dicotomy.py:152-168) needs, per midpoint, only two facts about f(new):
//   le0 : f(new) <= 0   (then b = new, else a = new; f(a) > 0 is an invariant of the loop)
//   bad : |f(new)| > tol (the global stop test ORs this over all pixels)
// An evaluator returns both.  The KL evaluator first SCREENS f in fp32 (one MUFU.RCP per phase instead
// of a correctly rounded fp64 quotient) and accepts the answer only when it is certain, i.e. when
// |f32| and | |f32| - tol | exceed a bound on |f32 - f_exact|; otherwise it evaluates f exactly like the
// reference (simplex_f).  Bound: fl32(x + den) 2^-24, rcp.approx 2^-23, fl32(num) 2^-24, product 2^-24
// => 3.0e-7 relative per term; (k-1) fp32 additions of partial sums <= s => 6e-8 (k-1) s; the final s - 1
// 6e-8 |f|.  The margin used is 1.25 x that bound: (4.5e-7 + 7.5e-8 (k-1)) s + 1e-7 |f| + 2e-8.
// Pixels whose num has entries outside [1e-30, 1e30] (fp32 under/overflow) are never screened.
// The trace also records the decisions, so that the replay of the it* global iterations is pure
// bracket arithmetic for every iteration the trace has seen.
// ------------------------------------------------------------------------------------------------
struct Cls {
    bool le0, bad;
};

template <int KP>
struct KlEval {
    const double (&num)[KP];
    const double (&den)[KP];
    float numf[KP];
    int k;
    double ls, tol;
    float lsf, tolf, mrel;
    bool screen;
    __device__ __forceinline__ KlEval(const double (&num_)[KP], const double (&den_)[KP], int k_, double ls_, double tol_)
        : num(num_), den(den_), k(k_), ls(ls_), tol(tol_) {
        lsf = (float)ls_;
        tolf = (float)tol_;
        mrel = 4.5e-7f + 7.5e-8f * (float)(k_ - 1);   // 1.25 x (2.98e-7 per term + 5.96e-8 per addition)
        screen = true;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            numf[kk] = (kk < k) ? (float)num[kk] : 0.f;
            if (kk < k && num[kk] != 0.0 && !(num[kk] >= 1e-30 && num[kk] <= 1e30)) screen = false;
        }
    }
    __device__ __forceinline__ double exact(double x) const { return simplex_f<double, KP>(num, den, x, k, ls); }
    // fp32 screen: returns false when the fp32 value cannot be trusted
    __device__ __forceinline__ bool screen_f(double x, float& f, float& margin) const {
        float sacc = 0.f;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) {
                const float t = __double2float_rn(x + den[kk]);
                float r;
                asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t));
                const float q = fmaxf(numf[kk] * r, lsf);
                sacc = (kk == 0) ? q : sacc + q;
            }
        f = sacc - 1.0f;
        margin = mrel * sacc + 1e-7f * fabsf(f) + 2e-8f;
        return true;
    }
    __device__ __forceinline__ Cls operator()(double x) const {
        if (screen) {
            float f, margin;
            screen_f(x, f, margin);
            const float af = fabsf(f);
            if (af > margin && fabsf(af - tolf) > margin + 1e-7f * tolf) return Cls{f <= 0.f, af > tolf};
        }
        const double fe = exact(x);
        return Cls{fe <= 0.0, fabs(fe) > tol};
    }
    __device__ __forceinline__ bool le0(double x) const {
        if (screen) {
            float f, margin;
            screen_f(x, f, margin);
            if (fabsf(f) > margin) return f <= 0.f;
        }
        return exact(x) <= 0.0;
    }
};

template <int KP>
struct AccEval {   // quadratic surrogate (dicotomy.py:57-81): always exact
    const double (&c)[KP];
    const double (&b)[KP];
    int k;
    double a, ls, tol;
    __device__ __forceinline__ AccEval(const double (&c_)[KP], const double (&b_)[KP], int k_, double a_, double ls_,
                                       double tol_)
        : c(c_), b(b_), k(k_), a(a_), ls(ls_), tol(tol_) {}
    __device__ __forceinline__ double exact(double x) const { return acc_f<KP>(c, b, x, k, a, ls); }
    __device__ __forceinline__ Cls operator()(double x) const {
        const double fe = exact(x);
        return Cls{fe <= 0.0, fabs(fe) > tol};
    }
    __device__ __forceinline__ bool le0(double x) const { return exact(x) <= 0.0; }
};

template <int KP>
struct PgEval {    // projected gradient (dicotomy.py:83-108): f(x) = sum_k max(a_k + x, ls) - 1, always exact
    const double (&av)[KP];
    int k;
    double ls, tol;
    __device__ __forceinline__ PgEval(const double (&a_)[KP], int k_, double ls_, double tol_)
        : av(a_), k(k_), ls(ls_), tol(tol_) {}
    __device__ __forceinline__ double exact(double x) const {
        double s = 0.0;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) {
                const double g = fmax(__dadd_rn(av[kk], x), ls);
                s = (kk == 0) ? g : __dadd_rn(s, g);
            }
        return __dsub_rn(s, 1.0);
    }
    __device__ __forceinline__ Cls operator()(double x) const {
        const double fe = exact(x);
        return Cls{fe <= 0.0, fabs(fe) > tol};
    }
    __device__ __forceinline__ bool le0(double x) const { return exact(x) <= 0.0; }
    // dicotomy.py:99-100: (nu_max, nu_min) = (1/k - min a, -max a)
    __device__ __forceinline__ void bracket(double& lo, double& hi) const {
        double mn = av[0], mx = av[0];
#pragma unroll
        for (int kk = 1; kk < KP; ++kk)
            if (kk < k) {
                mn = fmin(mn, av[kk]);
                mx = fmax(mx, av[kk]);
            }
        lo = __dsub_rn(__ddiv_rn(1.0, (double)k), mn);
        hi = -mx;
    }
};

// word 4 of a pixel's decision record: iterations seen by the trace | stationary flag
constexpr uint32_t BIS_STATIONARY = 1u << 8;

// sign and size class of f at a bracket end; the KL evaluator answers from its fp32 screen when that is certain
// (f(a) >= 1 and f(b) <= -1/2 by construction of the bracket, dicotomy.py:29-49, so it practically always is)
struct End {
    bool pos, neg, bad;
};
template <typename E>
__device__ __forceinline__ End end_of(const E& ev, double x) {
    const double f = ev.exact(x);
    return End{f > 0.0, f < 0.0, fabs(f) > ev.tol};
}
template <int KP>
__device__ __forceinline__ End end_of(const KlEval<KP>& ev, double x) {
    if (ev.screen) {
        float f, margin;
        ev.screen_f(x, f, margin);
        const float af = fabsf(f);
        if (af > margin && fabsf(af - ev.tolf) > margin + 1e-7f * ev.tolf) return End{f > 0.f, f < 0.f, af > ev.tolf};
    }
    const double f = ev.exact(x);
    return End{f > 0.0, f < 0.0, fabs(f) > ev.tol};
}

// ------------------------------------------------------------------------------------------------
// Root-anchored evaluator of the KL simplex function  f(x) = sum_k max(n_k / (x + d_k), ls) - 1.
//
// The lock-step loop of the reference needs, per midpoint, only the sign of f and whether |f| > tol.  f is convex and
// decreasing on the bracket (every t_k = x + d_k > 0 there), so both facts follow from WHERE the midpoint lies
// relative to the root nu* of f, which is computed once per pixel:
//   * Newton on g(x) = 1 / S(x) - 1, S = sum_k n_k / t_k.  g is concave and increasing (Cauchy-Schwarz:
//     2 S'^2 <= S S''), so from the left end of the bracket the iterates increase monotonically to nu* without
//     overshooting, and a single hyperbola is solved in one step; 4-6 fp64 iterations in practice.
//   * sign:   f(x) <= 0  <=>  x >= nu*                                       (monotone)
//   * size, left of the root  (e = nu* - x > 0):   D e <= f(x) <= D e + 0.52 F2 e^2     (tangent below a convex f;
//                                                    Taylor with f'' <= 1.031 f''(nu*) while e <= 0.01 min_k t_k)
//   * size, right of the root (e = x - nu* > 0):   D e - F2 e^2 / 2 <= |f(x)| <= D e   (f'' is decreasing), and
//                                                    |f(x)| >= 0.4999 e / (b0 - nu*)    (chord to the initial right
//                                                    end b0, where f <= -1/2 by construction, dicotomy.py:49)
//     with D = |f'(nu*)|, F2 = f''(nu*).
// A midpoint is classified from these bounds only when they decide it with a margin that covers the rounding of the
// reference's own evaluation (|x - nu*| > mx, see below) and of ours (1e-9 relative on tol); every other midpoint --
// the root within rounding distance, |f| within the bounds' gap of tol, no convergence, negative inputs -- goes
// through KlEval, i.e. the fp32 screen and then the bit-faithful evaluation.  The anchor therefore never changes a
// decision; it only avoids evaluating f where the answer is already certain.
//   mx = 1e-12 / D + (8 + 2k) 2^-52 (max(|a0|, |b0|) + max_k |d_k|): beyond it |f| >= D |x - nu*| > 1e-12 (the
//   reference's evaluation of f is accurate to a few k 2^-53) and the fp64 Newton iterate is that close to the true
//   root (its last step was <= 2 ulps; each evaluation of S carries <= k/2 ulps of x of noise when x + d_k cancels).
//   The size bounds additionally need D to be accurate to 1e-10, i.e. ulp(x) / min_k t_k small (`sized`).
// ------------------------------------------------------------------------------------------------
template <int KP>
struct KlAnchorEval {
    KlEval<KP> base;
    double nu, mx, tol;
    double eLlo, eLhi, eRlo, eRhi;     // |x - nu*| below / above which |f(x)| <= tol / > tol is certain, per side
    bool ok;
    // `warm`: a guess of the root (the pixel's root of the previous NMF iteration) or NaN.  From any point of the domain
    // the iteration is safe: right of the root the tangent of the concave g lands left of it, from there on the
    // iterates increase monotonically.
    __device__ __forceinline__ KlAnchorEval(const double (&num)[KP], const double (&den)[KP], int k, double ls, double tol_,
                                            double a0, double b0, double warm)
        : base(num, den, k, ls, tol_), tol(tol_) {
        ok = false;
        nu = mx = 0.0;
        eLlo = eRlo = 0.0;
        eLhi = eRhi = Num<double>::inf();
        bool valid = (a0 > -1e300) && (b0 < 1e300) && (a0 < b0);
        double dmax = 0.0;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) {
                valid = valid && (num[kk] >= 0.0) && (fabs(den[kk]) < 1e300);
                dmax = fmax(dmax, fabs(den[kk]));
            }
        if (!valid) return;
        double x = (warm > a0 && warm < b0) ? warm : a0, S = 0.0, Dv = 0.0, F2v = 0.0, tm = 1e300;
        bool conv = false;
#pragma unroll 1
        for (int it = 0; it < 24; ++it) {
            S = 0.0;
            Dv = 0.0;
            F2v = 0.0;
            tm = 1e300;
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
                if (kk < k) {
                    const double t = x + den[kk];
                    const double r = Num<double>::rcp(t);
                    const double q = num[kk] * r;
                    if (q > ls) {             // clamped terms are constants: no slope, no curvature
                        S += q;
                        const double qr = q * r;
                        Dv += qr;
                        F2v = fma(qr, r, F2v);
                        tm = fmin(tm, t);
                    } else {
                        S += ls;
                    }
                }
            if (!(S > 0.0) || !(Dv > 0.0) || !(tm > 0.0)) return;     // NaN / outside the domain: no anchor
            if (fabs(S - 1.0) <= 4e-15) {
                conv = true;
                break;
            }
            const double xn = x + S * (S - 1.0) * Num<double>::rcp(Dv);
            if (!(xn < 1e300)) return;
            if (!(xn > a0)) {                 // a warm start far right of the root overshot the domain: restart at a0
                if (x == a0) return;
                x = a0;
                continue;
            }
            // the step is within 2 ulps of x: converged as far as fp64 resolves the root (when x + d_k cancels, the
            // residual cannot get smaller than D ulp(x); mx below covers that distance)
            conv = fabs(xn - x) <= 4.5e-16 * fabs(x);
            x = xn;
            if (conv) break;
        }
        if (!conv || !(x > a0) || !(x < b0)) return;
        nu = x;
        const double D = Dv, F2 = 2.0 * F2v, invD = Num<double>::rcp(Dv);
        // (the last evaluation was at the previous iterate when the loop ended on a 2-ulp step: D, F2, tmin move by
        //  O(ulp(x) / tmin) relative, which `sized` bounds)
        const double span = fmax(fabs(a0), fabs(b0)) + dmax;
        mx = 1e-12 * invD + (double)(8 + 2 * k) * 2.3e-16 * span;
        ok = true;
        if (1e-15 * span <= 1e-10 * tm) {       // D is accurate to 1e-10: the size bounds can be used (else sign only)
            // |f| is monotone in the distance e from the root on either side, so every bound turns into a threshold on e:
            const double hi = tol * (1.0 + 1e-9), lo = tol * (1.0 - 1e-9);
            eLhi = hi * invD;                                                    // left:  f >= D e
            eLlo = fmin(0.01 * tm, lo * Num<double>::rcp(D + 0.52 * F2 * lo * invD)); //  f <= D e + 0.52 F2 e^2, e <= 0.01 tmin
            eRlo = lo * invD;                                                    // right: |f| <= D e
            const double q = F2 * hi * invD * invD;                              //        |f| >= D e - F2 e^2 / 2:
            const double chord_e = hi * (b0 - x) * (1.0 / 0.4999);               //        |f| >= 0.4999 e / (b0 - nu*)
            // for q < 1/4: D e - F2 e^2 / 2 >= (D - F2 hi / D) e > hi on (hi / (D (1 - q)), 2 hi / D], and beyond that
            // |f(e)| >= |f(2 hi / D)| >= 2 hi (1 - q) > hi
            eRhi = q < 0.25 ? fmin(chord_e, hi * invD * Num<double>::rcp(1.0 - q)) : chord_e;
            eLhi = fmax(eLhi, mx);
            eRhi = fmax(eRhi, mx);
        }
    }
    __device__ __forceinline__ double exact(double x) const { return base.exact(x); }
    __device__ __forceinline__ Cls operator()(double x) const {
        if (ok) {
            const double d = x - nu, e = fabs(d);
            if (e > mx) {
                const bool right = d > 0.0;
                if (e > (right ? eRhi : eLhi)) return Cls{right, true};
                if (e < (right ? eRlo : eLlo)) return Cls{right, false};
                // the sign is certain, the size class is not: evaluate like the reference
                return Cls{right, fabs(base.exact(x)) > tol};
            }
        }
        return base(x);
    }
    __device__ __forceinline__ bool le0(double x) const {
        if (ok && fabs(x - nu) > mx) return x > nu;
        return base.le0(x);
    }
};
// ends of the initial bracket: with a valid anchor a0 < nu* < b0 and |f| >= 1/2 there (dicotomy.py:29-49)
template <int KP>
__device__ __forceinline__ End end_of(const KlAnchorEval<KP>& ev, double x) {
    if (ev.ok) {
        const double d = x - ev.nu, e = fabs(d);
        if (e > ev.mx && e > (d > 0.0 ? ev.eRhi : ev.eLhi)) return End{d < 0.0, d > 0.0, true};
    }
    return end_of(ev.base, x);
}

// replay-side view of the anchor (h_apply): only the sign decisions are needed
template <int KP>
struct KlAnchorReplay {
    KlEval<KP> base;
    double nu, mx, tol;
    __device__ __forceinline__ KlAnchorReplay(const double (&num)[KP], const double (&den)[KP], int k, double ls, double tol_,
                                              double nu_, double mx_)
        : base(num, den, k, ls, tol_), nu(nu_), mx(mx_), tol(tol_) {}
    __device__ __forceinline__ double exact(double x) const { return base.exact(x); }
    __device__ __forceinline__ bool le0(double x) const {
        if (fabs(x - nu) > mx) return x > nu;      // mx = +inf when the pixel has no anchor
        return base.le0(x);
    }
};

// "Far" midpoints of a root-anchored evaluator: while |new - nu*| exceeds every size threshold (and the rounding margin
// mx), the evaluator's answer is {sign by side, |f| > tol} without looking at anything else -- see
// KlAnchorEval::operator().  far_info() hands the trace loop the root and that distance (false: no such shortcut).
template <typename E>
__device__ __forceinline__ bool far_info(const E&, double&, double&) {
    return false;
}
template <int KP>
__device__ __forceinline__ bool far_info(const KlAnchorEval<KP>& ev, double& nu, double& dist) {
    if (!ev.ok) return false;
    nu = ev.nu;
    dist = fmax(fmax(ev.eLhi, ev.eRhi), ev.mx);     // +inf when the size bounds are unusable: the fast loop never runs
    return true;
}

template <typename E>
__device__ __forceinline__ void bisect_trace_rec(double a, double b, const E& ev, int maxit, Mask128& bad, Mask128& dec,
                                                 uint32_t& seen, uint32_t& err) {
    // f at the two ends: only their signs and whether they are within tol matter (dicotomy.py:141-144)
    const End ea = end_of(ev, a), eb = end_of(ev, b);
    if (!ea.pos || !eb.neg) err |= ESPM_DEV_BRACKET;
    bool a_ok = !ea.bad, b_ok = !eb.bad;                     // is the end of the bracket already within tol?
    double nw = (a + b) * 0.5;
    int j = 0, widx = 0;
    uint32_t stat = 0u;
    uint32_t wb = 0u, wd = 0u, bit = 1u;    // bits of the current 32-iteration word
    // Fast loop over the far midpoints (typically the first ~17 of ~21 iterations): a dozen instructions each instead
    // of the general body below.  It takes exactly the decisions the general body would take: the evaluator returns
    // {new > nu*, bad} there; the moved end is not within tol, so `a_ok && b_ok` stays false; nu* stays inside [a, b],
    // so a stationary bracket (new == a or b) is at most one ulp from nu*, i.e. within mx, and ends this loop.
    {
        double nu_far = 0.0, dist = 0.0;
        if (far_info(ev, nu_far, dist) && !(a_ok && b_ok)) {
            while (j < maxit && j < 31) {
                const double d = nw - nu_far;
                if (!(fabs(d) > dist)) break;
                wb |= bit;
                if (d > 0.0) {
                    b = nw;
                    b_ok = false;
                    wd |= bit;
                } else {
                    a = nw;
                    a_ok = false;
                }
                nw = (a + b) * 0.5;
                bit <<= 1;
                ++j;
            }
        }
    }
    for (; j < maxit; ++j) {
        const Cls c = ev(nw);
        if (c.bad) wb |= bit;
        if (a_ok && b_ok) break;            // f is monotone: every later midpoint is within tol as well
        if (nw == a || nw == b) {           // stationary in floating point: new (and its bit) never change again
            if (c.bad) bad.set_from(j + 1, maxit);
            stat = BIS_STATIONARY;
            break;
        }
        if (c.le0) {
            b = nw;
            b_ok = !c.bad;
            wd |= bit;
        } else {
            a = nw;
            a_ok = !c.bad;
        }
        nw = (a + b) * 0.5;
        bit <<= 1;
        if (bit == 0u) {
            bad.or_word(widx, wb);
            dec.or_word(widx, wd);
            wb = wd = 0u;
            bit = 1u;
            ++widx;
        }
    }
    bad.or_word(widx, wb);
    dec.or_word(widx, wd);
    seen = (uint32_t)j | stat;
}

// new after exactly `its` updates of dicotomy.py:152-168: recorded decisions first, evaluations after
template <typename E>
__device__ __forceinline__ double bisect_replay_rec(double a, double b, const E& ev, int its, const Mask128& dec,
                                                    uint32_t seen) {
    const int e = (int)(seen & 0xffu);
    const int jb = its < e ? its : e;
    double nw = (a + b) * 0.5;
    int j = 0;
    for (; j < jb; ++j) {
        if (dec.get(j)) b = nw;
        else a = nw;
        nw = (a + b) * 0.5;
    }
    if (!(seen & BIS_STATIONARY)) {
        for (; j < its; ++j) {
            if (nw == a || nw == b) break;
            if (ev.le0(nw)) b = nw;
            else a = nw;
            nw = (a + b) * 0.5;
        }
    }
    return nw;
}

// updates.py:289: H' = (-b + sqrt(b^2 + 4 a c)) / (2 a)
__device__ __forceinline__ double hq_root(double c, double b, double a) {
    const double q = __dadd_rn(__dmul_rn(b, b), __dmul_rn(4.0 * a, c));
    return __ddiv_rn(__dadd_rn(-b, sqrt(q)), 2.0 * a);
}

// OR-reduce a per-thread mask over the block and merge it into the global mask / error word.
__device__ __forceinline__ void merge_mask(const Mask128& bits, uint32_t err, uint32_t* gmask, uint32_t* gflags) {
    __shared__ uint32_t sm_mask[5];
    if (threadIdx.x < 5) sm_mask[threadIdx.x] = 0u;
    __syncthreads();
    uint32_t v[5] = {bits.w[0], bits.w[1], bits.w[2], bits.w[3], err};
#pragma unroll
    for (int i = 0; i < 5; ++i) {
        const uint32_t r = __reduce_or_sync(0xffffffffu, v[i]);
        if ((threadIdx.x & 31) == 0 && r) atomicOr(&sm_mask[i], r);
    }
    __syncthreads();
    if (threadIdx.x < 4 && sm_mask[threadIdx.x] && gmask) atomicOr(&gmask[threadIdx.x], sm_mask[threadIdx.x]);
    if (threadIdx.x == 4 && sm_mask[4]) atomicOr(&gflags[0], sm_mask[4]);
}

// Block reduction of NV per-thread doubles (sum for i < n_sum, max afterwards) into out[NV].
// Fixed order (lane butterfly, then warps 0..7) => run-to-run deterministic.
template <int NV>
__device__ __forceinline__ void block_reduce_vals(const double (&vals)[NV], int n_sum, double* out) {
    __shared__ double sm_vals[PX_WARPS][NV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        const double r = (i < n_sum) ? warp_sum(vals[i]) : warp_max(vals[i]);
        if (lane == 0) sm_vals[warp][i] = r;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double r = sm_vals[0][threadIdx.x];
        for (int w = 1; w < PX_WARPS; ++w) {
            const double u = sm_vals[w][threadIdx.x];
            r = ((int)threadIdx.x < n_sum) ? r + u : (u > r ? u : r);
        }
        out[threadIdx.x] = r;
    }
}

// H' of one pixel from the multiplier nu of its simplex constraint (updates.py:152, 289, 387): ONE definition, used by the
// speculative replay inside h_finish and by h_apply, so that both produce the same bits.
template <typename TC, int KP>
__device__ __forceinline__ void h_from_nu(const espm_state& st, const double (&num)[KP], const double (&den)[KP], int k,
                                          double nu, double sigma, TC (&hn)[KP]) {
    if (st.flags & ESPM_FLAG_PG) {                                         // updates.py:381-387
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) hn[kk] = (kk < k) ? (TC)fmax(num[kk] + nu, st.log_shift) : TC(0);
    } else if ((st.flags & ESPM_FLAG_HQ) && (st.flags & ESPM_FLAG_LAPLACIAN)) {   // updates.py:286-289
        const double a = st.lambda_L * sigma;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            hn[kk] = (kk < k) ? (TC)fmax(hq_root(num[kk], den[kk] + nu, a), st.log_shift) : TC(0);
    } else {
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            hn[kk] = (kk < k) ? (TC)fmax(num[kk] / (den[kk] + nu), st.log_shift) : TC(0);
    }
}

template <typename TC, int KP>
__device__ __forceinline__ void store_h_next(const espm_state& st, int j, int k, const TC (&hn)[KP],
                                             double (&vals)[3 + 3 * KP]) {
    TC* Hn = reinterpret_cast<TC*>(st.H_next);
    TC* Ht = reinterpret_cast<TC*>(st.Ht);
    const TC* fx = reinterpret_cast<const TC*>(st.fixed_H);
    const TC ls = (TC)st.log_shift;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk)
        if (kk < k) {
            TC v = hn[kk];
            if (st.flags & ESPM_FLAG_FIXED_H) {  // updates.py:154-155
                const TC f = fx[(size_t)kk * st.ldh + j];
                if (f >= TC(0)) v = f;
            }
            Hn[(size_t)kk * st.ldh + j] = v;
            Ht[((size_t)(j / TILE_PX) * KP + kk) * TILE_PX + (j % TILE_PX)] = v;   // tile-major copy for the W pass
            if (st.flags & ESPM_FLAG_PEER) {
                // Laplacian halo: my first / last image row lands in the neighbours' H_next (peer stores)
                if (st.nb_prev_halo && j < st.ny)
                    reinterpret_cast<TC*>(st.nb_prev_halo)[(size_t)kk * st.nb_prev_ldh + j] = v;
                if (st.nb_next_halo && j >= st.p_loc - st.ny)
                    reinterpret_cast<TC*>(st.nb_next_halo)[(size_t)kk * st.nb_next_ldh + (j - (st.p_loc - st.ny))] = v;
            }
            vals[2 + kk] = (double)v;
            vals[2 + KP + kk] = (double)Num<TC>::vmax(v, ls);
            vals[3 + 2 * KP + kk] = (double)v;
        }
}

template <typename TC>
__device__ __forceinline__ void h_scalars_block(const espm_state& st, double* share);

// ------------------------------------------------------------------------------------------------
// h_finish: per-pixel assembly (updates.py:132-152) + loss regularisers + rel_H + bisection trace
// ------------------------------------------------------------------------------------------------
// OCC: CTAs per SM the kernel is compiled for.  4 (64 registers per thread) when the shard needs more than two CTAs per
// SM; 2 (128 registers: no spills, no rematerialised conversions in the root search) when the whole grid fits in
// 2 x #SM CTAs anyway -- the pixel shards of a multi-GPU fit, where the kernel is a pure latency chain.
template <typename TC, int KP, int OCC>
__global__ void __launch_bounds__(PX_THREADS, OCC) h_finish_kernel(const espm_state st) {
    pdl_wait();
    pdl_trigger();
    if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 6);
    const int j = blockIdx.x * PX_THREADS + threadIdx.x;
    const bool active = j < st.p_loc;
    const int k = st.k;
    const TC ls = (TC)st.log_shift;
    const TC* Hc = reinterpret_cast<const TC*>(st.H_cur);
    const TC* Hp = reinterpret_cast<const TC*>(st.H_prev);
    const double* hstats = reinterpret_cast<const double*>(st.hstats_cur);
    const TC* gwstats = reinterpret_cast<const TC*>(st.gwstats_cur);
    const bool lap = st.flags & ESPM_FLAG_LAPLACIAN;
    const bool use_mu = st.flags & ESPM_FLAG_MU;
    const bool simplex = st.flags & ESPM_FLAG_SIMPLEX_H;
    const bool hq = st.flags & ESPM_FLAG_HQ;   // algo="l2_surrogate" (updates.py:263-301)
    const bool quad = hq && lap;               // quadratic root / dichotomy_simplex_acc instead of num/(den+nu)
    const bool bmd = st.flags & ESPM_FLAG_BMD; // use_bregman (updates.py:120-125)
    const bool pg = st.flags & ESPM_FLAG_PG;   // proj_grad_step_h (updates.py:369-391)
    const bool l2h = st.flags & ESPM_FLAG_L2_H;  // Frobenius H step / gradient (updates.py:109-118, 330-332)
    const double sigma = st.sigma_dev ? *st.sigma_dev : st.sigma;   // gamma_ (device-resident under line search)
    // Speculative replay (simplex_H): the lock-step count it* of the bisection is a GLOBAL quantity -- known only once every
    // pixel (of every rank) has been traced -- but it hardly ever changes from one NMF iteration to the next.  dev_flags[6]
    // holds it* + 1 of the previous H update (0: none yet); this kernel replays that many iterations right after its
    // trace and writes H' (and its statistics) itself.  h_apply then only has to CONFIRM the count; it redoes the replay
    // when the guess was wrong.  dev_flags[7] tells h_apply which count was applied.
    const uint32_t spec = (simplex && !(st.flags & (ESPM_FLAG_EVAL_ONLY | ESPM_FLAG_NO_HSPEC))) ? st.dev_flags[6] : 0u;

    constexpr int NV = 3 + 3 * KP;
    double vals[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) vals[i] = 0.0;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) vals[3 + 2 * KP + kk] = -1e300;

    Mask128 bits;
    bits.clear();
    uint32_t err = 0u;

    if (active) {
        TC h[KP], HL[KP], num[KP], den[KP];
        double meanH = 0.0;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) meanH += hstats[kk];
        meanH /= ((double)k * (double)st.p_total);

        int deg = 0;
        bool up = false, down = false, left = false, right = false;
        if (st.ny > 0) {
            const int il = j / st.ny, col = j - il * st.ny;
            const int ig = st.row0 + il;
            left = col > 0;
            right = col < st.ny - 1;
            up = ig > 0;
            down = ig < st.nx - 1;
            deg = (int)left + (int)right + (int)up + (int)down;
        }
        double logreg = 0.0, lapl = 0.0, relh = 0.0;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            if (kk < k) {
                const TC* row = Hc + (size_t)kk * st.ldh;
                h[kk] = row[j];
                // ---- Laplacian stencil (utils.py:39-76; identity when shape_2d is None) ----
                if (st.ny > 0) {
                    TC nb = TC(0);
                    if (up) nb += row[j - st.ny];
                    if (left) nb += row[j - 1];
                    if (right) nb += row[j + 1];
                    if (down) nb += row[j + st.ny];
                    HL[kk] = (TC)deg * h[kk] - nb;
                } else {
                    HL[kk] = h[kk];
                }
                // ---- ratio sums of the H pass (sum of channel splits in fixed order) ----
                // (all splits are loaded before the first add: one L2 round trip instead of h_nsplit dependent ones)
                const TC* nr = reinterpret_cast<const TC*>(st.numraw) + (size_t)kk * st.p_pad + j;
                constexpr int SPU = 8;
                TC sv[SPU];
#pragma unroll
                for (int sp = 0; sp < SPU; ++sp) sv[sp] = (sp < st.h_nsplit) ? nr[(size_t)sp * KP * st.p_pad] : TC(0);
                TC s = sv[0];
#pragma unroll
                for (int sp = 1; sp < SPU; ++sp)
                    if (sp < st.h_nsplit) s += sv[sp];
                for (int sp = SPU; sp < st.h_nsplit; ++sp) s += nr[(size_t)sp * KP * st.p_pad];
                if (!(Num<TC>::vabs(s) < Num<TC>::inf())) err |= ESPM_DEV_NONFINITE;
                // ---- loss terms of the CURRENT iterate (measures.py:548, 577) ----
                if (use_mu) logreg += st.mu[kk] * (double)Num<TC>::vlog(h[kk] + (TC)st.eps_reg);
                if (lap) lapl += (double)(h[kk] * HL[kk]);
                if (st.flags & ESPM_FLAG_HAVE_HPREV) {  // base.py:324
                    const TC hp = Hp[(size_t)kk * st.ldh + j];
                    const double rr = (double)Num<TC>::vabs(h[kk] - hp) * Num<double>::rcp((double)h[kk] + st.tol * meanH);
                    relh = rr > relh ? rr : relh;
                }
                TC nm = s;
                TC dn = gwstats[kk];
                if (hq) {
                    // ---- updates.py:280-284: minus_c = H * s (s formed with y + ls), b; mu does not enter ----
                    if (lap) {
                        const TC lam = (TC)st.lambda_L;
                        dn = dn + lam * HL[kk] - (lam * (TC)sigma) * h[kk];
                    }
                    num[kk] = h[kk] * nm;
                    den[kk] = dn;
                    if (num[kk] < TC(0) || (!lap && den[kk] < TC(0))) err |= ESPM_DEV_NEGATIVE;
                } else if (pg) {
                    // ---- gradH (updates.py:316-345), new_H = H - 1/gamma * grad (updates.py:378) ----
                    TC g;
                    if (l2h) {
                        TC dd = TC(0);   // ((G W)^T (G W) H)_kk
#pragma unroll
                        for (int k2 = 0; k2 < KP; ++k2)
                            if (k2 < k) dd = fma((TC)st.gram_gw[kk * KP + k2], Hc[(size_t)k2 * st.ldh + j], dd);
                        g = dd - s;
                    } else {
                        g = -s + dn;
                    }
                    if (use_mu) g = g + (TC)st.mu[kk] / (h[kk] + (TC)st.eps_reg);
                    if (lap) {
                        // lambda_L * L is formed in FLOAT32 by the reference (utils.py:57 stores float32 entries)
                        const float lamf = (float)st.lambda_L;
                        const TC cdeg = (st.ny > 0) ? (TC)((float)deg * lamf) : (TC)lamf;
                        const TC nbs = (st.ny > 0) ? ((TC)deg * h[kk] - HL[kk]) : TC(0);   // sum of the neighbours
                        g = g + (cdeg * h[kk] - (TC)lamf * nbs);
                    }
                    num[kk] = h[kk] - (TC)(1.0 / st.gamma_h) * g;
                    den[kk] = g;   // the gradient itself (gradH of the operator-level API reads it back)
                } else if (l2h) {
                    // ---- updates.py:109-118: num = (G W)^T X, denum = (G W)^T (G W) H ----
                    TC dd = TC(0);
#pragma unroll
                    for (int k2 = 0; k2 < KP; ++k2)
                        if (k2 < k) dd = fma((TC)st.gram_gw[kk * KP + k2], Hc[(size_t)k2 * st.ldh + j], dd);
                    num[kk] = h[kk] * s;
                    den[kk] = dd;
                } else {
                    // ---- updates.py:120-142 ----
                    if (bmd) {   // sigmaR / H and the gradient of the data term (updates.py:121-125)
                        const TC t = reinterpret_cast<const TC*>(st.x_colsum)[j] / h[kk];
                        nm = t;
                        dn = (-s + dn) + t;
                    }
                    if (use_mu) dn = dn + (TC)st.mu[kk] / (h[kk] + (TC)st.eps_reg);
                    if (lap) {
                        const TC lam = (TC)st.lambda_L;
                        const TC ls_max = lam * (TC)sigma * (TC)hstats[2 * KP + kk];
                        nm = nm + ls_max;
                        dn = dn + ls_max + lam * HL[kk];
                    }
                    num[kk] = h[kk] * nm;
                    den[kk] = dn;
                    if (!bmd && (num[kk] < TC(0) || den[kk] < TC(0))) err |= ESPM_DEV_NEGATIVE;
                }
            } else {
                h[kk] = HL[kk] = num[kk] = TC(0);
                den[kk] = TC(1);
            }
        }
        vals[0] = logreg;
        vals[1] = lapl;
        vals[2 + 2 * KP] = relh;

        if (st.flags & ESPM_FLAG_EVAL_ONLY) {
            // loss terms only
        } else if (simplex) {
            TC* num_o = reinterpret_cast<TC*>(st.num);
            TC* den_o = reinterpret_cast<TC*>(st.den);
#pragma unroll
            for (int kk = 0; kk < KP; ++kk)
                if (kk < k) {
                    num_o[(size_t)kk * st.p_pad + j] = num[kk];
                    den_o[(size_t)kk * st.p_pad + j] = den[kk];
                }
            // The bisection itself always runs in fp64 (k x p data, negligible cost): in fp32 mode this
            // keeps the lock-step iteration count and nu aligned with the fp64 reference.
            double numd[KP], dend[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                numd[kk] = (double)num[kk];
                dend[kk] = (double)den[kk];
            }
            Mask128 dec;
            dec.clear();
            uint32_t seen = 0u;
            double nu_spec = 0.0;
            const int its_spec = (int)spec - 1;
            if (pg) {     // dicotomy.py:83-108 on new_H
                const PgEval<KP> ev(numd, k, st.log_shift, st.dicotomy_tol);
                double lo, hi;
                ev.bracket(lo, hi);
                bisect_trace_rec(lo, hi, ev, st.maxit, bits, dec, seen, err);
                if (spec) nu_spec = bisect_replay_rec(lo, hi, ev, its_spec, dec, seen);
            } else if (quad) {   // dicotomy.py:57-81 on (a, b, minus_c)
                const double qa = st.lambda_L * sigma;
                double lo, hi;
                acc_bracket<KP>(numd, dend, k, qa, lo, hi);
                const AccEval<KP> ev(numd, dend, k, qa, st.log_shift, st.dicotomy_tol);
                bisect_trace_rec(lo, hi, ev, st.maxit, bits, dec, seen, err);
                if (spec) nu_spec = bisect_replay_rec(lo, hi, ev, its_spec, dec, seen);
            } else {
                double lo, hi;
                simplex_bracket<double, KP>(numd, dend, k, lo, hi);
                // warm start of the root search: this pixel's root of the previous iteration (valid when its margin is)
                const double prev_mx = st.bisect_anchor[(size_t)st.p_pad + j];
                const double warm = (prev_mx > 0.0 && prev_mx < 1e300) ? st.bisect_anchor[j] : __longlong_as_double(-1LL);
                const KlAnchorEval<KP> ev(numd, dend, k, st.log_shift, st.dicotomy_tol, lo, hi, warm);
                bisect_trace_rec(lo, hi, ev, st.maxit, bits, dec, seen, err);
                st.bisect_anchor[j] = ev.nu;
                st.bisect_anchor[(size_t)st.p_pad + j] = ev.ok ? ev.mx : Num<double>::inf();
                if (spec) nu_spec = bisect_replay_rec(lo, hi, ev, its_spec, dec, seen);
            }
            uint32_t* rec = st.bisect_dec + j;
#pragma unroll
            for (int w = 0; w < 4; ++w) rec[(size_t)w * st.p_pad] = dec.w[w];
            rec[(size_t)4 * st.p_pad] = seen;
            if (spec) {
                TC hn[KP];
                h_from_nu<TC, KP>(st, numd, dend, k, nu_spec, sigma, hn);
                store_h_next<TC, KP>(st, j, k, hn, vals);
            }
        } else {
            if (pg) {   // keep new_H / grad readable (gradH, proj_grad_step_h of the operator-level API)
#pragma unroll
                for (int kk = 0; kk < KP; ++kk)
                    if (kk < k) {
                        reinterpret_cast<TC*>(st.num)[(size_t)kk * st.p_pad + j] = num[kk];
                        reinterpret_cast<TC*>(st.den)[(size_t)kk * st.p_pad + j] = den[kk];
                    }
            }
            TC hn[KP];  // updates.py:152 with nu = 0 (updates.py:289 for the quadratic surrogate)
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                if (kk >= k) hn[kk] = TC(0);
                else if (pg) hn[kk] = Num<TC>::vmax(num[kk], ls);                       // updates.py:387, nu = 0
                else if (quad)
                    hn[kk] = (TC)fmax(hq_root((double)num[kk], (double)den[kk], st.lambda_L * sigma), st.log_shift);
                else hn[kk] = Num<TC>::vmax(num[kk] / den[kk], ls);
            }
            store_h_next<TC, KP>(st, j, k, hn, vals);
        }
    }
    if (((st.flags & ESPM_FLAG_EVAL_ONLY) || simplex) && !spec) {
        // only the loss partials and rel_H are ours: the H_next statistics in px_part come from another kernel
        // (evaluation only) or from the h_apply that follows (simplex_H), which writes the other columns
        const double v3[3] = {vals[0], vals[1], vals[2 + 2 * KP]};
        __shared__ double tmp[3];
        block_reduce_vals<3>(v3, 2, tmp);
        __syncthreads();
        double* out = st.px_part + (size_t)blockIdx.x * NV;
        if (threadIdx.x < 2) out[threadIdx.x] = tmp[threadIdx.x];
        if (threadIdx.x == 2) out[2 + 2 * KP] = tmp[2];
    } else {
        block_reduce_vals<NV>(vals, px_part_nsum(KP), st.px_part + (size_t)blockIdx.x * NV);
    }
    merge_mask(bits, err, (simplex && !(st.flags & ESPM_FLAG_EVAL_ONLY)) ? st.bisect_mask : nullptr, st.dev_flags);
    // The last CTA to finish folds every partial into the scalar record (h_scalars_block),
    // in a fixed order that does not depend on which CTA that is.
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&st.dev_flags[2], 1u) == gridDim.x - 1;
    __syncthreads();
    if (is_last) {
        __threadfence();
        if ((st.flags & ESPM_FLAG_PEER) && simplex && !(st.flags & ESPM_FLAG_EVAL_ONLY) && (int)threadIdx.x < st.world) {
            // FIRST (the other ranks' h_apply waits for it): publish this rank's complete trace mask on every rank (its
            // own included), then raise the flag
            uint32_t* pf = st.peer_flags[threadIdx.x];
#pragma unroll
            for (int w = 0; w < 4; ++w) pf[ESPM_PF_MASK + 4 * st.rank + w] = __ldcg(st.bisect_mask + w);
            st_release_sys(pf + ESPM_PF_MFLAG + st.rank, st.seq_m);
        }
        // Pixel-sharded fit: the loss sums, rel_H and the error word of a record are per-shard quantities.  Every rank
        // leaves its share in slot [rank][rec_slot] of its OWN record inbox -- pinned host memory that every rank's
        // process has mapped -- and stamps it; each host folds the `world` shares in rank order once all stamps are
        // there.  No collective, no device-side wait, no store that leaves this GPU's host.
        double* share = nullptr;
        if ((st.flags & ESPM_FLAG_PEER) && st.rec_cap > 0 && st.peer_rec[st.rank])
            share = st.peer_rec[st.rank] + ((size_t)st.rank * st.rec_cap + st.rec_slot) * 8;
        h_scalars_block<TC>(st, share);
        if (threadIdx.x == 0) {
            time_stamp(st, 7);
            st.dev_flags[2] = 0u;
            if (simplex && !(st.flags & ESPM_FLAG_EVAL_ONLY)) st.dev_flags[7] = spec;   // the count this trace was applied with
        }
    }
    // halo rows pushed by store_h_next (the CTAs that own the first / last image row of the shard): one system fence per
    // CTA, by one thread after the barrier (fences are cumulative over what the barrier made visible to that thread)
    if ((st.flags & ESPM_FLAG_PEER) && (!simplex || spec)) {
        const int c0 = blockIdx.x * PX_THREADS, c1 = c0 + PX_THREADS;
        const bool pushed = (st.nb_prev_halo && c0 < st.ny) || (st.nb_next_halo && c1 > st.p_loc - st.ny);
        if (pushed) {
            __syncthreads();
            if (threadIdx.x == 0) __threadfence_system();
        }
    }
}

// ------------------------------------------------------------------------------------------------
// h_apply: replay it* iterations, H_next = max(num/(den+nu), ls)  (updates.py:152-155)
// ------------------------------------------------------------------------------------------------
template <typename TC, int KP>
__global__ void __launch_bounds__(PX_THREADS) h_apply_kernel(const espm_state st) {
    pdl_wait();
    pdl_trigger();
    if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 0);
    const int j = blockIdx.x * PX_THREADS + threadIdx.x;
    const int k = st.k;
    const TC ls = (TC)st.log_shift;
    constexpr int NV = 3 + 3 * KP;
    double vals[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) vals[i] = 0.0;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) vals[3 + 2 * KP + kk] = -1e300;
    int its;
    if (st.flags & ESPM_FLAG_PEER) {
        // lock-step count over ALL shards: wait for every rank's mask, OR them
        __shared__ uint32_t gmask[4];
        const uint32_t* pf = st.peer_flags[st.rank];
        wait_peer_flags(pf + ESPM_PF_MFLAG, st.world, st.seq_m, st.dev_flags);
        if (threadIdx.x < 4) {
            uint32_t m = 0u;
            for (int r = 0; r < st.world; ++r) m |= __ldcg(pf + ESPM_PF_MASK + 4 * r + threadIdx.x);
            gmask[threadIdx.x] = m;
        }
        __syncthreads();
        its = first_clear_bit(gmask, st.maxit);
    } else {
        its = first_clear_bit(st.bisect_mask, st.maxit);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 1);
    // dev_flags[7]: the count (+ 1) the preceding h_finish has already applied speculatively; dev_flags[6]: the guess
    // for the next H update.  Both are uniform over the grid (written by one thread of an EARLIER kernel / read by a
    // LATER one), so the early exit below is taken by every CTA or by none.
    if (blockIdx.x == 0 && threadIdx.x == 0) st.dev_flags[6] = (uint32_t)its + 1u;
    if (st.dev_flags[7] == (uint32_t)its + 1u) return;      // H', Ht, the halos and the statistics are in place
    if (j < st.p_loc) {
        double num[KP], den[KP];
        TC hn[KP];
        const TC* num_i = reinterpret_cast<const TC*>(st.num);
        const TC* den_i = reinterpret_cast<const TC*>(st.den);
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            num[kk] = (kk < k) ? (double)num_i[(size_t)kk * st.p_pad + j] : 0.0;
            den[kk] = (kk < k) ? (double)den_i[(size_t)kk * st.p_pad + j] : 1.0;
        }
        Mask128 dec;
        const uint32_t* rec = st.bisect_dec + j;
#pragma unroll
        for (int w = 0; w < 4; ++w) dec.w[w] = rec[(size_t)w * st.p_pad];
        const uint32_t seen = rec[(size_t)4 * st.p_pad];
        const double sigma = st.sigma_dev ? *st.sigma_dev : st.sigma;
        double nu;
        if (st.flags & ESPM_FLAG_PG) {                                         // updates.py:381-387
            const PgEval<KP> ev(num, k, st.log_shift, st.dicotomy_tol);
            double lo, hi;
            ev.bracket(lo, hi);
            nu = bisect_replay_rec(lo, hi, ev, its, dec, seen);
        } else if ((st.flags & ESPM_FLAG_HQ) && (st.flags & ESPM_FLAG_LAPLACIAN)) {   // updates.py:286-289
            const double a = st.lambda_L * sigma;
            double lo, hi;
            acc_bracket<KP>(num, den, k, a, lo, hi);
            nu = bisect_replay_rec(lo, hi, AccEval<KP>(num, den, k, a, st.log_shift, st.dicotomy_tol), its, dec, seen);
        } else {
            double lo, hi;
            simplex_bracket<double, KP>(num, den, k, lo, hi);
            const KlAnchorReplay<KP> ev(num, den, k, st.log_shift, st.dicotomy_tol, st.bisect_anchor[j],
                                        st.bisect_anchor[(size_t)st.p_pad + j]);
            nu = bisect_replay_rec(lo, hi, ev, its, dec, seen);
        }
        h_from_nu<TC, KP>(st, num, den, k, nu, sigma, hn);
        store_h_next<TC, KP>(st, j, k, hn, vals);
    }
    // only the H_next statistics are produced here; keep the loss partials written by h_finish
    __shared__ double tmp[NV];
    block_reduce_vals<NV>(vals, px_part_nsum(KP), tmp);
    __syncthreads();
    double* out = st.px_part + (size_t)blockIdx.x * NV;
    if (threadIdx.x < NV && threadIdx.x >= 2 && threadIdx.x != 2 + 2 * KP) out[threadIdx.x] = tmp[threadIdx.x];
    if (st.flags & ESPM_FLAG_PEER) {                         // halo rows pushed by store_h_next (see h_finish)
        const int c0 = blockIdx.x * PX_THREADS, c1 = c0 + PX_THREADS;
        const bool pushed = (st.nb_prev_halo && c0 < st.ny) || (st.nb_next_halo && c1 > st.p_loc - st.ny);
        if (pushed) {
            __syncthreads();
            if (threadIdx.x == 0) __threadfence_system();
        }
    }
}

// h_stats: statistics of H_next only (initialisation, operator-level API).
template <typename TC, int KP>
__global__ void __launch_bounds__(PX_THREADS) h_stats_kernel(const espm_state st) {
    const int j = blockIdx.x * PX_THREADS + threadIdx.x;
    const int k = st.k;
    const TC ls = (TC)st.log_shift;
    constexpr int NV = 3 + 3 * KP;
    double vals[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) vals[i] = 0.0;
#pragma unroll
    for (int kk = 0; kk < KP; ++kk) vals[3 + 2 * KP + kk] = -1e300;
    if (j < st.p_loc) {
        const TC* Hn = reinterpret_cast<const TC*>(st.H_next);
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) {
                const TC v = Hn[(size_t)kk * st.ldh + j];
                reinterpret_cast<TC*>(st.Ht)[((size_t)(j / TILE_PX) * KP + kk) * TILE_PX + (j % TILE_PX)] = v;
                vals[2 + kk] = (double)v;
                vals[2 + KP + kk] = (double)Num<TC>::vmax(v, ls);
                vals[3 + 2 * KP + kk] = (double)v;
            }
    }
    block_reduce_vals<NV>(vals, px_part_nsum(KP), st.px_part + (size_t)blockIdx.x * NV);
}

// ------------------------------------------------------------------------------------------------
// Reduce the px_part rows into hstats_next = {rowsum[kp], rowsumc[kp], rowmax[kp]} (one CTA).
// ------------------------------------------------------------------------------------------------
// Every thread takes whole px_part rows (blocks tid, tid + nthreads, ...): all its loads are independent, so the fold
// is one L2 round trip instead of px_blocks / 32 dependent ones; then lane butterfly and warps in index order
// (fixed order => deterministic).  Callable with up to 8 warps; hstats_out may be shared or global memory.
template <int KP>
__device__ __forceinline__ void reduce_hstats_block(const espm_state& st, double* hstats_out) {
    constexpr int NVAL = 3 * KP, STRIDE = 3 + 3 * KP;
    __shared__ double red[8][NVAL];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    double acc[NVAL];
#pragma unroll
    for (int v = 0; v < NVAL; ++v) acc[v] = (v >= 2 * KP) ? -1e300 : 0.0;
    for (int b = threadIdx.x; b < st.px_blocks; b += blockDim.x) {
        const double* row = st.px_part + (size_t)b * STRIDE;
        double u[NVAL];
#pragma unroll
        for (int v = 0; v < NVAL; ++v) u[v] = row[(v >= 2 * KP) ? (3 + v) : (2 + v)];
#pragma unroll
        for (int v = 0; v < NVAL; ++v) acc[v] = (v >= 2 * KP) ? (u[v] > acc[v] ? u[v] : acc[v]) : acc[v] + u[v];
    }
#pragma unroll
    for (int v = 0; v < NVAL; ++v) {
        const double r = (v >= 2 * KP) ? warp_max(acc[v]) : warp_sum(acc[v]);
        if (lane == 0) red[warp][v] = r;
    }
    __syncthreads();
    if ((int)threadIdx.x < NVAL) {
        const int v = threadIdx.x;
        double r = red[0][v];
        for (int w = 1; w < nwarps; ++w) r = (v >= 2 * KP) ? (red[w][v] > r ? red[w][v] : r) : r + red[w][v];
        hstats_out[v] = r;
    }
    __syncthreads();
}

template <typename TC, int KP>
__global__ void __launch_bounds__(256) hstats_reduce_kernel(const espm_state st) {
    reduce_hstats_block<KP>(st, reinterpret_cast<double*>(st.hstats_next));
}

// ------------------------------------------------------------------------------------------------
// h_scalars_block (last CTA of h_finish): loss parts of the current iterate + rel_H + bisection count into the
// scalar record
// ------------------------------------------------------------------------------------------------
// `share` (optional): this rank's slot of its OWN record inbox (pixel-sharded fits; host memory every rank's process has
// mapped): the additive / max / OR fields of the record that are per-shard quantities.  Written together with the record
// under ONE system fence, stamped like the record.
template <typename TC>
__device__ __forceinline__ void h_scalars_block(const espm_state& st, double* share) {
    __shared__ double sm[8][4];
    const int kp = st.kp, stride = px_part_stride(kp);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double xl = 0.0, lr = 0.0, lp = 0.0, rh = 0.0;
    for (int i = threadIdx.x; i < st.h_grid; i += blockDim.x) xl += st.xlogy_part[i];
    for (int b = threadIdx.x; b < st.px_blocks; b += blockDim.x) {
        const double* row = st.px_part + (size_t)b * stride;
        lr += row[0];
        lp += row[1];
        rh = row[2 + 2 * kp] > rh ? row[2 + 2 * kp] : rh;
    }
    xl = warp_sum(xl);
    lr = warp_sum(lr);
    lp = warp_sum(lp);
    rh = warp_max(rh);
    if (lane == 0) {
        sm[warp][0] = xl;
        sm[warp][1] = lr;
        sm[warp][2] = lp;
        sm[warp][3] = rh;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) {
            xl += sm[w][0];
            lr += sm[w][1];
            lp += sm[w][2];
            rh = sm[w][3] > rh ? sm[w][3] : rh;
        }
        const double* hstats = reinterpret_cast<const double*>(st.hstats_cur);
        const TC* gwstats = reinterpret_cast<const TC*>(st.gwstats_cur);
        double sumy = 0.0, meanh = 0.0;
        for (int kk = 0; kk < st.k; ++kk) {
            sumy += (double)gwstats[kp + kk] * hstats[kp + kk];  // measures.py:502, analytic
            meanh += hstats[kk];
        }
        double* rec = st.scalars;
        const double flags = (double)st.dev_flags[0];
        rec[ESPM_S_XLOGY] = xl;
        rec[ESPM_S_SUMY] = sumy;
        rec[ESPM_S_LOGREG] = lr;
        rec[ESPM_S_LAPL] = lp;
        rec[ESPM_S_REL_H] = rh;
        rec[ESPM_S_BISECT_ITS_H] =
            (st.flags & ESPM_FLAG_SIMPLEX_H) ? (double)first_clear_bit(st.bisect_mask, st.maxit) : 0.0;
        rec[ESPM_S_DEV_FLAGS] = flags;
        rec[ESPM_S_MEAN_H] = meanh / ((double)st.k * (double)st.p_total);
        if (share) {
            share[0] = xl;
            share[1] = lr;
            share[2] = lp;
            share[3] = rh;
            share[4] = flags;
        }
        // the record is complete (rel_W etc. were written by earlier kernels of the stream): stamp it
        __threadfence_system();
        *reinterpret_cast<volatile double*>(rec + ESPM_S_STAMP) = st.rec_stamp;
        if (share) *reinterpret_cast<volatile double*>(share + 7) = st.rec_stamp;
    }
}

// ------------------------------------------------------------------------------------------------
// w_reduce: s_sum[c][k] = sum_r s_part[r][c][k]; the last block reduces the H_next statistics.
// ------------------------------------------------------------------------------------------------
template <typename TC, int KP>
__global__ void __launch_bounds__(256) w_reduce_kernel(const espm_state st) {
    if (blockIdx.x == gridDim.x - 1) {
        reduce_hstats_block<KP>(st, reinterpret_cast<double*>(st.hstats_next));
        return;
    }
    const size_t total = (size_t)st.n_pad * st.kp;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    // slots of this channel block that a CTA of the W pass actually wrote (see w_pass_kernel)
    const int cb = (int)(i / ((size_t)st.cs * st.kp));
    const int first = (int)(((long long)cb * st.n_tiles) / st.w_upc);
    const int last = (int)((((long long)cb + 1) * st.n_tiles - 1) / st.w_upc);
    const TC* part = reinterpret_cast<const TC*>(st.s_part);
    TC s = part[i];
    for (int r = 1; r <= last - first; ++r) s += part[(size_t)r * total + i];
    reinterpret_cast<TC*>(st.s_sum)[i] = s;
}

// ------------------------------------------------------------------------------------------------
// GW = G.W (+ pad rows), clamped copy, column sums and flags.  Runs inside one CTA.
// ------------------------------------------------------------------------------------------------
template <typename TC>
__device__ void gw_prepare_block(const espm_state& st, const TC* W, double* sm /* >= 2*kp + 64 doubles */) {
    const int kp = st.kp, k = st.k, n = st.n, m = st.m;
    const TC ls = (TC)st.log_shift;
    const bool ident = st.flags & ESPM_FLAG_G_IDENTITY;
    const TC* G = reinterpret_cast<const TC*>(st.G);
    TC* GW = reinterpret_cast<TC*>(st.GW_next);
    TC* GWc = reinterpret_cast<TC*>(st.GWc_next);
    double cs[ESPM_MAX_K], csc[ESPM_MAX_K];
    for (int kk = 0; kk < ESPM_MAX_K; ++kk) cs[kk] = csc[kk] = 0.0;
    uint32_t flags = 0u;
    if (threadIdx.x == 0) st.dev_flags[1] = 0u;
    __syncthreads();
    for (int c = threadIdx.x; c < st.n_pad; c += blockDim.x) {
        bool all_zero = true;
        for (int kk = 0; kk < kp; ++kk) {
            TC v;
            if (c >= n) {
                v = (kk == 0) ? TC(1) : TC(0);  // pad channel: y = H[0] > 0, contributes nothing
            } else if (kk >= k) {
                v = TC(0);
            } else if (ident) {
                v = W[(size_t)c * k + kk];
            } else {
                TC acc = TC(0);
                for (int mm = 0; mm < m; ++mm) acc = fma(G[(size_t)c * m + mm], W[(size_t)mm * k + kk], acc);
                v = acc;
            }
            GW[(size_t)c * kp + kk] = v;
            const TC vc = (c < n && kk < k) ? Num<TC>::vmax(v, ls) : v;
            GWc[(size_t)c * kp + kk] = vc;
            if (c < n && kk < k) {
                cs[kk] += (double)v;
                csc[kk] += (double)vc;
                if (v < ls) flags |= ESPM_DEV_GW_BELOW_LS;
                if (v > TC(0)) all_zero = false;
            }
        }
        if (c < n && all_zero) flags |= ESPM_DEV_GW_ZERO_ROW;
    }
    // block reduction of the column sums (fixed order)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    double* red = sm;  // [nwarps][2*kp]
    for (int kk = 0; kk < k; ++kk) {
        const double a = warp_sum(cs[kk]), b = warp_sum(csc[kk]);
        if (lane == 0) {
            red[(size_t)warp * 2 * kp + kk] = a;
            red[(size_t)warp * 2 * kp + kp + kk] = b;
        }
    }
    const uint32_t f = __reduce_or_sync(0xffffffffu, flags);
    if (lane == 0 && f) atomicOr(&st.dev_flags[1], f);
    __syncthreads();
    TC* gwstats = reinterpret_cast<TC*>(st.gwstats_next);
    if ((int)threadIdx.x < 2 * kp) {
        const int kk = threadIdx.x % kp;
        double s = 0.0;
        if (kk < k)
            for (int w = 0; w < nwarps; ++w) s += red[(size_t)w * 2 * kp + threadIdx.x];
        gwstats[threadIdx.x] = (TC)s;
    }
    __syncthreads();
    if (threadIdx.x == 0) st.scalars[ESPM_S_GW_FLAGS] = (double)st.dev_flags[1];
}

template <typename TC>
__global__ void __launch_bounds__(1024) gw_prepare_kernel(const espm_state st) {
    __shared__ double sm[32 * 2 * ESPM_MAX_K];
    gw_prepare_block<TC>(st, reinterpret_cast<const TC*>(st.W_next), sm);
}

// colsum_G[m] = sum_c G[c][m]  (updates.py:60); one warp per column, Gt is m x n row-major.
template <typename TC>
__global__ void __launch_bounds__(256) colsum_g_kernel(const TC* Gt, int n, int m, TC* out) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= m) return;
    double s = 0.0;
    for (int c = lane; c < n; c += 32) s += (double)Gt[(size_t)warp * n + c];
    s = warp_sum(s);
    if (lane == 0) out[warp] = (TC)s;
}

// ------------------------------------------------------------------------------------------------
// w_finish: the W update (updates.py:58-76) + GW' for the next H pass, as ONE cooperative kernel of
// W_COOP_BLOCKS CTAs with ONE synchronisation point in the common case (plain KL rule, real G, no simplex_W,
// m k <= W_SM_MAX -- the "T path"):
//   before   one CTA per row of G^T: T[mm][:] = sum_c G[c][mm] S[c][:], S folded from the W-pass partial slots on the
//            fly; the last CTA folds the H' row statistics meanwhile.  Sharded: the k values of the row and the
//            statistics are PUSHED into slot [rank] of every rank's receive buffer, then the CTA raises its own flag word
//            on every rank
//   sync     one GPU: grid barrier.  Sharded: wait for the world x gridDim flag words (which is also the grid barrier)
//   after    W' = max(W * T / (colsum(G) (x) rowsum(H')), ls), fixed_W, rel_W: redundantly in every CTA from T (the ranks'
//            slots folded in rank order) and the statistics -- W' stays in shared memory, CTA 0 writes it out;
//            GW' = G W' (+ pad rows, clamped copy), per-CTA column sums / flags; the last CTA to finish folds the column
//            sums (one warp per column, fixed order) and the flags
// Other rules (identity G, Bregman, projected gradient, Frobenius): num / denum are formed before the barrier
// (`entry`), sharded fits push S itself (n x k) in phase 0 and fold the ranks' slots in phase A; simplex_W adds the
// lock-step bisection over the columns (trace, barrier, replay, barrier); m k > W_SM_MAX slices W' over the CTAs (one more
// barrier).
// ------------------------------------------------------------------------------------------------
constexpr int W_COOP_BLOCKS = 32;
constexpr int W_COOP_THREADS = 256;
constexpr int W_COOP_STRIDE = 2 * ESPM_MAX_K + 4;   // doubles per CTA row of coop_part: 2 KP column sums, [2 MAX_K] flags,
                                                  // [2 MAX_K + 1] sum of W' slice, [2 MAX_K + 2] rel_W of the slice
constexpr int W_SM_MAX = 1024;   // m*k up to which W' is kept in shared memory by every CTA

// Grid barrier for a cooperative launch: monotonically increasing arrival counter, every CTA arrives
// exactly once per barrier, so the target of an arrival is the next multiple of the grid size.
__device__ __forceinline__ void grid_barrier(uint32_t* ctr, uint32_t nblocks) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const uint32_t t = atomicAdd(ctr, 1u);
        const uint32_t target = (t / nblocks + 1u) * nblocks;
        while (*reinterpret_cast<volatile uint32_t*>(ctr) < target) {
        }
        __threadfence();
    }
    __syncthreads();
}

template <typename TC, int KP>
__global__ void __launch_bounds__(W_COOP_THREADS) w_finish_kernel(const espm_state st) {
    pdl_wait();      // results of the W pass (and of everything before it) are visible from here on
    pdl_trigger();   // lets the next H pass set up while we run
    if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 2);
    __shared__ double sm[8 * 2 * ESPM_MAX_K + 8];
    __shared__ int s_its;
    __shared__ uint32_t s_err;
    __shared__ double hs_sm[3 * ESPM_MAX_K];
    __shared__ TC wsm[W_SM_MAX];
    __shared__ bool s_last;
    const int k = st.k, m = st.m, n = st.n;
    const TC ls = (TC)st.log_shift;
    const bool ident = st.flags & ESPM_FLAG_G_IDENTITY;
    // fused mode: phase A folds the W-pass partial slots (single GPU) or the ranks' receive slots (peer exchange)
    // itself and every CTA has its own copy of the H' statistics
    const bool fly = (st.flags & ESPM_FLAG_FUSED_WREDUCE) != 0;
    const bool redundant_b = !(st.flags & ESPM_FLAG_SIMPLEX_W) && m * k <= W_SM_MAX;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int NWARPS = W_COOP_THREADS / 32;
    const int gthread = blockIdx.x * W_COOP_THREADS + threadIdx.x;
    const int gthreads = gridDim.x * W_COOP_THREADS;
    uint32_t* bar = st.dev_flags + 3;
    TC* S = reinterpret_cast<TC*>(st.s_sum);
    const TC* Gt = reinterpret_cast<const TC*>(st.Gt);
    const TC* W = reinterpret_cast<const TC*>(st.W_cur);
    const TC* colsumG = reinterpret_cast<const TC*>(st.colsum_G);
    double* hstats = reinterpret_cast<double*>(st.hstats_next);
    TC* wnum = reinterpret_cast<TC*>(st.w_num);
    TC* wden = reinterpret_cast<TC*>(st.w_den);
    TC* Wn = reinterpret_cast<TC*>(st.W_next);

    // ---- phase 0: fold the W-pass partial slots and the per-pixel statistics ----
    const bool peer = st.flags & ESPM_FLAG_PEER;
    const size_t recv_off = (size_t)(st.seq_s & 1u) * st.xchg_stride;   // parity of this exchange in every rank's buffer
    const bool w_bmd = st.flags & ESPM_FLAG_BMD, w_pg = st.flags & ESPM_FLAG_PG, w_l2 = st.flags & ESPM_FLAG_L2;
    // "T path" (plain KL update with a real G, W' small enough for shared memory: the C2 / C3 / C4 case).  The W pass left
    // partial sums of S = R H'^T; G^T is applied to the LOCAL S first, one CTA per row of G^T, while the last CTA folds the
    // H' statistics; num / denum are only formed after the synchronisation point (phase B), from T = G^T S and the
    // statistics.  Sharded (tx): the ranks exchange T_r = G^T S_r -- m x k values instead of n x k (108 floats instead
    // of 8192 at C3; G^T sum_r S_r = sum_r G^T S_r) -- every CTA pushes the k values of its row into slot [rank] of every
    // rank's receive buffer and raises ITS OWN flag word there (no ticket, no second fence); the wait for all
    // world x gridDim flag words doubles as the grid barrier of the single-GPU path, and the slots are folded in rank
    // order (identical W' on every rank, no broadcast).
    const bool tp = fly && !ident && redundant_b && !(w_bmd || w_pg || w_l2) && m <= st.n_pad;
    const bool tx = tp && peer;
    const size_t my_slot_off = recv_off + (size_t)st.rank * st.xchg_slot;
    // W-pass partial slots of every channel block (see w_pass_kernel), once per CTA: no 64-bit divisions per channel
    __shared__ int cb_nr[256];
    const int n_cb = st.n_pad / st.cs;
    const bool cb_tab = fly && n_cb <= 256;
    if (cb_tab) {
        for (int cb = threadIdx.x; cb < n_cb; cb += W_COOP_THREADS) {
            const int first = (int)(((long long)cb * st.n_tiles) / st.w_upc);
            const int last = (int)((((long long)cb + 1) * st.n_tiles - 1) / st.w_upc);
            cb_nr[cb] = last - first;
        }
        __syncthreads();
    }
    if (tp) {
        if (blockIdx.x == gridDim.x - 1) {
            reduce_hstats_block<KP>(st, hs_sm);
            if ((int)threadIdx.x < 3 * KP) {
                if (tx) {
                    for (int r = 0; r < st.world; ++r)
                        reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(st.peer_xchg[r]) + my_slot_off + st.xchg_hs_off)[threadIdx.x] =
                            hs_sm[threadIdx.x];
                } else {
                    hstats[threadIdx.x] = hs_sm[threadIdx.x];
                }
            }
            __syncthreads();
        }
    } else if (peer) {
        // Sharded: PUSH model.  Every rank folds its own partial slots and stores the result into slot [rank] of the
        // receive buffer of EVERY rank (its own included) -- remote stores over NVLink are fire-and-forget, so no
        // thread ever waits for a remote load.  The last CTA to finish pushing raises this rank's flag everywhere;
        // every CTA then waits for all flags and from there on reads only LOCAL memory: phase A folds the `world`
        // slots in rank order (identical sums on every rank, no broadcast), exactly like the single-GPU path folds the
        // W-pass partial slots.  No grid barrier before phase A.
        const size_t total = (size_t)st.n_pad * KP;
        const TC* part = reinterpret_cast<const TC*>(st.s_part);
        const size_t my_off = recv_off + (size_t)st.rank * st.xchg_slot;
        for (size_t i = gthread; i < total; i += gthreads) {
            const int cb = (int)(i / ((size_t)st.cs * KP));
            const int first = (int)(((long long)cb * st.n_tiles) / st.w_upc);
            const int last = (int)((((long long)cb + 1) * st.n_tiles - 1) / st.w_upc);
            TC v = part[i];
            for (int r = 1; r <= last - first; ++r) v += part[(size_t)r * total + i];
            for (int r = 0; r < st.world; ++r)
                reinterpret_cast<TC*>(reinterpret_cast<unsigned char*>(st.peer_xchg[r]) + my_off)[i] = v;
        }
        if (blockIdx.x == gridDim.x - 1) {
            reduce_hstats_block<KP>(st, hs_sm);
            if ((int)threadIdx.x < 3 * KP)
                for (int r = 0; r < st.world; ++r)
                    reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(st.peer_xchg[r]) + my_off + st.xchg_hs_off)[threadIdx.x] =
                        hs_sm[threadIdx.x];
        }
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&st.dev_flags[5], 1u) == gridDim.x - 1;
        __syncthreads();
        if (s_last) {     // every CTA of this rank has pushed (and fenced): publish
            __threadfence_system();
            if ((int)threadIdx.x < st.world) st_release_sys(st.peer_flags[threadIdx.x] + ESPM_PF_SFLAG + st.rank, st.seq_s);
            if (threadIdx.x == 0) st.dev_flags[5] = 0u;
        }
        wait_peer_flags(st.peer_flags[st.rank] + ESPM_PF_SFLAG, st.world, st.seq_s, st.dev_flags);
        // global H' statistics: every CTA folds the ranks' slots for itself (rank order)
        if ((int)threadIdx.x < 3 * KP) {
            const bool is_max = (int)threadIdx.x >= 2 * KP;
            const unsigned char* base = reinterpret_cast<const unsigned char*>(st.peer_xchg[st.rank]) + recv_off + st.xchg_hs_off;
            double v = 0.0;
            for (int r = 0; r < st.world; ++r) {
                const double u = __ldcg(reinterpret_cast<const double*>(base + (size_t)r * st.xchg_slot) + threadIdx.x);
                v = (r == 0) ? u : (is_max ? (u > v ? u : v) : v + u);
            }
            hs_sm[threadIdx.x] = v;
            if (blockIdx.x == gridDim.x - 1) hstats[threadIdx.x] = v;
        }
        __syncthreads();
    } else if (st.flags & ESPM_FLAG_FUSED_WREDUCE) {
        reduce_hstats_block<KP>(st, hs_sm);                   // every CTA, for itself
        __syncthreads();
        if (blockIdx.x == gridDim.x - 1 && (int)threadIdx.x < 3 * KP) hstats[threadIdx.x] = hs_sm[threadIdx.x];
    }

    // ---- phase A: num = W * (G^T S), den = colsum(G) (x) rowsum(H')   (updates.py:58-60) ----
    bool nonfinite = false;
    // num / denum of one entry from v = (G^T S)[mm][kk] and cs_h = colsum(G)[mm] * rowsum(H')[kk]; trow = (G^T G W)[mm][:]
    auto entry = [&](int mm, int kk, TC v, TC cs_h, const TC (&trow)[KP]) {
        const int i = mm * k + kk;
        TC ggwhh = TC(0);
        if (w_l2) {   // (G^T G W H H^T)[mm][kk]  (updates.py:30-32)
#pragma unroll
            for (int k2 = 0; k2 < KP; ++k2)
                if (k2 < k) ggwhh = fma(trow[k2], (TC)st.gram_h[k2 * KP + kk], ggwhh);
        }
        if (w_pg) {          // gradW + projected step (updates.py:303-314, 357)
            const TC grad = w_l2 ? TC(2) * (ggwhh - v) : (-v + cs_h);
            wnum[i] = W[i] - (TC)(1.0 / st.gamma_w) * grad;
            wden[i] = grad;   // the gradient itself (gradW of the operator-level API reads it back)
        } else if (w_l2) {   // new_W = W / GGWHH * GXH (updates.py:36)
            wnum[i] = (W[i] / ggwhh) * v;
            wden[i] = TC(1);
        } else if (w_bmd) {  // updates.py:40-48
            const TC sr = ident ? reinterpret_cast<const TC*>(st.x_rowsum)[mm] : (TC)st.x_total;
            const TC gradg = -v + cs_h;
            wnum[i] = sr * W[i];
            wden[i] = gradg * W[i] + sr;
        } else {             // updates.py:59-60
            wnum[i] = W[i] * v;
            wden[i] = cs_h;
        }
    };
    const double* hs = fly ? hs_sm : hstats;
    // S[c][:] -- from s_sum, or (fly) summed from the W-pass partial slots in slot order, exactly like phase 0
    const size_t s_total = (size_t)st.n_pad * KP;
    const TC* s_part = reinterpret_cast<const TC*>(st.s_part);
    auto load_srow = [&](int c, TC (&srow)[KP]) {
        if (peer && !tx) {
            // slots of the ranks in this rank's receive buffer (written by the peers, read through L2 only)
            const unsigned char* base = reinterpret_cast<const unsigned char*>(st.peer_xchg[st.rank]) + recv_off;
            ldcg_row<TC, KP>(srow, reinterpret_cast<const TC*>(base) + (size_t)c * KP);
#pragma unroll 4
            for (int r = 1; r < st.world; ++r) {
                TC u[KP];
                ldcg_row<TC, KP>(u, reinterpret_cast<const TC*>(base + (size_t)r * st.xchg_slot) + (size_t)c * KP);
#pragma unroll
                for (int kk = 0; kk < KP; ++kk) srow[kk] += u[kk];
            }
        } else if (fly) {
            const int cb = c / st.cs;
            int nr;                                // slots 0..nr hold partial sums of this channel block
            if (cb_tab) {
                nr = cb_nr[cb];
            } else {
                const int first = (int)(((long long)cb * st.n_tiles) / st.w_upc);
                const int last = (int)((((long long)cb + 1) * st.n_tiles - 1) / st.w_upc);
                nr = last - first;
            }
            constexpr int RU = 6;                  // slots loaded at once (independent loads: one L2 round trip)
            TC t[RU][KP];
            lds_row<TC, KP>(srow, s_part + (size_t)c * KP);
#pragma unroll
            for (int r = 0; r < RU; ++r) {
                if (r < nr) lds_row<TC, KP>(t[r], s_part + (size_t)(r + 1) * s_total + (size_t)c * KP);
            }
#pragma unroll
            for (int r = 0; r < RU; ++r) {
                if (r < nr) {
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk) srow[kk] += t[r][kk];
                }
            }
            for (int r = RU + 1; r <= nr; ++r) {
                TC u[KP];
                lds_row<TC, KP>(u, s_part + (size_t)r * s_total + (size_t)c * KP);
#pragma unroll
                for (int kk = 0; kk < KP; ++kk) srow[kk] += u[kk];
            }
        } else {
            lds_row<TC, KP>(srow, S + (size_t)c * KP);
        }
    };
    if (ident) {
        for (int i = gthread; i < m * k; i += gthreads) {
            const int mm = i / k, kk = i - mm * k;
            TC srow[KP];
            load_srow(mm, srow);
            TC sv = srow[0];
#pragma unroll
            for (int k2 = 1; k2 < KP; ++k2)
                if (k2 == kk) sv = srow[k2];
            nonfinite |= !(Num<TC>::vabs(sv) < Num<TC>::inf());
            TC trow[KP];
#pragma unroll
            for (int k2 = 0; k2 < KP; ++k2) trow[k2] = (k2 < k) ? W[mm * k + k2] : TC(0);   // G^T G = I
            entry(mm, kk, sv, (TC)hs[kk], trow);
        }
    } else {
        // one CTA per row of G^T: the 8 warps split the channels, partial sums meet in shared memory (fixed order)
        TC* accsm = reinterpret_cast<TC*>(sm);   // [NWARPS][KP]
        for (int mm = blockIdx.x; mm < m; mm += gridDim.x) {
            TC acc[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) acc[kk] = TC(0);
#pragma unroll 4
            for (int c = threadIdx.x; c < n; c += W_COOP_THREADS) {
                const TC g = Gt[(size_t)mm * n + c];
                TC srow[KP];
                load_srow(c, srow);
#pragma unroll
                for (int kk = 0; kk < KP; ++kk) acc[kk] = fma(g, srow[kk], acc[kk]);
            }
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                const TC v = warp_sum(acc[kk]);
                if (lane == 0) accsm[warp * KP + kk] = v;
            }
            __syncthreads();
            if (warp == 0) {
                TC trow[KP];
#pragma unroll
                for (int k2 = 0; k2 < KP; ++k2) trow[k2] = TC(0);
                if (w_l2) {   // row mm of (G^T G) W
                    const TC* GG = reinterpret_cast<const TC*>(st.GG);
                    for (int m2 = lane; m2 < m; m2 += 32) {
                        const TC g = GG[(size_t)mm * m + m2];
#pragma unroll
                        for (int k2 = 0; k2 < KP; ++k2)
                            if (k2 < k) trow[k2] = fma(g, W[m2 * k + k2], trow[k2]);
                    }
#pragma unroll
                    for (int k2 = 0; k2 < KP; ++k2) trow[k2] = warp_sum(trow[k2]);
                }
                if (lane < k) {
                    TC v = accsm[lane];
                    for (int w = 1; w < NWARPS; ++w) v += accsm[w * KP + lane];
                    nonfinite |= !(Num<TC>::vabs(v) < Num<TC>::inf());
                    if (tx) {     // this rank's (G^T S)[mm][lane] into slot [rank] of every rank's receive buffer
                        for (int r = 0; r < st.world; ++r)
                            reinterpret_cast<TC*>(reinterpret_cast<unsigned char*>(st.peer_xchg[r]) + my_slot_off)[mm * KP + lane] = v;
                    } else if (tp) {
                        S[mm * KP + lane] = v;        // (s_sum is free in fused mode: it holds T = G^T S until phase B)
                    } else {
                        entry(mm, lane, v, colsumG[mm] * (TC)hs[lane], trow);
                    }
                }
            }
            __syncthreads();
        }
    }
    // x / 0 in the W pass (updates.py:53-56): the caller redoes the step with ESPM_FLAG_CLAMP_Y
    if (__any_sync(0xffffffffu, nonfinite) && lane == 0)
        atomicOr(&st.dev_flags[0], ESPM_DEV_NONFINITE | ESPM_DEV_NONFINITE_W);
    if (tx) {
        // every thread of this CTA is past its remote stores: threads 0..world-1 each raise this CTA's flag word on one
        // rank.  st.release is cumulative over the stores the barrier ordered before it; the `world` releases run in
        // parallel, so the CTA pays one round trip, and nothing waits for a ticket of the whole grid.
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 3);
        __syncthreads();
        if ((int)threadIdx.x < st.world)
            st_release_sys(st.peer_flags[threadIdx.x] + ESPM_PF_TFLAG + 32 * st.rank + blockIdx.x, st.seq_s);
        // wait for the flag words of every CTA of every rank (bounded, like wait_peer_flags)
        {
            const uint32_t* tf = st.peer_flags[st.rank] + ESPM_PF_TFLAG;
            for (int w = threadIdx.x; w < 32 * st.world; w += W_COOP_THREADS) {
                if ((w & 31) >= (int)gridDim.x) continue;
                const long long t0 = clock64();
                while ((int32_t)(ld_acquire_sys(tf + w) - st.seq_s) < 0) {
                    if (clock64() - t0 > (1ll << 31)) {
                        atomicOr(st.dev_flags, ESPM_DEV_PEER_TIMEOUT);
                        break;
                    }
                    __nanosleep(32);
                }
            }
            __syncthreads();
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 4);
        // global H' statistics: every CTA folds the ranks' slots for itself (rank order)
        if ((int)threadIdx.x < 3 * KP) {
            const bool is_max = (int)threadIdx.x >= 2 * KP;
            const unsigned char* base = reinterpret_cast<const unsigned char*>(st.peer_xchg[st.rank]) + recv_off + st.xchg_hs_off;
            double v = 0.0;
            for (int r = 0; r < st.world; ++r) {
                const double u = __ldcg(reinterpret_cast<const double*>(base + (size_t)r * st.xchg_slot) + threadIdx.x);
                v = (r == 0) ? u : (is_max ? (u > v ? u : v) : v + u);
            }
            hs_sm[threadIdx.x] = v;
            if (blockIdx.x == gridDim.x - 1) hstats[threadIdx.x] = v;
        }
        __syncthreads();
    } else if (tp) {
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 3);
        grid_barrier(bar, gridDim.x);
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 4);
        if ((int)threadIdx.x < 3 * KP) hs_sm[threadIdx.x] = __ldcg(hstats + threadIdx.x);   // written by the last CTA
        __syncthreads();
    } else {
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 3);
        grid_barrier(bar, gridDim.x);
        if (blockIdx.x == 0 && threadIdx.x == 0) time_stamp(st, 4);
    }

    if (threadIdx.x == 0) {
        s_its = 0;
        s_err = 0u;
    }
    __syncthreads();
    // ---- simplex_W (updates.py:61-68): lock-step bisection over the k columns of (num, den), dicotomy.py:4-55,111-173.
    // One CTA per column: all 256 threads share the sum over the rows, so a column costs rows/256 quotients per thread
    // and evaluation instead of rows/32 (the whole bisection used to run in the warps of CTA 0: 0.15 ms at C5).  The
    // global stop test couples the columns only through the iteration count, so -- like the H update -- every column is
    // TRACED on its own (which iterations still have |f| > tol, which way each one went), the traces are OR-ed after one
    // grid barrier, and every column is replayed for the common count.
    if (st.flags & ESPM_FLAG_SIMPLEX_W) {
        const bool sub = st.flags & ESPM_FLAG_SIMPLEX_ROWS;
        const int nrows = sub ? st.n_simplex_rows : m;
        auto row_of = [&](int i) { return sub ? st.simplex_rows[i] : i; };
        double* redsm = sm;   // [NWARPS] partial sums, [NWARPS..] scratch of the bracket
        uint32_t* pub = reinterpret_cast<uint32_t*>(st.coop_part + (size_t)blockIdx.x * W_COOP_STRIDE);
        Mask128 bad, dec;
        bad.clear();
        dec.clear();
        uint32_t seen = 0u;
        double lo = 0.0, hi = 0.0;
        const int kk = blockIdx.x;      // this CTA's column (grids of W_COOP_BLOCKS >= ESPM_MAX_K CTAs)
        struct ColEval {               // block-collective evaluator: every thread gets the same value
            const TC* wnum;
            const TC* wden;
            const int* rows;
            double* red;
            int k, kk, nrows;
            double ls, tol;
            __device__ __forceinline__ double exact(double x) const {
                double sacc = 0.0;
                for (int i = threadIdx.x; i < nrows; i += W_COOP_THREADS) {
                    const int o = (rows ? rows[i] : i) * k + kk;
                    sacc += fmax(simplex_quot<double>((double)__ldcg(wnum + o), x + (double)__ldcg(wden + o)), ls);
                }
                sacc = warp_sum(sacc);
                if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sacc;
                __syncthreads();
                double t = red[0];
                for (int w = 1; w < W_COOP_THREADS / 32; ++w) t += red[w];
                __syncthreads();
                return t - 1.0;
            }
            __device__ __forceinline__ Cls operator()(double x) const {
                const double fe = exact(x);
                return Cls{fe <= 0.0, fabs(fe) > tol};
            }
            __device__ __forceinline__ bool le0(double x) const { return exact(x) <= 0.0; }
        };
        const ColEval ev{wnum, wden, sub ? st.simplex_rows : nullptr, redsm, k, kk, nrows, st.log_shift,
                         st.dicotomy_tol_w};
        if (kk < k) {
            // bracket of dicotomy.py:29-49 over the rows of this column
            double amax = -Num<double>::inf(), nmax = -Num<double>::inf(), dmin = Num<double>::inf(), nsum = 0.0;
            bool neg = false;
            for (int i = threadIdx.x; i < nrows; i += W_COOP_THREADS) {
                const int o = row_of(i) * k + kk;
                const double nv = (double)__ldcg(wnum + o), dv = (double)__ldcg(wden + o);
                if (nv > 0.0) amax = fmax(amax, nv / 2.0 - dv);
                nmax = fmax(nmax, nv);
                dmin = fmin(dmin, dv);
                nsum += nv;
                neg |= (nv < 0.0) || (dv < 0.0);
            }
            amax = warp_max(amax);
            nmax = warp_max(nmax);
            dmin = -warp_max(-dmin);
            nsum = warp_sum(nsum);
            if (lane == 0) {
                redsm[NWARPS + warp] = amax;
                redsm[2 * NWARPS + warp] = nmax;
                redsm[3 * NWARPS + warp] = dmin;
                redsm[4 * NWARPS + warp] = nsum;
            }
            const int any_neg = __syncthreads_or((int)neg);
            amax = redsm[NWARPS], nmax = redsm[2 * NWARPS], dmin = redsm[3 * NWARPS], nsum = redsm[4 * NWARPS];
            for (int w = 1; w < NWARPS; ++w) {
                amax = fmax(amax, redsm[NWARPS + w]);
                nmax = fmax(nmax, redsm[2 * NWARPS + w]);
                dmin = fmin(dmin, redsm[3 * NWARPS + w]);
                nsum += redsm[4 * NWARPS + w];
            }
            __syncthreads();
            lo = amax;
            hi = (double)nrows * nmax / 0.5 - dmin;
            uint32_t e = 0u;
            if (any_neg || !(nsum > 0.0)) e |= ESPM_DEV_NEGATIVE;
            bisect_trace_rec(lo, hi, ev, st.maxit, bad, dec, seen, e);
            if (threadIdx.x == 0) {
#pragma unroll
                for (int w = 0; w < 4; ++w) pub[w] = bad.w[w];
                if (e) atomicOr(&st.dev_flags[0], e);
            }
        }
        grid_barrier(bar, gridDim.x);
        uint32_t gmask[4] = {0u, 0u, 0u, 0u};
        for (int c = 0; c < k; ++c) {
            const uint32_t* pc = reinterpret_cast<const uint32_t*>(st.coop_part + (size_t)c * W_COOP_STRIDE);
#pragma unroll
            for (int w = 0; w < 4; ++w) gmask[w] |= __ldcg(pc + w);
        }
        const int its = first_clear_bit(gmask, st.maxit);
        if (threadIdx.x == 0) s_its = its;   // every CTA: the last one to finish writes the record
        if (kk < k) {
            const double nu = bisect_replay_rec(lo, hi, ev, its, dec, seen);
            // denum[rows] += nu (updates.py:65,68)
            for (int i = threadIdx.x; i < nrows; i += W_COOP_THREADS) {
                const int o = row_of(i) * k + kk;
                wden[o] = __ldcg(wden + o) + (TC)nu;
            }
        }
        grid_barrier(bar, gridDim.x);
    }

    // ---- phase B: W' = max(num/den, ls), fixed_W (updates.py:70-76); rel_W (base.py:323) ----
    // small m k without bisection: every CTA computes all of W' into shared memory (no barrier before phase C);
    // otherwise every CTA takes a slice (a single CTA needed 40 us for the 2048 x 8 entries of C5), one barrier.
    const TC* fw = reinterpret_cast<const TC*>(st.fixed_W);
    auto w_entry = [&](int i) {
        const TC nv = __ldcg(wnum + i), dv = __ldcg(wden + i);   // L2: written by other CTAs in this launch
        TC v = Num<TC>::vmax((st.flags & ESPM_FLAG_PG) ? nv : nv / dv, ls);
        if (st.flags & ESPM_FLAG_FIXED_W) {
            const TC f = fw[i];
            if (f >= TC(0)) v = f;
        }
        return v;
    };
    auto block_sum = [&](double v) {      // fixed order; every thread gets the result
        v = warp_sum(v);
        if (lane == 0) sm[warp] = v;
        __syncthreads();
        double t = sm[0];
        for (int w = 1; w < NWARPS; ++w) t += sm[w];
        __syncthreads();
        return t;
    };
    auto block_max = [&](double v) {
        v = warp_max(v);
        if (lane == 0) sm[warp] = v;
        __syncthreads();
        double t = sm[0];
        for (int w = 1; w < NWARPS; ++w) t = sm[w] > t ? sm[w] : t;
        __syncthreads();
        return t;
    };
    // T-exchange path: num / denum of entry i from the ranks' slots of G^T S (rank order) and the global H' statistics
    auto w_entry_tx = [&](int i) {
        const int mm = i / k, kk = i - mm * k;
        TC gs;
        if (tx) {
            const unsigned char* base = reinterpret_cast<const unsigned char*>(st.peer_xchg[st.rank]) + recv_off;
            gs = __ldcg(reinterpret_cast<const TC*>(base) + mm * KP + kk);
            for (int r = 1; r < st.world; ++r)
                gs += __ldcg(reinterpret_cast<const TC*>(base + (size_t)r * st.xchg_slot) + mm * KP + kk);
        } else {
            gs = __ldcg(S + mm * KP + kk);
        }
        const TC nv = W[i] * gs, dv = colsumG[mm] * (TC)hs_sm[kk];      // updates.py:59-60
        if (blockIdx.x == 0) {
            wnum[i] = nv;
            wden[i] = dv;
        }
        TC v = Num<TC>::vmax(nv / dv, ls);
        if (st.flags & ESPM_FLAG_FIXED_W) {
            const TC f = fw[i];
            if (f >= TC(0)) v = f;
        }
        return v;
    };
    if (redundant_b) {
        double wsum = 0.0;
        for (int i = threadIdx.x; i < m * k; i += W_COOP_THREADS) {
            const TC v = tp ? w_entry_tx(i) : w_entry(i);
            if (blockIdx.x == 0) Wn[i] = v;
            wsm[i] = v;
            wsum += (double)v;
        }
        __syncthreads();
        if (blockIdx.x == 0) {   // the scalars of the record are CTA 0's business
            const double meanW = block_sum(wsum) / (double)(m * k);
            double rel = 0.0;
            for (int i = threadIdx.x; i < m * k; i += W_COOP_THREADS) {
                const double wn = (double)wsm[i], wo = (double)W[i];
                const double r = fabs(wn - wo) / (wn + st.tol * meanW);
                rel = r > rel ? r : rel;
            }
            rel = block_max(rel);
            if (threadIdx.x == 0) {
                st.scalars[ESPM_S_REL_W] = rel;
                st.scalars[ESPM_S_BISECT_ITS_W] = (double)s_its;
                st.scalars[ESPM_S_MEAN_W] = meanW;
            }
        }
    } else {
        const int total = m * k, per = (total + (int)gridDim.x - 1) / (int)gridDim.x;
        const int i0 = blockIdx.x * per, i1 = (i0 + per < total) ? i0 + per : total;
        double* row = st.coop_part + (size_t)blockIdx.x * W_COOP_STRIDE;
        double wsum = 0.0;
        for (int i = i0 + threadIdx.x; i < i1; i += W_COOP_THREADS) {
            const TC v = w_entry(i);
            Wn[i] = v;
            wsum += (double)v;
        }
        wsum = block_sum(wsum);
        if (threadIdx.x == 0) row[2 * ESPM_MAX_K + 1] = wsum;
        grid_barrier(bar, gridDim.x);
        double meanW = 0.0;
        for (int b = 0; b < (int)gridDim.x; ++b) meanW += __ldcg(st.coop_part + (size_t)b * W_COOP_STRIDE + 2 * ESPM_MAX_K + 1);
        meanW /= (double)total;
        double rel = 0.0;
        for (int i = i0 + threadIdx.x; i < i1; i += W_COOP_THREADS) {
            const double wn = (double)Wn[i], wo = (double)W[i];   // Wn[i]: this thread's own store
            const double r = fabs(wn - wo) / (wn + st.tol * meanW);
            rel = r > rel ? r : rel;
        }
        rel = block_max(rel);
        if (threadIdx.x == 0) row[2 * ESPM_MAX_K + 2] = rel;
    }
    __syncthreads();

    // ---- phase C: GW' = G W' for the next H pass (updates.py:107), one channel per thread ----
    {
        const TC* Wsrc = redundant_b ? wsm : Wn;
        TC* GW = reinterpret_cast<TC*>(st.GW_next);
        TC* GWc = reinterpret_cast<TC*>(st.GWc_next);
        double cs[KP], csc[KP];
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) cs[kk] = csc[kk] = 0.0;
        uint32_t flags = 0u;
        for (int c = gthread; c < st.n_pad; c += gthreads) {
            TC v[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) v[kk] = TC(0);
            if (c >= n) {
                v[0] = TC(1);  // pad channel: y = H[0] > 0, contributes nothing
            } else if (ident) {
#pragma unroll
                for (int kk = 0; kk < KP; ++kk)
                    if (kk < k) v[kk] = Wsrc[(size_t)c * k + kk];
            } else {
#pragma unroll 8
                for (int mm = 0; mm < m; ++mm) {
                    const TC g = Gt[(size_t)mm * n + c];   // coalesced over the channels of a warp
#pragma unroll
                    for (int kk = 0; kk < KP; ++kk)
                        if (kk < k) v[kk] = fma(g, Wsrc[(size_t)mm * k + kk], v[kk]);
                }
            }
            bool all_zero = true;
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                const bool real = c < n && kk < k;
                const TC vc = real ? Num<TC>::vmax(v[kk], ls) : v[kk];
                GW[(size_t)c * KP + kk] = v[kk];
                GWc[(size_t)c * KP + kk] = vc;
                if (real) {
                    cs[kk] += (double)v[kk];
                    csc[kk] += (double)vc;
                    if (v[kk] < ls) flags |= ESPM_DEV_GW_BELOW_LS;
                    if (v[kk] > TC(0)) all_zero = false;
                }
            }
            if (c < n && all_zero) flags |= ESPM_DEV_GW_ZERO_ROW;
        }
        // per-CTA column sums (fixed order) -> coop_part[block][2*KP + 1]
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            const double a = warp_sum(cs[kk]), b = warp_sum(csc[kk]);
            if (lane == 0) {
                sm[warp * 2 * KP + kk] = a;
                sm[warp * 2 * KP + KP + kk] = b;
            }
        }
        const uint32_t f = __reduce_or_sync(0xffffffffu, flags);
        if (threadIdx.x == 0) s_err = 0u;
        __syncthreads();
        if (lane == 0 && f) atomicOr(&s_err, f);
        __syncthreads();
        double* part = st.coop_part + (size_t)blockIdx.x * W_COOP_STRIDE;
        if (threadIdx.x < 2 * KP) {
            double a = 0.0;
            for (int w = 0; w < NWARPS; ++w) a += sm[w * 2 * KP + threadIdx.x];
            part[threadIdx.x] = a;
        }
        if (threadIdx.x == 0) part[2 * ESPM_MAX_K] = (double)s_err;
    }
    // ---- phase D (the last CTA to get here): column sums over the CTAs in index order ----
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&st.dev_flags[4], 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last) {
        __threadfence();
        TC* gwstats = reinterpret_cast<TC*>(st.gwstats_next);
        // one warp per column: lane b fetches CTA b's partial (ONE L2 round trip for the whole fold instead of gridDim
        // dependent ones), butterfly sum in a fixed order
        for (int v = warp; v < 2 * KP + 1; v += NWARPS) {
            const int col = v < 2 * KP ? v : 2 * ESPM_MAX_K;      // last "column": the CTAs' flag words
            double a = 0.0;
            uint32_t fb = 0u;
            for (int b = lane; b < (int)gridDim.x; b += 32) {
                const double x = __ldcg(st.coop_part + (size_t)b * W_COOP_STRIDE + col);
                if (v < 2 * KP) a += x;
                else fb |= (uint32_t)x;
            }
            if (v < 2 * KP) {
                a = warp_sum(a);
                if (lane == 0) gwstats[v] = (TC)a;
            } else {
                fb = __reduce_or_sync(0xffffffffu, fb);
                if (lane == 0) s_err = fb;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            time_stamp(st, 5);
            const uint32_t f = s_err;
            st.dev_flags[1] = f;
            st.scalars[ESPM_S_GW_FLAGS] = (double)f;
            if (!redundant_b) {   // scalars of the sliced phase B, folded in CTA order
                double ws = 0.0, rel = 0.0;
                for (int b = 0; b < (int)gridDim.x; ++b) {
                    ws += __ldcg(st.coop_part + (size_t)b * W_COOP_STRIDE + 2 * ESPM_MAX_K + 1);
                    const double r = __ldcg(st.coop_part + (size_t)b * W_COOP_STRIDE + 2 * ESPM_MAX_K + 2);
                    rel = r > rel ? r : rel;
                }
                st.scalars[ESPM_S_REL_W] = rel;
                st.scalars[ESPM_S_BISECT_ITS_W] = (double)s_its;
                st.scalars[ESPM_S_MEAN_W] = ws / (double)(m * k);
            }
            st.dev_flags[4] = 0u;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Gram matrix of k vectors: out[a][b] = sum_r A(r, a) A(r, b), A(r, a) = A[r * ld_r + a * ld_a].
// One CTA per (a, b) pair; fixed-order reduction.  Used for (G W)^T (G W) and H H^T (updates.py:31, 115).
// ------------------------------------------------------------------------------------------------
template <typename TC>
__global__ void __launch_bounds__(256) gram_kernel(const TC* A, long long rows, long long ld_r, long long ld_a, int k,
                                                   int kp, double* out) {
    const int a = blockIdx.x / k, b = blockIdx.x % k;
    __shared__ double sm[8];
    double acc = 0.0;
    for (long long r = threadIdx.x; r < rows; r += blockDim.x)
        acc = fma((double)A[r * ld_r + a * ld_a], (double)A[r * ld_r + b * ld_a], acc);
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sm[w];
        out[a * kp + b] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// Line search on the Laplacian surrogate (smooth_nmf.py:376-382; surrogates.py:5-53, 66-149), Ht = H_cur
// (the iterate the surrogate was built at), H = H_next:
//   t1 = sum (Ht L) Ht, t2 = sum (Ht L) H, b_inf = trace(H L H^T) / 2,
//   t3 = sum_k max_j(H_kj) sum_j dgkl(Ht_kj, H_kj)   (log_surrogate, bmd)   |   sum (Ht - H)^2   (l2_surrogate)
//   d = (2 t2 - t1 + sigma t3) / 2 - b_inf;   gamma_ <- gamma_ / 1.05 if d > 0 else gamma_ * 1.5
// (diff_surrogate is called with its default lambda_L = 1, smooth_nmf.py:378.)
// ------------------------------------------------------------------------------------------------
template <typename TC, int KP>
__global__ void __launch_bounds__(PX_THREADS) linesearch_kernel(const espm_state st) {
    const int j = blockIdx.x * PX_THREADS + threadIdx.x;
    const int k = st.k;
    const bool quad = st.flags & ESPM_FLAG_HQ;
    constexpr int NV = 4 + KP;   // t1, t2, trace(H L H), (quad: sum sq) , per-phase dgkl row sums
    double vals[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) vals[i] = 0.0;
    if (j < st.p_loc) {
        const TC* Ho = reinterpret_cast<const TC*>(st.H_cur);
        const TC* Hn = reinterpret_cast<const TC*>(st.H_next);
        int deg = 0;
        bool up = false, down = false, left = false, right = false;
        if (st.ny > 0) {
            const int il = j / st.ny, col = j - il * st.ny;
            const int ig = st.row0 + il;
            left = col > 0;
            right = col < st.ny - 1;
            up = ig > 0;
            down = ig < st.nx - 1;
            deg = (int)left + (int)right + (int)up + (int)down;
        }
#pragma unroll
        for (int kk = 0; kk < KP; ++kk)
            if (kk < k) {
                const TC* ro = Ho + (size_t)kk * st.ldh;
                const TC* rn = Hn + (size_t)kk * st.ldh;
                const double ho = (double)ro[j], hn = (double)rn[j];
                double lo = ho, ln = hn;   // (Ht L)_j and (H L)_j; identity when shape_2d is None
                if (st.ny > 0) {
                    double so = 0.0, sn = 0.0;
                    if (up) { so += (double)ro[j - st.ny]; sn += (double)rn[j - st.ny]; }
                    if (left) { so += (double)ro[j - 1]; sn += (double)rn[j - 1]; }
                    if (right) { so += (double)ro[j + 1]; sn += (double)rn[j + 1]; }
                    if (down) { so += (double)ro[j + st.ny]; sn += (double)rn[j + st.ny]; }
                    lo = (double)deg * ho - so;
                    ln = (double)deg * hn - sn;
                }
                if (st.flags & ESPM_FLAG_PG) {   // quadratic surrogate of the projected gradient (surrogates.py:153-171)
                    const double g = (double)reinterpret_cast<const TC*>(st.den)[(size_t)kk * st.p_pad + j];
                    vals[0] += (hn - ho) * g;
                    vals[1] += (hn - ho) * (hn - ho);
                    continue;
                }
                vals[0] += lo * ho;
                vals[1] += lo * hn;
                vals[2] += ln * hn;
                if (quad) vals[3] += (ho - hn) * (ho - hn);
                else vals[4 + kk] = ho * log(ho / hn) - ho + hn;
            }
    }
    block_reduce_vals<NV>(vals, NV, st.ls_part + (size_t)blockIdx.x * NV);
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(&st.dev_flags[4], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // fold the per-CTA partials in index order; rowmax(H_next) from the px_part rows written by the H update
    __shared__ double tot[NV + KP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int stride = px_part_stride(KP);
    for (int v = warp; v < NV + KP; v += PX_WARPS) {
        const bool is_max = v >= NV;
        double r = is_max ? -1e300 : 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) {
            const double u = is_max ? st.px_part[(size_t)b * stride + 3 + 2 * KP + (v - NV)] : st.ls_part[(size_t)b * NV + v];
            r = is_max ? (u > r ? u : r) : r + u;
        }
        r = is_max ? warp_max(r) : warp_sum(r);
        if (lane == 0) tot[v] = r;
    }
    __syncthreads();
    if (st.flags & ESPM_FLAG_LS_PARTIAL) {
        // sharded: the sums of this rank only; the caller adds the ranks (max for the row maxima) and decides
        if ((int)threadIdx.x < NV + KP) st.ls_part[(size_t)gridDim.x * NV + threadIdx.x] = tot[threadIdx.x];
        if (threadIdx.x == 0) st.dev_flags[4] = 0u;
        return;
    }
    if (threadIdx.x == 0 && (st.flags & ESPM_FLAG_PG)) {
        st.scalars[ESPM_S_LS_D] = tot[0];
        st.scalars[ESPM_S_GAMMA] = tot[1];
        st.dev_flags[4] = 0u;
    } else if (threadIdx.x == 0) {
        const double sigma = *st.sigma_dev;
        double t3 = tot[3];
        if (!quad) {
            t3 = 0.0;
            for (int kk = 0; kk < k; ++kk) t3 += tot[NV + kk] * tot[4 + kk];
        }
        const double d = 0.5 * (2.0 * tot[1] - tot[0] + sigma * t3) - 0.5 * tot[2];
        const double g = d > 0.0 ? sigma / 1.05 : sigma * 1.5;
        *st.sigma_dev = g;
        st.scalars[ESPM_S_GAMMA] = g;
        st.scalars[ESPM_S_LS_D] = d;
        st.dev_flags[4] = 0u;
    }
}

// ------------------------------------------------------------------------------------------------
// Standalone dichotomy_simplex(num, den) -> nu  (dicotomy.py:4-55), two kernels: trace, replay.
// acc_a > 0 selects dichotomy_simplex_acc(a, b = den, minus_c = num) (dicotomy.py:57-81, fp64 only).
// ------------------------------------------------------------------------------------------------
template <typename TC, int KP>
__global__ void __launch_bounds__(PX_THREADS) dicho_trace_kernel(const TC* num_i, const TC* den_i, long long p, int k,
                                                                 double ls_d, double tol_d, int maxit, double acc_a,
                                                                 uint32_t* gmask, uint32_t* gflags) {
    const long long j = (long long)blockIdx.x * PX_THREADS + threadIdx.x;
    Mask128 bits;
    bits.clear();
    uint32_t err = 0u;
    if (j < p) {
        TC num[KP], den[KP];
        TC nsum = TC(0);
        const bool acc = acc_a > 0.0, pgm = acc_a < 0.0;
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            num[kk] = (kk < k) ? num_i[(size_t)kk * p + j] : TC(0);
            den[kk] = (kk < k && !pgm) ? den_i[(size_t)kk * p + j] : TC(1);
            if (kk < k && !pgm) {
                nsum += num[kk];
                if (num[kk] < TC(0) || (!acc && den[kk] < TC(0))) err |= ESPM_DEV_NEGATIVE;
            }
        }
        if (acc_a < 0.0) {   // projected gradient: num holds a (dicotomy.py:83-108)
            double av[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) av[kk] = (double)num[kk];
            const PgEval<KP> ev(av, k, ls_d, tol_d);
            double lo, hi;
            ev.bracket(lo, hi);
            Mask128 dec;
            dec.clear();
            uint32_t seen;
            err = 0u;
            bisect_trace_rec(lo, hi, ev, maxit, bits, dec, seen, err);
        } else if (acc) {
            double c[KP], b[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                c[kk] = (double)num[kk];
                b[kk] = (double)den[kk];
            }
            acc_trace<KP>(c, b, k, acc_a, ls_d, tol_d, maxit, bits, err);
        } else {
            if (!(nsum > TC(0))) err |= ESPM_DEV_NEGATIVE;  // dicotomy.py:19
            simplex_trace<TC, KP>(num, den, k, (TC)ls_d, (TC)tol_d, maxit, bits, err);
        }
    }
    merge_mask(bits, err, gmask, gflags);
}

template <typename TC, int KP>
__global__ void __launch_bounds__(PX_THREADS) dicho_apply_kernel(const TC* num_i, const TC* den_i, long long p, int k,
                                                                 double ls_d, int maxit, double acc_a,
                                                                 const uint32_t* gmask, TC* nu_out, int* its_out) {
    const long long j = (long long)blockIdx.x * PX_THREADS + threadIdx.x;
    const int its = first_clear_bit(gmask, maxit);
    if (j == 0 && its_out) *its_out = its;
    if (j < p) {
        TC num[KP], den[KP];
#pragma unroll
        for (int kk = 0; kk < KP; ++kk) {
            num[kk] = (kk < k) ? num_i[(size_t)kk * p + j] : TC(0);
            den[kk] = (kk < k && !(acc_a < 0.0)) ? den_i[(size_t)kk * p + j] : TC(1);
        }
        if (acc_a < 0.0) {
            double av[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) av[kk] = (double)num[kk];
            const PgEval<KP> ev(av, k, ls_d, 0.0);
            double lo, hi;
            ev.bracket(lo, hi);
            Mask128 none;
            none.clear();
            nu_out[j] = (TC)bisect_replay_rec(lo, hi, ev, its, none, 0u);
        } else if (acc_a > 0.0) {
            double c[KP], b[KP];
#pragma unroll
            for (int kk = 0; kk < KP; ++kk) {
                c[kk] = (double)num[kk];
                b[kk] = (double)den[kk];
            }
            nu_out[j] = (TC)acc_replay<KP>(c, b, k, acc_a, ls_d, its);
        } else {
            nu_out[j] = simplex_replay<TC, KP>(num, den, k, (TC)ls_d, its);
        }
    }
}

}  // namespace espm
