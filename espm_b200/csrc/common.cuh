// Shared device helpers for the espm_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include <cstdlib>
#include <utility>

#include "../../include/espm_b200.h"

#ifndef __CUDA_ARCH__
#define ESPM_DEVICE_ARCH 0
#else
#define ESPM_DEVICE_ARCH __CUDA_ARCH__
#endif

namespace espm {

constexpr int TILE_PX = ESPM_TILE_PX;        // pixels per tile
constexpr int STAGE_BYTES = ESPM_STAGE_BYTES; // X bytes per pipeline stage
constexpr int N_CONSUMER_WARPS = 8;
constexpr int N_CONSUMER_THREADS = N_CONSUMER_WARPS * 32;
constexpr int XPASS_THREADS = N_CONSUMER_THREADS + 32;  // + one TMA producer warp

// ---------------------------------------------------------------- error plumbing (host)
void set_error(const char* fmt, ...);
#define ESPM_CUDA_CHECK(expr)                                                               \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            espm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                            __LINE__);                                                      \
            return ESPM_ERR_CUDA;                                                           \
        }                                                                                   \
    } while (0)

// Runs the statement with `constexpr int KP` set to the padded component count kp (one instance per supported width);
// any other kp is an error.  Variadic so that the statement may hold template argument lists.
#define ESPM_KP_SWITCH(kp, ...)                                         \
    switch (kp) {                                                       \
        case 2: { constexpr int KP = 2; __VA_ARGS__; break; }           \
        case 3: { constexpr int KP = 3; __VA_ARGS__; break; }           \
        case 4: { constexpr int KP = 4; __VA_ARGS__; break; }           \
        case 5: { constexpr int KP = 5; __VA_ARGS__; break; }           \
        case 6: { constexpr int KP = 6; __VA_ARGS__; break; }           \
        case 8: { constexpr int KP = 8; __VA_ARGS__; break; }           \
        case 12: { constexpr int KP = 12; __VA_ARGS__; break; }         \
        case 16: { constexpr int KP = 16; __VA_ARGS__; break; }         \
        default:                                                        \
            set_error("unsupported padded component count kp=%d", kp);  \
            return ESPM_ERR_BAD_ARG;                                    \
    }

// ---------------------------------------------------------------- mbarrier / bulk-copy PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// TMA bulk copy global -> shared (contiguous bytes, 16 B aligned, size % 16 == 0); completion is
// signalled on `bar` through complete_tx.  SASS: UBLKCP.
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                             uint64_t* bar, uint64_t l2_policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
            "r"(smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(l2_policy)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// The per-iteration kernels are launched with cudaLaunchAttributeProgrammaticStreamSerialization: a kernel's CTAs
// may be scheduled while the previous kernel of the stream drains.  pdl_wait() (griddepcontrol.wait) is the FIRST
// statement of every such kernel -- nothing of the predecessor is read or overwritten before it returns, so the only
// effect is that launch latency and CTA start-up overlap the predecessor's tail.  pdl_trigger() lets the next kernel
// of the stream do the same with us.  Both are no-ops for kernels launched without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// ---------------------------------------------------------------- arithmetic traits
template <typename T>
struct Num;
template <>
struct Num<float> {
    // x / y for the streaming passes: MUFU.RCP + FMUL (<= 2 ulp; the fp32 mode's bar is 1e-5)
    static __device__ __forceinline__ float ratio(float x, float y) { return __fdividef(x, y); }
    static __device__ __forceinline__ float log2_fast(float y) { return __log2f(y); }
    static __device__ __forceinline__ float vmax(float a, float b) { return fmaxf(a, b); }
    static __device__ __forceinline__ float vmin(float a, float b) { return fminf(a, b); }
    static __device__ __forceinline__ float vabs(float a) { return fabsf(a); }
    static __device__ __forceinline__ float vsqrt(float a) { return sqrtf(a); }
    static __device__ __forceinline__ float vlog(float a) { return logf(a); }
    static __device__ __forceinline__ float inf() { return __int_as_float(0x7f800000); }
};
template <>
struct Num<double> {
    // fp64 reciprocal: MUFU.RCP64H seed (rcp.approx.ftz.f64, ~20 good bits, full exponent range) + two
    // Newton steps in fp64 => <= 1 ulp.  y == 0 gives NaN/inf like the division would (callers flag
    // non-finite results); 7 instructions instead of the ~25 of an IEEE fp64 division.
    static __device__ __forceinline__ double rcp(double y) {
        double r;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));
        double e = fma(-y, r, 1.0);
        r = fma(r, e, r);
        e = fma(-y, r, 1.0);
        r = fma(r, e, r);
        return r;
    }
    // x / y of the streaming passes: the seed is good to 2^-19.9 (scripts/probes/rcp_probe.cu), so ONE cubic step
    // r (1 + e + e^2), e = 1 - y r, leaves e^3 = 2^-59.7: 3 DFMA instead of 4, max error 1 ulp on the reciprocal
    // (measured over 2^24 arguments); the step tolerance of the fp64 mode is 1e-10.
    static __device__ __forceinline__ double ratio(double x, double y) {
        double r;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(y));
        const double e = fma(-y, r, 1.0);
        const double t = fma(e, e, e);
        return x * fma(r, t, r);
    }
    static __device__ __forceinline__ double log2_fast(double y) { return log2(y); }
    static __device__ __forceinline__ double vmax(double a, double b) { return fmax(a, b); }
    static __device__ __forceinline__ double vmin(double a, double b) { return fmin(a, b); }
    static __device__ __forceinline__ double vabs(double a) { return fabs(a); }
    static __device__ __forceinline__ double vsqrt(double a) { return sqrt(a); }
    static __device__ __forceinline__ double vlog(double a) { return log(a); }
    static __device__ __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000LL); }
};

// Table-driven log2 of a double for the streaming H pass (the CUDA library log2 is ~35 DP-pipe instructions, which
// made the fp64 H pass DP-bound at 0.41 of the HBM peak): y = 2^e m, i = top 7 mantissa bits of m,
// r = m * inv_i - 1 with inv_i = 1 / (1 + (i + 0.5) / 128)  (|r| <= 2^-8, one exact FMA),
// log2(y) = e - log2(inv_i) + r * P(r), P of degree 4 fitted to log2(1 + r) / r on |r| <= 2^-8 (truncation
// 3e-17).  8 DP instructions; absolute error <= 2 ulp of the result (the final additions), checked against a
// long-double evaluation in tests/test_log2_table.py.  Zero / subnormal / negative / non-finite arguments take
// the library path.
constexpr int LOG2TAB_N = 128;
// The 16-byte entries are replicated LOG2TAB_R = 4 times in shared memory: a lane reads copy (lane & 3), and copy c of
// entry i lives at 16-byte slot (i & 63) * 8 + c * 2 + (i >> 6), i.e. in bank groups {2c, 2c + 1}.  An LDS.128 is
// served per quarter warp (8 lanes), so lookups with unrelated i collide only between the two lanes that share a copy
// (expected 1.5 wavefronts per quarter instead of 2.6 for a single copy: the single-copy table spent 40 % of the
// kernel's shared-memory wavefronts on bank conflicts, profiles/r01f_summary.md).
constexpr int LOG2TAB_R = 4;
constexpr int LOG2TAB_BYTES = LOG2TAB_N * LOG2TAB_R * 16;
__device__ __forceinline__ void log2tab_fill(double2* tab, int tid, int nthreads) {
    for (int i = tid; i < LOG2TAB_N; i += nthreads) {
        const double inv = 1.0 / (1.0 + ((double)i + 0.5) * (1.0 / LOG2TAB_N));
        const double2 v = make_double2(inv, -log2(inv));
#pragma unroll
        for (int c = 0; c < LOG2TAB_R; ++c) tab[(i & 63) * 8 + c * 2 + (i >> 6)] = v;
    }
}
// this lane's view of the table: byte offset of its copy folded into the base pointer
__device__ __forceinline__ const double2* log2tab_lane(const double2* tab, int lane) { return tab + (lane & 3) * 2; }
// entry of mantissa index i = hi[19:13] in the lane's copy: slot (i & 63) * 8 + (i >> 6)
__device__ __forceinline__ double2 log2tab_get(const double2* lane_tab, int hi) {
    const unsigned off = (((unsigned)hi >> 6) & 0x1f80u) | (((unsigned)hi >> 15) & 0x10u);   // bytes
    return *reinterpret_cast<const double2*>(reinterpret_cast<const unsigned char*>(lane_tab) + off);
}
// polynomial coefficients in constant memory: DFMA takes them as c[bank][offset] operands (64-bit immediates
// would cost two UMOVs each)
static __device__ __constant__ double LOG2_C[5] = {0x1.71547652b82ffp+0, -0x1.715476529026dp-1, 0x1.ec709dc2ea15bp-2,
                                                   -0x1.7155b049ac044p-2, 0x1.277837d2b64aap-2};
// Branch-free core: valid for normal positive y.  `range` accumulates max((unsigned)(hi - 0x00100000)); the caller
// tests log2_range_bad(range) once per batch and redoes the batch with the library log2 if it fires.
// `tab` is the lane's view (log2tab_lane).
__device__ __forceinline__ double log2_tab_core(double y, const double2* tab, unsigned& range) {
    const int hi = __double2hiint(y);
    const unsigned t = (unsigned)hi - 0x00100000u;
    range = t > range ? t : range;
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(y));
    const double2 tv = log2tab_get(tab, hi);
    const double r = fma(m, tv.x, -1.0);
    double p = LOG2_C[4];
    p = fma(p, r, LOG2_C[3]);
    p = fma(p, r, LOG2_C[2]);
    p = fma(p, r, LOG2_C[1]);
    p = fma(p, r, LOG2_C[0]);
    return fma(p, r, tv.y + (double)((hi >> 20) - 1023));
}
__device__ __forceinline__ bool log2_range_bad(unsigned range) { return range >= 0x7fe00000u; }
__device__ __forceinline__ double log2_tab(double y, const double2* tab) {
    unsigned range = 0u;
    const double v = log2_tab_core(y, tab, range);
    return log2_range_bad(range) ? log2(y) : v;
}
// max(x, b) for x >= 0, b >= 0 (no NaN): the IEEE order of non-negative doubles is the order of their bit patterns,
// so this is integer compare + select instead of the 7-instruction DSETP.MAX sequence.
__device__ __forceinline__ double max_nonneg(double x, double b) {
    const long long xb = __double_as_longlong(x), bb = __double_as_longlong(b);
    return __longlong_as_double(xb > bb ? xb : bb);
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        T u = __shfl_xor_sync(0xffffffffu, v, o);
        v = v > u ? v : u;
    }
    return v;
}

// Geometry of the X-pass kernels for a (storage, compute) type pair.  A pipeline stage always holds CS = 32 channels
// (16 for f64 storage) x 128 pixels, i.e. ONE contiguous bulk copy of 16 KiB (f32 / f64), 8 KiB (uint16) or 4 KiB
// (uint8): compact count storage changes the bytes per stage, not the work distribution of the consumer warps.
template <typename TX, typename TC>
struct PassGeom {
    static constexpr int PPL = (sizeof(TC) == 8) ? 2 : 4;          // pixels per lane
    static constexpr int HALVES = 4 / PPL;                         // warps covering one 128-px row
    static constexpr int NSLOT = N_CONSUMER_WARPS / HALVES;        // channel rows processed at once
    static constexpr int CS = (sizeof(TX) == 8) ? 16 : 32;         // channels per stage
    static constexpr int X_BYTES = CS * TILE_PX * (int)sizeof(TX); // bytes of X per stage (<= STAGE_BYTES)
    static constexpr int CPW = CS / NSLOT;                         // channels per warp per stage
};
static_assert(PassGeom<float, float>::X_BYTES == STAGE_BYTES && PassGeom<double, double>::X_BYTES == STAGE_BYTES, "stage size");

// host-side helpers implemented in api.cu
int plan_stage_channels(int x_dtype);

}  // namespace espm
