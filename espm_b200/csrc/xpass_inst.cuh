// Host dispatch of the X-pass kernels, and the table row that bundles every X-streaming kernel family of one
// (storage, compute) type pair.  Each pair is one translation unit (stream_<pair>.cu), so the pairs compile in parallel.
#pragma once
#include "xpass.cuh"

namespace espm {

enum XPassKind { XPASS_H = 0, XPASS_W = 1 };

struct XPassLaunch {
    int kind;   // XPassKind
    int kp;
    int safe;
    int grid;
    int smem;
    int mode;   // XMODE_*
};

template <typename TX, typename TC, int KP, bool SAFE>
static int xpass_do(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream) {
    void (*kern)(const XPassArgs) =
        (l.kind == XPASS_H) ? h_pass_kernel<TX, TC, KP, SAFE, XMODE_KL> : w_pass_kernel<TX, TC, KP, SAFE, XMODE_KL>;
    if constexpr (!SAFE) {
        // Frobenius variants (no division, so no clamped instances)
        if (l.mode == XMODE_FROB)
            kern = (l.kind == XPASS_H) ? h_pass_kernel<TX, TC, KP, false, XMODE_FROB> : w_pass_kernel<TX, TC, KP, false, XMODE_FROB>;
        else if (l.mode == XMODE_KL_FROB && l.kind == XPASS_H)
            kern = h_pass_kernel<TX, TC, KP, false, XMODE_KL_FROB>;
    } else if (l.mode != XMODE_KL) {
        set_error("the Frobenius X passes have no clamped (SAFE) instances");
        return ESPM_ERR_UNSUPPORTED;
    }
    {
        // the opt-in shared-memory size is a per-function attribute: set it when it changes, not on every launch
        // (slot = kernel of this instantiation; one device per process is the rule, but the device is checked)
        static int last_smem[8], last_dev[8];
        static bool init = false;
        if (!init) {
            for (int i = 0; i < 8; ++i) last_smem[i] = last_dev[i] = -1;
            init = true;
        }
        const int slot = (l.kind == XPASS_H ? 0 : 4) + (l.mode & 3);
        int dev = 0;
        ESPM_CUDA_CHECK(cudaGetDevice(&dev));
        if (last_smem[slot] != l.smem || last_dev[slot] != dev) {
            ESPM_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, l.smem));
            last_smem[slot] = l.smem;
            last_dev[slot] = dev;
        }
    }
    if (occ_out) {
        ESPM_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ_out, kern, XPASS_THREADS, l.smem));
        return ESPM_OK;
    }
    ESPM_CUDA_CHECK(launch_pdl(kern, dim3(l.grid), dim3(XPASS_THREADS), (size_t)l.smem, stream, *a));
    return ESPM_OK;
}

template <typename TX, typename TC>
static int xpass_entry(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream) {
    if (l.safe) {
        ESPM_KP_SWITCH(l.kp, return xpass_do<TX, TC, KP, true>(l, a, occ_out, stream));
    } else {
        ESPM_KP_SWITCH(l.kp, return xpass_do<TX, TC, KP, false>(l, a, occ_out, stream));
    }
    return ESPM_OK;
}

// sizes needed by the planner (host)
struct XPassSizes {
    int h_stride, w_stride;  // bytes per pipeline stage
    int h_tail, w_tail;      // bytes after the ring (epilogue staging)
    int fixed;               // barriers + misc
    int cs, halves;
    int h_occ, w_occ;        // CTAs per SM the kernels are compiled for
};

template <typename TX, typename TC, int KP>
static void xpass_sizes_kp(int safe, XPassSizes* o) {
    using S0 = XPassSmem<TX, TC, KP, false>;
    using S1 = XPassSmem<TX, TC, KP, true>;
    o->h_stride = safe ? S1::H_STRIDE : S0::H_STRIDE;
    o->w_stride = S0::W_STRIDE;
    o->h_tail = S0::HTAIL_BYTES;
    o->w_tail = S0::WTAIL_BYTES;
    o->fixed = S0::BAR_BYTES + S0::MISC_BYTES;
    o->cs = S0::G::CS;
    o->halves = S0::G::HALVES;
    o->h_occ = S0::OCC_BASE;
    o->w_occ = S0::W_OCC < S1::W_OCC ? S0::W_OCC : S1::W_OCC;
}

template <typename TX, typename TC>
static int xpass_sizes(int kp, int safe, XPassSizes* o) {
    ESPM_KP_SWITCH(kp, xpass_sizes_kp<TX, TC, KP>(safe, o));
    return ESPM_OK;
}

// The launchers of one (storage, compute) pair; one row per pair is defined in stream_<pair>.cu.
// fit_stats, w_info and the residual products with bytes_out != NULL only report the scratch bytes of the launch.
struct StreamPair {
    int x_dtype, c_dtype;   // ESPM_F32 / ESPM_F64 / ESPM_U8 / ESPM_U16
    int (*xpass)(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t s);
    int (*xpass_sizes)(int kp, int safe, XPassSizes* o);
    // pixel_out [4][p_loc], channel_out [4][n]
    int (*fit_stats)(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s);
    // out: [k + 2 k (k + 1) / 2][p_loc] doubles (std rows, packed C, packed F)
    int (*h_info)(const espm_state* st, int simplex, double* out, cudaStream_t s);
    // out: [k (k + 1) / 2][n] doubles (packed A_c)
    int (*w_info)(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
    // products of the Pearson residual: left out [r][p_loc] = R^T Q (Q [n][r]), right out [n][r] = R P^T (P [r][p_loc])
    int (*resid_left)(const espm_state* st, const double* Q, int r, double* out, void* scratch, int64_t* bytes_out,
                      cudaStream_t s);
    int (*resid_right)(const espm_state* st, const double* P, int r, double* out, void* scratch, int64_t* bytes_out,
                       cudaStream_t s);
};
extern const StreamPair stream_f32f32, stream_f32f64, stream_f64f64;
// compact count storage (SURVEY.md section 8f-4): uint8 / uint16 X with fp32 arithmetic
extern const StreamPair stream_u8f32, stream_u16f32;

}  // namespace espm
