// Explicit instantiation helpers for the X-pass kernels: one translation unit per (storage, compute)
// type pair so that the 48 template instances compile in parallel.
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

template <typename TX, typename TC, bool SAFE>
static int xpass_by_kp(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream) {
    switch (l.kp) {
        case 2: return xpass_do<TX, TC, 2, SAFE>(l, a, occ_out, stream);
        case 3: return xpass_do<TX, TC, 3, SAFE>(l, a, occ_out, stream);
        case 4: return xpass_do<TX, TC, 4, SAFE>(l, a, occ_out, stream);
        case 5: return xpass_do<TX, TC, 5, SAFE>(l, a, occ_out, stream);
        case 6: return xpass_do<TX, TC, 6, SAFE>(l, a, occ_out, stream);
        case 8: return xpass_do<TX, TC, 8, SAFE>(l, a, occ_out, stream);
        case 12: return xpass_do<TX, TC, 12, SAFE>(l, a, occ_out, stream);
        case 16: return xpass_do<TX, TC, 16, SAFE>(l, a, occ_out, stream);
        default:
            set_error("unsupported padded component count kp=%d", l.kp);
            return ESPM_ERR_BAD_ARG;
    }
}

template <typename TX, typename TC>
static int xpass_entry(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream) {
    return l.safe ? xpass_by_kp<TX, TC, true>(l, a, occ_out, stream) : xpass_by_kp<TX, TC, false>(l, a, occ_out, stream);
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
    switch (kp) {
        case 2: xpass_sizes_kp<TX, TC, 2>(safe, o); return ESPM_OK;
        case 3: xpass_sizes_kp<TX, TC, 3>(safe, o); return ESPM_OK;
        case 4: xpass_sizes_kp<TX, TC, 4>(safe, o); return ESPM_OK;
        case 5: xpass_sizes_kp<TX, TC, 5>(safe, o); return ESPM_OK;
        case 6: xpass_sizes_kp<TX, TC, 6>(safe, o); return ESPM_OK;
        case 8: xpass_sizes_kp<TX, TC, 8>(safe, o); return ESPM_OK;
        case 12: xpass_sizes_kp<TX, TC, 12>(safe, o); return ESPM_OK;
        case 16: xpass_sizes_kp<TX, TC, 16>(safe, o); return ESPM_OK;
        default: set_error("unsupported padded component count kp=%d", kp); return ESPM_ERR_BAD_ARG;
    }
}

// defined in xpass_f32f32.cu / xpass_f32f64.cu / xpass_f64f64.cu
int xpass_f32f32(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream);
int xpass_f32f64(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream);
int xpass_f64f64(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream);
// compact count storage (SURVEY.md section 8f-4): uint8 / uint16 X with fp32 arithmetic
int xpass_u8f32(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream);
int xpass_u16f32(const XPassLaunch& l, const XPassArgs* a, int* occ_out, cudaStream_t stream);

}  // namespace espm
