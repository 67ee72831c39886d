// Launch helpers for the k x p / m x k kernels, instantiated once per arithmetic type.
#pragma once
#include "small.cuh"

namespace espm {

enum SmallOp {
    OP_H_FINISH = 0,
    OP_H_APPLY,
    OP_H_STATS,
    OP_W_REDUCE,
    OP_W_FINISH,
    OP_GW_PREPARE,
    OP_LINESEARCH,
    OP_GRAM_GW,
    OP_GRAM_H,
};

struct DichoArgs {
    int k, kp, maxit;
    long long p;
    const void* num;
    const void* den;
    double log_shift, tol;
    double acc_a;   // > 0: dichotomy_simplex_acc with this `a` (num = minus_c, den = b)
    void* nu_out;
    uint32_t* mask4;
    uint32_t* dev_flags;
    int* its_out;
};

template <typename TC>
static int small_launch_t(int op, const espm_state* st, cudaStream_t s) {
    const int kp = st->kp;
    switch (op) {
        case OP_H_FINISH:
            if (st->n_sms > 0 && st->px_blocks <= 2 * st->n_sms) {
                ESPM_KP_SWITCH(kp, ESPM_CUDA_CHECK(launch_pdl(h_finish_kernel<TC, KP, 2>, dim3(st->px_blocks), dim3(PX_THREADS), 0, s, *st)));
            } else {
                ESPM_KP_SWITCH(kp, ESPM_CUDA_CHECK(launch_pdl(h_finish_kernel<TC, KP, 4>, dim3(st->px_blocks), dim3(PX_THREADS), 0, s, *st)));
            }
            break;
        case OP_H_APPLY:
            ESPM_KP_SWITCH(kp, ESPM_CUDA_CHECK(launch_pdl(h_apply_kernel<TC, KP>, dim3(st->px_blocks), dim3(PX_THREADS), 0, s, *st)));
            break;
        case OP_H_STATS:
            ESPM_KP_SWITCH(kp, (h_stats_kernel<TC, KP><<<st->px_blocks, PX_THREADS, 0, s>>>(*st)));
            ESPM_KP_SWITCH(kp, (hstats_reduce_kernel<TC, KP><<<1, 256, 0, s>>>(*st)));
            break;
        case OP_W_REDUCE: {
            const size_t total = (size_t)st->n_pad * st->kp;
            const int blocks = (int)((total + 255) / 256) + 1;
            ESPM_KP_SWITCH(kp, (w_reduce_kernel<TC, KP><<<blocks, 256, 0, s>>>(*st)));
            break;
        }
        case OP_W_FINISH: {
            // cooperative launch: the kernel separates its phases with grid barriers
            espm_state copy = *st;
            void* args[] = {&copy};
            const void* fn = nullptr;
            ESPM_KP_SWITCH(kp, (fn = (const void*)w_finish_kernel<TC, KP>));
            // cooperative (grid barriers) AND programmatic dependent launch: the CTAs become resident while the W
            // pass drains and wait in griddepcontrol.wait
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(W_COOP_BLOCKS);
            cfg.blockDim = dim3(W_COOP_THREADS);
            cfg.dynamicSmemBytes = 0;
            cfg.stream = s;
            cudaLaunchAttribute attr[2];
            attr[0].id = cudaLaunchAttributeCooperative;
            attr[0].val.cooperative = 1;
            attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            attr[1].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 2;
            ESPM_CUDA_CHECK(cudaLaunchKernelExC(&cfg, fn, args));
            break;
        }
        case OP_GW_PREPARE:
            gw_prepare_kernel<TC><<<1, 1024, 0, s>>>(*st);
            break;
        case OP_LINESEARCH:
            ESPM_KP_SWITCH(kp, (linesearch_kernel<TC, KP><<<st->px_blocks, PX_THREADS, 0, s>>>(*st)));
            break;
        case OP_GRAM_GW:   // over the n real channels of GW_cur [n_pad][kp]
            gram_kernel<TC><<<st->k * st->k, 256, 0, s>>>((const TC*)st->GW_cur, st->n, st->kp, 1, st->k, st->kp,
                                                            st->gram_gw);
            break;
        case OP_GRAM_H:    // over the p_loc pixels of H_next [k][ldh]
            gram_kernel<TC><<<st->k * st->k, 256, 0, s>>>((const TC*)st->H_next, st->p_loc, 1, st->ldh, st->k, st->kp,
                                                            st->gram_h);
            break;
        default:
            set_error("unknown small op %d", op);
            return ESPM_ERR_BAD_ARG;
    }
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

template <typename TC>
static int dicho_launch_t(const DichoArgs& d, cudaStream_t s) {
    const int blocks = (int)((d.p + PX_THREADS - 1) / PX_THREADS);
    ESPM_CUDA_CHECK(cudaMemsetAsync(d.mask4, 0, 4 * sizeof(uint32_t), s));
    ESPM_KP_SWITCH(d.kp, (dicho_trace_kernel<TC, KP><<<blocks, PX_THREADS, 0, s>>>(
                             (const TC*)d.num, (const TC*)d.den, d.p, d.k, d.log_shift, d.tol, d.maxit, d.acc_a,
                             d.mask4, d.dev_flags)));
    ESPM_CUDA_CHECK(cudaGetLastError());
    ESPM_KP_SWITCH(d.kp, (dicho_apply_kernel<TC, KP><<<blocks, PX_THREADS, 0, s>>>(
                             (const TC*)d.num, (const TC*)d.den, d.p, d.k, d.log_shift, d.maxit, d.acc_a, d.mask4,
                             (TC*)d.nu_out, d.its_out)));
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

template <typename TC>
static int colsum_launch_t(const espm_state* st, void* out, cudaStream_t s) {
    const int warps_per_block = 8;
    const int blocks = (st->m + warps_per_block - 1) / warps_per_block;
    colsum_g_kernel<TC><<<blocks, 256, 0, s>>>((const TC*)st->Gt, st->n, st->m, (TC*)out);
    ESPM_CUDA_CHECK(cudaGetLastError());
    return ESPM_OK;
}

// defined in small_f32.cu / small_f64.cu
int small_launch_f32(int op, const espm_state* st, cudaStream_t s);
int small_launch_f64(int op, const espm_state* st, cudaStream_t s);
int dicho_launch_f32(const DichoArgs& d, cudaStream_t s);
int dicho_launch_f64(const DichoArgs& d, cudaStream_t s);
int colsum_launch_f32(const espm_state* st, void* out, cudaStream_t s);
int colsum_launch_f64(const espm_state* st, void* out, cudaStream_t s);

}  // namespace espm
