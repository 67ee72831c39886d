// Host-side declarations of the phase information launchers (winfo_f32.cu / winfo_f64.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/espm_b200.h"

namespace espm {
// out: [k (k + 1) / 2][n] doubles (packed A_c); with bytes_out set, only the scratch size is written
int w_info_f32f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
int w_info_u8f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
int w_info_u16f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
int w_info_f32f64(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
int w_info_f64f64(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s);
}  // namespace espm
