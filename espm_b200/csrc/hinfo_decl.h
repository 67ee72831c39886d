// Host-side declarations of the abundance information launchers (hinfo_f32.cu / hinfo_f64.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/espm_b200.h"

namespace espm {
// out: [k + 2 k (k + 1) / 2][p_loc] doubles (std rows, packed C, packed F)
int h_info_f32f32(const espm_state* st, int simplex, double* out, cudaStream_t s);
int h_info_u8f32(const espm_state* st, int simplex, double* out, cudaStream_t s);
int h_info_u16f32(const espm_state* st, int simplex, double* out, cudaStream_t s);
int h_info_f32f64(const espm_state* st, int simplex, double* out, cudaStream_t s);
int h_info_f64f64(const espm_state* st, int simplex, double* out, cudaStream_t s);
}  // namespace espm
