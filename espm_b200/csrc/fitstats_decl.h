// Host-side declarations of the goodness-of-fit launchers (fitstats_f32.cu / fitstats_f64.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/espm_b200.h"

namespace espm {
// bytes_out != NULL: only report the scratch bytes the launch needs
int fit_stats_f32f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s);
int fit_stats_u8f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                    cudaStream_t s);
int fit_stats_u16f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s);
int fit_stats_f32f64(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s);
int fit_stats_f64f64(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s);
}  // namespace espm
