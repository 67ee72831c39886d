// Goodness-of-fit kernels with fp32 arithmetic: f32, uint8 and uint16 storage of X.
#include "fitstats.cuh"
#include "fitstats_decl.h"
namespace espm {
int fit_stats_f32f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s) {
    return fit_stats_entry<float, float>(st, pixel_out, channel_out, scratch, bytes_out, s);
}
int fit_stats_u8f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                    cudaStream_t s) {
    return fit_stats_entry<uint8_t, float>(st, pixel_out, channel_out, scratch, bytes_out, s);
}
int fit_stats_u16f32(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s) {
    return fit_stats_entry<uint16_t, float>(st, pixel_out, channel_out, scratch, bytes_out, s);
}
}  // namespace espm
