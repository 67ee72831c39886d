// Goodness-of-fit kernels with fp64 arithmetic: f32 and f64 storage of X.
#include "fitstats.cuh"
#include "fitstats_decl.h"
namespace espm {
int fit_stats_f32f64(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s) {
    return fit_stats_entry<float, double>(st, pixel_out, channel_out, scratch, bytes_out, s);
}
int fit_stats_f64f64(const espm_state* st, double* pixel_out, double* channel_out, void* scratch, int64_t* bytes_out,
                     cudaStream_t s) {
    return fit_stats_entry<double, double>(st, pixel_out, channel_out, scratch, bytes_out, s);
}
}  // namespace espm
