// Abundance information kernels with fp64 arithmetic: f32 and f64 storage of X.
#include "hinfo.cuh"
#include "hinfo_decl.h"
namespace espm {
int h_info_f32f64(const espm_state* st, int simplex, double* out, cudaStream_t s) {
    return h_info_entry<float, double>(st, simplex, out, s);
}
int h_info_f64f64(const espm_state* st, int simplex, double* out, cudaStream_t s) {
    return h_info_entry<double, double>(st, simplex, out, s);
}
}  // namespace espm
