// Abundance information kernels with fp32 arithmetic: f32, uint8 and uint16 storage of X.
#include "hinfo.cuh"
#include "hinfo_decl.h"
namespace espm {
int h_info_f32f32(const espm_state* st, int simplex, double* out, cudaStream_t s) {
    return h_info_entry<float, float>(st, simplex, out, s);
}
int h_info_u8f32(const espm_state* st, int simplex, double* out, cudaStream_t s) {
    return h_info_entry<uint8_t, float>(st, simplex, out, s);
}
int h_info_u16f32(const espm_state* st, int simplex, double* out, cudaStream_t s) {
    return h_info_entry<uint16_t, float>(st, simplex, out, s);
}
}  // namespace espm
