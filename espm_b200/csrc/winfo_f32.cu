// Phase information kernels with fp32 arithmetic: f32, uint8 and uint16 storage of X.
#include "winfo.cuh"
#include "winfo_decl.h"
namespace espm {
int w_info_f32f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s) {
    return w_info_entry<float, float>(st, out, scratch, bytes_out, s);
}
int w_info_u8f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s) {
    return w_info_entry<uint8_t, float>(st, out, scratch, bytes_out, s);
}
int w_info_u16f32(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s) {
    return w_info_entry<uint16_t, float>(st, out, scratch, bytes_out, s);
}
}  // namespace espm
