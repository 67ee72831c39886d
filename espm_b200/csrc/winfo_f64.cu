// Phase information kernels with fp64 arithmetic: f32 and f64 storage of X.
#include "winfo.cuh"
#include "winfo_decl.h"
namespace espm {
int w_info_f32f64(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s) {
    return w_info_entry<float, double>(st, out, scratch, bytes_out, s);
}
int w_info_f64f64(const espm_state* st, double* out, void* scratch, int64_t* bytes_out, cudaStream_t s) {
    return w_info_entry<double, double>(st, out, scratch, bytes_out, s);
}
}  // namespace espm
