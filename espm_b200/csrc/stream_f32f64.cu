// Every X-streaming kernel for f32 storage of X and fp64 arithmetic (see xpass_inst.cuh).
#include "fitstats.cuh"
#include "resid.cuh"
#include "winfo.cuh"
#include "xpass_inst.cuh"
namespace espm {
const StreamPair stream_f32f64 = {ESPM_F32, ESPM_F64,
    xpass_entry<float, double>, xpass_sizes<float, double>,
    fit_stats_entry<float, double>, h_info_entry<float, double>, w_info_entry<float, double>,
    resid_left_entry<float, double>, resid_right_entry<float, double>};
}  // namespace espm
