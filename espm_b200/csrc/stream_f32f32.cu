// Every X-streaming kernel for f32 storage of X and fp32 arithmetic (see xpass_inst.cuh).
#include "fitstats.cuh"
#include "resid.cuh"
#include "winfo.cuh"
#include "xpass_inst.cuh"
namespace espm {
const StreamPair stream_f32f32 = {ESPM_F32, ESPM_F32,
    xpass_entry<float, float>, xpass_sizes<float, float>,
    fit_stats_entry<float, float>, h_info_entry<float, float>, w_info_entry<float, float>,
    resid_left_entry<float, float>, resid_right_entry<float, float>};
}  // namespace espm
