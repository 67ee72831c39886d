// Every X-streaming kernel for uint16 storage of X and fp32 arithmetic (see xpass_inst.cuh).
#include "fitstats.cuh"
#include "resid.cuh"
#include "winfo.cuh"
#include "xpass_inst.cuh"
namespace espm {
const StreamPair stream_u16f32 = {ESPM_U16, ESPM_F32,
    xpass_entry<uint16_t, float>, xpass_sizes<uint16_t, float>,
    fit_stats_entry<uint16_t, float>, h_info_entry<uint16_t, float>, w_info_entry<uint16_t, float>,
    resid_left_entry<uint16_t, float>, resid_right_entry<uint16_t, float>};
}  // namespace espm
