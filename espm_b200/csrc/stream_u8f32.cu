// Every X-streaming kernel for uint8 storage of X and fp32 arithmetic (see xpass_inst.cuh).
#include "fitstats.cuh"
#include "resid.cuh"
#include "winfo.cuh"
#include "xpass_inst.cuh"
namespace espm {
const StreamPair stream_u8f32 = {ESPM_U8, ESPM_F32,
    xpass_entry<uint8_t, float>, xpass_sizes<uint8_t, float>,
    fit_stats_entry<uint8_t, float>, h_info_entry<uint8_t, float>, w_info_entry<uint8_t, float>,
    resid_left_entry<uint8_t, float>, resid_right_entry<uint8_t, float>};
}  // namespace espm
