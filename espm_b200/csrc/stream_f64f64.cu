// Every X-streaming kernel for f64 storage of X and fp64 arithmetic (see xpass_inst.cuh).
#include "fitstats.cuh"
#include "resid.cuh"
#include "winfo.cuh"
#include "xpass_inst.cuh"
namespace espm {
const StreamPair stream_f64f64 = {ESPM_F64, ESPM_F64,
    xpass_entry<double, double>, xpass_sizes<double, double>,
    fit_stats_entry<double, double>, h_info_entry<double, double>, w_info_entry<double, double>,
    resid_left_entry<double, double>, resid_right_entry<double, double>};
}  // namespace espm
