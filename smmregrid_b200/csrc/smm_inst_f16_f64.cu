// smm_inst_f16_f64.cu -- kernel launchers for x = IEEE binary16 (float32 semantics), y = double
// (one translation unit per type pair so that the library builds in parallel; see smm_internal.h).
#include "smm_launch.cuh"

namespace smm {
SMM_DECLARE_LAUNCHERS(, F16, double)
}  // namespace smm
