// smm_inst_i16f64_f32.cu -- kernel launchers for x = int16 / uint16 CF-packed, decoded to float64, y = float
// (one translation unit per type pair so that the library builds in parallel; see smm_internal.h).
#include "smm_launch.cuh"

namespace smm {
SMM_DECLARE_LAUNCHERS(, I16F64, float)
}  // namespace smm
