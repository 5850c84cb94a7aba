// smm_inst_i16f32_f64.cu -- kernel launchers for x = int16 / uint16 CF-packed, decoded to float32, y = double
// (one translation unit per type pair so that the library builds in parallel; see smm_internal.h).
#include "smm_launch.cuh"

namespace smm {
SMM_DECLARE_LAUNCHERS(, I16F32, double)
}  // namespace smm
