// smm_inst_bf16_f64.cu -- kernel launchers for x = bfloat16 (float32 semantics), y = double
// (one translation unit per type pair so that the library builds in parallel; see smm_internal.h).
#include "smm_launch.cuh"

namespace smm {
SMM_DECLARE_LAUNCHERS(, BF16, double)
}  // namespace smm
