// smm_aux_kernels.cuh -- the kernels outside the weight application (included by smm_api.cu only):
//   mask_sum_kernel       mask_tensordot (weights.py:47-52): sequential ascending-src sum per row.
//   nan_variation_kernel  detect_nan_variation_dims (util.py:57-85) for one axis.
//   widen16_kernel        exact float16 / bfloat16 -> float32 copy of a slab (the float32 path of
//                         half sources whose 2-byte rows cannot be staged).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace smm {

// ------------------------------------------------------------------ mask_tensordot

// weights.py:47-52.  One thread per destination row, links in ascending-src order, separate
// multiply and add: bit-identical to the reference's accumulation, so `t < 0.5` is too.
__global__ void mask_sum_kernel(const int32_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                                const double *__restrict__ val, const int32_t *__restrict__ src_imask,
                                int32_t *__restrict__ dst_imask, int32_t *__restrict__ any_masked,
                                int64_t n_dst)
{
    const int64_t row = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (row >= n_dst) return;
    double t = 0.0;
    const int j1 = rowptr[row + 1];
    for (int j = rowptr[row]; j < j1; ++j)
        t = __dadd_rn(t, __dmul_rn(static_cast<double>(src_imask[col[j]]), val[j]));
    const int32_t m = t < 0.5 ? 0 : 1;
    dst_imask[row] = m;
    if (m == 0) atomicOr(any_masked, 1);
}

// detect_nan_variation_dims (smmregrid/util.py:57-85) for one axis: x viewed as
// [outer, n_axis, inner]; counts the (outer, inner) positions whose NaN-ness changes somewhere
// along the axis (`isnull().astype(int8).diff(dim).astype(bool).any(dim).sum()`).  isnull is
// NaN only: +-inf is not missing.  One thread per position, coalesced over `inner`.
template <typename TX>
__global__ void nan_variation_kernel(const TX *__restrict__ x, int64_t outer, int64_t n_axis, int64_t inner,
                                     unsigned long long *__restrict__ count)
{
    const int64_t pos = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    bool varies = false;
    if (pos < outer * inner) {
        const int64_t o = pos / inner, i = pos - o * inner;
        const TX *p = x + o * n_axis * inner + i;
        const bool first = p[0] != p[0];
        for (int64_t k = 1; k < n_axis && !varies; ++k) {
            const TX v = p[k * inner];
            varies = (v != v) != first;
        }
    }
    const unsigned n = __popc(__ballot_sync(0xffffffffu, varies));
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(count, static_cast<unsigned long long>(n));
}

// y[b][i] = x[b][i] widened exactly to float32, i < n, b < blockIdx.y's rows (one grid row per batch row).
template <bool BF16>
__global__ void widen16_kernel(const uint16_t *__restrict__ x, int64_t ldx, int64_t n, float *__restrict__ y, int64_t ldy)
{
    const uint16_t *xr = x + static_cast<int64_t>(blockIdx.y) * ldx;
    float *yr = y + static_cast<int64_t>(blockIdx.y) * ldy;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const uint16_t r = xr[i];
        float v;
        if constexpr (BF16) v = __uint_as_float(static_cast<uint32_t>(r) << 16);
        else asm("cvt.f32.f16 %0, %1;" : "=f"(v) : "h"(r));
        yr[i] = v;
    }
}

}  // namespace smm
