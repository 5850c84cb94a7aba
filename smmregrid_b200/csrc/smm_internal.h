// smm_internal.h -- declarations shared by the translation units of the library (not part of
// the ABI).  The kernel launchers are templates over the (x, y) element types; each of the eight
// type pairs (x: float, double, I16F32, I16F64; y: float, double) is instantiated in its own
// translation unit (smm_inst_*.cu) so the library builds in parallel.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "smm_common.h"

namespace smm {

// thread-local error message of the ABI + the library-wide launch counter (smm_api.cu)
int smm_fail(int code, const std::string &msg);
void smm_count_launches(int n);

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess)                                                                \
            return ::smm::smm_fail(e__ == cudaErrorMemoryAllocation ? 4 /*SMM_ERR_ALLOC*/ : 3, \
                                   std::string(#expr) + ": " + cudaGetErrorString(e__));       \
    } while (0)

constexpr int kMaxDevices = 64;

// One level of an operator on the device.
struct LevelDev {
    int64_t n_src = 0, n_dst = 0, nnz = 0, touched = 0;
    int32_t max_row_nnz = 0;
    int32_t *rowptr = nullptr, *col = nullptr;
    double *val = nullptr;
    bool staged = false;
    std::string why_not_staged;
    int32_t lpr = 0, kpl = 0, rpt = 0, nct = 0, ntiles = 0, max_segs = 0;
    int64_t max_elems = 0, sum_elems = 0;
    TileDesc *tiles = nullptr;
    Seg *segs = nullptr;
    double *wplan = nullptr;
    uint16_t *iplan = nullptr;
    int32_t *rowmap = nullptr;          // tile slot -> row (re-ordered plans) | packed plans: the rowslot table
    bool packed = false, reordered = false;
    bool ordlong = false;               // reference-order plan for long rows: a thread per row, links in shared memory (ordered_kernel)
    int32_t *tcols = nullptr, *blk_ptr = nullptr, *rcol = nullptr;   // compact (two-pass) plan of gather levels
    int32_t compact_blocks = 0;
    int32_t *gather_rows = nullptr;     // split plans: the long rows the gather kernel serves next to the staged launch
    int32_t n_gather_rows = 0;
    int64_t gather_nnz = 0;
    int32_t *imask = nullptr;
    double *frac = nullptr;
    bool has_imask = false, has_frac = false;
    int64_t device_bytes = 0;
};

// packed element types (smm_kernels.cuh): raw 16-bit sources decoding to float / double
struct I16F32;
struct I16F64;

struct JobSpec {
    int32_t level;
    const void *x;
    void *y;
    int32_t masked;
};

// staged_kernel<TX, TY, lpr, kpl, nct, packed, ord> on `grid` work items
template <typename TX, typename TY>
int launch_staged_t(int dev, int lpr, int kpl, int nct, bool packed, bool ord, dim3 grid, size_t smem,
                    cudaStream_t st, const JobBatch &jb, const ApplyArgs &a);

// ordered_kernel<TX, TY, rows_per_tile> (reference-order sums, a thread per row, links in shared memory)
template <typename TX, typename TY>
int launch_ordered_t(int dev, int rows_per_tile, int threads_per_row, dim3 grid, size_t smem, cudaStream_t st,
                     const JobBatch &jb, const ApplyArgs &a);

// gather_kernel<TX, TY, lpr, ord>
template <typename TX, typename TY>
int launch_gather_t(int lpr, bool ord, dim3 grid, cudaStream_t st, const JobBatch &jb, const ApplyArgs &a);

// the two passes of the compact path over B batch rows; `xt` holds touched x kCompactBC elements of
// what x holds (xs_t<TX>: raw 16 bits for packed sources, decoded in pass 2 with `dec`)
template <typename TX, typename TY>
int launch_compact_t(int dev, const LevelDev &L, const JobSpec &sp, void *xt, int64_t B, int64_t xbs,
                     int64_t ybs, double area_min, const Decode &dec, cudaStream_t st);

#define SMM_DECLARE_LAUNCHERS(EXTERN, TX, TY)                                                              \
    EXTERN template int launch_staged_t<TX, TY>(int, int, int, int, bool, bool, dim3, size_t, cudaStream_t, \
                                                const JobBatch &, const ApplyArgs &);                      \
    EXTERN template int launch_gather_t<TX, TY>(int, bool, dim3, cudaStream_t, const JobBatch &,           \
                                                const ApplyArgs &);                                        \
    EXTERN template int launch_ordered_t<TX, TY>(int, int, int, dim3, size_t, cudaStream_t,                \
                                                 const JobBatch &, const ApplyArgs &);                     \
    EXTERN template int launch_compact_t<TX, TY>(int, const LevelDev &, const JobSpec &, void *, int64_t,  \
                                                 int64_t, int64_t, double, const Decode &, cudaStream_t);

}  // namespace smm
