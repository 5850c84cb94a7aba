// smm_launch.cuh -- definitions of the kernel launchers declared in smm_internal.h.  Included by
// the eight smm_inst_*.cu translation units only, each of which instantiates one (x, y) type pair
// (x: float, double, or packed 16-bit decoding to float / double; see XElem).
#pragma once
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <mutex>

#include "smm_internal.h"
#include "smm_kernels.cuh"

namespace smm {

// The dynamic shared memory a kernel may use is process-wide state of the kernel on the current
// device, shared by every thread that launches it, and launches of one kernel need different sizes
// (the stage count and rows per stage follow B).  So the attribute is only ever raised, to the
// largest size asked for so far, under a lock: a caller that set a smaller size after another had
// raised it would make the other's launch fail.  optin[dev] is that high-water mark, read without
// the lock by launches that need no more; devices beyond kMaxDevices go through the lock each time.
template <typename Kernel>
int raise_smem_optin(Kernel kfn, std::atomic<size_t> (&optin)[kMaxDevices], int dev, size_t smem)
{
    const bool tracked = dev >= 0 && dev < kMaxDevices;
    if (tracked && optin[dev].load(std::memory_order_acquire) >= smem) return 0;
    static std::mutex mu;
    std::lock_guard<std::mutex> lock(mu);
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, kfn));
    const size_t have = static_cast<size_t>(fa.maxDynamicSharedSizeBytes);
    if (have < smem)
        CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    if (tracked) optin[dev].store(std::max(have, smem), std::memory_order_release);
    return 0;
}

template <typename TX, typename TY>
int launch_staged_t(int dev, int lpr, int kpl, int nct, bool packed, bool ord, dim3 grid, size_t smem,
                    cudaStream_t st, const JobBatch &jb, const ApplyArgs &a)
{
#define SMM_CASE_PO(L_, K_, N_, P_, O_)                                                           \
    if (lpr == L_ && kpl == K_ && nct == N_ && packed == P_ && ord == O_) {                       \
        auto kfn = staged_kernel<TX, TY, L_, K_, N_, P_, O_>;                                     \
        static std::atomic<size_t> optin[kMaxDevices];                                            \
        if (const int rc = raise_smem_optin(kfn, optin, dev, smem)) return rc;                    \
        kfn<<<grid, N_ + 32 * producer_warps(N_), smem, st>>>(jb, a);                             \
        CUDA_TRY(cudaGetLastError());                                                             \
        smm_count_launches(1);                                                                    \
        return 0;                                                                                 \
    }
    // fast sums: 256 and 512 consumer threads; reference-order sums (ORD): 256 only
#define SMM_CASE(L_, K_) SMM_CASE_PO(L_, K_, 256, false, false) SMM_CASE_PO(L_, K_, 512, false, false) \
                         SMM_CASE_PO(L_, K_, 256, false, true)
    SMM_CASE_PO(1, 16, 256, true, false) SMM_CASE_PO(1, 16, 512, true, false) SMM_CASE_PO(1, 16, 256, true, true)
    SMM_CASE(1, 4) SMM_CASE(2, 4) SMM_CASE(1, 8) SMM_CASE(1, 12) SMM_CASE(1, 16) SMM_CASE(2, 12)
    SMM_CASE(2, 14) SMM_CASE(2, 16) SMM_CASE(4, 12) SMM_CASE(4, 16) SMM_CASE(8, 12) SMM_CASE(8, 14)
    SMM_CASE(8, 16) SMM_CASE(16, 16) SMM_CASE(32, 16)
#undef SMM_CASE
#undef SMM_CASE_PO
    return smm_fail(1, "no staged kernel for this lane configuration");
}

template <typename TX, typename TY>
int launch_ordered_t(int dev, int rows_per_tile, int threads_per_row, dim3 grid, size_t smem, cudaStream_t st,
                     const JobBatch &jb, const ApplyArgs &a)
{
#define SMM_ORD_CASE_T(R_, T_)                                                                    \
    if (rows_per_tile == R_ && threads_per_row == T_) {                                           \
        auto kfn = ordered_kernel<TX, TY, R_, T_>;                                                \
        static std::atomic<size_t> optin[kMaxDevices];                                            \
        if (const int rc = raise_smem_optin(kfn, optin, dev, smem)) return rc;                    \
        kfn<<<grid, R_ * T_ + 32 * kOrderedProducerWarps, smem, st>>>(jb, a);                     \
        CUDA_TRY(cudaGetLastError());                                                             \
        smm_count_launches(1);                                                                    \
        return 0;                                                                                 \
    }
#define SMM_ORD_CASE(R_) SMM_ORD_CASE_T(R_, 1) SMM_ORD_CASE_T(R_, 2)
    SMM_ORD_CASE(32) SMM_ORD_CASE(64) SMM_ORD_CASE(128) SMM_ORD_CASE(256)
#undef SMM_ORD_CASE
#undef SMM_ORD_CASE_T
    return smm_fail(1, "no ordered kernel for this tile height");
}

template <typename TX, typename TY>
int launch_gather_t(int lpr, bool ord, dim3 grid, cudaStream_t st, const JobBatch &jb, const ApplyArgs &a)
{
    if (ord) gather_kernel<TX, TY, 1, true><<<grid, kGatherThreads, 0, st>>>(jb, a);
    else if (lpr == 1) gather_kernel<TX, TY, 1><<<grid, kGatherThreads, 0, st>>>(jb, a);
    else if (lpr == 4) gather_kernel<TX, TY, 4><<<grid, kGatherThreads, 0, st>>>(jb, a);
    else gather_kernel<TX, TY, 32><<<grid, kGatherThreads, 0, st>>>(jb, a);
    CUDA_TRY(cudaGetLastError());
    smm_count_launches(1);
    return 0;
}

// Two-pass apply of one gather-family level (see compact_kernel): per chunk of <= 64 batch rows,
// transpose the touched source columns into XT, then apply the links from XT.
template <typename TX, typename TY>
int launch_compact_t(int dev, const LevelDev &L, const JobSpec &sp, void *xt_raw, int64_t B, int64_t xbs,
                     int64_t ybs, double area_min, const Decode &dec, cudaStream_t st)
{
    using XS = xs_t<TX>;          // pass 1 copies what x holds: packed sources stay raw in XT
    XS *xt = static_cast<XS *>(xt_raw);
    const size_t smem = static_cast<size_t>(kCompactBC) * compact_stride(sizeof(XS)) * sizeof(XS);
    static std::atomic<size_t> optin[kMaxDevices];
    if (const int rc = raise_smem_optin(compact_kernel<XS>, optin, dev, smem)) return rc;
    const unsigned grid2 = static_cast<unsigned>((L.n_dst + kCompactRows - 1) / kCompactRows);
    // bulk (TMA) copies of the slab rows need 16-byte aligned row pieces; SMM_COMPACT_BULK=0 forces element copies
    static const bool bulk_env = [] { const char *e = getenv("SMM_COMPACT_BULK"); return !(e && e[0] == '0'); }();
    const int bulk = bulk_env && reinterpret_cast<uintptr_t>(sp.x) % 16 == 0 && (xbs * sizeof(XS)) % 16 == 0 &&
                     (kCompactW * sizeof(XS)) % 16 == 0;
    // 8-byte elements: half the batch rows per pass keeps the pass-1 tile at the size that lets three
    // blocks share an SM (one block's transposition overlaps the others' copies)
    static const int rows64 = [] { const char *e = getenv("SMM_COMPACT_F64_ROWS"); return e ? atoi(e) : 32; }();
    const int step = (sizeof(XS) == 8 && bulk && rows64 > 0 && rows64 < kCompactBC) ? rows64 : kCompactBC;
    for (int64_t b0 = 0; b0 < B; b0 += step) {
        const int bc = static_cast<int>(B - b0 < step ? B - b0 : step);
        compact_kernel<XS><<<static_cast<unsigned>(L.compact_blocks), kCompactThreads,
                             static_cast<size_t>(bc) * compact_stride(sizeof(XS)) * sizeof(XS), st>>>(
            static_cast<const XS *>(sp.x) + b0 * xbs, xbs, L.n_src, bc, L.tcols, L.blk_ptr, xt, bulk);
        compact_apply_kernel<TX, TY><<<grid2, kCompactThreads, 0, st>>>(
            xt, bc, L.rowptr, L.rcol, L.val, L.imask, L.frac, sp.masked, area_min, L.n_dst,
            static_cast<TY *>(sp.y) + b0 * ybs, ybs, L.nnz >= 2 * L.n_dst ? 1 : 0, dec);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return smm_fail(3, std::string("compact apply: ") + cudaGetErrorString(e));
        smm_count_launches(2);
    }
    return 0;
}

}  // namespace smm
