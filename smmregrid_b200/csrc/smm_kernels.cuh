// smm_kernels.cuh -- sm_100a kernels of the weight-application path.
//
//   staged_kernel   Y = X.W for operators whose tiles have a compact source footprint
//                   (structured / locally ordered sources).  Four producer warps stream the
//                   tile's footprint of up to 8 batch rows per stage into shared memory with
//                   1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx, L2
//                   evict-first); the consumer warps hold the tile's link weights and
//                   footprint offsets in REGISTERS for the whole batch loop, so per batch row
//                   the only HBM traffic is the X stream in and the tile's rows out.  LPR
//                   lanes share one destination row; operators without a row above 16 links
//                   use the PACKED layout instead (a thread owns up to four rows).
//   gather_kernel   generic CSR fallback: direct ld.global.nc gathers, kGatherBT batch rows
//                   register-blocked per thread (scattered sources, oversized rows,
//                   unaligned slabs).
//   compact_kernel + compact_apply_kernel
//                   two-pass alternative to the gathers for scattered sources with enough batch
//                   rows: touched columns transposed into a compact buffer, then links applied
//                   with lanes over the batch, in the reference's summation order.
//   (mask_sum_kernel and nan_variation_kernel, the two init-time kernels, are in smm_aux_kernels.cuh)
//
// Numerics (smmregrid/regrid.py:544-570): non-finite x -> 1e20 in x's dtype, float64
// products/accumulation, NaN where dst_grid_imask == 0 / dst_grid_frac < remap_area_min /
// Y > 1e19.  The fast path multiplies raw values and sums a row's links lane-split +
// tree-reduced; a non-finite sum (some source was NaN/inf) makes the warp redo its links with
// the fill, and whenever a sum is within 1e-9 relative of the 1e19 threshold the row is
// REPLAYED in the reference's order (ascending src, separate multiply and add) so the NaN
// decision is bit-identical.
//
// Summation order.  The fast sums differ from the reference's by rounding only as long as the
// products of a row do not cancel.  Operators with weights of both signs (bicubic, second-order
// conservative) are therefore planned and evaluated in the REFERENCE'S OWN ORDER (template
// parameter ORD: links in ascending source order, separate multiply and add, one dependent
// chain per row -- a lane holds a contiguous run of the row's links and hands its partial sum
// to the next lane), which makes every value bit-identical to the reference loop.  Callers can
// request that order for any operator (SMM_SUM_REFERENCE), e.g. for fields that change sign.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <cuda/std/type_traits>

#include "smm_common.h"

namespace smm {

// ------------------------------------------------------------------ PTX helpers

__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 1-D TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes,
                                             uint32_t bar, uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1], %2, [%3], %4;" ::"r"(dst),
        "l"(src), "r"(bytes), "r"(bar), "l"(policy)
        : "memory");
}

// ------------------------------------------------------------------ numerics helpers

// regrid.py:545-547: np.ma.fix_invalid + filled -> 1e20 in the input dtype.
__device__ __forceinline__ float fill_invalid(float v) { return (fabsf(v) <= 3.402823466e+38f) ? v : 1e20f; }
__device__ __forceinline__ double fill_invalid(double v) { return (fabs(v) <= 1.7976931348623157e+308) ? v : 1e20; }

// ------------------------------------------------------------------ source element types
//
// TX is float, double, or a PACKED type: raw 16-bit CF-packed values (smm_decode) that every read
// of x decodes to float (I16F32) or double (I16F64).  xs_t<TX> is what x holds in memory (staged,
// gathered, transposed into XT), xv_t<TX> what the arithmetic sees.  For float / double every
// helper below is exactly the plain load.
struct I16F32 {};
struct I16F64 {};
template <typename TX> struct XElem { using S = TX; using V = TX; static constexpr bool kPacked = false; };
template <> struct XElem<I16F32> { using S = uint16_t; using V = float; static constexpr bool kPacked = true; };
template <> struct XElem<I16F64> { using S = uint16_t; using V = double; static constexpr bool kPacked = true; };
template <typename TX> using xs_t = typename XElem<TX>::S;
template <typename TX> using xv_t = typename XElem<TX>::V;

// CF decode of one raw value (see Decode): fill values -> NaN, else (v * scale) + offset in V, each
// operation rounded once (no FMA contraction), as numpy does it in the decoded dtype.
template <typename V>
__device__ __forceinline__ V decode16(uint32_t r, const Decode &d)
{
    // v exactly, without the (quarter-rate) integer conversion: 2^23 + (r ^ sign_xor) as float bits,
    // minus 2^23 (+ 2^15 for int16: the xor moved the sign bit into a bias)
    const float v = __fsub_rn(__int_as_float(static_cast<int>(0x4B000000u | (r ^ d.sign_xor))), d.bias_f);
    V x;
    if constexpr (sizeof(V) == 4) x = __fadd_rn(__fmul_rn(v, d.scale_f), d.offset_f);
    else x = __dadd_rn(__dmul_rn(static_cast<double>(v), d.scale), d.offset);
    // one predicate for the four compares (bitwise: no short-circuit, so one select below)
    const int ri = static_cast<int>(r);
    const bool fill = (ri == d.fill[0]) | (ri == d.fill[1]) | (ri == d.fill[2]) | (ri == d.fill[3]);
    if constexpr (sizeof(V) == 4) return fill ? CUDART_NAN_F : x;
    else return fill ? CUDART_NAN : x;
}

// plain (generic) read of one source element; packed types pass their Decode
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_g(const xs_t<TX> *p) { return *p; }
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_g(const xs_t<TX> *p, const Decode &d)
{
    if constexpr (XElem<TX>::kPacked) return decode16<xv_t<TX>>(*p, d);
    else return *p;
}

// Gather load of one source element, with the smallest L2 prefetch-size hint (SASS LDG.E.LTC64B):
// a random 4-byte gather was measured to pull 128 bytes from DRAM without it.  B200, B = 64:
// C5dis 5.59 -> 4.98 ms, C5nn 1.43 -> 1.29 ms; the 256-byte hint costs 7 %.  SMM_GATHER_L2 = 0
// (no hint) | 64 | 128 | 256 at compile time.
#ifndef SMM_GATHER_L2
#define SMM_GATHER_L2 64
#endif
template <typename TX> __device__ __forceinline__ TX ld_nc(const TX *p);
template <> __device__ __forceinline__ float ld_nc<float>(const float *p)
{
#if SMM_GATHER_L2 == 64
    float v; asm volatile("ld.global.nc.L2::64B.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 128
    float v; asm volatile("ld.global.nc.L2::128B.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 256
    float v; asm volatile("ld.global.nc.L2::256B.f32 %0, [%1];" : "=f"(v) : "l"(p)); return v;
#else
    return __ldg(p);
#endif
}
template <> __device__ __forceinline__ double ld_nc<double>(const double *p)
{
#if SMM_GATHER_L2 == 64
    double v; asm volatile("ld.global.nc.L2::64B.f64 %0, [%1];" : "=d"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 128
    double v; asm volatile("ld.global.nc.L2::128B.f64 %0, [%1];" : "=d"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 256
    double v; asm volatile("ld.global.nc.L2::256B.f64 %0, [%1];" : "=d"(v) : "l"(p)); return v;
#else
    return __ldg(p);
#endif
}
template <> __device__ __forceinline__ uint16_t ld_nc<uint16_t>(const uint16_t *p)
{
#if SMM_GATHER_L2 == 64
    uint16_t v; asm volatile("ld.global.nc.L2::64B.u16 %0, [%1];" : "=h"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 128
    uint16_t v; asm volatile("ld.global.nc.L2::128B.u16 %0, [%1];" : "=h"(v) : "l"(p)); return v;
#elif SMM_GATHER_L2 == 256
    uint16_t v; asm volatile("ld.global.nc.L2::256B.u16 %0, [%1];" : "=h"(v) : "l"(p)); return v;
#else
    return __ldg(p);
#endif
}

// gather read of one source element, decoded for packed types
template <typename TX>
__device__ __forceinline__ xv_t<TX> ld_nc_x(const xs_t<TX> *p, const Decode &d)
{
    if constexpr (XElem<TX>::kPacked) return decode16<xv_t<TX>>(ld_nc(p), d);
    else return ld_nc(p);
}

// Reference-order evaluation of one destination row: links in ascending-src order, separate
// multiply and add in float64 (pydata/sparse ndarray.COO loop; no FMA contraction).  Packed
// sources pass their Decode (`d`: empty for float / double).
template <typename TX, typename... D>
__device__ __noinline__ double replay_row(const int32_t *__restrict__ rowptr,
                                          const int32_t *__restrict__ col,
                                          const double *__restrict__ val, int row,
                                          const xs_t<TX> *__restrict__ xrow, const D &...d)
{
    double acc = 0.0;
    const int j1 = rowptr[row + 1];
    for (int j = rowptr[row]; j < j1; ++j) {
        const xv_t<TX> v = fill_invalid(ldx_g<TX>(xrow + col[j], d...));
        acc = __dadd_rn(acc, __dmul_rn(static_cast<double>(v), val[j]));
    }
    return acc;
}
template <typename TX>
__device__ __forceinline__ double replay(const int32_t *rowptr, const int32_t *col, const double *val, int row,
                                         const xs_t<TX> *xrow, const Decode &d)
{
    if constexpr (XElem<TX>::kPacked) return replay_row<TX>(rowptr, col, val, row, xrow, d);
    else return replay_row<TX>(rowptr, col, val, row, xrow);
}

__device__ __forceinline__ bool near_threshold(double acc) { return fabs(acc - 1e19) <= 1e10; }

// Epilogue of one destination value (regrid.py:553-570): imask / frac (folded into `dead`), then
// `> 1e19 -> NaN`.  One comparison keeps ordinary values on the short path; only sums in the
// neighbourhood of the threshold are replayed in the reference's summation order (`replay()`).
template <typename TY, bool ORD = false, typename Replay>
__device__ __forceinline__ TY finish(double acc, bool dead, Replay replay)
{
    if (acc > 9.9e18) {
        if (!ORD && near_threshold(acc)) acc = replay();      // ORD: acc already is the reference-order sum
        if (acc > 1e19) acc = CUDART_NAN;
    }
    return static_cast<TY>(dead ? CUDART_NAN : acc);
}

// Store of one result: streaming (st.global.cs) -- y is written once and not read back here.
// Measured against plain / .wt / .cg stores: C2 +1.3 %, C3 +0.7 %, C4 +0.1 %.
// SMM_STORE_MODE: 0 plain, 1 .cs, 2 .wt, 3 .cg.
#ifndef SMM_STORE_MODE
#define SMM_STORE_MODE 1
#endif
template <typename TY>
__device__ __forceinline__ void store_y(TY *p, TY v)
{
#if SMM_STORE_MODE == 1
    __stcs(p, v);
#elif SMM_STORE_MODE == 2
    __stwt(p, v);
#elif SMM_STORE_MODE == 3
    __stcg(p, v);
#else
    *p = v;
#endif
}

__device__ __forceinline__ const LevelJob &find_job(const JobBatch &jb, int item, int &j)
{
    int lo = 0, hi = jb.njobs - 1;                 // last job with item0 <= item
#pragma unroll 1
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (item >= jb.jobs[mid].item0) lo = mid; else hi = mid - 1;
    }
    j = lo;
    return jb.jobs[j];
}

// ------------------------------------------------------------------ staged kernel

template <typename TX> __device__ __forceinline__ TX lds(uint32_t addr);
template <> __device__ __forceinline__ float lds<float>(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
template <> __device__ __forceinline__ double lds<double>(uint32_t addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
template <> __device__ __forceinline__ uint16_t lds<uint16_t>(uint32_t addr)
{
    uint16_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
// an already loaded source element, decoded for packed types
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_v(xs_t<TX> v) { return v; }
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_v(xs_t<TX> v, const Decode &d)
{
    if constexpr (XElem<TX>::kPacked) return decode16<xv_t<TX>>(v, d);
    else return v;
}

// shared-memory read of one staged source element, decoded for packed types
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_s(uint32_t addr) { return lds<TX>(addr); }
template <typename TX>
__device__ __forceinline__ xv_t<TX> ldx_s(uint32_t addr, const Decode &d)
{
    if constexpr (XElem<TX>::kPacked) return decode16<xv_t<TX>>(lds<uint16_t>(addr), d);
    else return lds<TX>(addr);
}

// Sum of one lane's register-resident links against the staged footprint at shared address
// `sb`.  kFill = false is the fast path: raw values, no non-finite test (any NaN/inf input
// makes the sum non-finite, which the caller detects and redoes with kFill = true).
template <int LPR>
__device__ __forceinline__ double group_sum(double acc)
{
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

// keeps a value in a register: stops the compiler from re-deriving the shared window base
// (S2UR SR_CgaCtaId + shifts) in front of every mbarrier operation of the batch loop
__device__ __forceinline__ uint32_t pin_reg(uint32_t v)
{
    asm volatile("mov.b32 %0, %0;" : "+r"(v));
    return v;
}

// Sum of one lane's register-resident links against the staged footprint at shared address
// `sb`.  kFill = false is the fast path: raw values, no non-finite test (any NaN/inf input
// makes the sum non-finite, which the caller detects and redoes with kFill = true).
template <typename TX, int KPL, bool kFill>
__device__ __forceinline__ double lane_sum(uint32_t sb, const uint32_t (&off)[KPL], const double (&w)[KPL], const Decode &d)
{
    static_assert(KPL % 2 == 0, "links per lane come in pairs");
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int k = 0; k < KPL; k += 2) {
        xv_t<TX> v0 = ldx_s<TX>(sb + off[k + 0], d);
        xv_t<TX> v1 = ldx_s<TX>(sb + off[k + 1], d);
        if (kFill) { v0 = fill_invalid(v0); v1 = fill_invalid(v1); }
        acc[k % 4 + 0] = fma(static_cast<double>(v0), w[k + 0], acc[k % 4 + 0]);
        acc[k % 4 + 1] = fma(static_cast<double>(v1), w[k + 1], acc[k % 4 + 1]);
    }
    return (acc[0] + acc[1]) + (acc[2] + acc[3]);
}

// Packed rows: a thread's 16 links are four sub-rows of four; one partial sum per sub-row.
template <typename TX, bool kFill>
__device__ __forceinline__ void lane_sum4(uint32_t sb, const uint32_t (&off)[16], const double (&w)[16], double (&s4)[4],
                                          const Decode &d)
{
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        xv_t<TX> v0 = ldx_s<TX>(sb + off[4 * u + 0], d);
        xv_t<TX> v1 = ldx_s<TX>(sb + off[4 * u + 1], d);
        xv_t<TX> v2 = ldx_s<TX>(sb + off[4 * u + 2], d);
        xv_t<TX> v3 = ldx_s<TX>(sb + off[4 * u + 3], d);
        if (kFill) { v0 = fill_invalid(v0); v1 = fill_invalid(v1); v2 = fill_invalid(v2); v3 = fill_invalid(v3); }
        const double e = fma(static_cast<double>(v1), w[4 * u + 1], static_cast<double>(v0) * w[4 * u + 0]);
        const double o = fma(static_cast<double>(v3), w[4 * u + 3], static_cast<double>(v2) * w[4 * u + 2]);
        s4[u] = e + o;
    }
}

// ---- reference-order variants (ORD plans: slot k of lane l holds link l*KPL + k of the row's
// ascending-source list; padding slots carry weight 0 behind the last link)

// products of one lane's links, each rounded once (no FMA contraction)
template <typename TX, int KPL, bool kFill>
__device__ __forceinline__ void lane_products(uint32_t sb, const uint32_t (&off)[KPL], const double (&w)[KPL],
                                              double (&p)[KPL], const Decode &d)
{
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
        xv_t<TX> v = ldx_s<TX>(sb + off[k], d);
        if (kFill) v = fill_invalid(v);
        p[k] = __dmul_rn(static_cast<double>(v), w[k]);
    }
}

// One dependent chain per row through the LPR lanes of its group, in link order.  Every lane of
// the group returns the row's sum.
template <int LPR, int KPL>
__device__ __forceinline__ double ordered_group_sum(const double (&p)[KPL], int l_in)
{
    double acc = 0.0;
    if constexpr (LPR == 1) {
#pragma unroll
        for (int k = 0; k < KPL; ++k) acc = __dadd_rn(acc, p[k]);
        return acc;
    } else {
#pragma unroll 1
        for (int l = 0; l < LPR; ++l) {
            if (l_in == l) {
#pragma unroll
                for (int k = 0; k < KPL; ++k) acc = __dadd_rn(acc, p[k]);
            }
            const double up = __shfl_up_sync(0xffffffffu, acc, 1, LPR);
            if (l_in == l + 1) acc = up;
        }
        return __shfl_sync(0xffffffffu, acc, LPR - 1, LPR);
    }
}

template <typename TX, int LPR, int KPL, bool kFill>
__device__ __forceinline__ double lane_sum_ordered(uint32_t sb, const uint32_t (&off)[KPL], const double (&w)[KPL], int l_in,
                                                   const Decode &d)
{
    double p[KPL];
    lane_products<TX, KPL, kFill>(sb, off, w, p, d);
    return ordered_group_sum<LPR, KPL>(p, l_in);
}

// Packed rows in reference order: the chain of a row runs through its consecutive sub-rows
// (`cont` bit u: sub-row u continues the row of sub-row u-1); s4[u] = the chain after sub-row u.
template <typename TX, bool kFill>
__device__ __forceinline__ void lane_chain4(uint32_t sb, const uint32_t (&off)[16], const double (&w)[16], uint32_t cont,
                                            double (&s4)[4], const Decode &d)
{
    double c = 0.0;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        c = (cont & (1u << u)) ? c : 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            xv_t<TX> v = ldx_s<TX>(sb + off[4 * u + j], d);
            if (kFill) v = fill_invalid(v);
            c = __dadd_rn(c, __dmul_rn(static_cast<double>(v), w[4 * u + j]));
        }
        s4[u] = c;
    }
}

// Opt-in renormalising mode (extension, off by default; SURVEY.md §8f): the sums a lane needs to
// EXCLUDE non-finite sources instead of filling them: sum of w*x over finite x, sum of w over
// finite x, sum of all w.
// Kept out of line and fed from the plan arrays (not from the caller's register image) so that
// this cold path costs the hot loop no registers.
template <typename TX, int KPL, int NCT, typename... D>
__device__ __noinline__ void lane_sum_valid(const double *__restrict__ wplan, const uint16_t *__restrict__ iplan,
                                            size_t base, uint32_t sb, double *out3, const D &...d)
{
    double wx = 0.0, wv = 0.0, wa = 0.0;
#pragma unroll 2
    for (int k = 0; k < KPL; ++k) {
        const double wk = __ldg(wplan + base + static_cast<size_t>(k) * NCT);
        const uint32_t o = static_cast<uint32_t>(__ldg(iplan + base + static_cast<size_t>(k) * NCT)) *
                           static_cast<uint32_t>(sizeof(xs_t<TX>));
        const xv_t<TX> v = ldx_s<TX>(sb + o, d...);
        wa += wk;
        if (fill_invalid(v) == v) { wx = fma(static_cast<double>(v), wk, wx); wv += wk; }   // false for NaN, +-inf
    }
    out3[0] = wx; out3[1] = wv; out3[2] = wa;
}

// renormalised value of a row from its group-reduced sums; NaN below the valid-weight threshold
__device__ __forceinline__ double renormalise(double wx, double wv, double wa, double min_valid)
{
    if (wv == wa) return wx;                           // nothing was missing (also rows without links)
    if (!(fabs(wv) >= min_valid * fabs(wa)) || wv == 0.0) return CUDART_NAN;
    return wx * (wa / wv);
}

__device__ __forceinline__ bool not_finite(double v) { return !(fabs(v) <= 1.7976931348623157e+308); }

// CTA roles: NCT/32 consumer warps (two warpgroups for NCT = 256) | one warpgroup of 4 TMA
// producer warps.
//
// Issuing one bulk copy costs a warp ~100 cycles of serial latency (uniform-register operand
// moves + TMA hand-off) and a tile's footprint is 10-20 segments per batch row, so a single
// producer warp caps the CTA well below the HBM rate (measured: 5.6 TB/s with one producer
// warp, 6.5 TB/s with four).  The segments of a stage are therefore split over four producer
// warps whose issue latencies overlap.
//
// Registers: two CTAs of 12 warps per SM = 6 warps per SM sub-partition -> 80 registers per
// thread at launch; the producer warpgroup then shrinks to 40 and the consumer warpgroups
// grow to 96 (setmaxnreg), which the link weights + offsets held in registers need.
// producer warps per CTA: 4 with NCT = 256 (two CTAs per SM), SMM_PRODUCERS_512 with NCT = 512
#ifndef SMM_PRODUCERS_512
#define SMM_PRODUCERS_512 4
#endif
__host__ __device__ constexpr int producer_warps(int nct) { return nct == 512 ? SMM_PRODUCERS_512 : 4; }
constexpr int kProducerRegs = 40;
#ifndef SMM_CONSUMER_REGS_512
#define SMM_CONSUMER_REGS_512 104
#endif
// NCT = 512 launches 640 threads x 96 registers; the 56 x 128 the producers give back let the 512
// consumers grow to 104 (4 consumer warps x 104 + 1 producer warp x 40 per sub-partition <= 512).
__host__ __device__ constexpr int consumer_regs(int nct) { return nct == 512 ? SMM_CONSUMER_REGS_512 : 96; }

// per-tile segment table in bytes: {dst offset in the stage, length, source offset in the row}
struct SegB { uint32_t dst, len; uint64_t src; };

// TMA producer warp `p` of `nwarps`: for every stage of up to NB consecutive batch rows of the work
// item, wait for the stage to be free, then stream the tile's footprint with 1-D bulk copies
// (producer p issues copies p, p + active, ... one per lane); completion is counted in bytes on
// the stage's `full` mbarrier.
template <typename TX>
__device__ __forceinline__ void produce_stages(const LevelJob &job, const ApplyArgs &a, const TileDesc &td,
                                               const SegB *ssegs, uint32_t full_addr, uint32_t empty_addr,
                                               uint32_t stages_addr, int p, int nwarps, int lane, int64_t b0, int64_t b1)
{
    // small footprints need fewer issuing warps (<= 3 copies each); the others retire at once
    const int per_stage = td.nseg * a.rows_per_stage;
    const int active = per_stage >= 3 * nwarps ? nwarps : (per_stage + 2) / 3 > 0 ? (per_stage + 2) / 3 : 1;
    if (p >= active) return;
    const uint64_t policy = l2_evict_first_policy();
    const char *xbase = static_cast<const char *>(job.x);
    const uint32_t tile_bytes = static_cast<uint32_t>(td.elems) * sizeof(xs_t<TX>);
    const int NB = a.rows_per_stage;
    const int S = a.nstages;
    const int64_t xrow_stride = a.x_bstride * static_cast<int64_t>(sizeof(xs_t<TX>));
    int s = 0;
    uint32_t ph = 0;
    for (int64_t g = b0; g < b1; g += NB) {          // one stage = up to NB consecutive batch rows
        const int nb = (g + NB <= b1) ? NB : static_cast<int>(b1 - g);
        mbar_wait(empty_addr + 8 * s, ph ^ 1u);
        const uint32_t fb = full_addr + 8 * s;
        // the phase cannot complete before this arrive, so copies of the other producers that
        // land earlier only drive the transaction count transiently negative
        if (p == 0 && lane == 0) mbar_arrive_expect_tx(fb, tile_bytes * static_cast<uint32_t>(nb));
        const char *xg = xbase + g * xrow_stride;
        const uint32_t sbase = stages_addr + static_cast<uint32_t>(s) * a.stage_bytes;
        const int ncopies = nb * td.nseg;
        for (int i = p + active * lane; i < ncopies; i += 32 * active) {
            const int n = i / td.nseg;
            const SegB e = ssegs[i - n * td.nseg];
            tma_bulk_g2s(sbase + static_cast<uint32_t>(n) * a.row_bytes + e.dst, xg + n * xrow_stride + e.src, e.len,
                         fb, policy);
        }
        if (++s == S) { s = 0; ph ^= 1u; }
    }
}

// PACKED (LPR = 1, KPL = 16): a thread owns up to four short destination rows, one per 4-link
// sub-row (a longer row continues into the next sub-rows); job.rowmap then holds
// [ntiles][4][NCT] = destination row of a sub-row, -1 empty, -2 continuation of the previous one.
template <typename TX, typename TY, int LPR, int KPL, int NCT, bool PACKED = false, bool ORD = false>
__global__ void __launch_bounds__(NCT + 32 * producer_warps(NCT), NCT == 256 ? 2 : 1)
staged_kernel(const __grid_constant__ JobBatch jb, const __grid_constant__ ApplyArgs a)
{
    constexpr int kProducerWarps = producer_warps(NCT);
    constexpr int kThreads = NCT + 32 * kProducerWarps;
    constexpr int kConsumerWarps = NCT / 32;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    // blockIdx.y = level of the grouped launch, blockIdx.x = its work item: everything that
    // steers the batch loop (tile, chunk, b0, b1, stage base) then derives from block indices and
    // kernel parameters only, stays in uniform registers, and the per-link shared-memory load
    // becomes LDS [R_off + UR_base] without a per-link address instruction
    const LevelJob &job = jb.jobs[blockIdx.z];
    const int tile = blockIdx.x;
    const int chunk = blockIdx.y;
    if (tile >= job.nblocks) return;
    const int64_t b0 = static_cast<int64_t>(chunk) * a.chunk;
    const int64_t b1 = (b0 + a.chunk < a.B) ? b0 + a.chunk : a.B;
    const TileDesc td = job.tiles[tile];

    SegB *ssegs = reinterpret_cast<SegB *>(smem + kSmemHeader);
    const uint32_t smem_addr = pin_reg(smem_u32(smem));
    const uint32_t full_addr = smem_addr, empty_addr = smem_addr + 8 * kMaxStages;
    const uint32_t stages_addr = smem_u32(smem) + a.stage_off;      // not pinned: stays uniform
    const int S = a.nstages;

    for (int i = tid; i < td.nseg; i += kThreads) {
        const Seg sg = job.segs[td.seg0 + i];
        ssegs[i] = SegB{sg.dst * static_cast<uint32_t>(sizeof(xs_t<TX>)), sg.len * static_cast<uint32_t>(sizeof(xs_t<TX>)),
                        static_cast<uint64_t>(sg.src) * sizeof(xs_t<TX>)};
    }
    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full_addr + 8 * s, 1);
            mbar_init(empty_addr + 8 * s, kConsumerWarps);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp >= kConsumerWarps) {
        // ---------------- producer warps: TMA bulk copies of the footprint, one stage per batch
        // row; producer p issues segments p, p + 4, ... (one per lane)
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kProducerRegs));
        produce_stages<TX>(job, a, td, ssegs, full_addr, empty_addr, stages_addr, warp - kConsumerWarps, kProducerWarps,
                           lane, b0, b1);
    } else {
        // ---------------- consumer warps: links live in registers for the whole batch loop
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(consumer_regs(NCT)));
        const int r_in = tid / LPR;
        const int l_in = tid % LPR;
        const bool valid = r_in < td.nrows;
        // td.row0 is the tile's first slot; plans built on a re-ordered row sequence map slots to rows
        const int row = (!PACKED && job.rowmap && valid) ? job.rowmap[td.row0 + r_in] : td.row0 + r_in;

        double w[KPL];
        uint32_t off[KPL];
        {
            const size_t base = static_cast<size_t>(tile) * KPL * NCT + tid;
#pragma unroll
            for (int k = 0; k < KPL; ++k) {
                w[k] = __ldg(job.wplan + base + static_cast<size_t>(k) * NCT);
                off[k] = stages_addr + static_cast<uint32_t>(__ldg(job.iplan + base + static_cast<size_t>(k) * NCT)) *
                                           static_cast<uint32_t>(sizeof(xs_t<TX>));      // address of the link in stage 0, row 0
            }
        }
        if constexpr (PACKED) {
            static_assert(LPR == 1 && KPL == 16, "packed rows: 4 sub-rows of 4 links per thread");
            int rs[4];                  // destination row per sub-row (-1 none)
            uint32_t flags = 0;         // bit u: sub-row u continues u-1; bit 4+u: row of sub-row u is dead
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                rs[u] = __ldg(job.rowmap + (static_cast<size_t>(tile) * 4 + u) * NCT + tid);
                if (rs[u] == -2) flags |= 1u << u;
                if (rs[u] >= 0) {
                    bool dead = false;
                    if (job.masked && job.imask[rs[u]] == 0) dead = true;
                    if (a.remap_area_min > 0.0 && job.frac[rs[u]] < a.remap_area_min) dead = true;
                    if (dead) flags |= 16u << u;
                }
            }
            uint32_t dm[4];             // 0x7ff80000 for the sub-rows of dead rows, else 0
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                dm[u] = (flags & (16u << u)) ? 0x7ff80000u : 0u;
                asm volatile("" : "+r"(dm[u]));          // opaque: kept in a register, not re-derived from `flags` per batch row
            }
            TY *yb = static_cast<TY *>(job.y) + b0 * a.y_bstride;
            const xs_t<TX> *xp = static_cast<const xs_t<TX> *>(job.x) + b0 * a.x_bstride;
            const bool stream_only = (a.debug_flags & 1u) != 0;
            const int NB = a.rows_per_stage;
            bool prefer_fill = false;
            uint32_t n_done = 0;
            int s = 0;
            uint32_t ph = 0;
            for (int64_t g = b0; g < b1; g += NB) {
                const int nb = (g + NB <= b1) ? NB : static_cast<int>(b1 - g);
                mbar_wait(full_addr + 8 * s, ph);
                uint32_t sb = static_cast<uint32_t>(s) * a.stage_bytes;      // uniform: LDS [R_link + UR_sb]
#pragma unroll 1
                for (int n = 0; n < nb; ++n, sb += a.row_bytes, yb += a.y_bstride, xp += a.x_bstride) {
                    double s4[4] = {0.0, 0.0, 0.0, 0.0};
                    if (!stream_only) {
                        // same fast / filled / adaptive scheme as the lane-per-row consumers below
                        const bool probe = !prefer_fill || (n_done & 15u) == 0;
                        ++n_done;
                        if (probe) {
                            if constexpr (ORD) lane_chain4<TX, false>(sb, off, w, flags, s4, a.dec);
                            else lane_sum4<TX, false>(sb, off, w, s4, a.dec);
                            prefer_fill = __any_sync(0xffffffffu, not_finite((s4[0] + s4[1]) + (s4[2] + s4[3])));
                        }
                        if (prefer_fill) {                                          // one copy of the filled sum
                            if constexpr (ORD) lane_chain4<TX, true>(sb, off, w, flags, s4, a.dec);
                            else lane_sum4<TX, true>(sb, off, w, s4, a.dec);
                        }
                    }
                    if (n == nb - 1) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(empty_addr + 8 * s);
                    }
                    // a row's value = its first sub-row + the continuation sub-rows behind it
                    // (ORD: the chain already ran through the continuation sub-rows; the row's value
                    // is the chain after its last sub-row)
                    double acc[4];
                    acc[3] = s4[3];
                    if constexpr (ORD) {
                        acc[2] = (flags & 8u) ? acc[3] : s4[2];
                        acc[1] = (flags & 4u) ? acc[2] : s4[1];
                        acc[0] = (flags & 2u) ? acc[1] : s4[0];
                    } else {
                        acc[2] = s4[2] + ((flags & 8u) ? acc[3] : 0.0);
                        acc[1] = s4[1] + ((flags & 4u) ? acc[2] : 0.0);
                        acc[0] = s4[0] + ((flags & 2u) ? acc[1] : 0.0);
                    }
                    // one warp-wide test keeps the threshold logic (finish) off the common path,
                    // which is then four predicated stores
                    // (compared on the high words: 0x43E12C7B'00000000 is just below 9.9e18, NaN counts as hot)
                    const int hi_max = max(max(__double2hiint(acc[0]), __double2hiint(acc[1])),
                                           max(__double2hiint(acc[2]), __double2hiint(acc[3])));
                    if (__any_sync(0xffffffffu, hi_max >= 0x43E12C7B)) {
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            if (rs[u] >= 0)
                                store_y(yb + rs[u], finish<TY, ORD>(acc[u], (flags & (16u << u)) != 0,
                                                                    [&]() { return replay<TX>(job.rowptr, job.col, job.val, rs[u], xp, a.dec); }));
                        }
                    } else {
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            // a dead row's value becomes NaN by OR-ing exponent + quiet bit into its high
                            // word: one LOP3 per store where the select on `flags` costs a test and two selects
                            if (rs[u] >= 0)
                                store_y(yb + rs[u], static_cast<TY>(__hiloint2double(__double2hiint(acc[u]) | static_cast<int>(dm[u]),
                                                                                     __double2loint(acc[u]))));
                        }
                    }
                }
                if (++s == S) { s = 0; ph ^= 1u; }
            }
            return;
        }
        bool dead = false;
        if (valid) {
            if (job.masked && job.imask[row] == 0) dead = true;
            if (a.remap_area_min > 0.0 && job.frac[row] < a.remap_area_min) dead = true;
        }
        TY *yp = static_cast<TY *>(job.y) + row + b0 * a.y_bstride;      // this row's output, batch row b
        const xs_t<TX> *xp = static_cast<const xs_t<TX> *>(job.x) + b0 * a.x_bstride;    // source row b (replay only)
        const bool stream_only = (a.debug_flags & 1u) != 0;

        const int NB = a.rows_per_stage;
        bool prefer_fill = false;      // warp-uniform: the previous batch row needed the 1e20 fill
        uint32_t n_done = 0;
        int s = 0;
        uint32_t ph = 0;
        for (int64_t g = b0; g < b1; g += NB) {          // one stage = up to NB consecutive batch rows
            const int nb = (g + NB <= b1) ? NB : static_cast<int>(b1 - g);
            mbar_wait(full_addr + 8 * s, ph);
            uint32_t sb = static_cast<uint32_t>(s) * a.stage_bytes;          // uniform: LDS [R_link + UR_sb]
#pragma unroll 1
            for (int n = 0; n < nb; ++n, sb += a.row_bytes, yp += a.y_bstride, xp += a.x_bstride) {
                double acc = 0.0;
                bool renormed = false;
                if (!stream_only) {
                    // fast path: raw values.  A non-finite partial means some source value was NaN/inf
                    // (regrid.py:545-547 fills those with 1e20): redo the warp's links with the fill --
                    // or, in the opt-in renormalising mode, without the missing sources.
                    // Missing values are usually static (land/sea masks): a warp that needed the
                    // fill for one batch row goes straight to the single-pass filled sum for the
                    // following ones and re-probes the cheap path every 16 rows.
                    const bool probe = !prefer_fill || (n_done & 15u) == 0;
                    ++n_done;
                    auto row_sum = [&](auto fill) -> double {        // ORD: already the whole row's sum
                        if constexpr (ORD) return lane_sum_ordered<TX, LPR, KPL, decltype(fill)::value>(sb, off, w, l_in, a.dec);
                        else return lane_sum<TX, KPL, decltype(fill)::value>(sb, off, w, a.dec);
                    };
                    if (!probe) {
                        acc = row_sum(cuda::std::true_type{});
                    } else {
                        prefer_fill = false;
                        acc = row_sum(cuda::std::false_type{});
                        if (__any_sync(0xffffffffu, not_finite(acc))) {
                            if (a.renorm_min_valid < 0.0) {
                                acc = row_sum(cuda::std::true_type{});
                                prefer_fill = true;
                            } else {
                                double s3[3];
                                const size_t base = static_cast<size_t>(tile) * KPL * NCT + tid;
                                if constexpr (XElem<TX>::kPacked)
                                    lane_sum_valid<TX, KPL, NCT>(job.wplan, job.iplan, base, stages_addr + sb, s3, a.dec);
                                else
                                    lane_sum_valid<TX, KPL, NCT>(job.wplan, job.iplan, base, stages_addr + sb, s3);
                                acc = renormalise(group_sum<LPR>(s3[0]), group_sum<LPR>(s3[1]), group_sum<LPR>(s3[2]),
                                                  a.renorm_min_valid);
                                renormed = true;
                            }
                        }
                    }
                }
                if (n == nb - 1) {                   // last row read: the stage may be refilled
                    __syncwarp();
                    if (lane == 0) mbar_arrive(empty_addr + 8 * s);
                }
                if (renormed) {
                    if (l_in == 0 && valid) store_y(yp, static_cast<TY>(dead ? CUDART_NAN : acc));
                } else {
                    if constexpr (!ORD) acc = group_sum<LPR>(acc);
                    if (l_in == 0 && valid && !(a.debug_flags & 2u)) {       // bit 1 (profiling aid): no stores
                        if (a.renorm_min_valid < 0.0)
                            store_y(yp, finish<TY, ORD>(acc, dead, [&]() { return replay<TX>(job.rowptr, job.col, job.val, row, xp, a.dec); }));
                        else
                            store_y(yp, static_cast<TY>(dead ? CUDART_NAN : acc));      // no fill, so no 1e19 rule
                    }
                }
            }
            if (++s == S) { s = 0; ph ^= 1u; }
        }
    }
}

// ------------------------------------------------------------------ ordered (reference-order) kernel, long rows
//
// Reference-order sums for rows too long for a thread's registers.  The staged kernel spreads such
// a row over LPR lanes, and a chain that has to visit the lanes one after the other leaves all but
// one lane in LPR idle.  Here a THREAD owns a row (R rows per tile = R consumer threads) and walks
// its links -- the k-th link of thread t at [k][t] of an image of (float64 weight, stage byte offset)
// pairs the CTA keeps in SHARED memory for the whole batch loop (conflict-free: the lanes of a warp
// read consecutive words) -- adding the products one by one in ascending source order.  Two batch
// rows are chained at a time (the image is read once for both; two independent dependency chains).
// Same producers, stages and epilogue as staged_kernel; plan = the lane-per-row register image with
// LPR = 1 and KPL = K = the longest row (ApplyArgs::ord_k), slot k = the row's k-th link.

__device__ __forceinline__ double lds_f64(uint32_t addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// links in flight per thread: the chain itself is serial (one DADD per link and batch row), what
// overlaps is the offset -> value -> convert -> multiply pipeline of the following links.  Measured
// on B200 (reference-order sums forced, f32 -> f64): C4 2577 / 3060 / 3266 GB/s and C2 4260 / 4362 /
// 3950 GB/s with 4 / 8 / 16 links unrolled.
#ifndef SMM_ORD_UNROLL
#define SMM_ORD_UNROLL 8
#endif
constexpr int kOrdUnroll = SMM_ORD_UNROLL;

template <typename TX, int R, bool kFill>
__device__ __forceinline__ void chain_pair(uint32_t wa, uint32_t oa, int K, uint32_t s0, uint32_t s1, double &a0, double &a1,
                                           const Decode &d)
{
    a0 = 0.0;
    a1 = 0.0;
#pragma unroll kOrdUnroll
    for (int k = 0; k < K; ++k, wa += R * 8, oa += R * 4) {
        const double w = lds_f64(wa);
        const uint32_t o = lds_u32(oa);
        xv_t<TX> v0 = ldx_s<TX>(s0 + o, d);
        xv_t<TX> v1 = ldx_s<TX>(s1 + o, d);
        if (kFill) { v0 = fill_invalid(v0); v1 = fill_invalid(v1); }
        a0 = __dadd_rn(a0, __dmul_rn(static_cast<double>(v0), w));
        a1 = __dadd_rn(a1, __dmul_rn(static_cast<double>(v1), w));
    }
}

template <typename TX, int R, bool kFill>
__device__ __forceinline__ double chain_one(uint32_t wa, uint32_t oa, int K, uint32_t s0, const Decode &d)
{
    double acc = 0.0;
#pragma unroll kOrdUnroll
    for (int k = 0; k < K; ++k, wa += R * 8, oa += R * 4) {
        const double w = lds_f64(wa);
        xv_t<TX> v = ldx_s<TX>(s0 + lds_u32(oa), d);
        if (kFill) v = fill_invalid(v);
        acc = __dadd_rn(acc, __dmul_rn(static_cast<double>(v), w));
    }
    return acc;
}

constexpr int kOrderedProducerWarps = 4;

// Consumer loop of ordered_kernel with TWO threads per row: thread group HALF (0 | 1; R threads
// each, whole warps) chains batch row HALF of every pair of staged rows, so twice as many warps
// share the latency of the dependent offset -> value -> convert -> multiply -> add pipeline.  A
// separate instantiation per HALF keeps the stage offset of "my" row a uniform register.
template <typename TX, typename TY, int R, int HALF>
__device__ __forceinline__ void ordered_consume_half(const LevelJob &job, const ApplyArgs &a, const TileDesc &td,
                                                     uint32_t wimg_addr, uint32_t oimg_addr, uint32_t full_addr,
                                                     uint32_t empty_addr, int t, int lane, int64_t b0, int64_t b1)
{
    asm volatile("barrier.sync.aligned %0, %1;" ::"n"(1 + HALF), "n"(R) : "memory");      // convergence, see ordered_kernel
    const bool valid = t < td.nrows;
    const int row = (job.rowmap && valid) ? job.rowmap[td.row0 + t] : td.row0 + t;
    bool dead = false;
    if (valid) {
        if (job.masked && job.imask[row] == 0) dead = true;
        if (a.remap_area_min > 0.0 && job.frac[row] < a.remap_area_min) dead = true;
    }
    TY *yp = static_cast<TY *>(job.y) + row + (b0 + HALF) * a.y_bstride;
    const uint32_t wa = wimg_addr + static_cast<uint32_t>(t) * 8u;
    const uint32_t oa = oimg_addr + static_cast<uint32_t>(t) * 4u;
    const int NB = a.rows_per_stage, S = a.nstages, K = a.ord_k;
    bool prefer_fill = false;
    uint32_t n_done = 0;
    int s = 0;
    uint32_t ph = 0;
    for (int64_t g = b0; g < b1; g += NB) {
        const int nb = (g + NB <= b1) ? NB : static_cast<int>(b1 - g);
        mbar_wait(full_addr + 8 * s, ph);
        uint32_t sb = static_cast<uint32_t>(s) * a.stage_bytes + HALF * a.row_bytes;      // uniform
#pragma unroll 1
        for (int n = HALF; n < nb + HALF; n += 2, sb += 2 * a.row_bytes, yp += 2 * a.y_bstride) {
            const bool mine = n < nb;                        // (an odd last pair has no row for HALF 1)
            double acc = 0.0;
            if (mine) {
                const bool probe = !prefer_fill || (n_done & 15u) == 0;
                ++n_done;
                if (!probe) {
                    acc = chain_one<TX, R, true>(wa, oa, K, sb, a.dec);
                } else {
                    prefer_fill = false;
                    acc = chain_one<TX, R, false>(wa, oa, K, sb, a.dec);
                    if (__any_sync(0xffffffffu, not_finite(acc))) {
                        acc = chain_one<TX, R, true>(wa, oa, K, sb, a.dec);
                        prefer_fill = true;
                    }
                }
            }
            if (n + 2 >= nb + HALF) {                        // this group's last row of the stage is read
                __syncwarp();
                if (lane == 0) mbar_arrive(empty_addr + 8 * s);
            }
            if (mine && valid) store_y(yp, finish<TY, true>(acc, dead, []() { return 0.0; }));
        }
        if (++s == S) { s = 0; ph ^= 1u; }
    }
}

template <typename TX, typename TY, int R, int TPR = 1>     // TPR = threads per row (1: a thread chains both rows of a pair)
__global__ void __launch_bounds__(R * TPR + 32 * kOrderedProducerWarps, 1)
ordered_kernel(const __grid_constant__ JobBatch jb, const __grid_constant__ ApplyArgs a)
{
    constexpr int kThreads = R * TPR + 32 * kOrderedProducerWarps;
    constexpr int kConsumerWarps = R * TPR / 32;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int lane = tid & 31;

    const LevelJob &job = jb.jobs[blockIdx.z];
    const int tile = blockIdx.x;
    const int chunk = blockIdx.y;
    if (tile >= job.nblocks) return;
    const int64_t b0 = static_cast<int64_t>(chunk) * a.chunk;
    const int64_t b1 = (b0 + a.chunk < a.B) ? b0 + a.chunk : a.B;
    const TileDesc td = job.tiles[tile];
    const int K = a.ord_k;

    SegB *ssegs = reinterpret_cast<SegB *>(smem + kSmemHeader);
    double *wimg = reinterpret_cast<double *>(smem + a.wimg_off);
    uint32_t *oimg = reinterpret_cast<uint32_t *>(smem + a.oimg_off);
    const uint32_t smem_addr = smem_u32(smem);
    const uint32_t full_addr = smem_addr, empty_addr = smem_addr + 8 * kMaxStages;
    const uint32_t stages_addr = smem_addr + a.stage_off;
    const int S = a.nstages;

    for (int i = tid; i < td.nseg; i += kThreads) {
        const Seg sg = job.segs[td.seg0 + i];
        ssegs[i] = SegB{sg.dst * static_cast<uint32_t>(sizeof(xs_t<TX>)), sg.len * static_cast<uint32_t>(sizeof(xs_t<TX>)),
                        static_cast<uint64_t>(sg.src) * sizeof(xs_t<TX>)};
    }
    {   // the tile's link image: [K][R] weights and stage byte offsets
        const size_t ibase = static_cast<size_t>(tile) * K * R;
        for (int i = tid; i < K * R; i += kThreads) {
            wimg[i] = __ldg(job.wplan + ibase + i);
            // absolute shared address of the link in stage 0, row 0: what is added per batch row is a
            // pure function of the stage and row counters and stays in a uniform register
            oimg[i] = stages_addr + static_cast<uint32_t>(__ldg(job.iplan + ibase + i)) * static_cast<uint32_t>(sizeof(xs_t<TX>));
        }
    }
    if (tid == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(full_addr + 8 * s, 1);
            mbar_init(empty_addr + 8 * s, kConsumerWarps);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp >= kConsumerWarps) {
        produce_stages<TX>(job, a, td, ssegs, full_addr, empty_addr, stages_addr, warp - kConsumerWarps,
                           kOrderedProducerWarps, lane, b0, b1);
        return;
    }
    if constexpr (TPR == 2) {
        if (tid < R)
            ordered_consume_half<TX, TY, R, 0>(job, a, td, smem_u32(wimg), smem_u32(oimg), full_addr, empty_addr, tid,
                                               lane, b0, b1);
        else
            ordered_consume_half<TX, TY, R, 1>(job, a, td, smem_u32(wimg), smem_u32(oimg), full_addr, empty_addr,
                                               tid - R, lane, b0, b1);
        return;
    }
    // (the role branch above is warp-uniform, which the compiler cannot see: an ALIGNED barrier
    // among the consumer warps tells it that they are converged, so that the batch loop's control
    // and the stage offsets may live in uniform registers -- staged_kernel gets the same effect from
    // its setmaxnreg.sync.aligned)
    asm volatile("barrier.sync.aligned 1, %0;" ::"n"(R) : "memory");
    const bool valid = tid < td.nrows;
    const int row = (job.rowmap && valid) ? job.rowmap[td.row0 + tid] : td.row0 + tid;
    bool dead = false;
    if (valid) {
        if (job.masked && job.imask[row] == 0) dead = true;
        if (a.remap_area_min > 0.0 && job.frac[row] < a.remap_area_min) dead = true;
    }
    TY *yp = static_cast<TY *>(job.y) + row + b0 * a.y_bstride;
    const uint32_t wa = smem_u32(wimg) + static_cast<uint32_t>(tid) * 8u;
    const uint32_t oa = smem_u32(oimg) + static_cast<uint32_t>(tid) * 4u;
    const int NB = a.rows_per_stage;
    bool prefer_fill = false;      // warp-uniform: the previous pair needed the 1e20 fill
    uint32_t n_done = 0;
    int s = 0;
    uint32_t ph = 0;
    for (int64_t g = b0; g < b1; g += NB) {
        const int nb = (g + NB <= b1) ? NB : static_cast<int>(b1 - g);
        mbar_wait(full_addr + 8 * s, ph);
        uint32_t sb = static_cast<uint32_t>(s) * a.stage_bytes;          // uniform: LDS [R_link + UR_sb]
#pragma unroll 1
        for (int n = 0; n < nb; n += 2, sb += 2 * a.row_bytes) {
            const bool two = n + 1 < nb;
            const uint32_t s1 = two ? sb + a.row_bytes : sb;
            double a0, a1;
            // fast path on raw values; a non-finite sum (some source was NaN / inf) makes the warp
            // redo the pair with the 1e20 fill, and stay on the filled chain while that keeps happening
            const bool probe = !prefer_fill || (n_done & 15u) == 0;
            ++n_done;
            if (!probe) {
                chain_pair<TX, R, true>(wa, oa, K, sb, s1, a0, a1, a.dec);
            } else {
                prefer_fill = false;
                chain_pair<TX, R, false>(wa, oa, K, sb, s1, a0, a1, a.dec);
                if (__any_sync(0xffffffffu, not_finite(a0) || not_finite(a1))) {
                    chain_pair<TX, R, true>(wa, oa, K, sb, s1, a0, a1, a.dec);
                    prefer_fill = true;
                }
            }
            if (n + 2 >= nb) {                           // last rows read: the stage may be refilled
                __syncwarp();
                if (lane == 0) mbar_arrive(empty_addr + 8 * s);
            }
            if (valid) {
                store_y(yp, finish<TY, true>(a0, dead, []() { return 0.0; }));
                if (two) store_y(yp + a.y_bstride, finish<TY, true>(a1, dead, []() { return 0.0; }));
            }
            yp += (two ? 2 : 1) * a.y_bstride;
        }
        if (++s == S) { s = 0; ph ^= 1u; }
    }
}

// ------------------------------------------------------------------ gather kernel

// ORD (always with LPR = 1): a thread walks its row's links in ascending source order with
// separate multiply and add -- the reference's own summation order.
template <typename TX, typename TY, int LPR, bool ORD = false>
__global__ void __launch_bounds__(kGatherThreads)
gather_kernel(const __grid_constant__ JobBatch jb, const __grid_constant__ ApplyArgs a)
{
    constexpr int BT = kGatherBT;
    constexpr int RPB = kGatherThreads / LPR;   // destination rows per block
    int jidx;
    const LevelJob &job = find_job(jb, blockIdx.x, jidx);
    const int local = blockIdx.x - job.item0;
    const int rblock = local % job.nblocks;
    const int chunk = local / job.nblocks;
    const int64_t b0 = static_cast<int64_t>(chunk) * a.chunk;
    const int64_t b1 = (b0 + a.chunk < a.B) ? b0 + a.chunk : a.B;

    const int tid = threadIdx.x;
    const int l_in = tid % LPR;
    // the job serves every row of the level, or the rows of a list (the long rows of a split plan)
    const int64_t slot = static_cast<int64_t>(rblock) * RPB + tid / LPR;
    const bool valid = slot < (job.nrows > 0 ? static_cast<int64_t>(job.nrows) : a.n_dst);
    const int row = valid ? (job.nrows > 0 ? job.rowmap[slot] : static_cast<int>(slot)) : 0;

    int j0 = 0, j1 = 0;
    bool dead = false;
    if (valid) {
        j0 = job.rowptr[row];
        j1 = job.rowptr[row + 1];
        if (job.masked && job.imask[row] == 0) dead = true;
        if (a.remap_area_min > 0.0 && job.frac[row] < a.remap_area_min) dead = true;
    }
    const xs_t<TX> *xbase = static_cast<const xs_t<TX> *>(job.x);
    TY *yrow = static_cast<TY *>(job.y) + row;
    const bool do_fill = a.renorm_min_valid < 0.0;

    for (int64_t b = b0; b < b1; b += BT) {
        const xs_t<TX> *xr[BT];
#pragma unroll
        for (int t = 0; t < BT; ++t) {
            const int64_t bb = (b + t < b1) ? b + t : b1 - 1;
            xr[t] = xbase + bb * a.x_bstride;
        }
        double acc[BT];
#pragma unroll
        for (int t = 0; t < BT; ++t) acc[t] = 0.0;
        for (int j = j0 + l_in; j < j1; j += LPR) {
            const int c = __ldg(job.col + j);
            const double wv = __ldg(job.val + j);
            xv_t<TX> v[BT];
#pragma unroll
            for (int t = 0; t < BT; ++t) v[t] = ld_nc_x<TX>(xr[t] + c, a.dec);
#pragma unroll
            for (int t = 0; t < BT; ++t) {  // renormalising mode keeps raw values: a non-finite sum flags the row
                const double xv = static_cast<double>(do_fill ? fill_invalid(v[t]) : v[t]);
                if constexpr (ORD) acc[t] = __dadd_rn(acc[t], __dmul_rn(xv, wv));
                else acc[t] = fma(xv, wv, acc[t]);
            }
        }
#pragma unroll
        for (int t = 0; t < BT; ++t) {
#pragma unroll
            for (int o = LPR / 2; o > 0; o >>= 1) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
        }
        if (a.renorm_min_valid >= 0.0) {
            // opt-in renormalising mode: rows whose plain sum is non-finite are redone without the
            // missing sources (sequentially by the row's first lane: rare rows, simple code)
            if (l_in == 0 && valid) {
#pragma unroll
                for (int t = 0; t < BT; ++t) {
                    if (b + t >= b1) continue;
                    double r = acc[t];
                    if (not_finite(r)) {
                        double wx = 0.0, wv = 0.0, wa = 0.0;
                        for (int j = j0; j < j1; ++j) {
                            const xv_t<TX> v = ldx_g<TX>(xr[t] + job.col[j], a.dec);
                            const double wj = job.val[j];
                            wa += wj;
                            if (fill_invalid(v) == v) { wx = fma(static_cast<double>(v), wj, wx); wv += wj; }
                        }
                        r = renormalise(wx, wv, wa, a.renorm_min_valid);
                    }
                    yrow[(b + t) * a.y_bstride] = static_cast<TY>(dead ? CUDART_NAN : r);
                }
            }
            continue;
        }
        if (l_in == 0 && valid) {
#pragma unroll
            for (int t = 0; t < BT; ++t) {
                if (b + t < b1)
                    yrow[(b + t) * a.y_bstride] = finish<TY, ORD>(acc[t], dead, [&]() {
                        return replay<TX>(job.rowptr, job.col, job.val, row, xr[t], a.dec);
                    });
            }
        }
    }
}

// ------------------------------------------------------------------ compact (two-pass) path
//
// Scattered sources (unstructured grids in file order): a direct gather pulls a 64-byte sector
// per 4-byte element.  With enough batch rows it is cheaper to (1) read the slab once, fully
// coalesced, and write the TOUCHED source columns transposed into a compact buffer
// XT[n_touched][BC] (BC = batch rows of the chunk, <= 64: every column becomes one contiguous
// run), then (2) apply the links from XT, where a link is one coalesced run of BC values, with
// lanes over the batch.  Pass 2 sums each (row, batch row) in the reference's own order
// (ascending source, separate multiply and add), so the results are bit-identical to a
// reference-order evaluation and no threshold replay is needed.

constexpr int kCompactThreads = 256;
constexpr int kCompactRows = 32;        // destination rows per pass-2 block

// Pass 1.  Block i owns source columns [i*W, (i+1)*W) and the touched columns among them,
// tcols[blk_ptr[i] .. blk_ptr[i+1]) (ascending; their rank in tcols is the row of XT).
// The block's [bc][W] piece of the slab comes in as bc 1-D TMA bulk copies (one per batch row,
// W * sizeof(TX) bytes each, all in flight at once, completion counted on one mbarrier) when the
// rows are 16-byte aligned (`bulk`), else as 4-byte asynchronous element copies (LDGSTS).  Packed
// 16-bit sources are transposed RAW (XT holds the 16-bit values; pass 2 decodes them); their
// element copies are plain loads and stores, as cp.async has no 2-byte form.
constexpr int kCompactStride = kCompactW + 4;       // tile row stride in elements: a multiple of 16 bytes
// (2-byte elements: kCompactW + 8, the next stride that keeps the rows 16-byte aligned)
__host__ __device__ constexpr int compact_stride(size_t elem_bytes) { return elem_bytes == 2 ? kCompactW + 8 : kCompactStride; }

template <typename TX>
__global__ void __launch_bounds__(kCompactThreads)
compact_kernel(const TX *__restrict__ x, int64_t x_bstride, int64_t n_src, int bc,
               const int32_t *__restrict__ tcols, const int32_t *__restrict__ blk_ptr, TX *__restrict__ xt,
               int bulk)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ int16_t tcol_s[kCompactW];
    static_assert(kCompactW <= 32768, "touched columns of a block are kept as 16-bit offsets");
    constexpr int kStride = compact_stride(sizeof(TX));
    TX *tile = reinterpret_cast<TX *>(smem_raw);                 // [bc][kStride]
    const int t0 = blk_ptr[blockIdx.x], t1 = blk_ptr[blockIdx.x + 1];
    if (t0 == t1) return;                                        // nothing touched here: not read at all
    const int64_t c0 = static_cast<int64_t>(blockIdx.x) * kCompactW;
    const int w = static_cast<int>((n_src - c0 < kCompactW) ? n_src - c0 : kCompactW);
    const int tid = threadIdx.x;
    const bool use_bulk = bulk && (w * sizeof(TX)) % 16 == 0;    // block-uniform
    const uint32_t bar_addr = smem_u32(&bar);
    if (use_bulk) {
        if (tid == 0) {
            mbar_init(bar_addr, 1);
            mbar_fence_init();
        }
        __syncthreads();
        if (tid < 32) {
            if (tid == 0) mbar_arrive_expect_tx(bar_addr, static_cast<uint32_t>(bc) * w * sizeof(TX));
            const uint64_t pol = l2_evict_first_policy();
            for (int b = tid; b < bc; b += 32)
                tma_bulk_g2s(smem_u32(tile + b * kStride), x + c0 + b * x_bstride,
                             static_cast<uint32_t>(w * sizeof(TX)), bar_addr, pol);
        }
    }
    // the block's touched columns (at most W of them), fetched while the copies are in flight:
    // the transposition below then depends on shared memory only
    for (int i = tid; i < t1 - t0; i += kCompactThreads) tcol_s[i] = static_cast<int16_t>(tcols[t0 + i] - c0);
    if (use_bulk) {
        __syncthreads();
        mbar_wait(bar_addr, 0);
    } else {
        // thread (col, row group): the threads of a warp copy 32 consecutive columns of one batch
        // row (one 128-byte line per LDGSTS instruction); with fewer than 256 columns per block the
        // remaining threads take every (256 / W)-th batch row
        constexpr int kRowGroups = kCompactThreads / kCompactW > 0 ? kCompactThreads / kCompactW : 1;
        if constexpr (sizeof(TX) == 2) {
            for (int col = tid % kCompactW; col < w; col += kCompactThreads) {
                const TX *xc = x + c0 + col;
#pragma unroll 8
                for (int b = (kCompactW < kCompactThreads ? tid / kCompactW : 0); b < bc; b += kRowGroups)
                    tile[b * kStride + col] = __ldg(xc + b * x_bstride);
            }
        } else {
            for (int col = tid % kCompactW; col < w; col += kCompactThreads) {
                const TX *xc = x + c0 + col;
                const uint32_t dst0 = smem_u32(tile + col);
#pragma unroll 8
                for (int b = (kCompactW < kCompactThreads ? tid / kCompactW : 0); b < bc; b += kRowGroups)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(dst0 + static_cast<uint32_t>(b * kStride * sizeof(TX))),
                                 "l"(xc + b * x_bstride), "n"(sizeof(TX))
                                 : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
    }
    const int warp = tid >> 5, lane = tid & 31;
    for (int t = t0 + warp; t < t1; t += kCompactThreads / 32) {
        const int c = tcol_s[t - t0];
        TX *dst = xt + static_cast<int64_t>(t) * kCompactBC;
        if (lane < bc) dst[lane] = tile[lane * kStride + c];
        if (kCompactBC > 32 && lane + 32 < bc) dst[lane + 32] = tile[(lane + 32) * kStride + c];
    }
}

// Pass 2.  Block = 32 destination rows x bc batch rows; warp w takes rows w, w + 8, ...; lanes are
// batch rows.  rcol[j] = rank of link j's source column in tcols.  The block's row pointers and
// its links (a contiguous piece of the CSR; up to kCompactLinks of them) are staged in shared
// memory first, so that a row costs one round trip to memory (its XT runs) instead of three.
// The pass is bound by instruction issue (DESIGN.md 4.2), so the link loop is
// kept lean: raw values first (RAW) -- the sums of a row whose sources are all finite are exactly
// the filled sums -- and the 1e20 fill (regrid.py:545-547) only in a redo of the rows whose raw
// sum came out non-finite; no batch-range predicates when the chunk is full (FULL); the links
// read with plain shared-memory loads when they are staged (STAGED).
constexpr int kCompactLinks = 1024;

// the row again, with non-finite values replaced by 1e20 (out of line: keeps the common loop small).
// Four links at a time, their loads unconditional and ahead of any use: with predicated loads the
// compiler puts each value's non-finite test right behind its load and the links go one round trip
// to memory at a time.  (XT rows are kCompactBC wide whatever bc is, slots behind the last link
// re-read it; what lanes >= bc compute is never stored.)
template <typename TX, typename... D>
__device__ __noinline__ double2 compact_row_filled(const xs_t<TX> *__restrict__ xt, const int32_t *rc, const double *vl,
                                                   int j0, int j1, int lane, const D &...d)
{
    using XS = xs_t<TX>;
    double a0 = 0.0, a1 = 0.0;
    for (int j = j0; j < j1; j += 4) {
        xv_t<TX> v0[4], v1[4];
        double w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int jj = j + u < j1 ? j + u : j1 - 1;
            const XS *src = xt + static_cast<int64_t>(rc[jj]) * kCompactBC + lane;
            w[u] = vl[jj];
            v0[u] = ldx_v<TX>(__ldg(src), d...);
            v1[u] = ldx_v<TX>(kCompactBC > 32 ? __ldg(src + 32) : XS(0), d...);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (j + u < j1) {
                a0 = __dadd_rn(a0, __dmul_rn(static_cast<double>(fill_invalid(v0[u])), w[u]));
                a1 = __dadd_rn(a1, __dmul_rn(static_cast<double>(fill_invalid(v1[u])), w[u]));
            }
        }
    }
    return make_double2(a0, a1);
}

template <typename TX, typename TY, bool FULL, bool STAGED, bool RAW>
__device__ __forceinline__ void compact_rows(const xs_t<TX> *__restrict__ xt, int bc, const int32_t *rp, const int32_t *rc,
                                             const double *vl, const uint8_t *dead_s, int nrows, int warp, int lane,
                                             TY (*out)[kCompactRows + 1], const Decode &d)
{
    using XS = xs_t<TX>;
    for (int rl = warp; rl < nrows; rl += kCompactThreads / 32) {
        double a0 = 0.0, a1 = 0.0;
        const int j0 = rp[rl], j1 = rp[rl + 1];
#pragma unroll 4
        for (int j = j0; j < j1; ++j) {
            const XS *src = xt + static_cast<int64_t>(rc[j]) * kCompactBC + lane;
            const double wj = vl[j];
            xv_t<TX> v0, v1;
            if (FULL) {
                v0 = ldx_v<TX>(__ldg(src), d);
                v1 = ldx_v<TX>(kCompactBC > 32 ? __ldg(src + 32) : XS(0), d);
            } else {
                v0 = ldx_v<TX>(lane < bc ? __ldg(src) : XS(0), d);
                v1 = ldx_v<TX>(lane + 32 < bc ? __ldg(src + 32) : XS(0), d);
            }
            if (!RAW) { v0 = fill_invalid(v0); v1 = fill_invalid(v1); }
            a0 = __dadd_rn(a0, __dmul_rn(static_cast<double>(v0), wj));      // reference order, no FMA
            a1 = __dadd_rn(a1, __dmul_rn(static_cast<double>(v1), wj));
        }
        // (a warp that remembers "the last row needed the fill" and skips the raw pass was measured:
        // it costs the clean case more than it saves the other)
        if (RAW && __any_sync(0xffffffffu, not_finite(a0) || not_finite(a1))) {
            double2 f;
            if constexpr (XElem<TX>::kPacked) f = compact_row_filled<TX>(xt, rc, vl, j0, j1, lane, d);
            else f = compact_row_filled<TX>(xt, rc, vl, j0, j1, lane);
            a0 = f.x;
            a1 = f.y;
        }
        if (a0 > 1e19) a0 = CUDART_NAN;                                       // regrid.py:570
        if (a1 > 1e19) a1 = CUDART_NAN;
        const bool dead = dead_s[rl] != 0;
        out[lane][rl] = static_cast<TY>(dead ? CUDART_NAN : a0);
        if (kCompactBC > 32) out[(lane + 32) % kCompactBC][rl] = static_cast<TY>(dead ? CUDART_NAN : a1);
    }
}

template <typename TX, typename TY>
__global__ void __launch_bounds__(kCompactThreads, 6)       // 6 blocks per SM: the out-of-line filled row must not raise the register count
compact_apply_kernel(const xs_t<TX> *__restrict__ xt, int bc, const int32_t *__restrict__ rowptr,
                     const int32_t *__restrict__ rcol, const double *__restrict__ val,
                     const int32_t *__restrict__ imask, const double *__restrict__ frac, int masked,
                     double remap_area_min, int64_t n_dst, TY *__restrict__ y, int64_t y_bstride, int raw_first,
                     const __grid_constant__ Decode dec)
{
    __shared__ TY out[kCompactBC][kCompactRows + 1];
    __shared__ double val_s[kCompactLinks];
    __shared__ int32_t rcol_s[kCompactLinks];
    __shared__ int32_t rp[kCompactRows + 1];
    __shared__ uint8_t dead_s[kCompactRows];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t row0 = static_cast<int64_t>(blockIdx.x) * kCompactRows;
    const int nrows = static_cast<int>((n_dst - row0 < kCompactRows) ? n_dst - row0 : kCompactRows);
    if (tid <= nrows) rp[tid] = rowptr[row0 + tid];
    if (tid < nrows) {
        bool dead = false;
        if (masked && imask[row0 + tid] == 0) dead = true;
        if (remap_area_min > 0.0 && frac[row0 + tid] < remap_area_min) dead = true;
        dead_s[tid] = dead;
    }
    __syncthreads();
    const int jb0 = rp[0], nl = rp[nrows] - jb0;
    const bool staged = nl <= kCompactLinks;                    // block-uniform
    if (staged) {
        for (int i = tid; i < nl; i += kCompactThreads) {
            rcol_s[i] = __ldg(rcol + jb0 + i);
            val_s[i] = __ldg(val + jb0 + i);
        }
        __syncthreads();
    }
    const bool full = bc == kCompactBC;
    // raw_first (rows of two or more links on average): sum raw values and redo the rows that came
    // out non-finite; with one link per row the per-row work dominates and the fill stays in line
    if (staged && full && raw_first)
        compact_rows<TX, TY, true, true, true>(xt, bc, rp, rcol_s - jb0, val_s - jb0, dead_s, nrows, warp, lane, out, dec);
    else if (staged && full)
        compact_rows<TX, TY, true, true, false>(xt, bc, rp, rcol_s - jb0, val_s - jb0, dead_s, nrows, warp, lane, out, dec);
    else if (staged)
        compact_rows<TX, TY, false, true, false>(xt, bc, rp, rcol_s - jb0, val_s - jb0, dead_s, nrows, warp, lane, out, dec);
    else
        compact_rows<TX, TY, false, false, false>(xt, bc, rp, rcol, val, dead_s, nrows, warp, lane, out, dec);
    __syncthreads();
    for (int b = warp; b < bc; b += kCompactThreads / 32)
        if (lane < nrows) y[b * y_bstride + row0 + lane] = out[b][lane];
}

}  // namespace smm
