// smm_api.cu -- C ABI (include/smmregrid_b200.h) over the sm_100a kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#if defined(__x86_64__) || defined(_M_X64)
#include <emmintrin.h>
#endif

#include "../../include/smmregrid_b200.h"
#include "smm_internal.h"
#include "smm_aux_kernels.cuh"
#include "smm_plan.h"

using namespace smm;

namespace smm {

// the kernel launchers live in the smm_inst_*.cu translation units
SMM_DECLARE_LAUNCHERS(extern, float, float)
SMM_DECLARE_LAUNCHERS(extern, float, double)
SMM_DECLARE_LAUNCHERS(extern, double, float)
SMM_DECLARE_LAUNCHERS(extern, double, double)
SMM_DECLARE_LAUNCHERS(extern, I16F32, float)
SMM_DECLARE_LAUNCHERS(extern, I16F32, double)
SMM_DECLARE_LAUNCHERS(extern, I16F64, float)
SMM_DECLARE_LAUNCHERS(extern, I16F64, double)
SMM_DECLARE_LAUNCHERS(extern, F16, float)
SMM_DECLARE_LAUNCHERS(extern, F16, double)
SMM_DECLARE_LAUNCHERS(extern, BF16, float)
SMM_DECLARE_LAUNCHERS(extern, BF16, double)

namespace {
thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};
}  // namespace

int smm_fail(int code, const std::string &msg)
{
    g_err = msg;
    return code;
}

void smm_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

}  // namespace smm

namespace {

int fail(int code, const std::string &msg) { return smm_fail(code, msg); }

struct HostSlot {
    void *dx = nullptr, *dy = nullptr;
    size_t cap_x = 0, cap_y = 0;
    void *px = nullptr, *py = nullptr;      // pinned bounce buffers for pageable host arrays
    size_t cap_px = 0, cap_py = 0;
    cudaEvent_t ev_in = nullptr, ev_k = nullptr, ev_out = nullptr;   // H2D done | apply done | D2H done
};

}  // namespace

struct smm_handle {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    bool ref_order = false;              // rows are summed in the reference's order (SMM_SUM_REFERENCE)
    bool cache_hit = false;              // CSR + plans were read from the on-disk plan cache
    int gather_lanes[2] = {1, 1};        // lanes per row of fast-sum gather launches: whole levels | row lists
    std::vector<LevelDev> levels;
    // stream-ordered pool for the compact path's transposed buffer; keeps its memory between
    // applies (re-mapping ~1 GB per call cost 8 ms against 1.9 ms of kernels), freed with the handle
    mutable std::mutex pool_mu;
    mutable cudaMemPool_t pool = nullptr;
    std::mutex host_mu;
    HostSlot slots[kHostSlots];
    cudaStream_t s_in[2] = {nullptr, nullptr};                       // host pipeline: H2D (alternating) ...
    cudaStream_t s_k = nullptr, s_out = nullptr;                     // ... applies | D2H
};

namespace {

template <typename T>
int upload(T **dptr, const std::vector<T> &v, int64_t &bytes)
{
    *dptr = nullptr;
    const size_t n = std::max<size_t>(v.size(), 1) * sizeof(T);
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(dptr), n));
    if (!v.empty()) CUDA_TRY(cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    bytes += static_cast<int64_t>(n);
    return SMM_OK;
}

void free_level(LevelDev &L)
{
    cudaFree(L.rowptr); cudaFree(L.col); cudaFree(L.val);
    cudaFree(L.tiles); cudaFree(L.segs); cudaFree(L.wplan); cudaFree(L.iplan); cudaFree(L.rowmap);
    cudaFree(L.imask); cudaFree(L.frac);
    cudaFree(L.tcols); cudaFree(L.blk_ptr); cudaFree(L.rcol); cudaFree(L.gather_rows);
    L = LevelDev{};
}

int upload_level(const HostCsr &csr, const HostPlan &plan, LevelDev &L)
{
    L.n_src = csr.n_src; L.n_dst = csr.n_dst; L.nnz = static_cast<int64_t>(csr.col.size());
    L.touched = csr.touched_src; L.max_row_nnz = csr.max_row_nnz;
    int rc;
    if ((rc = upload(&L.rowptr, csr.rowptr, L.device_bytes))) return rc;
    if ((rc = upload(&L.col, csr.col, L.device_bytes))) return rc;
    if ((rc = upload(&L.val, csr.val, L.device_bytes))) return rc;
    L.staged = plan.ok;
    L.why_not_staged = plan.why;
    L.lpr = plan.lpr; L.kpl = plan.kpl; L.rpt = plan.rows_per_tile; L.nct = plan.nct;
    if (plan.ok) {
        L.ntiles = static_cast<int32_t>(plan.tiles.size());
        L.max_segs = plan.max_tile_segments;
        L.max_elems = plan.max_tile_elems;
        L.sum_elems = plan.sum_tile_elems;
        if ((rc = upload(&L.tiles, plan.tiles, L.device_bytes))) return rc;
        if ((rc = upload(&L.segs, plan.segs, L.device_bytes))) return rc;
        if ((rc = upload(&L.wplan, plan.wplan, L.device_bytes))) return rc;
        if ((rc = upload(&L.iplan, plan.iplan, L.device_bytes))) return rc;
        L.packed = plan.packed;
        L.reordered = plan.reordered;
        L.ordlong = plan.ordlong;
        if (plan.packed) { if ((rc = upload(&L.rowmap, plan.rowslot, L.device_bytes))) return rc; }
        else if (!plan.rowmap.empty() && (rc = upload(&L.rowmap, plan.rowmap, L.device_bytes))) return rc;
        L.n_gather_rows = static_cast<int32_t>(plan.gather_rows.size());
        if (L.n_gather_rows > 0) {
            if ((rc = upload(&L.gather_rows, plan.gather_rows, L.device_bytes))) return rc;
            for (int32_t r : plan.gather_rows) L.gather_nnz += csr.rowptr[r + 1] - csr.rowptr[r];
        }
    }
    if (!plan.ok && L.nnz > 0) {
        // scattered sources: the two-pass compact path needs the touched columns and link ranks
        CompactPlan cp;
        build_compact(csr, kCompactW, cp);
        L.compact_blocks = static_cast<int32_t>(cp.blk_ptr.size()) - 1;
        if ((rc = upload(&L.tcols, cp.tcols, L.device_bytes))) return rc;
        if ((rc = upload(&L.blk_ptr, cp.blk_ptr, L.device_bytes))) return rc;
        if ((rc = upload(&L.rcol, cp.rcol, L.device_bytes))) return rc;
    }
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&L.imask), static_cast<size_t>(L.n_dst) * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&L.frac), static_cast<size_t>(L.n_dst) * sizeof(double)));
    L.device_bytes += L.n_dst * 12;
    return SMM_OK;
}

int open_device(int device, smm_handle *h)
{
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(SMM_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e) +
                                      " (smmregrid_b200 has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(SMM_ERR_INVALID, "device index out of range");
    cudaDeviceProp p;
    CUDA_TRY(cudaGetDeviceProperties(&p, device));
    if (p.major != 10)
        return fail(SMM_ERR_CUDA, "smmregrid_b200 kernels are built for sm_100a only; device is sm_" +
                                      std::to_string(p.major) + std::to_string(p.minor));
    h->device = device;
    h->sm_count = p.multiProcessorCount;
    h->smem_optin = p.sharedMemPerBlockOptin;
    return SMM_OK;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// One layout for every level of a weight set, so that a grouped launch runs a single kernel:
// lanes per row / links per lane from the longest row, or -- no row above 16 links anywhere --
// the packed-rows layout (a thread owns up to 4 rows).
struct PlanChoice {
    bool cfg = false, packed = false;
    int32_t lpr = 0, kpl = 0;
};

PlanChoice choose_plan(const std::vector<HostCsr> &csrs, const PlanSettings &s)
{
    PlanChoice pc;
    int32_t max_row = 0;
    int64_t pslots = 0;
    for (const HostCsr &c : csrs) {
        max_row = std::max(max_row, c.max_row_nnz);
        const int64_t ps = packed_slots(c);
        pslots = (ps < 0 || pslots < 0) ? -1 : pslots + ps;
    }
    pc.cfg = choose_lanes(s, max_row, pc.lpr, pc.kpl);
    pc.packed = pc.cfg && prefer_packed(s, pslots);
    return pc;
}

// Tile plans of all levels, one layout for the whole weight set so that a grouped launch runs a
// single kernel.  Candidates, in order of preference:
//   packed        every row has <= 16 links: a thread owns up to 4 rows;
//   split         a few rows are longer (at most 1/8 of the rows, 40 % of the links: the fans of
//                 cells around the grid poles of a tripolar ocean grid): the short rows are packed,
//                 the long ones are listed for the gather kernel (HostPlan::gather_rows);
//   ordered-long  (reference-order sums only) a thread per row, links in shared memory;
//   lanes per row from the longest row.
// A packed tile holds 4x the rows, so its footprint may not fit where the lane-per-row tile's
// does: if any level's packed plan is unusable for that reason, all levels fall back to the next
// candidate.
void plan_levels(const std::vector<HostCsr> &csrs, int64_t n_dst, int sm_count, bool ref_order,
                 const PlanSettings &s, std::vector<HostPlan> &plans)
{
    const PlanChoice pc = choose_plan(csrs, s);
    plans.assign(csrs.size(), HostPlan{});
    bool split = false;
    if (pc.cfg && !pc.packed) {
        int64_t rows = 0, rows_long = 0, nnz = 0, nnz_long = 0;
        for (const HostCsr &c : csrs)
            for (int64_t r = 0; r < c.n_dst; ++r) {
                const int32_t n = c.rowptr[r + 1] - c.rowptr[r];
                ++rows; nnz += n;
                if (n > 16) { ++rows_long; nnz_long += n; }
            }
        split = rows_long > 0 && rows_long * 8 <= rows && nnz_long * 5 <= nnz * 2;
        if (s.split >= 0) split = rows_long > 0 && s.split == 1;
    }
    // levels are independent: a few host threads take them in turn (75 ocean levels: ~13 s -> ~1 s)
    const int nthreads = std::max(1, std::min({host_cpus(), 16, static_cast<int>(csrs.size())}));
    // reference-order sums for rows beyond the packed layout: a thread per row with the links in
    // shared memory (ordered_kernel) when an image of K = longest row links x R rows x 12 bytes fits
    // ~100 KB for some R in {256, 128, 64, 32}; else the lane-by-lane chain of staged_kernel<ORD>
    int32_t ord_k = 0, ord_rows = 0;
    if (ref_order && pc.cfg && !pc.packed && s.ordlong) {
        for (const HostCsr &c : csrs) ord_k = std::max(ord_k, c.max_row_nnz);
        for (int32_t r : {256, 128, 64, 32})
            if (ord_rows == 0 && static_cast<int64_t>(ord_k) * r * 12 <= 100 * 1024) ord_rows = r;
        if (s.ord_rows) ord_rows = s.ord_rows;
    }
    enum Mode { kSplit, kPacked, kOrdLong, kLanes };
    std::vector<Mode> modes;
    if (split) modes.push_back(kSplit);
    if (pc.packed) modes.push_back(kPacked);
    if (ord_rows > 0) modes.push_back(kOrdLong);
    modes.push_back(kLanes);
    for (Mode mode : modes) {
        // packed plans: 256 consumer threads, two CTAs per SM (measured: bilinear 1440x721 -> 3600x1800
        // +4 %, 1:1 conservative +3 %, C3 +9 % over 512), unless SMM_CONSUMER_THREADS overrides;
        // reference-order kernels exist for 256 consumer threads only
        const int32_t nct = mode == kOrdLong ? ord_rows
                            : mode == kLanes ? (ref_order ? 256 : default_consumer_threads(s, n_dst, pc.cfg ? pc.lpr : 0, sm_count))
                                             : (ref_order ? 256 : default_consumer_threads(s, 0, 1, sm_count));
        std::atomic<bool> retry{false};
        parallel_for(nthreads, static_cast<int64_t>(csrs.size()), [&](int64_t i) {
            if (retry.load()) return;
            plans[i] = HostPlan{};
            plans[i].ref_order = ref_order;
            if (!pc.cfg) { plans[i].why = "a destination row has more than 512 links"; return; }
            if (mode == kSplit) {
                std::vector<int32_t> lrows, srows;
                long_rows(csrs[i], lrows, srows);
                build_plan(csrs[i], -1, pc.kpl, nct, ref_order, s, plans[i], &srows);
                plans[i].gather_rows = std::move(lrows);
                if (!plans[i].ok) retry.store(true);           // any failure: the whole set takes the next layout
            } else if (mode == kOrdLong) {
                build_plan(csrs[i], 1, ord_k, nct, true, s, plans[i]);
                plans[i].ordlong = plans[i].ok;
                if (!plans[i].ok && !csrs[i].col.empty()) retry.store(true);
            } else {
                build_plan(csrs[i], mode == kPacked ? -1 : pc.lpr, pc.kpl, nct, ref_order, s, plans[i]);
                // only a footprint that is too large can be cured by smaller tiles
                if (mode == kPacked && !plans[i].ok && plans[i].why.rfind("tile footprint", 0) == 0) retry.store(true);
            }
        });
        if (!retry.load()) return;
    }
}

// SMM_SUM_AUTO: reference order when some weight is negative (the products of a row can cancel)
bool resolve_ref_order(int32_t summation, const PlanSettings &s, const std::vector<HostCsr> &csrs)
{
    if (s.summation != SMM_SUM_AUTO) summation = s.summation;
    if (summation == SMM_SUM_REFERENCE) return true;
    if (summation == SMM_SUM_FAST) return false;
    for (const HostCsr &c : csrs)
        if (c.has_negative) return true;
    return false;
}


// Host side of smm_create_levels, shared with the host-only introspection entry point: CSR and
// tile plans of every level, through the on-disk cache when a directory is given.
int build_host_operator(int32_t n_levels, const int64_t *link_length, int64_t nl_max, int64_t n_src, int64_t n_dst,
                        const int32_t *src_address, const int32_t *dst_address, const double *remap_matrix,
                        int32_t num_wgts, int32_t index_base, const smm_create_opts *opts, int sm_count,
                        const PlanSettings &s, std::vector<HostCsr> &csrs, std::vector<HostPlan> &plans, bool &ref_order, bool &cache_hit)
{
    const int32_t summation = opts ? opts->summation : SMM_SUM_AUTO;
    if (summation != SMM_SUM_AUTO && summation != SMM_SUM_FAST && summation != SMM_SUM_REFERENCE)
        return fail(SMM_ERR_INVALID, "smm_create_opts.summation must be SMM_SUM_AUTO, SMM_SUM_FAST or SMM_SUM_REFERENCE");
    const std::string cache_dir = (opts && opts->plan_cache_dir) ? opts->plan_cache_dir : "";
    csrs.assign(static_cast<size_t>(n_levels), HostCsr{});
    plans.clear();
    cache_hit = false;
    PlanCacheKey cache_key;
    bool usable_arrays = true;          // the cache key hashes the arrays: they must be there
    for (int32_t i = 0; i < n_levels; ++i)
        if (link_length[i] > 0 && (!src_address || !dst_address || !remap_matrix)) usable_arrays = false;
    const bool use_cache = !cache_dir.empty() && usable_arrays && n_src > 0 && n_dst > 0 && num_wgts >= 1;
    if (use_cache) {
        cache_key = plan_cache_key(n_levels, link_length, nl_max, n_src, n_dst, src_address, dst_address,
                                   remap_matrix, num_wgts, index_base, summation, sm_count, s);
        cache_hit = plan_cache_load(cache_dir, cache_key, n_levels, n_src, n_dst, csrs, plans, ref_order);
        if (cache_hit) return SMM_OK;
        csrs.assign(static_cast<size_t>(n_levels), HostCsr{});
    }
    {
        // levels are independent: built by a few host threads; the first failing level is reported
        std::vector<int> rcs(static_cast<size_t>(n_levels), SMM_OK);
        std::vector<std::string> errs(static_cast<size_t>(n_levels));
        const int nthreads = std::max(1, std::min({host_cpus(), 16, static_cast<int>(n_levels)}));
        parallel_for(nthreads, n_levels, [&](int64_t i) {
            const int64_t o = i * nl_max;
            rcs[i] = build_csr(n_src, n_dst, link_length[i], src_address ? src_address + o : nullptr,
                               dst_address ? dst_address + o : nullptr,
                               remap_matrix ? remap_matrix + o * num_wgts : nullptr, num_wgts, index_base,
                               csrs[i], errs[i]);
        });
        for (int32_t i = 0; i < n_levels; ++i)
            if (rcs[i]) return fail(rcs[i], (n_levels > 1 ? "level " + std::to_string(i) + ": " : "") + errs[i]);
    }
    ref_order = resolve_ref_order(summation, s, csrs);
    plan_levels(csrs, n_dst, sm_count, ref_order, s, plans);
    if (use_cache) plan_cache_store(cache_dir, cache_key, csrs, plans, ref_order);   // best effort
    return SMM_OK;
}

// ------------------------------------------------------------------ launch dispatch

// (packed 16-bit x: the element type follows the decoded dtype, opt.dec_dtype)
#define SMM_DTYPE_DISPATCH(FN, ...)                                                                           \
    ((x_dtype == SMM_I16)                                                                                     \
         ? ((opt.dec_dtype == SMM_F32)                                                                        \
                ? (y_dtype == SMM_F32 ? FN<I16F32, float>(__VA_ARGS__) : FN<I16F32, double>(__VA_ARGS__))     \
                : (y_dtype == SMM_F32 ? FN<I16F64, float>(__VA_ARGS__) : FN<I16F64, double>(__VA_ARGS__)))    \
     : (x_dtype == SMM_F16) ? (y_dtype == SMM_F32 ? FN<F16, float>(__VA_ARGS__) : FN<F16, double>(__VA_ARGS__))    \
     : (x_dtype == SMM_BF16) ? (y_dtype == SMM_F32 ? FN<BF16, float>(__VA_ARGS__) : FN<BF16, double>(__VA_ARGS__)) \
     : (x_dtype == SMM_F32 && y_dtype == SMM_F32) ? FN<float, float>(__VA_ARGS__)                             \
     : (x_dtype == SMM_F32 && y_dtype == SMM_F64) ? FN<float, double>(__VA_ARGS__)                            \
     : (x_dtype == SMM_F64 && y_dtype == SMM_F32) ? FN<double, float>(__VA_ARGS__)                            \
                                                  : FN<double, double>(__VA_ARGS__))

// bytes of one x element as it sits in memory (SMM_I16: the raw 16 bits)
size_t x_elem_bytes(int32_t x_dtype)
{
    return (x_dtype == SMM_I16 || x_dtype == SMM_F16 || x_dtype == SMM_BF16) ? 2 : x_dtype == SMM_F32 ? 4 : 8;
}

bool is_half(int32_t x_dtype) { return x_dtype == SMM_F16 || x_dtype == SMM_BF16; }

// Batch rows per work item.  A work item pays a fixed prologue (its tile's register image,
// barriers: `prologue_us`) and the launch pays about half an item of tail per wave, so with an
// estimated launch time T the cost is minimal near sqrt(T / (2 * prologue)) waves.  (Measured
// on B200: the former fixed ~32-wave target cost 8-12 % at 64-512 batch rows on C2.)
// `slots` = CTAs resident on the device, `bytes_per_row` = HBM bytes one batch row moves.
int64_t pick_chunks(int64_t B, int64_t blocks_total, int64_t slots, double bytes_per_row, double prologue_us,
                    int64_t multiple, int64_t &chunk)
{
    const LaunchSettings &ls = launch_settings();
    const double t_us = static_cast<double>(B) * bytes_per_row / 6.5e6;     // at ~6.5 TB/s
    double waves = ls.waves > 0 ? ls.waves : std::sqrt(t_us / (2.0 * prologue_us));
    waves = std::min(32.0, std::max(1.0, waves));
    const double items = waves * static_cast<double>(slots);
    int64_t nchunks = static_cast<int64_t>(items / static_cast<double>(std::max<int64_t>(blocks_total, 1)) + 0.5);
    const int64_t max_chunks = std::max<int64_t>(1, B / ls.min_rows_per_item);
    nchunks = std::max<int64_t>(1, std::min<int64_t>({nchunks, max_chunks, 65535}));      // (grid.y of the staged launch)
    chunk = (B + nchunks - 1) / nchunks;
    chunk = (chunk + multiple - 1) / multiple * multiple;
    return (B + chunk - 1) / chunk;
}

constexpr int kCompactUnavailable = -1;   // launch_compact: nothing was launched, use the gather kernel

// Per-call options, resolved (smm_apply_opts; NULL = defaults).
struct ApplyOpts {
    int kernel = 0;                 // 0 automatic | SMM_KERNEL_*
    double renorm_min_valid = -1.0; // < 0: reference semantics (fill 1e20)
    int32_t dec_dtype = SMM_F64;    // SMM_I16 x: the decoded dtype D
    Decode dec{};                   // SMM_I16 x: the decode parameters as the kernels read them
};

// smm_decode -> Decode, after checking it against x_dtype
int resolve_decode(const smm_decode *d, int32_t x_dtype, ApplyOpts &out)
{
    if (x_dtype == SMM_I16 && !d) return fail(SMM_ERR_INVALID, "x_dtype SMM_I16 needs smm_apply_opts.decode");
    if (!d) return SMM_OK;
    if (x_dtype != SMM_I16) return fail(SMM_ERR_INVALID, "smm_apply_opts.decode is only valid with x_dtype SMM_I16");
    if (d->dtype != SMM_F32 && d->dtype != SMM_F64)
        return fail(SMM_ERR_INVALID, "smm_decode.dtype must be SMM_F32 or SMM_F64");
    if (d->n_fill < 0 || d->n_fill > 4) return fail(SMM_ERR_INVALID, "smm_decode.n_fill must be within [0, 4]");
    if (!std::isfinite(d->scale_factor) || !std::isfinite(d->add_offset))
        return fail(SMM_ERR_INVALID, "smm_decode.scale_factor and add_offset must be finite");
    const float sf = static_cast<float>(d->scale_factor), of = static_cast<float>(d->add_offset);
    if (d->dtype == SMM_F32 && (static_cast<double>(sf) != d->scale_factor || static_cast<double>(of) != d->add_offset))
        return fail(SMM_ERR_INVALID, "smm_decode: scale_factor and add_offset must be exact float32 values when dtype is SMM_F32");
    out.dec_dtype = d->dtype;
    out.dec.scale = d->scale_factor; out.dec.offset = d->add_offset;
    out.dec.scale_f = sf; out.dec.offset_f = of;
    out.dec.sign_xor = d->is_unsigned ? 0u : 0x8000u;
    out.dec.bias_f = d->is_unsigned ? 8388608.0f : 8421376.0f;
    // compared on the raw 16 bits; a value outside the raw type's range matches nothing
    const int32_t lo = d->is_unsigned ? 0 : -32768, hi = d->is_unsigned ? 65535 : 32767;
    for (int i = 0; i < 4; ++i)
        out.dec.fill[i] = (i < d->n_fill && d->fill[i] >= lo && d->fill[i] <= hi) ? (d->fill[i] & 0xffff) : -1;
    return SMM_OK;
}

int resolve_opts(const smm_apply_opts *o, int32_t x_dtype, ApplyOpts &out)
{
    out = ApplyOpts{};
    if (int rc = resolve_decode(o ? o->decode : nullptr, x_dtype, out)) return rc;
    if (!o) return SMM_OK;
    if (o->kernel != 0 && o->kernel != SMM_KERNEL_STAGED && o->kernel != SMM_KERNEL_GATHER &&
        o->kernel != SMM_KERNEL_COMPACT)
        return fail(SMM_ERR_INVALID, "smm_apply_opts.kernel must be 0, SMM_KERNEL_STAGED, SMM_KERNEL_GATHER or SMM_KERNEL_COMPACT");
    out.kernel = o->kernel;
    if (o->renormalize) {
        if (!(o->min_valid_fraction >= 0.0 && o->min_valid_fraction <= 1.0))
            return fail(SMM_ERR_INVALID, "smm_apply_opts.min_valid_fraction must be within [0, 1]");
        out.renorm_min_valid = o->min_valid_fraction;
    }
    return SMM_OK;
}

// The handle's stream-ordered pool for transient device buffers (created on first use); null when
// the device has no stream-ordered pools.
cudaMemPool_t handle_pool(const smm_handle *h)
{
    std::lock_guard<std::mutex> lock(h->pool_mu);
    if (!h->pool) {
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = h->device;
        uint64_t keep = UINT64_MAX;
        if (cudaMemPoolCreate(&h->pool, &props) != cudaSuccess ||
            cudaMemPoolSetAttribute(h->pool, cudaMemPoolAttrReleaseThreshold, &keep) != cudaSuccess) {
            cudaGetLastError();
            if (h->pool) { cudaMemPoolDestroy(h->pool); h->pool = nullptr; }
        }
    }
    return h->pool;
}

// Two-pass apply of one gather-family level (see compact_kernel).  The transposed buffer XT comes
// from the handle's stream-ordered pool, so concurrent applies on other streams stay independent.
int launch_compact(const smm_handle *h, const LevelDev &L, const JobSpec &sp, int32_t x_dtype, int32_t y_dtype,
                   int64_t B, int64_t xbs, int64_t ybs, double area_min, const ApplyOpts &opt, cudaStream_t st)
{
    cudaMemPool_t pool = handle_pool(h);
    if (!pool) return kCompactUnavailable;           // no stream-ordered pools here: direct gathers instead
    void *xt = nullptr;
    const size_t sx = x_elem_bytes(x_dtype);
    const size_t xt_bytes = std::max<size_t>(static_cast<size_t>(L.touched), 1) * kCompactBC * sx;
    if (cudaMallocFromPoolAsync(&xt, xt_bytes, pool, st) != cudaSuccess) {
        cudaGetLastError();
        return kCompactUnavailable;                  // not enough memory for the transposed buffer
    }
    const int rc = SMM_DTYPE_DISPATCH(launch_compact_t, h->device, L, sp, xt, B, xbs, ybs, area_min, opt.dec, st);
    cudaFreeAsync(xt, st);
    return rc;
}

int launch_jobs(const smm_handle *h, const std::vector<JobSpec> &specs, int32_t x_dtype,
                int32_t y_dtype, int64_t B, int64_t xbs, int64_t ybs, double area_min,
                const ApplyOpts &opt, cudaStream_t st);

constexpr int64_t kWidenBytes = int64_t{256} << 20;     // float32 rows widened per chunk (launch_widened)

// The float32 path of one half-source level on float32 copies of its rows, widened exactly into a
// buffer from the handle's pool, up to kWidenBytes at a time (see route_jobs).
int launch_widened(const smm_handle *h, const JobSpec &s, int32_t x_dtype, int32_t y_dtype, int64_t B, int64_t xbs,
                   int64_t ybs, double area_min, const ApplyOpts &opt, cudaStream_t st)
{
    const int64_t n = h->levels[s.level].n_src;          // a multiple of 4 here: float32 rows stay 16-byte aligned
    const int64_t rows = std::max<int64_t>(1, std::min<int64_t>({B, kWidenBytes / (4 * n), 65535}));
    cudaMemPool_t pool = handle_pool(h);
    float *buf = nullptr;
    if (!pool || cudaMallocFromPoolAsync(reinterpret_cast<void **>(&buf), static_cast<size_t>(rows * n) * 4, pool, st) != cudaSuccess) {
        cudaGetLastError();
        return fail(SMM_ERR_ALLOC, "no device memory for the float32 copy of half-precision rows that cannot be staged");
    }
    const size_t sy = y_dtype == SMM_F32 ? 4 : 8;
    int rc = SMM_OK;
    for (int64_t b0 = 0; b0 < B && rc == SMM_OK; b0 += rows) {
        const int64_t nb = std::min(rows, B - b0);
        const uint16_t *x = static_cast<const uint16_t *>(s.x) + b0 * xbs;
        const dim3 grid(static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 1024)), static_cast<unsigned>(nb));
        if (x_dtype == SMM_BF16) widen16_kernel<true><<<grid, 256, 0, st>>>(x, xbs, n, buf, n);
        else widen16_kernel<false><<<grid, 256, 0, st>>>(x, xbs, n, buf, n);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { rc = fail(SMM_ERR_CUDA, std::string("widen16_kernel: ") + cudaGetErrorString(e)); break; }
        smm_count_launches(1);
        const std::vector<JobSpec> w{JobSpec{s.level, buf, static_cast<char *>(s.y) + static_cast<size_t>(b0 * ybs) * sy, s.masked}};
        rc = launch_jobs(h, w, SMM_F32, y_dtype, nb, n, ybs, area_min, opt, st);
    }
    cudaFreeAsync(buf, st);
    return rc;
}

// shared memory of the link image of ordered-long plans: kpl x nct x (8 + 4) bytes
size_t image_bytes(const LevelDev &L) { return L.ordlong ? round_up(static_cast<size_t>(L.kpl) * L.nct * 12, 128) : 0; }

// shared memory a staged launch needs for two stages of one batch row each
size_t two_stage_smem(size_t max_segs, size_t max_elems, size_t image, size_t es)
{
    return kSmemHeader + round_up(max_segs * sizeof(Seg), 128) + image + 2 * round_up(max_elems * es, 128);
}

// The kernel family that applies one level of a call.
enum Route { kWidened, kStaged, kCompact, kGather };

// Appends the route of every spec.  Half sources get the kernel family float32 data would get: their
// results are the float32 path's bit for bit, and the fast sums of the families differ in the last
// bits.  So every choice of a family is made with the element size `sd` of the float32 slab of the
// same B and ldx, at a 16-byte aligned address (plus the level's offset in the caller's x); stages,
// rows per stage and work items, which change no value, are sized with the real 2 bytes.
int route_jobs(const smm_handle *h, const std::vector<JobSpec> &specs, int32_t x_dtype, int64_t B, int64_t xbs,
               const ApplyOpts &opt, std::vector<Route> &route)
{
    const bool half_x = is_half(x_dtype);
    const size_t sx = x_elem_bytes(x_dtype), sd = half_x ? 4 : sx;
    for (const JobSpec &s : specs) {
        const LevelDev &L = h->levels[s.level];
        bool ok = L.staged && opt.kernel != SMM_KERNEL_GATHER;
        // the renormalising extension is not implemented for packed-rows and ordered-long plans: gather kernel
        ok = ok && !((L.packed || L.ordlong) && opt.renorm_min_valid >= 0.0);
        // TMA bulk copies need 16-byte aligned rows and lengths
        const bool aligned = (reinterpret_cast<uintptr_t>(s.x) % 16 == 0) && ((xbs * sx) % 16 == 0) &&
                             ((L.n_src * sx) % 16 == 0);
        ok = ok && (half_x ? (s.x_off * 4) % 16 == 0 && (xbs * 4) % 16 == 0 && (L.n_src * 4) % 16 == 0 : aligned);
        // at least two stages must fit
        ok = ok && two_stage_smem(L.max_segs, L.max_elems, image_bytes(L), sd) <= h->smem_optin;
        if (!ok && opt.kernel == SMM_KERNEL_STAGED)
            return fail(SMM_ERR_INVALID, "staged kernel forced but unavailable for level " +
                                             std::to_string(s.level) + ": " +
                                             (L.staged ? std::string("slab alignment / footprint size")
                                                       : L.why_not_staged));
        // a half level that float32 would stage but whose 2-byte rows cannot be (x not 16-byte aligned,
        // ldx or n_src not a multiple of 8) takes the float32 path on widened rows: rows never depend
        // on the batching, so the chunked float32 applies give the float32 results
        if (ok) { route.push_back(aligned ? kStaged : kWidened); continue; }
        // The two-pass compact path for scattered sources with enough batch rows.  Cost per batch row
        // in HBM-byte equivalents, calibrated on B200 (C5nn / C5dis, f32 and f64): a random gather
        // costs ~120 bytes (a 64-byte sector at about half the streaming rate); the two passes move
        // the slab (at the streaming rate: TMA bulk copies), the touched columns twice-ish and the
        // links (random 256-byte runs), together ~1.2x the bytes at the streaming rate.  Runs of
        // fewer than 16 batch values are not worth it.
        const double gather_cost = static_cast<double>(L.nnz) * 120.0;
        const double compact_cost = 1.2 * (static_cast<double>(L.n_src) + static_cast<double>(L.touched) +
                                           static_cast<double>(L.nnz)) * static_cast<double>(sd);
        bool compact = L.rcol && opt.renorm_min_valid < 0.0 && opt.kernel != SMM_KERNEL_GATHER;
        if (opt.kernel != SMM_KERNEL_COMPACT) compact = compact && B >= 16 && gather_cost > compact_cost;
        route.push_back(compact ? kCompact : kGather);
    }
    return SMM_OK;
}

// The job of one level in a grouped launch, `nblocks` blocks of it (the launcher sets its first work item)
LevelJob level_job(const LevelDev &L, const JobSpec &s, int64_t nblocks)
{
    LevelJob j{};
    j.nblocks = static_cast<int32_t>(nblocks);
    j.tiles = L.tiles; j.segs = L.segs; j.wplan = L.wplan; j.iplan = L.iplan; j.rowmap = L.rowmap;
    j.rowptr = L.rowptr; j.col = L.col; j.val = L.val;
    j.imask = L.imask; j.frac = L.frac;
    j.x = s.x; j.y = s.y; j.masked = s.masked;
    return j;
}

// Shared-memory layout and batch split of a staged launch of `njobs` levels in the plan layout of `L`
// (the last of them): fills the staged fields of `a`, the dynamic shared memory and threads per row.
int size_staged(const smm_handle *h, const LevelDev &L, size_t max_segs, size_t max_elems, int64_t tiles,
                size_t njobs, size_t sx, size_t sy, ApplyArgs &a, size_t &smem, int &tpr)
{
    const LaunchSettings &ls = launch_settings();
    const size_t segs_off = kSmemHeader + round_up(max_segs * sizeof(Seg), 128);
    const size_t stage_off = segs_off + image_bytes(L);
    a.n_src = L.n_src; a.n_dst = L.n_dst;
    a.ord_k = L.kpl;
    a.wimg_off = static_cast<uint32_t>(segs_off);
    a.oimg_off = static_cast<uint32_t>(segs_off + static_cast<size_t>(L.kpl) * L.nct * 8);
    const size_t row_bytes = std::max<size_t>(128, round_up(max_elems * sx, 128));
    // stage several batch rows together (up to 8, ~56 KB per stage) so that the per-stage
    // barrier and loop overhead of the consumers is amortised: C3 2156 -> 2671 GB/s, C2 5565 -> 6111
    int nb_rows = ls.rows_per_stage > 0 ? ls.rows_per_stage : static_cast<int>((56u << 10) / row_bytes);
    const size_t smem_half = (228u * 1024u - 2u * 1024u) / 2u - 1024u;   // two CTAs per SM (NCT = 256)
    {   // ...but never at the price of pipeline depth (>= 4 stages) or of the second CTA per SM
        const size_t budget = (L.nct == 256 ? smem_half : h->smem_optin) - std::min(stage_off, smem_half);
        nb_rows = static_cast<int>(std::min<size_t>(nb_rows, std::max<size_t>(1, budget / (4 * row_bytes))));
    }
    nb_rows = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>({nb_rows, 8, a.B})));
    if (L.ordlong) {    // ordered kernel: one CTA per SM, batch rows chained in pairs: an even number of
                        // rows per stage, as many as leave three stages
        nb_rows = (a.B >= 2 && stage_off + 4 * row_bytes <= h->smem_optin) ? 2 : 1;
        while (nb_rows >= 2 && nb_rows + 2 <= 8 && nb_rows + 2 <= a.B &&
               stage_off + 3 * static_cast<size_t>(nb_rows + 2) * row_bytes <= h->smem_optin)
            nb_rows += 2;
    }
    const size_t stage_bytes = row_bytes * nb_rows;
    int64_t chunk = 0;             // batch rows per work item: whole stages
    const double row_bytes_hbm = static_cast<double>(njobs) *
                                 (static_cast<double>(a.n_src) * sx + static_cast<double>(a.n_dst) * sy);
    const int ctas_per_sm = (!L.ordlong && L.nct == 256) ? 2 : 1;
    const int64_t nchunks = pick_chunks(a.B, tiles, static_cast<int64_t>(h->sm_count) * ctas_per_sm,
                                        row_bytes_hbm, L.ordlong ? 6.0 : (L.nct == 256 ? 2.5 : 4.0), nb_rows, chunk);
    a.chunk = chunk; a.nchunks = static_cast<int32_t>(nchunks);
    size_t S = (!L.ordlong && L.nct == 256 && smem_half > stage_off) ? (smem_half - stage_off) / stage_bytes : 0;
    if (S < 3) S = (h->smem_optin - stage_off) / stage_bytes;        // one CTA per SM
    S = std::min<size_t>(S, kMaxStages);
    S = std::min<size_t>(S, static_cast<size_t>(ls.max_stages));
    if (S < 2) return fail(SMM_ERR_INVALID, "internal: staged footprint does not fit");
    a.nstages = static_cast<int32_t>(S);
    a.stage_bytes = static_cast<uint32_t>(stage_bytes);
    a.row_bytes = static_cast<uint32_t>(row_bytes);
    a.rows_per_stage = nb_rows;
    a.stage_off = static_cast<uint32_t>(stage_off);
    smem = stage_off + S * stage_bytes;
    // two threads per row (one per batch row of a pair) while that leaves at most 8 consumer warps:
    // C4 (64 rows per tile) 3060 -> 3989 GB/s, C2 (256 rows: 16 warps re-reading the image) 4368 -> 3518
    tpr = (L.ordlong && nb_rows >= 2 && (ls.ord_tpr == 2 || (ls.ord_tpr == 0 && L.nct <= 128))) ? 2 : 1;
    return SMM_OK;
}

// Staged launches: up to kMaxJobs levels at a time (balanced when there are more), and a group is
// closed early when the segment table of one level and the footprint of another would not fit two
// stages TOGETHER (each level fits on its own, see route_jobs).
int launch_staged(const smm_handle *h, const std::vector<JobSpec> &staged, int32_t x_dtype, int32_t y_dtype,
                  const ApplyOpts &opt, ApplyArgs a, cudaStream_t st)
{
    const size_t sx = x_elem_bytes(x_dtype), sy = y_dtype == SMM_F32 ? 4 : 8;
    const size_t groups = (staged.size() + kMaxJobs - 1) / kMaxJobs;
    const size_t per_group = groups ? (staged.size() + groups - 1) / groups : 1;   // balanced
    for (size_t g0 = 0; g0 < staged.size();) {
        JobBatch jb{};
        int64_t tiles = 0, max_tiles = 0;
        size_t max_segs = 0, max_elems = 0, g1 = g0;
        for (; g1 < staged.size() && g1 - g0 < per_group; ++g1) {
            const LevelDev &L = h->levels[staged[g1].level];
            const size_t ms = std::max<size_t>(max_segs, L.max_segs), me = std::max<size_t>(max_elems, L.max_elems);
            if (g1 > g0 && two_stage_smem(ms, me, image_bytes(L), sx) > h->smem_optin) break;
            max_segs = ms; max_elems = me;
            tiles += L.ntiles;
            max_tiles = std::max<int64_t>(max_tiles, L.ntiles);
            jb.jobs[g1 - g0] = level_job(L, staged[g1], L.ntiles);
        }
        const LevelDev &L = h->levels[staged[g1 - 1].level];
        jb.njobs = static_cast<int32_t>(g1 - g0);
        g0 = g1;
        size_t smem = 0;
        int tpr = 1;
        if (const int rc = size_staged(h, L, max_segs, max_elems, tiles, jb.njobs, sx, sy, a, smem, tpr)) return rc;
        if (max_tiles == 0) continue;
        // grid: x = tile, y = batch chunk, z = level of the group (blocks beyond a level's tile
        // count exit at once).  No index arithmetic in the kernel: what steers its batch loop stays
        // in uniform registers.
        const dim3 grid(static_cast<unsigned>(max_tiles), static_cast<unsigned>(a.nchunks), static_cast<unsigned>(jb.njobs));
        const int rc = L.ordlong ? SMM_DTYPE_DISPATCH(launch_ordered_t, h->device, L.nct, tpr, grid, smem, st, jb, a)
                                 : SMM_DTYPE_DISPATCH(launch_staged_t, h->device, L.lpr, L.kpl, L.nct, L.packed,
                                                      h->ref_order, grid, smem, st, jb, a);
        if (rc) return rc;
    }
    return SMM_OK;
}

// Gather launches of whole levels, or (`lists`) of the long rows of split plans, kMaxJobs levels at a time
int launch_gather(const smm_handle *h, const std::vector<JobSpec> &list, bool lists, int32_t x_dtype,
                  int32_t y_dtype, const ApplyOpts &opt, ApplyArgs a, cudaStream_t st)
{
    const bool ord = h->ref_order;     // reference order: one thread walks a row's links in sequence
    const int lpr = ord ? 1 : h->gather_lanes[lists ? 1 : 0];
    const int rpb = kGatherThreads / lpr;
    for (size_t g0 = 0; g0 < list.size(); g0 += kMaxJobs) {
        const size_t g1 = std::min(list.size(), g0 + kMaxJobs);
        JobBatch jb{};
        jb.njobs = static_cast<int32_t>(g1 - g0);
        int64_t nnz = 0, rows = 0, blocks_total = 0;
        for (size_t g = g0; g < g1; ++g) {
            const LevelDev &L = h->levels[list[g].level];
            const int64_t nrows = lists ? L.n_gather_rows : L.n_dst, nblocks = (nrows + rpb - 1) / rpb;
            LevelJob &j = jb.jobs[g - g0] = level_job(L, list[g], nblocks);
            if (lists) { j.rowmap = L.gather_rows; j.nrows = L.n_gather_rows; }
            nnz += lists ? L.gather_nnz : L.nnz;
            rows += nrows;
            blocks_total += nblocks;
            a.n_src = L.n_src; a.n_dst = L.n_dst;
        }
        int64_t chunk = 0;
        // gather kernel: up to 8 CTAs of 256 threads per SM, a light prologue, traffic dominated by the gathers
        const double row_bytes_hbm = static_cast<double>(nnz) * 64.0 + static_cast<double>(rows) * (y_dtype == SMM_F32 ? 4 : 8);
        const int64_t nchunks = pick_chunks(a.B, blocks_total, static_cast<int64_t>(h->sm_count) * 8, row_bytes_hbm, 1.0,
                                            kGatherBT, chunk);
        a.chunk = chunk; a.nchunks = static_cast<int32_t>(nchunks);
        int64_t item = 0;
        for (int32_t k = 0; k < jb.njobs; ++k) {
            jb.jobs[k].item0 = static_cast<int32_t>(item);
            item += static_cast<int64_t>(jb.jobs[k].nblocks) * nchunks;
        }
        if (item > INT32_MAX) return fail(SMM_ERR_INVALID, "too many work items in one launch");
        if (item == 0) continue;
        const dim3 grid(static_cast<unsigned>(item));
        const int rc = SMM_DTYPE_DISPATCH(launch_gather_t, lpr, ord, grid, st, jb, a);
        if (rc) return rc;
    }
    return SMM_OK;
}

// One apply of the specs' levels to B batch rows, in this order: widened levels, staged groups,
// compact levels, gathers of whole levels, gathers of the split plans' row lists.
int launch_jobs(const smm_handle *h, const std::vector<JobSpec> &specs, int32_t x_dtype,
                int32_t y_dtype, int64_t B, int64_t xbs, int64_t ybs, double area_min,
                const ApplyOpts &opt, cudaStream_t st)
{
    std::vector<Route> route;
    if (const int rc = route_jobs(h, specs, x_dtype, B, xbs, opt, route)) return rc;
    // the specs of one route, or (split plans) the staged ones whose long rows are listed for gathers
    auto select = [&](Route r, bool lists = false) {
        std::vector<JobSpec> out;
        for (size_t i = 0; i < specs.size(); ++i)
            if (route[i] == r && (!lists || h->levels[specs[i].level].n_gather_rows > 0)) out.push_back(specs[i]);
        return out;
    };
    for (const JobSpec &s : select(kWidened))
        if (const int rc = launch_widened(h, s, x_dtype, y_dtype, B, xbs, ybs, area_min, opt, st)) return rc;
    ApplyArgs a{};
    a.B = B; a.x_bstride = xbs; a.y_bstride = ybs; a.remap_area_min = area_min;
    a.renorm_min_valid = opt.renorm_min_valid;
    a.dec = opt.dec;
    a.debug_flags = launch_settings().debug_flags;
    if (const int rc = launch_staged(h, select(kStaged), x_dtype, y_dtype, opt, a, st)) return rc;
    for (size_t i = 0; i < specs.size(); ++i) {
        if (route[i] != kCompact) continue;
        const int rc = launch_compact(h, h->levels[specs[i].level], specs[i], x_dtype, y_dtype, B, xbs, ybs, area_min, opt, st);
        if (rc == kCompactUnavailable) route[i] = kGather;        // the level takes the gather kernel instead
        else if (rc) return rc;
    }
    if (const int rc = launch_gather(h, select(kGather), false, x_dtype, y_dtype, opt, a, st)) return rc;
    return launch_gather(h, select(kStaged, true), true, x_dtype, y_dtype, opt, a, st);
}

// true when cudaMemcpyAsync can DMA straight from/to the pointer (pinned or registered)
bool is_pinned(const void *p)
{
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// Large host copy with non-temporal stores: the destination (a pinned bounce buffer the DMA engine
// reads next) is written once and not read by the CPU again, so bypassing the cache saves the
// read-for-ownership of every destination line (+18 % over memcpy, measured with 4-8 threads).
void copy_streaming(char *dst, const char *src, size_t n)
{
#if defined(__x86_64__) || defined(_M_X64)
    if (n >= 4096) {
        size_t head = (64 - (reinterpret_cast<uintptr_t>(dst) & 63)) & 63;
        std::memcpy(dst, src, head);
        dst += head; src += head; n -= head;
        const size_t blocks = n / 64;
        for (size_t i = 0; i < blocks; ++i, src += 64, dst += 64) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src) + 0);
            const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src) + 1);
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src) + 2);
            const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src) + 3);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst) + 0, a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst) + 1, b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst) + 2, c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(dst) + 3, d);
        }
        _mm_sfence();
        n -= blocks * 64;
    }
#endif
    std::memcpy(dst, src, n);
}

// rows x row_bytes strided copy split over a few threads (pageable <-> pinned staging)
void parallel_copy_rows(char *dst, size_t dst_stride, const char *src, size_t src_stride, size_t row_bytes,
                        int64_t rows, int nthreads)
{
    const size_t total = static_cast<size_t>(rows) * row_bytes;
    if (nthreads <= 1 || total < (size_t{4} << 20)) {
        for (int64_t r = 0; r < rows; ++r) std::memcpy(dst + r * dst_stride, src + r * src_stride, row_bytes);
        return;
    }
    // split by bytes so a few huge rows still spread over all threads
    parallel_for(nthreads, nthreads, [&](int64_t t) {
        const size_t lo = total * t / nthreads, hi = total * (t + 1) / nthreads;
        size_t pos = lo;
        while (pos < hi) {
            const size_t r = pos / row_bytes, o = pos % row_bytes;
            const size_t n = std::min(row_bytes - o, hi - pos);
            copy_streaming(dst + r * dst_stride + o, src + r * src_stride + o, n);
            pos += n;
        }
    });
}

int check_level(const smm_handle *h, int32_t level)
{
    if (!h) return fail(SMM_ERR_INVALID, "null handle");
    if (level < 0 || level >= static_cast<int32_t>(h->levels.size()))
        return fail(SMM_ERR_INVALID, "level " + std::to_string(level) + " out of range [0, " +
                                         std::to_string(h->levels.size()) + ")");
    return SMM_OK;
}

// Checks the four apply entry points share: dtypes, options, B (and n_sel of the grouped calls,
// which pass it) and remap_area_min.  `empty`: nothing to apply, SMM_OK before any pointer is read.
int check_apply(int32_t x_dtype, int32_t y_dtype, const smm_apply_opts *opts, int64_t B, const int32_t *n_sel,
                double area_min, ApplyOpts &opt, bool &empty)
{
    if ((x_dtype != SMM_F32 && x_dtype != SMM_F64 && x_dtype != SMM_I16 && !is_half(x_dtype)) ||
        (y_dtype != SMM_F32 && y_dtype != SMM_F64))
        return fail(SMM_ERR_DTYPE, "x_dtype must be SMM_F32 (0), SMM_F64 (1), SMM_I16 (2), SMM_F16 (3) or SMM_BF16 (4), "
                                   "y_dtype SMM_F32 or SMM_F64");
    if (int rc = resolve_opts(opts, x_dtype, opt)) return rc;
    if (B < 0 || (n_sel && *n_sel < 0)) return fail(SMM_ERR_INVALID, n_sel ? "n_sel and B must be >= 0" : "B must be >= 0");
    if ((empty = B == 0 || (n_sel && *n_sel == 0)) || (area_min >= 0.0 && area_min <= 1.0)) return SMM_OK;
    return fail(SMM_ERR_INVALID, "The remap_area_min provided must be between 0.0 and 1.0");
}

// A masked apply needs the level's dst_grid_imask, a remap_area_min > 0 its dst_grid_frac.
int check_dst_arrays(const smm_handle *h, int32_t level, bool masked, double area_min)
{
    const LevelDev &L = h->levels[level];
    if (masked && !L.has_imask)
        return fail(SMM_ERR_INVALID, "masked apply but dst_grid_imask was never set for level " + std::to_string(level));
    if (area_min > 0.0 && !L.has_frac)
        return fail(SMM_ERR_INVALID, "remap_area_min > 0 but dst_grid_frac was never set for level " + std::to_string(level));
    return SMM_OK;
}

}  // namespace

namespace {

// Host <-> device streaming pipeline shared by smm_apply_host and smm_apply_levels_host.
// A batch row is `row_x` bytes of source (rows `x_stride` bytes apart) and `row_y` bytes of
// result; `launch(dx, dy, nb, stream)` applies the operator to nb batch rows held contiguously
// on the device.
//
// Streams per engine: the host->device copies alternate between two streams `s_in[0/1]` (the
// PCIe link is the bottleneck of the whole pipeline: it must never wait for a kernel or a
// device->host copy, and with two copies in flight the set-up latency of one hides behind the
// transfer of the other), the applies run on `s_k`, the (50x smaller) results return on `s_out`;
// events order them per chunk, and a ring of kHostSlots device buffers lets the copy of
// chunk i+1.. proceed while chunk i is applied.  Pinned (or registered) host arrays are DMA'd
// directly.  Pageable arrays -- what numpy / xarray hand over -- go through pinned bounce buffers
// filled by a few host threads, which overlaps the host copy of chunk i+1 with the PCIe
// transfer and kernel of chunk i (cudaMemcpyAsync straight from pageable memory is synchronous
// and ~3-5x slower).
template <typename Launch>
int host_pipeline(smm_handle *h, const void *x, size_t row_x, size_t x_stride, void *y, size_t row_y,
                  size_t y_stride, int64_t B, int64_t chunk_rows, Launch launch)
{
    const LaunchSettings &ls = launch_settings();
    const HostCallSettings hs = host_call_settings();
    const auto t_enter = std::chrono::steady_clock::now();
    auto ms_since = [&](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    const bool x_pinned = is_pinned(x), y_pinned = is_pinned(y);
    if (chunk_rows <= 0) {
        // ~128 MB of source per chunk for direct DMA (the fill of the pipeline -- the first chunk's
        // copy -- is the only part that does not overlap), ~64 MB when staging; at least 4 rows
        const int64_t mb = hs.chunk_mb > 0 ? hs.chunk_mb : (x_pinned ? 128 : 64);
        chunk_rows = std::max<int64_t>(4, (mb << 20) / std::max<int64_t>(1, static_cast<int64_t>(row_x)));
    }
    chunk_rows = std::min(chunk_rows, B);
    std::lock_guard<std::mutex> lock(h->host_mu);
    DeviceGuard g(h->device);
    const size_t need_x = static_cast<size_t>(chunk_rows) * row_x;
    const size_t need_y = static_cast<size_t>(chunk_rows) * row_y;
    for (cudaStream_t *sp : {&h->s_in[0], &h->s_in[1], &h->s_k, &h->s_out})
        if (!*sp) CUDA_TRY(cudaStreamCreateWithFlags(sp, cudaStreamNonBlocking));
    const int nslots = static_cast<int>(std::min<int64_t>(ls.host_slots, (B + chunk_rows - 1) / chunk_rows));
    for (int s = 0; s < nslots; ++s) {
        HostSlot &sl = h->slots[s];
        for (cudaEvent_t *ev : {&sl.ev_in, &sl.ev_k, &sl.ev_out})
            if (!*ev) CUDA_TRY(cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
        if (sl.cap_x < need_x) {
            cudaFree(sl.dx); sl.dx = nullptr; sl.cap_x = 0;
            CUDA_TRY(cudaMalloc(&sl.dx, need_x));
            sl.cap_x = need_x;
        }
        if (sl.cap_y < need_y) {
            cudaFree(sl.dy); sl.dy = nullptr; sl.cap_y = 0;
            CUDA_TRY(cudaMalloc(&sl.dy, need_y));
            sl.cap_y = need_y;
        }
        if (!x_pinned && sl.cap_px < need_x) {
            cudaFreeHost(sl.px); sl.px = nullptr; sl.cap_px = 0;
            CUDA_TRY(cudaHostAlloc(&sl.px, need_x, cudaHostAllocDefault));
            sl.cap_px = need_x;
        }
        if (!y_pinned && sl.cap_py < need_y) {
            cudaFreeHost(sl.py); sl.py = nullptr; sl.cap_py = 0;
            CUDA_TRY(cudaHostAlloc(&sl.py, need_y, cudaHostAllocDefault));
            sl.cap_py = need_y;
        }
    }
    const int nthreads = hs.copy_threads;
    struct Pending { char *ys = nullptr; int64_t nb = 0; bool used = false; };
    Pending pending[kHostSlots];
    // waits for the slot's last result copy and, when staging, hands the rows to the caller
    auto drain = [&](int s) -> int {
        if (!pending[s].used) return SMM_OK;
        CUDA_TRY(cudaEventSynchronize(h->slots[s].ev_out));
        if (!y_pinned && pending[s].nb)
            parallel_copy_rows(pending[s].ys, y_stride, static_cast<const char *>(h->slots[s].py), row_y, row_y,
                               pending[s].nb, 1);
        pending[s] = Pending{};
        return SMM_OK;
    };
    // one chunk through the three streams (a lambda so that every failure below leaves through the
    // common drain of the streams: queued copies must not outlive the call)
    auto run = [&]() -> int {
        int rc, slot = 0;
        int64_t ichunk = 0;
        for (int64_t b0 = 0; b0 < B; b0 += chunk_rows, slot = (slot + 1) % nslots, ++ichunk) {
            const int64_t nb = std::min(chunk_rows, B - b0);
            HostSlot &sl = h->slots[slot];
            cudaStream_t s_in = h->s_in[ichunk % ls.host_in_streams];
            const char *xs = static_cast<const char *>(x) + static_cast<size_t>(b0) * x_stride;
            char *ys = static_cast<char *>(y) + static_cast<size_t>(b0) * y_stride;
            const bool reused = pending[slot].used;
            // the result bounce buffer (or nothing) of this slot's previous chunk goes out first;
            // results of other chunks that have already arrived are handed over now as well, while
            // the link is busy with input, instead of piling up for the end of the call
            if (!y_pinned) {
                if ((rc = drain(slot))) return rc;
                for (int s2 = 0; s2 < nslots; ++s2)
                    if (pending[s2].used && cudaEventQuery(h->slots[s2].ev_out) == cudaSuccess && (rc = drain(s2))) return rc;
                cudaGetLastError();      // (cudaErrorNotReady of a query is not an error)
            }
            if (reused) CUDA_TRY(cudaStreamWaitEvent(s_in, sl.ev_k, 0));         // dx free: its kernel is done
            if (x_pinned) {
                if (x_stride == row_x)   // contiguous rows: one linear copy runs at the full PCIe rate
                    CUDA_TRY(cudaMemcpyAsync(sl.dx, xs, static_cast<size_t>(nb) * row_x, cudaMemcpyHostToDevice, s_in));
                else
                    CUDA_TRY(cudaMemcpy2DAsync(sl.dx, row_x, xs, x_stride, row_x, nb, cudaMemcpyHostToDevice, s_in));
            } else {
                if (reused) CUDA_TRY(cudaEventSynchronize(sl.ev_in));            // px free: its DMA is done
                parallel_copy_rows(static_cast<char *>(sl.px), row_x, xs, x_stride, row_x, nb, nthreads);
                CUDA_TRY(cudaMemcpyAsync(sl.dx, sl.px, static_cast<size_t>(nb) * row_x, cudaMemcpyHostToDevice, s_in));
            }
            CUDA_TRY(cudaEventRecord(sl.ev_in, s_in));
            CUDA_TRY(cudaStreamWaitEvent(h->s_k, sl.ev_in, 0));
            if (reused) CUDA_TRY(cudaStreamWaitEvent(h->s_k, sl.ev_out, 0));     // dy free: its copy-out is done
            if ((rc = launch(sl.dx, sl.dy, nb, h->s_k))) return rc;
            CUDA_TRY(cudaEventRecord(sl.ev_k, h->s_k));
            CUDA_TRY(cudaStreamWaitEvent(h->s_out, sl.ev_k, 0));
            if (y_pinned) {
                if (y_stride == row_y)
                    CUDA_TRY(cudaMemcpyAsync(ys, sl.dy, static_cast<size_t>(nb) * row_y, cudaMemcpyDeviceToHost, h->s_out));
                else
                    CUDA_TRY(cudaMemcpy2DAsync(ys, y_stride, sl.dy, row_y, row_y, nb, cudaMemcpyDeviceToHost, h->s_out));
            } else {
                CUDA_TRY(cudaMemcpyAsync(sl.py, sl.dy, static_cast<size_t>(nb) * row_y, cudaMemcpyDeviceToHost, h->s_out));
            }
            CUDA_TRY(cudaEventRecord(sl.ev_out, h->s_out));
            pending[slot] = Pending{ys, y_pinned ? 0 : nb, true};
        }
        for (int s = 0; s < nslots; ++s)
            if ((rc = drain(s))) return rc;
        return SMM_OK;
    };
    const double ms_setup = ms_since(t_enter);
    const int rc = run();
    if (ls.host_trace)
        std::fprintf(stderr, "[smm host pipeline] B=%lld chunk_rows=%lld slots=%d pinned x/y=%d/%d setup %.3f ms total %.3f ms (%.2f GB/s in)\n",
                     static_cast<long long>(B), static_cast<long long>(chunk_rows), nslots, int(x_pinned), int(y_pinned), ms_setup,
                     ms_since(t_enter), static_cast<double>(B) * row_x / (ms_since(t_enter) * 1e6));
    if (rc) {
        // nothing queued may still touch the caller's buffers (or the bounce buffers) after the
        // failure has been reported
        const std::string msg = g_err;
        cudaStreamSynchronize(h->s_in[0]); cudaStreamSynchronize(h->s_in[1]);
        cudaStreamSynchronize(h->s_k); cudaStreamSynchronize(h->s_out);
        cudaGetLastError();
        g_err = msg;
        return rc;
    }
    return SMM_OK;
}

}  // namespace

// ====================================================================== C ABI

extern "C" {

int smm_create(int64_t n_src, int64_t n_dst, int64_t nnz, const int32_t *src_address,
               const int32_t *dst_address, const double *remap_matrix, int32_t num_wgts,
               int32_t index_base, int32_t device, const smm_create_opts *opts, smm_handle **out)
{
    const int64_t ll = nnz;
    return smm_create_levels(1, &ll, nnz, n_src, n_dst, src_address, dst_address, remap_matrix,
                             num_wgts, index_base, device, opts, out);
}

int smm_create_levels(int32_t n_levels, const int64_t *link_length, int64_t nl_max, int64_t n_src,
                      int64_t n_dst, const int32_t *src_address, const int32_t *dst_address,
                      const double *remap_matrix, int32_t num_wgts, int32_t index_base,
                      int32_t device, const smm_create_opts *opts, smm_handle **out)
{
    const PlanSettings settings = plan_settings();
    if (!out) return fail(SMM_ERR_INVALID, "null output handle pointer");
    *out = nullptr;
    if (n_levels < 1 || !link_length || nl_max < 0)
        return fail(SMM_ERR_INVALID, "smm_create_levels: n_levels >= 1, link_length and nl_max >= 0 required");
    for (int32_t i = 0; i < n_levels; ++i)
        if (link_length[i] < 0 || link_length[i] > nl_max)
            return fail(SMM_ERR_INVALID, "link_length[" + std::to_string(i) + "] outside [0, nl_max]");

    smm_handle *h = new (std::nothrow) smm_handle();
    if (!h) return fail(SMM_ERR_ALLOC, "host allocation failed");
    int rc = open_device(device, h);
    if (rc) { delete h; return rc; }

    std::vector<HostCsr> csrs;
    std::vector<HostPlan> plans;
    rc = build_host_operator(n_levels, link_length, nl_max, n_src, n_dst, src_address, dst_address, remap_matrix,
                             num_wgts, index_base, opts, h->sm_count, settings, csrs, plans, h->ref_order, h->cache_hit);
    if (rc) { delete h; return rc; }
    h->levels.resize(static_cast<size_t>(n_levels));
    DeviceGuard g(device);              // the caller's current device is left as it was
    for (int32_t i = 0; i < n_levels; ++i) {
        rc = upload_level(csrs[i], plans[i], h->levels[i]);
        if (rc) { smm_destroy(h); return rc; }
        csrs[i] = HostCsr{};
        plans[i] = HostPlan{};
    }
    // Lanes per row of the gather kernel, from the mean row length of the weight set's gather-family
    // levels (of all levels when every one has a staged plan) and of the split plans' row lists.
    // The lanes split a row's fast sum: chosen once per handle, a level's bits do not depend on
    // which other levels share a call.
    int64_t nnz[3] = {0, 0, 0}, rows[3] = {0, 0, 0};      // gather-family levels | staged levels | row lists
    for (const LevelDev &L : h->levels) {
        nnz[L.staged ? 1 : 0] += L.nnz; rows[L.staged ? 1 : 0] += L.n_dst;
        nnz[2] += L.gather_nnz; rows[2] += L.n_gather_rows;
    }
    auto lanes = [](int64_t n, int64_t r) { const double avg = r ? static_cast<double>(n) / r : 0.0;
                                            return avg <= 2.0 ? 1 : (avg <= 24.0 ? 4 : 32); };
    h->gather_lanes[0] = rows[0] ? lanes(nnz[0], rows[0]) : lanes(nnz[1], rows[1]);
    h->gather_lanes[1] = lanes(nnz[2], rows[2]);
    *out = h;
    return SMM_OK;
}

int smm_destroy(smm_handle *h)
{
    if (!h) return SMM_OK;
    {
        DeviceGuard g(h->device);
        for (LevelDev &L : h->levels) free_level(L);
        if (h->pool) { cudaDeviceSynchronize(); cudaMemPoolDestroy(h->pool); }
        for (HostSlot &s : h->slots) {
            cudaFree(s.dx); cudaFree(s.dy);
            cudaFreeHost(s.px); cudaFreeHost(s.py);
            for (cudaEvent_t ev : {s.ev_in, s.ev_k, s.ev_out})
                if (ev) cudaEventDestroy(ev);
        }
        for (cudaStream_t st : {h->s_in[0], h->s_in[1], h->s_k, h->s_out})
            if (st) cudaStreamDestroy(st);
    }
    delete h;
    return SMM_OK;
}

int smm_get_info(const smm_handle *h, int32_t level, smm_info *out)
{
    int rc = check_level(h, level);
    if (rc) return rc;
    if (!out) return fail(SMM_ERR_INVALID, "null smm_info");
    const LevelDev &L = h->levels[level];
    std::memset(out, 0, sizeof(*out));
    out->n_src = L.n_src; out->n_dst = L.n_dst; out->nnz = L.nnz;
    out->n_levels = static_cast<int32_t>(h->levels.size());
    out->kernel = L.staged ? SMM_KERNEL_STAGED : SMM_KERNEL_GATHER;
    out->summation = h->ref_order ? SMM_SUM_REFERENCE : SMM_SUM_FAST;
    out->plan_cache_hit = h->cache_hit ? 1 : 0;
    out->gather_rows = L.staged ? L.n_gather_rows : 0;
    out->lanes_per_row = L.lpr; out->links_per_lane = L.kpl; out->rows_per_tile = L.rpt;
    out->n_tiles = L.ntiles; out->max_row_nnz = L.max_row_nnz;
    out->max_tile_segments = L.max_segs; out->max_tile_elems = L.max_elems;
    out->consumer_threads = L.nct;
    out->rows_reordered = (L.staged && L.reordered) ? 1 : 0;
    out->packed_rows = (L.staged && L.packed) ? 1 : 0;
    out->sum_tile_elems = L.sum_elems; out->touched_src = L.touched;
    out->device_bytes = L.device_bytes;
    return SMM_OK;
}

int smm_mask_sum(smm_handle *h, int32_t level, const int32_t *src_imask, int32_t *dst_imask_out,
                 int32_t *any_masked_out)
{
    int rc = check_level(h, level);
    if (rc) return rc;
    if (!src_imask) return fail(SMM_ERR_INVALID, "null src_imask");
    DeviceGuard g(h->device);
    LevelDev &L = h->levels[level];
    CUDA_TRY(cudaDeviceSynchronize());          // the level's dst_grid_imask is rewritten: no apply may be in flight
    int32_t *d_src = nullptr, *d_flag = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_src), static_cast<size_t>(L.n_src) * sizeof(int32_t)));
    cudaError_t e = cudaMalloc(reinterpret_cast<void **>(&d_flag), sizeof(int32_t));
    if (e != cudaSuccess) { cudaFree(d_src); return fail(SMM_ERR_ALLOC, cudaGetErrorString(e)); }
    e = cudaMemcpy(d_src, src_imask, static_cast<size_t>(L.n_src) * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(d_flag, 0, sizeof(int32_t));
    if (e == cudaSuccess) {
        const int threads = 256;
        const unsigned blocks = static_cast<unsigned>((L.n_dst + threads - 1) / threads);
        mask_sum_kernel<<<blocks, threads>>>(L.rowptr, L.col, L.val, d_src, L.imask, d_flag, L.n_dst);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        e = cudaGetLastError();
    }
    int32_t flag = 0;
    if (e == cudaSuccess) e = cudaMemcpy(&flag, d_flag, sizeof(int32_t), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && dst_imask_out)
        e = cudaMemcpy(dst_imask_out, L.imask, static_cast<size_t>(L.n_dst) * sizeof(int32_t),
                       cudaMemcpyDeviceToHost);
    cudaFree(d_src); cudaFree(d_flag);
    if (e != cudaSuccess) return fail(SMM_ERR_CUDA, std::string("smm_mask_sum: ") + cudaGetErrorString(e));
    L.has_imask = true;
    if (any_masked_out) *any_masked_out = flag;
    return SMM_OK;
}

int smm_nan_variation(const void *x, int32_t x_dtype, int64_t outer, int64_t n_axis, int64_t inner,
                      int64_t *count_out, smm_stream_t stream)
{
    if (!count_out) return fail(SMM_ERR_INVALID, "null count_out");
    *count_out = 0;
    if (x_dtype != SMM_F32 && x_dtype != SMM_F64) return fail(SMM_ERR_DTYPE, "x_dtype must be SMM_F32 or SMM_F64");
    if (outer < 0 || n_axis < 0 || inner < 0) return fail(SMM_ERR_INVALID, "negative extent");
    const int64_t npos = outer * inner;
    if (npos == 0 || n_axis < 2) return SMM_OK;
    if (!x) return fail(SMM_ERR_INVALID, "null x");
    if ((npos + 255) / 256 > INT32_MAX) return fail(SMM_ERR_INVALID, "too many positions for one launch");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    unsigned long long *d_count = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_count), sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), st);
    if (e == cudaSuccess) {
        const unsigned grid = static_cast<unsigned>((npos + 255) / 256);
        if (x_dtype == SMM_F32)
            nan_variation_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float *>(x), outer, n_axis, inner, d_count);
        else
            nan_variation_kernel<double><<<grid, 256, 0, st>>>(static_cast<const double *>(x), outer, n_axis, inner, d_count);
        e = cudaGetLastError();
        if (e == cudaSuccess) g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    unsigned long long host = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&host, d_count, sizeof(host), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_count);
    if (e != cudaSuccess) return fail(SMM_ERR_CUDA, std::string("smm_nan_variation: ") + cudaGetErrorString(e));
    *count_out = static_cast<int64_t>(host);
    return SMM_OK;
}

int smm_set_dst_mask(smm_handle *h, int32_t level, const int32_t *dst_grid_imask, const double *dst_grid_frac)
{
    int rc = check_level(h, level);
    if (rc) return rc;
    DeviceGuard g(h->device);
    LevelDev &L = h->levels[level];
    // applies run on non-blocking streams, which the synchronous copies below do not order against
    CUDA_TRY(cudaDeviceSynchronize());
    if (dst_grid_imask) {
        CUDA_TRY(cudaMemcpy(L.imask, dst_grid_imask, static_cast<size_t>(L.n_dst) * sizeof(int32_t),
                            cudaMemcpyHostToDevice));
        L.has_imask = true;
    }
    if (dst_grid_frac) {
        CUDA_TRY(cudaMemcpy(L.frac, dst_grid_frac, static_cast<size_t>(L.n_dst) * sizeof(double),
                            cudaMemcpyHostToDevice));
        L.has_frac = true;
    }
    return SMM_OK;
}

int smm_apply(const smm_handle *h, int32_t level, const void *x, int32_t x_dtype, int64_t B,
              int64_t ldx, void *y, int32_t y_dtype, int64_t ldy, int32_t masked,
              double remap_area_min, const smm_apply_opts *opts, smm_stream_t stream)
{
    ApplyOpts opt;
    bool empty;
    int rc = check_level(h, level);
    if (rc || (rc = check_apply(x_dtype, y_dtype, opts, B, nullptr, remap_area_min, opt, empty)) || empty) return rc;
    const LevelDev &L = h->levels[level];
    if (!x || !y) return fail(SMM_ERR_INVALID, "null x or y");
    if (ldx < L.n_src || ldy < L.n_dst) return fail(SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst");
    if ((rc = check_dst_arrays(h, level, masked, remap_area_min))) return rc;
    DeviceGuard g(h->device);
    std::vector<JobSpec> specs{JobSpec{level, x, y, masked ? 1 : 0}};
    return launch_jobs(h, specs, x_dtype, y_dtype, B, ldx, ldy, remap_area_min, opt,
                       static_cast<cudaStream_t>(stream));
}

int smm_apply_levels(const smm_handle *h, int32_t n_sel, const int32_t *level_index, const void *x,
                     int32_t x_dtype, int64_t B, int64_t x_batch_stride, int64_t x_level_stride,
                     void *y, int32_t y_dtype, int64_t y_batch_stride, int64_t y_level_stride,
                     const uint8_t *masked, double remap_area_min, const smm_apply_opts *opts,
                     smm_stream_t stream)
{
    if (!h) return fail(SMM_ERR_INVALID, "null handle");
    ApplyOpts opt;
    bool empty;
    int rc = check_apply(x_dtype, y_dtype, opts, B, &n_sel, remap_area_min, opt, empty);
    if (rc || empty) return rc;
    if (!level_index || !x || !y) return fail(SMM_ERR_INVALID, "null level_index, x or y");
    const size_t sx = x_elem_bytes(x_dtype), sy = y_dtype == SMM_F32 ? 4 : 8;
    std::vector<JobSpec> specs;
    specs.reserve(static_cast<size_t>(n_sel));
    for (int32_t i = 0; i < n_sel; ++i) {
        JobSpec s;
        s.level = level_index[i];
        s.x = static_cast<const char *>(x) + static_cast<int64_t>(i) * x_level_stride * static_cast<int64_t>(sx);
        s.y = static_cast<char *>(y) + static_cast<int64_t>(i) * y_level_stride * static_cast<int64_t>(sy);
        s.masked = masked ? (masked[i] ? 1 : 0) : 0;
        s.x_off = static_cast<int64_t>(i) * x_level_stride;
        if ((rc = check_level(h, s.level)) || (rc = check_dst_arrays(h, s.level, s.masked, remap_area_min))) return rc;
        specs.push_back(s);
    }
    DeviceGuard g(h->device);
    return launch_jobs(h, specs, x_dtype, y_dtype, B, x_batch_stride, y_batch_stride, remap_area_min, opt,
                       static_cast<cudaStream_t>(stream));
}

int smm_apply_host(const smm_handle *hc, int32_t level, const void *x, int32_t x_dtype, int64_t B,
                   int64_t ldx, void *y, int32_t y_dtype, int64_t ldy, int32_t masked,
                   double remap_area_min, const smm_apply_opts *opts, int64_t chunk_rows)
{
    ApplyOpts opt;
    bool empty;
    int rc = check_level(hc, level);
    if (rc || (rc = check_apply(x_dtype, y_dtype, opts, B, nullptr, remap_area_min, opt, empty)) || empty) return rc;
    if (!x || !y) return fail(SMM_ERR_INVALID, "null x or y");
    smm_handle *h = const_cast<smm_handle *>(hc);
    const LevelDev &L = h->levels[level];
    if (ldx < L.n_src || ldy < L.n_dst) return fail(SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst");
    if ((rc = check_dst_arrays(h, level, masked, remap_area_min))) return rc;
    const size_t sx = x_elem_bytes(x_dtype), sy = y_dtype == SMM_F32 ? 4 : 8;
    return host_pipeline(h, x, L.n_src * sx, ldx * sx, y, L.n_dst * sy, ldy * sy, B, chunk_rows,
                         [&](void *dx, void *dy, int64_t nb, cudaStream_t st) -> int {
                             std::vector<JobSpec> specs{JobSpec{level, dx, dy, masked ? 1 : 0}};
                             return launch_jobs(h, specs, x_dtype, y_dtype, nb, L.n_src, L.n_dst, remap_area_min, opt, st);
                         });
}

int smm_apply_levels_host(const smm_handle *hc, int32_t n_sel, const int32_t *level_index, const void *x,
                          int32_t x_dtype, int64_t B, void *y, int32_t y_dtype, const uint8_t *masked,
                          double remap_area_min, const smm_apply_opts *opts, int64_t chunk_rows)
{
    if (!hc) return fail(SMM_ERR_INVALID, "null handle");
    ApplyOpts opt;
    bool empty;
    int rc = check_apply(x_dtype, y_dtype, opts, B, &n_sel, remap_area_min, opt, empty);
    if (rc || empty) return rc;
    if (!level_index || !x || !y) return fail(SMM_ERR_INVALID, "null level_index, x or y");
    for (int32_t i = 0; i < n_sel; ++i)
        if ((rc = check_level(hc, level_index[i])) || (rc = check_dst_arrays(hc, level_index[i], masked && masked[i], remap_area_min)))
            return rc;
    smm_handle *h = const_cast<smm_handle *>(hc);
    const int64_t n_src = h->levels[0].n_src, n_dst = h->levels[0].n_dst;
    const size_t sx = x_elem_bytes(x_dtype), sy = y_dtype == SMM_F32 ? 4 : 8;
    const size_t row_x = static_cast<size_t>(n_sel) * n_src * sx, row_y = static_cast<size_t>(n_sel) * n_dst * sy;
    return host_pipeline(h, x, row_x, row_x, y, row_y, row_y, B, chunk_rows,
                         [&](void *dx, void *dy, int64_t nb, cudaStream_t st) -> int {
                             std::vector<JobSpec> specs;
                             specs.reserve(static_cast<size_t>(n_sel));
                             for (int32_t i = 0; i < n_sel; ++i)
                                 specs.push_back(JobSpec{level_index[i],
                                                         static_cast<const char *>(dx) + static_cast<size_t>(i) * n_src * sx,
                                                         static_cast<char *>(dy) + static_cast<size_t>(i) * n_dst * sy,
                                                         masked ? (masked[i] ? 1 : 0) : 0, static_cast<int64_t>(i) * n_src});
                             return launch_jobs(h, specs, x_dtype, y_dtype, nb, static_cast<int64_t>(n_sel) * n_src,
                                                static_cast<int64_t>(n_sel) * n_dst, remap_area_min, opt, st);
                         });
}

// ---- host-only introspection (no device): CSR + plan exactly as smm_create builds them

struct smm_host_plan {
    HostCsr csr;
    HostPlan plan;
    bool cache_hit = false;
};

int smm_host_plan_build(int64_t n_src, int64_t n_dst, int64_t nnz, const int32_t *src_address,
                        const int32_t *dst_address, const double *remap_matrix, int32_t num_wgts,
                        int32_t index_base, const smm_create_opts *opts, smm_host_plan **out)
{
    const PlanSettings settings = plan_settings();
    if (!out) return fail(SMM_ERR_INVALID, "null output pointer");
    *out = nullptr;
    if (nnz < 0) return fail(SMM_ERR_INVALID, "smm_create: n_src, n_dst must be > 0, nnz >= 0, num_wgts >= 1");
    smm_host_plan *p = new (std::nothrow) smm_host_plan();
    if (!p) return fail(SMM_ERR_ALLOC, "host allocation failed");
    std::vector<HostCsr> csrs;
    std::vector<HostPlan> plans;
    bool ref_order = false;
    const int64_t ll = nnz;
    const int rc = build_host_operator(1, &ll, nnz, n_src, n_dst, src_address, dst_address, remap_matrix, num_wgts,
                                       index_base, opts, 148, settings, csrs, plans, ref_order, p->cache_hit);
    if (rc) { delete p; return rc; }
    p->csr = std::move(csrs[0]);
    p->plan = std::move(plans[0]);
    *out = p;
    return SMM_OK;
}

int smm_host_plan_info(const smm_host_plan *p, smm_info *out, int64_t *n_segs_out)
{
    if (!p || !out) return fail(SMM_ERR_INVALID, "null argument");
    std::memset(out, 0, sizeof(*out));
    out->n_src = p->csr.n_src; out->n_dst = p->csr.n_dst;
    out->nnz = static_cast<int64_t>(p->csr.col.size());
    out->n_levels = 1;
    out->kernel = p->plan.ok ? SMM_KERNEL_STAGED : SMM_KERNEL_GATHER;
    out->lanes_per_row = p->plan.lpr; out->links_per_lane = p->plan.kpl;
    out->rows_per_tile = p->plan.rows_per_tile;
    out->n_tiles = p->plan.ok ? static_cast<int32_t>(p->plan.tiles.size()) : 0;
    out->max_row_nnz = p->csr.max_row_nnz;
    out->max_tile_segments = p->plan.max_tile_segments;
    out->consumer_threads = p->plan.nct;
    out->rows_reordered = (p->plan.ok && p->plan.reordered) ? 1 : 0;
    out->packed_rows = (p->plan.ok && p->plan.packed) ? 1 : 0;
    out->summation = p->plan.ref_order ? SMM_SUM_REFERENCE : SMM_SUM_FAST;
    out->plan_cache_hit = p->cache_hit ? 1 : 0;
    out->gather_rows = p->plan.ok ? static_cast<int32_t>(p->plan.gather_rows.size()) : 0;
    out->max_tile_elems = p->plan.max_tile_elems;
    out->sum_tile_elems = p->plan.sum_tile_elems;
    out->touched_src = p->csr.touched_src;
    if (n_segs_out) *n_segs_out = p->plan.ok ? static_cast<int64_t>(p->plan.segs.size()) : 0;
    return SMM_OK;
}

int smm_host_plan_copy(const smm_host_plan *p, int32_t *rowptr, int32_t *col, double *val,
                       int32_t *tiles, uint32_t *segs, double *wplan, uint16_t *iplan)
{
    if (!p) return fail(SMM_ERR_INVALID, "null plan");
    auto cp = [](void *dst, const void *src, size_t n) { if (dst && n) std::memcpy(dst, src, n); };
    cp(rowptr, p->csr.rowptr.data(), p->csr.rowptr.size() * sizeof(int32_t));
    cp(col, p->csr.col.data(), p->csr.col.size() * sizeof(int32_t));
    cp(val, p->csr.val.data(), p->csr.val.size() * sizeof(double));
    if (p->plan.ok) {
        static_assert(sizeof(TileDesc) == 32 && sizeof(Seg) == 16, "layout is part of the ABI");
        cp(tiles, p->plan.tiles.data(), p->plan.tiles.size() * sizeof(TileDesc));
        cp(segs, p->plan.segs.data(), p->plan.segs.size() * sizeof(Seg));
        cp(wplan, p->plan.wplan.data(), p->plan.wplan.size() * sizeof(double));
        cp(iplan, p->plan.iplan.data(), p->plan.iplan.size() * sizeof(uint16_t));
    }
    return SMM_OK;
}

int smm_host_plan_rowmap(const smm_host_plan *p, int32_t *rowmap)
{
    if (!p || !rowmap) return fail(SMM_ERR_INVALID, "null argument");
    if (p->plan.ok && !p->plan.rowmap.empty()) std::memcpy(rowmap, p->plan.rowmap.data(), p->plan.rowmap.size() * sizeof(int32_t));
    return SMM_OK;
}

int smm_host_plan_gather_rows(const smm_host_plan *p, int32_t *rows)
{
    if (!p || !rows) return fail(SMM_ERR_INVALID, "null argument");
    if (p->plan.ok && !p->plan.gather_rows.empty())
        std::memcpy(rows, p->plan.gather_rows.data(), p->plan.gather_rows.size() * sizeof(int32_t));
    return SMM_OK;
}

int smm_host_plan_rowslot(const smm_host_plan *p, int32_t *rowslot)
{
    if (!p || !rowslot) return fail(SMM_ERR_INVALID, "null argument");
    if (p->plan.ok && !p->plan.rowslot.empty()) std::memcpy(rowslot, p->plan.rowslot.data(), p->plan.rowslot.size() * sizeof(int32_t));
    return SMM_OK;
}

int smm_host_plan_compact(const smm_host_plan *p, int64_t *n_touched_out, int64_t *n_blocks_out,
                          int32_t *tcols, int32_t *blk_ptr, int32_t *rcol)
{
    if (!p) return fail(SMM_ERR_INVALID, "null plan");
    CompactPlan cp;
    build_compact(p->csr, kCompactW, cp);
    if (n_touched_out) *n_touched_out = static_cast<int64_t>(cp.tcols.size());
    if (n_blocks_out) *n_blocks_out = static_cast<int64_t>(cp.blk_ptr.size()) - 1;
    auto cpv = [](int32_t *dst, const std::vector<int32_t> &v) { if (dst && !v.empty()) std::memcpy(dst, v.data(), v.size() * sizeof(int32_t)); };
    cpv(tcols, cp.tcols); cpv(blk_ptr, cp.blk_ptr); cpv(rcol, cp.rcol);
    return SMM_OK;
}

void smm_host_plan_free(smm_host_plan *p) { delete p; }

int smm_copy_ceiling(int32_t device, void *host, int64_t bytes, int32_t direction, int32_t reps,
                     double *seconds_out)
{
    if (!host || bytes <= 0 || reps < 1 || !seconds_out || (direction != 0 && direction != 1))
        return fail(SMM_ERR_INVALID, "smm_copy_ceiling: host buffer, bytes > 0, reps >= 1, direction 0|1 required");
    if (!is_pinned(host)) return fail(SMM_ERR_INVALID, "smm_copy_ceiling: the host buffer must be pinned");
    DeviceGuard g(device);
    void *d = nullptr;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CUDA_TRY(cudaMalloc(&d, static_cast<size_t>(bytes)));
    cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    const cudaMemcpyKind kind = direction == 0 ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost;
    void *dst = direction == 0 ? d : host;
    const void *src = direction == 0 ? host : d;
    if (e == cudaSuccess) e = cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), kind, st);      // warm-up
    if (e == cudaSuccess) e = cudaEventRecord(e0, st);
    for (int32_t r = 0; r < reps && e == cudaSuccess; ++r) e = cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), kind, st);
    if (e == cudaSuccess) e = cudaEventRecord(e1, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    float ms = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (st) cudaStreamDestroy(st);
    cudaFree(d);
    if (e != cudaSuccess) return fail(SMM_ERR_CUDA, std::string("smm_copy_ceiling: ") + cudaGetErrorString(e));
    *seconds_out = 1e-3 * static_cast<double>(ms) / reps;
    return SMM_OK;
}

int64_t smm_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

const char *smm_last_error(void) { return g_err.c_str(); }

const char *smm_version(void) { return "smmregrid_b200 0.2.0 (sm_100a)"; }

}  // extern "C"
