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
#include <thread>
#include <vector>

#include <sched.h>
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

constexpr int kHostSlots = 4;

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
    int32_t lpr = 0, kpl = 0, nct = 256;
};

PlanChoice choose_plan(const std::vector<HostCsr> &csrs, int64_t n_dst, int sm_count, bool ref_order)
{
    PlanChoice pc;
    int32_t max_row = 0;
    int64_t pslots = 0;
    for (const HostCsr &c : csrs) {
        max_row = std::max(max_row, c.max_row_nnz);
        const int64_t ps = packed_slots(c);
        pslots = (ps < 0 || pslots < 0) ? -1 : pslots + ps;
    }
    pc.cfg = choose_lanes(max_row, pc.lpr, pc.kpl);
    const int64_t nlev = static_cast<int64_t>(std::max<size_t>(csrs.size(), 1));
    pc.packed = pc.cfg && prefer_packed(pslots);
    // packed plans: always 256 consumer threads, two CTAs per SM (measured: bilinear 1440x721 ->
    // 3600x1800 +4 %, 1:1 conservative +3 %, C3 +9 % over 512); n_dst = 0 leaves only the
    // SMM_CONSUMER_THREADS override
    pc.nct = pc.packed ? default_consumer_threads(0, 1, sm_count)
                       : default_consumer_threads(n_dst, pc.cfg ? pc.lpr : 0, sm_count);
    if (ref_order) pc.nct = 256;         // reference-order kernels exist for 256 consumer threads only
    (void)nlev;
    return pc;
}

int host_threads_all()
{
    cpu_set_t set;
    return sched_getaffinity(0, sizeof(set), &set) == 0 ? std::max(1, CPU_COUNT(&set)) : 1;
}

int env_int_plan(const char *name, int dflt)
{
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
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
                 std::vector<HostPlan> &plans)
{
    PlanChoice pc = choose_plan(csrs, n_dst, sm_count, ref_order);
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
        if (const char *e = std::getenv("SMM_SPLIT")) split = rows_long > 0 && e[0] == '1';      // experiments: 0 | 1
    }
    // levels are independent: a few host threads take them in turn (75 ocean levels: ~13 s -> ~1 s)
    const int nthreads = std::max(1, std::min({host_threads_all(), 16, static_cast<int>(csrs.size())}));
    // reference-order sums for rows beyond the packed layout: a thread per row with the links in
    // shared memory (ordered_kernel) when an image of K = longest row links x R rows x 12 bytes fits
    // ~100 KB for some R in {256, 128, 64, 32}; else the lane-by-lane chain of staged_kernel<ORD>
    int32_t ord_k = 0, ord_rows = 0;
    if (ref_order && pc.cfg && !pc.packed && env_int_plan("SMM_ORDLONG", 1) != 0) {
        for (const HostCsr &c : csrs) ord_k = std::max(ord_k, c.max_row_nnz);
        for (int32_t r : {256, 128, 64, 32})
            if (ord_rows == 0 && static_cast<int64_t>(ord_k) * r * 12 <= 100 * 1024) ord_rows = r;
        if (const int forced = env_int_plan("SMM_ORD_ROWS", 0)) ord_rows = forced;
    }
    enum Mode { kSplit, kPacked, kOrdLong, kLanes };
    std::vector<Mode> modes;
    if (split) modes.push_back(kSplit);
    if (pc.packed) modes.push_back(kPacked);
    if (ord_rows > 0) modes.push_back(kOrdLong);
    modes.push_back(kLanes);
    for (Mode mode : modes) {
        const int32_t nct = mode == kOrdLong ? ord_rows
                            : mode == kLanes ? (ref_order ? 256 : default_consumer_threads(n_dst, pc.cfg ? pc.lpr : 0, sm_count))
                                             : (ref_order ? 256 : default_consumer_threads(0, 1, sm_count));
        std::atomic<size_t> next{0};
        std::atomic<bool> retry{false};
        auto work = [&]() {
            for (size_t i = next.fetch_add(1); i < csrs.size() && !retry.load(); i = next.fetch_add(1)) {
                plans[i] = HostPlan{};
                plans[i].ref_order = ref_order;
                if (!pc.cfg) { plans[i].why = "a destination row has more than 512 links"; continue; }
                if (mode == kSplit) {
                    std::vector<int32_t> lrows, srows;
                    long_rows(csrs[i], lrows, srows);
                    build_plan(csrs[i], -1, pc.kpl, nct, ref_order, plans[i], &srows);
                    plans[i].gather_rows = std::move(lrows);
                    if (!plans[i].ok) retry.store(true);           // any failure: the whole set takes the next layout
                } else if (mode == kOrdLong) {
                    build_plan(csrs[i], 1, ord_k, nct, true, plans[i]);
                    plans[i].ordlong = plans[i].ok;
                    if (!plans[i].ok && !csrs[i].col.empty()) retry.store(true);
                } else {
                    build_plan(csrs[i], mode == kPacked ? -1 : pc.lpr, pc.kpl, nct, ref_order, plans[i]);
                    // only a footprint that is too large can be cured by smaller tiles
                    if (mode == kPacked && !plans[i].ok && plans[i].why.rfind("tile footprint", 0) == 0) retry.store(true);
                }
            }
        };
        if (nthreads == 1) {
            work();
        } else {
            std::vector<std::thread> pool;
            for (int t = 0; t < nthreads; ++t) pool.emplace_back(work);
            for (auto &th : pool) th.join();
        }
        if (!retry.load()) return;
    }
}

// SMM_SUM_AUTO: reference order when some weight is negative (the products of a row can cancel)
bool resolve_ref_order(int32_t summation, const std::vector<HostCsr> &csrs)
{
    if (const char *e = std::getenv("SMM_SUMMATION")) {          // experiments: fast | reference
        if (e[0] == 'f') return false;
        if (e[0] == 'r') return true;
    }
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
                        std::vector<HostCsr> &csrs, std::vector<HostPlan> &plans, bool &ref_order, bool &cache_hit)
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
                                   remap_matrix, num_wgts, index_base, summation, sm_count);
        cache_hit = plan_cache_load(cache_dir, cache_key, n_levels, n_src, n_dst, csrs, plans, ref_order);
        if (cache_hit) return SMM_OK;
        csrs.assign(static_cast<size_t>(n_levels), HostCsr{});
    }
    {
        // levels are independent: built by a few host threads; the first failing level is reported
        std::vector<int> rcs(static_cast<size_t>(n_levels), SMM_OK);
        std::vector<std::string> errs(static_cast<size_t>(n_levels));
        std::atomic<int32_t> next{0};
        auto work = [&]() {
            for (int32_t i = next.fetch_add(1); i < n_levels; i = next.fetch_add(1)) {
                const int64_t o = static_cast<int64_t>(i) * nl_max;
                rcs[i] = build_csr(n_src, n_dst, link_length[i], src_address ? src_address + o : nullptr,
                                   dst_address ? dst_address + o : nullptr,
                                   remap_matrix ? remap_matrix + o * num_wgts : nullptr, num_wgts, index_base,
                                   csrs[i], errs[i]);
            }
        };
        const int nthreads = std::max(1, std::min({host_threads_all(), 16, static_cast<int>(n_levels)}));
        if (nthreads == 1) {
            work();
        } else {
            std::vector<std::thread> pool;
            for (int t = 0; t < nthreads; ++t) pool.emplace_back(work);
            for (auto &th : pool) th.join();
        }
        for (int32_t i = 0; i < n_levels; ++i)
            if (rcs[i]) return fail(rcs[i], (n_levels > 1 ? "level " + std::to_string(i) + ": " : "") + errs[i]);
    }
    ref_order = resolve_ref_order(summation, csrs);
    plan_levels(csrs, n_dst, sm_count, ref_order, plans);
    if (use_cache) plan_cache_store(cache_dir, cache_key, csrs, plans, ref_order);   // best effort
    return SMM_OK;
}

// ------------------------------------------------------------------ launch dispatch

int env_int(const char *name, int dflt)
{
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
}

// (packed 16-bit x: the element type follows the decoded dtype, opt.dec_dtype)
#define SMM_DTYPE_DISPATCH(FN, ...)                                                                           \
    ((x_dtype == SMM_I16)                                                                                     \
         ? ((opt.dec_dtype == SMM_F32)                                                                        \
                ? (y_dtype == SMM_F32 ? FN<I16F32, float>(__VA_ARGS__) : FN<I16F32, double>(__VA_ARGS__))     \
                : (y_dtype == SMM_F32 ? FN<I16F64, float>(__VA_ARGS__) : FN<I16F64, double>(__VA_ARGS__)))    \
     : (x_dtype == SMM_F32 && y_dtype == SMM_F32) ? FN<float, float>(__VA_ARGS__)                             \
     : (x_dtype == SMM_F32 && y_dtype == SMM_F64) ? FN<float, double>(__VA_ARGS__)                            \
     : (x_dtype == SMM_F64 && y_dtype == SMM_F32) ? FN<double, float>(__VA_ARGS__)                            \
                                                  : FN<double, double>(__VA_ARGS__))

// bytes of one x element as it sits in memory (SMM_I16: the raw 16 bits)
size_t x_elem_bytes(int32_t x_dtype) { return x_dtype == SMM_I16 ? 2 : x_dtype == SMM_F32 ? 4 : 8; }

// Batch rows per work item.  A work item pays a fixed prologue (its tile's register image,
// barriers: `prologue_us`) and the launch pays about half an item of tail per wave, so with an
// estimated launch time T the cost is minimal near sqrt(T / (2 * prologue)) waves.  (Measured
// on B200: the former fixed ~32-wave target cost 8-12 % at 64-512 batch rows on C2.)
// `slots` = CTAs resident on the device, `bytes_per_row` = HBM bytes one batch row moves.
int64_t pick_chunks(int64_t B, int64_t blocks_total, int64_t slots, double bytes_per_row, double prologue_us,
                    int64_t multiple, int64_t &chunk)
{
    static const int k_min_rows = std::max(1, env_int("SMM_MIN_ROWS_PER_ITEM", 8));
    static const int k_waves = env_int("SMM_WAVES", 0);                    // experiments: fixed wave count
    const double t_us = static_cast<double>(B) * bytes_per_row / 6.5e6;     // at ~6.5 TB/s
    double waves = k_waves > 0 ? k_waves : std::sqrt(t_us / (2.0 * prologue_us));
    waves = std::min(32.0, std::max(1.0, waves));
    const double items = waves * static_cast<double>(slots);
    int64_t nchunks = static_cast<int64_t>(items / static_cast<double>(std::max<int64_t>(blocks_total, 1)) + 0.5);
    const int64_t max_chunks = std::max<int64_t>(1, B / k_min_rows);
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

// Two-pass apply of one gather-family level (see compact_kernel).  The transposed buffer XT comes
// from the handle's stream-ordered pool, so concurrent applies on other streams stay independent.
int launch_compact(const smm_handle *h, const LevelDev &L, const JobSpec &sp, int32_t x_dtype, int32_t y_dtype,
                   int64_t B, int64_t xbs, int64_t ybs, double area_min, const ApplyOpts &opt, cudaStream_t st)
{
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
                return kCompactUnavailable;          // no stream-ordered pools here: direct gathers instead
            }
        }
    }
    void *xt = nullptr;
    const size_t sx = x_elem_bytes(x_dtype);
    const size_t xt_bytes = std::max<size_t>(static_cast<size_t>(L.touched), 1) * kCompactBC * sx;
    if (cudaMallocFromPoolAsync(&xt, xt_bytes, h->pool, st) != cudaSuccess) {
        cudaGetLastError();
        return kCompactUnavailable;                  // not enough memory for the transposed buffer
    }
    const int rc = SMM_DTYPE_DISPATCH(launch_compact_t, h->device, L, sp, xt, B, xbs, ybs, area_min, opt.dec, st);
    cudaFreeAsync(xt, st);
    return rc;
}

int launch_jobs(const smm_handle *h, const std::vector<JobSpec> &specs, int32_t x_dtype,
                int32_t y_dtype, int64_t B, int64_t xbs, int64_t ybs, double area_min,
                const ApplyOpts &opt, cudaStream_t st)
{
    if (B == 0 || specs.empty()) return SMM_OK;
    const size_t sx = x_elem_bytes(x_dtype);
    const bool ord = h->ref_order;
    // shared memory a staged launch needs for `nstages` stages of one batch row each (`image` = the
    // link image of ordered-long plans: kpl x nct x (8 + 4) bytes)
    auto image_bytes = [](const LevelDev &L) -> size_t {
        return L.ordlong ? round_up(static_cast<size_t>(L.kpl) * L.nct * 12, 128) : 0;
    };
    auto staged_smem = [&](size_t max_segs, size_t max_elems, size_t nstages, size_t image = 0) {
        return kSmemHeader + round_up(max_segs * sizeof(Seg), 128) + image + nstages * round_up(max_elems * sx, 128);
    };
    std::vector<JobSpec> staged, gather, gather_lists;      // gather_lists: the long rows of split plans
    for (const JobSpec &s : specs) {
        const LevelDev &L = h->levels[s.level];
        if (s.masked && !L.has_imask)
            return fail(SMM_ERR_INVALID, "masked apply but dst_grid_imask was never set for level " +
                                             std::to_string(s.level));
        if (area_min > 0.0 && !L.has_frac)
            return fail(SMM_ERR_INVALID, "remap_area_min > 0 but dst_grid_frac was never set for level " +
                                             std::to_string(s.level));
        bool ok = L.staged && opt.kernel != SMM_KERNEL_GATHER;
        // the renormalising extension is not implemented for packed-rows and ordered-long plans: gather kernel
        ok = ok && !((L.packed || L.ordlong) && opt.renorm_min_valid >= 0.0);
        // TMA bulk copies need 16-byte aligned rows and lengths
        ok = ok && (reinterpret_cast<uintptr_t>(s.x) % 16 == 0) && ((xbs * sx) % 16 == 0) &&
             ((L.n_src * sx) % 16 == 0);
        // at least two stages must fit
        ok = ok && staged_smem(L.max_segs, L.max_elems, 2, image_bytes(L)) <= h->smem_optin;
        if (!ok && opt.kernel == SMM_KERNEL_STAGED)
            return fail(SMM_ERR_INVALID, "staged kernel forced but unavailable for level " +
                                             std::to_string(s.level) + ": " +
                                             (L.staged ? std::string("slab alignment / footprint size")
                                                       : L.why_not_staged));
        (ok ? staged : gather).push_back(s);
        if (ok && L.n_gather_rows > 0) gather_lists.push_back(s);
    }

    ApplyArgs a{};
    a.B = B; a.x_bstride = xbs; a.y_bstride = ybs; a.remap_area_min = area_min;
    a.renorm_min_valid = opt.renorm_min_valid;
    a.dec = opt.dec;
    // experiment switches are read once per process, not per launch
    static const uint32_t k_debug_flags = static_cast<uint32_t>(env_int("SMM_DEBUG_STREAM_ONLY", 0)) & 3u;
    static const int k_max_stages = std::max(2, env_int("SMM_MAX_STAGES", kMaxStages));
    a.debug_flags = k_debug_flags;   // bit 0: staged consumers skip the arithmetic (profiling aid)

    auto fill_job = [&](const JobSpec &s, LevelJob &j) {
        const LevelDev &L = h->levels[s.level];
        j.tiles = L.tiles; j.segs = L.segs; j.wplan = L.wplan; j.iplan = L.iplan; j.rowmap = L.rowmap;
        j.rowptr = L.rowptr; j.col = L.col; j.val = L.val;
        j.imask = L.imask; j.frac = L.frac;
        j.x = s.x; j.y = s.y; j.masked = s.masked; j.nrows = 0;
    };

    // ---- staged launches: up to kMaxJobs levels at a time (balanced when there are more), and a
    // group is closed early when the segment table of one level and the footprint of another would
    // not fit two stages TOGETHER (each level fits on its own, see above)
    const size_t staged_groups = (staged.size() + kMaxJobs - 1) / kMaxJobs;
    const size_t staged_per = staged_groups ? (staged.size() + staged_groups - 1) / staged_groups : 1;   // balanced
    for (size_t g0 = 0; g0 < staged.size();) {
        size_t g1 = g0;
        JobBatch jb{};
        int64_t tiles_total = 0;
        size_t max_segs = 0, max_elems = 0;
        int lpr = 0, kpl = 0, nct = 256;
        bool packed = false, ordl = false;
        size_t image = 0;
        for (; g1 < staged.size() && g1 - g0 < staged_per; ++g1) {
            const LevelDev &L = h->levels[staged[g1].level];
            const size_t ms = std::max<size_t>(max_segs, L.max_segs), me = std::max<size_t>(max_elems, L.max_elems);
            if (g1 > g0 && staged_smem(ms, me, 2, image_bytes(L)) > h->smem_optin) break;
            max_segs = ms; max_elems = me;
            tiles_total += L.ntiles;
            lpr = L.lpr; kpl = L.kpl; nct = L.nct; packed = L.packed; ordl = L.ordlong;
            image = image_bytes(L);
            a.n_src = L.n_src; a.n_dst = L.n_dst;
        }
        const size_t segs_off = kSmemHeader + round_up(max_segs * sizeof(Seg), 128);
        const size_t stage_off = segs_off + image;
        a.ord_k = kpl;
        a.wimg_off = static_cast<uint32_t>(segs_off);
        a.oimg_off = static_cast<uint32_t>(segs_off + static_cast<size_t>(kpl) * nct * 8);
        const size_t row_bytes = std::max<size_t>(128, round_up(max_elems * sx, 128));
        // stage several batch rows together (up to 8, ~56 KB per stage) so that the per-stage
        // barrier and loop overhead of the consumers is amortised: C3 2156 -> 2671 GB/s, C2 5565 -> 6111
        static const int k_rows_per_stage = env_int("SMM_ROWS_PER_STAGE", 0);
        int nb_rows = k_rows_per_stage > 0 ? k_rows_per_stage : static_cast<int>((56u << 10) / row_bytes);
        const size_t half = (228u * 1024u - 2u * 1024u) / 2u - 1024u;   // two CTAs per SM (NCT = 256)
        {   // ...but never at the price of pipeline depth (>= 4 stages) or of the second CTA per SM
            const size_t budget = (nct == 256 ? half : h->smem_optin) - std::min(stage_off, half);
            nb_rows = static_cast<int>(std::min<size_t>(nb_rows, std::max<size_t>(1, budget / (4 * row_bytes))));
        }
        nb_rows = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>({nb_rows, 8, B})));
        if (ordl) {     // ordered kernel: one CTA per SM, batch rows chained in pairs: an even number of rows
                        // per stage, as many as leave three stages
            nb_rows = (B >= 2 && stage_off + 4 * row_bytes <= h->smem_optin) ? 2 : 1;
            while (nb_rows >= 2 && nb_rows + 2 <= 8 && nb_rows + 2 <= B &&
                   stage_off + 3 * static_cast<size_t>(nb_rows + 2) * row_bytes <= h->smem_optin)
                nb_rows += 2;
        }
        const size_t stage_bytes = row_bytes * nb_rows;
        int64_t chunk = 0;             // batch rows per work item: whole stages
        const double row_bytes_hbm = static_cast<double>(g1 - g0) *
                                     (static_cast<double>(a.n_src) * sx + static_cast<double>(a.n_dst) * (y_dtype == SMM_F32 ? 4 : 8));
        const int ctas_per_sm = (!ordl && nct == 256) ? 2 : 1;
        const int64_t nchunks = pick_chunks(B, tiles_total, static_cast<int64_t>(h->sm_count) * ctas_per_sm,
                                            row_bytes_hbm, ordl ? 6.0 : (nct == 256 ? 2.5 : 4.0), nb_rows, chunk);
        a.chunk = chunk; a.nchunks = static_cast<int32_t>(nchunks);
        size_t S = (!ordl && nct == 256 && half > stage_off) ? (half - stage_off) / stage_bytes : 0;
        if (S < 3) S = (h->smem_optin - stage_off) / stage_bytes;        // one CTA per SM
        S = std::min<size_t>(S, kMaxStages);
        S = std::min<size_t>(S, static_cast<size_t>(k_max_stages));
        if (S < 2) return fail(SMM_ERR_INVALID, "internal: staged footprint does not fit");
        a.nstages = static_cast<int32_t>(S);
        a.stage_bytes = static_cast<uint32_t>(stage_bytes);
        a.row_bytes = static_cast<uint32_t>(row_bytes);
        a.rows_per_stage = nb_rows;
        a.stage_off = static_cast<uint32_t>(stage_off);
        const size_t smem = stage_off + S * stage_bytes;
        // grid: x = tile, y = batch chunk, z = level of the group (blocks beyond a level's tile
        // count exit at once).  No index arithmetic in the kernel: what steers its batch loop stays
        // in uniform registers.
        int64_t max_tiles = 0;
        jb.njobs = static_cast<int32_t>(g1 - g0);
        for (size_t g = g0; g < g1; ++g) {
            LevelJob &j = jb.jobs[g - g0];
            fill_job(staged[g], j);
            j.nblocks = h->levels[staged[g].level].ntiles;
            j.item0 = 0;
            max_tiles = std::max<int64_t>(max_tiles, j.nblocks);
        }
        g0 = g1;
        if (max_tiles == 0) continue;
        const dim3 grid(static_cast<unsigned>(max_tiles), static_cast<unsigned>(nchunks), static_cast<unsigned>(jb.njobs));
        // two threads per row (one per batch row of a pair) while that leaves at most 8 consumer warps:
        // C4 (64 rows per tile) 3060 -> 3989 GB/s, C2 (256 rows: 16 warps re-reading the image) 4368 -> 3518
        static const int k_ord_tpr = env_int("SMM_ORD_TPR", 0);
        const int tpr = (ordl && nb_rows >= 2 && (k_ord_tpr == 2 || (k_ord_tpr == 0 && nct <= 128))) ? 2 : 1;
        const int rc = ordl ? SMM_DTYPE_DISPATCH(launch_ordered_t, h->device, nct, tpr, grid, smem, st, jb, a)
                            : SMM_DTYPE_DISPATCH(launch_staged_t, h->device, lpr, kpl, nct, packed, ord, grid, smem, st, jb, a);
        if (rc) return rc;
    }

    // ---- compact (two-pass) launches: scattered sources with enough batch rows, one level at a time
    {
        std::vector<JobSpec> plain;
        for (const JobSpec &sp : gather) {
            const LevelDev &L = h->levels[sp.level];
            // Cost per batch row in HBM-byte equivalents, calibrated on B200 (C5nn / C5dis, f32 and
            // f64): a random gather costs ~120 bytes (a 64-byte sector at about half the streaming
            // rate); the two passes move the slab (at the streaming rate: TMA bulk copies), the
            // touched columns twice-ish and the links (random 256-byte runs), together ~1.2x the
            // bytes at the streaming rate.  Runs of fewer than 16 batch values are not worth it.
            const double gather_cost = static_cast<double>(L.nnz) * 120.0;
            const double compact_cost = 1.2 * (static_cast<double>(L.n_src) + static_cast<double>(L.touched) +
                                               static_cast<double>(L.nnz)) * static_cast<double>(sx);
            bool use = L.rcol && opt.renorm_min_valid < 0.0 && opt.kernel != SMM_KERNEL_GATHER;
            if (opt.kernel != SMM_KERNEL_COMPACT) use = use && B >= 16 && gather_cost > compact_cost;
            if (!use) { plain.push_back(sp); continue; }
            const int rc = launch_compact(h, L, sp, x_dtype, y_dtype, B, xbs, ybs, area_min, opt, st);
            if (rc == kCompactUnavailable) { plain.push_back(sp); continue; }
            if (rc) return rc;
        }
        gather.swap(plain);
    }

    // ---- gather launches: whole levels, then the row lists of split plans
    for (int pass = 0; pass < 2; ++pass) {
    const std::vector<JobSpec> &list = pass == 0 ? gather : gather_lists;
    const bool lists = pass == 1;
    // reference order: one thread walks a row's links in sequence
    const int lpr = ord ? 1 : h->gather_lanes[pass];
    for (size_t g0 = 0; g0 < list.size(); g0 += kMaxJobs) {
        const size_t g1 = std::min(list.size(), g0 + kMaxJobs);
        JobBatch jb{};
        int64_t nnz = 0, rows = 0;
        for (size_t g = g0; g < g1; ++g) {
            const LevelDev &L = h->levels[list[g].level];
            nnz += lists ? L.gather_nnz : L.nnz;
            rows += lists ? L.n_gather_rows : L.n_dst;
            a.n_src = L.n_src; a.n_dst = L.n_dst;
        }
        const int rpb = kGatherThreads / lpr;
        auto rows_of = [&](const LevelDev &L) -> int64_t { return lists ? L.n_gather_rows : L.n_dst; };
        int64_t blocks_total = 0;
        for (size_t g = g0; g < g1; ++g)
            blocks_total += (rows_of(h->levels[list[g].level]) + rpb - 1) / rpb;
        int64_t chunk = 0;
        // gather kernel: up to 8 CTAs of 256 threads per SM, a light prologue, traffic dominated by the gathers
        const double row_bytes_hbm = static_cast<double>(nnz) * 64.0 + static_cast<double>(rows) * (y_dtype == SMM_F32 ? 4 : 8);
        const int64_t nchunks = pick_chunks(B, blocks_total, static_cast<int64_t>(h->sm_count) * 8, row_bytes_hbm, 1.0,
                                            kGatherBT, chunk);
        a.chunk = chunk; a.nchunks = static_cast<int32_t>(nchunks);
        a.nstages = 0; a.stage_bytes = 0; a.stage_off = 0; a.row_bytes = 0; a.rows_per_stage = 1;
        int64_t item = 0;
        jb.njobs = static_cast<int32_t>(g1 - g0);
        for (size_t g = g0; g < g1; ++g) {
            const LevelDev &L = h->levels[list[g].level];
            LevelJob &j = jb.jobs[g - g0];
            fill_job(list[g], j);
            if (lists) { j.rowmap = L.gather_rows; j.nrows = L.n_gather_rows; }
            j.nblocks = static_cast<int32_t>((rows_of(L) + rpb - 1) / rpb);
            j.item0 = static_cast<int32_t>(item);
            item += static_cast<int64_t>(j.nblocks) * nchunks;
        }
        if (item > INT32_MAX) return fail(SMM_ERR_INVALID, "too many work items in one launch");
        if (item == 0) continue;
        const dim3 grid(static_cast<unsigned>(item));
        const int rc = SMM_DTYPE_DISPATCH(launch_gather_t, lpr, ord, grid, st, jb, a);
        if (rc) return rc;
    }
    }
    return SMM_OK;
}

// true when cudaMemcpyAsync can DMA straight from/to the pointer (pinned or registered)
bool is_pinned(const void *p)
{
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

int host_threads()
{
    cpu_set_t set;
    int n = 1;
    if (sched_getaffinity(0, sizeof(set), &set) == 0) n = CPU_COUNT(&set);
    return std::max(1, std::min(n, env_int("SMM_HOST_COPY_THREADS", 12)));
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
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; ++t) {
        pool.emplace_back([=]() {
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
    for (auto &th : pool) th.join();
}

int check_dtypes(int32_t x_dtype, int32_t y_dtype)
{
    if ((x_dtype != SMM_F32 && x_dtype != SMM_F64 && x_dtype != SMM_I16) || (y_dtype != SMM_F32 && y_dtype != SMM_F64))
        return fail(SMM_ERR_DTYPE, "x_dtype must be SMM_F32 (0), SMM_F64 (1) or SMM_I16 (2), y_dtype SMM_F32 or SMM_F64");
    return SMM_OK;
}

int check_level(const smm_handle *h, int32_t level)
{
    if (!h) return fail(SMM_ERR_INVALID, "null handle");
    if (level < 0 || level >= static_cast<int32_t>(h->levels.size()))
        return fail(SMM_ERR_INVALID, "level " + std::to_string(level) + " out of range [0, " +
                                         std::to_string(h->levels.size()) + ")");
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
    static const bool k_trace = env_int("SMM_HOST_TRACE", 0) != 0;      // diagnostics: phase times on stderr
    const auto t_enter = std::chrono::steady_clock::now();
    auto ms_since = [&](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    const bool x_pinned = is_pinned(x), y_pinned = is_pinned(y);
    if (chunk_rows <= 0) {
        // ~128 MB of source per chunk for direct DMA (the fill of the pipeline -- the first chunk's
        // copy -- is the only part that does not overlap), ~64 MB when staging; at least 4 rows;
        // SMM_HOST_CHUNK_MB overrides
        const int64_t mb = std::max(1, env_int("SMM_HOST_CHUNK_MB", x_pinned ? 128 : 64));
        chunk_rows = std::max<int64_t>(4, (mb << 20) / std::max<int64_t>(1, static_cast<int64_t>(row_x)));
    }
    chunk_rows = std::min(chunk_rows, B);
    std::lock_guard<std::mutex> lock(h->host_mu);
    DeviceGuard g(h->device);
    const size_t need_x = static_cast<size_t>(chunk_rows) * row_x;
    const size_t need_y = static_cast<size_t>(chunk_rows) * row_y;
    for (cudaStream_t *sp : {&h->s_in[0], &h->s_in[1], &h->s_k, &h->s_out})
        if (!*sp) CUDA_TRY(cudaStreamCreateWithFlags(sp, cudaStreamNonBlocking));
    static const int k_in_streams = std::max(1, std::min(2, env_int("SMM_HOST_IN_STREAMS", 2)));
    static const int k_slots = std::max(2, std::min(kHostSlots, env_int("SMM_HOST_SLOTS", kHostSlots)));
    const int nslots = static_cast<int>(std::min<int64_t>(k_slots, (B + chunk_rows - 1) / chunk_rows));
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
    const int nthreads = host_threads();
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
            cudaStream_t s_in = h->s_in[ichunk % k_in_streams];
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
    if (k_trace)
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
                             num_wgts, index_base, opts, h->sm_count, csrs, plans, h->ref_order, h->cache_hit);
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
    int rc = check_level(h, level);
    if (rc) return rc;
    if ((rc = check_dtypes(x_dtype, y_dtype))) return rc;
    ApplyOpts opt;
    if ((rc = resolve_opts(opts, x_dtype, opt))) return rc;
    if (B < 0) return fail(SMM_ERR_INVALID, "B must be >= 0");
    if (B == 0) return SMM_OK;
    const LevelDev &L = h->levels[level];
    if (!x || !y) return fail(SMM_ERR_INVALID, "null x or y");
    if (ldx < L.n_src || ldy < L.n_dst) return fail(SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst");
    if (!(remap_area_min >= 0.0 && remap_area_min <= 1.0))
        return fail(SMM_ERR_INVALID, "The remap_area_min provided must be between 0.0 and 1.0");
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
    int rc;
    if ((rc = check_dtypes(x_dtype, y_dtype))) return rc;
    ApplyOpts opt;
    if ((rc = resolve_opts(opts, x_dtype, opt))) return rc;
    if (n_sel < 0 || B < 0) return fail(SMM_ERR_INVALID, "n_sel and B must be >= 0");
    if (n_sel == 0 || B == 0) return SMM_OK;
    if (!level_index || !x || !y) return fail(SMM_ERR_INVALID, "null level_index, x or y");
    if (!(remap_area_min >= 0.0 && remap_area_min <= 1.0))
        return fail(SMM_ERR_INVALID, "The remap_area_min provided must be between 0.0 and 1.0");
    const size_t sx = x_elem_bytes(x_dtype), sy = y_dtype == SMM_F32 ? 4 : 8;
    std::vector<JobSpec> specs;
    specs.reserve(static_cast<size_t>(n_sel));
    for (int32_t i = 0; i < n_sel; ++i) {
        if ((rc = check_level(h, level_index[i]))) return rc;
        JobSpec s;
        s.level = level_index[i];
        s.x = static_cast<const char *>(x) + static_cast<int64_t>(i) * x_level_stride * static_cast<int64_t>(sx);
        s.y = static_cast<char *>(y) + static_cast<int64_t>(i) * y_level_stride * static_cast<int64_t>(sy);
        s.masked = masked ? (masked[i] ? 1 : 0) : 0;
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
    int rc = check_level(hc, level);
    if (rc) return rc;
    if ((rc = check_dtypes(x_dtype, y_dtype))) return rc;
    ApplyOpts opt;
    if ((rc = resolve_opts(opts, x_dtype, opt))) return rc;
    if (B < 0) return fail(SMM_ERR_INVALID, "B must be >= 0");
    if (B == 0) return SMM_OK;
    if (!x || !y) return fail(SMM_ERR_INVALID, "null x or y");
    if (!(remap_area_min >= 0.0 && remap_area_min <= 1.0))
        return fail(SMM_ERR_INVALID, "The remap_area_min provided must be between 0.0 and 1.0");
    smm_handle *h = const_cast<smm_handle *>(hc);
    const LevelDev &L = h->levels[level];
    if (ldx < L.n_src || ldy < L.n_dst) return fail(SMM_ERR_INVALID, "ldx < n_src or ldy < n_dst");
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
    int rc;
    if ((rc = check_dtypes(x_dtype, y_dtype))) return rc;
    ApplyOpts opt;
    if ((rc = resolve_opts(opts, x_dtype, opt))) return rc;
    if (n_sel < 0 || B < 0) return fail(SMM_ERR_INVALID, "n_sel and B must be >= 0");
    if (n_sel == 0 || B == 0) return SMM_OK;
    if (!level_index || !x || !y) return fail(SMM_ERR_INVALID, "null level_index, x or y");
    if (!(remap_area_min >= 0.0 && remap_area_min <= 1.0))
        return fail(SMM_ERR_INVALID, "The remap_area_min provided must be between 0.0 and 1.0");
    for (int32_t i = 0; i < n_sel; ++i)
        if ((rc = check_level(hc, level_index[i]))) return rc;
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
                                                         masked ? (masked[i] ? 1 : 0) : 0});
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
                                       index_base, opts, 148, csrs, plans, ref_order, p->cache_hit);
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
