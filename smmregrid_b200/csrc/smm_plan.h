// smm_plan.h -- host-side construction of the device operator from CDO link arrays.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "smm_common.h"

namespace smm {

// CSR by destination row with ascending source columns and summed duplicates: the per-row
// view of what sparse.COO(coords=[src,dst], data) holds (smmregrid/weights.py:37-39).
struct HostCsr {
    int64_t n_src = 0, n_dst = 0;
    std::vector<int32_t> rowptr;   // n_dst + 1
    std::vector<int32_t> col;
    std::vector<double> val;
    int32_t max_row_nnz = 0;
    int64_t touched_src = 0;
    bool has_negative = false;     // some weight < 0: sums may cancel (bicubic, second-order conservative)
};

// Compact (two-pass) plan of a level served by the gather family: the touched source columns in
// ascending order, their range per block of `block_cols` source columns, and every link's
// column replaced by its rank among the touched columns (see compact_kernel).
struct CompactPlan {
    std::vector<int32_t> tcols;      // [touched_src]
    std::vector<int32_t> blk_ptr;    // [ceil(n_src / block_cols) + 1]
    std::vector<int32_t> rcol;       // [nnz]
};
void build_compact(const HostCsr &csr, int32_t block_cols, CompactPlan &out);

// Returns 0 on success, SMM_ERR_* otherwise (message in err).
int build_csr(int64_t n_src, int64_t n_dst, int64_t nnz, const int32_t *src_address,
              const int32_t *dst_address, const double *remap_matrix, int32_t num_wgts,
              int32_t index_base, HostCsr &out, std::string &err);

// Tile plan of the staged kernel.
struct HostPlan {
    bool ok = false;          // false: level is served by the gather kernel only
    std::string why;          // reason when !ok
    int32_t lpr = 0, kpl = 0, rows_per_tile = 0;
    int32_t nct = 0;          // consumer threads per CTA the register image is laid out for
    std::vector<TileDesc> tiles;
    std::vector<Seg> segs;
    std::vector<int32_t> rowmap;   // empty: tile t holds rows [t*R, ...); else destination row of every tile slot
    bool reordered = false;        // rows were tiled in mean-source-address order
    bool packed = false;           // packed-rows plan: one thread owns up to 4 short rows (4 link slots each)
    bool ref_order = false;        // links placed for reference-order summation (lane l, slot k = link l*kpl + k)
    bool ordlong = false;          // ref_order plan with one lane per row and kpl = the longest row, nct = rows per
                                   // tile (32..256): the image lives in shared memory (ordered_kernel)
    int64_t nrows = 0;             // destination rows this plan covers (n_dst unless it is one part of a split plan)
    // Split plans: operators whose rows are mostly short (<= 16 links) with a few long ones (the
    // fan of cells around a grid pole of a tripolar ocean grid) tile the short rows with the
    // packed layout (this plan) and leave the long rows, listed here in ascending order, to the
    // gather kernel (a second, small launch).  Empty for ordinary plans.
    std::vector<int32_t> gather_rows;
    std::vector<int32_t> rowslot;  // packed: [ntiles][4][nct] destination row of a sub-row, -1 empty, -2 continuation
    std::vector<double> wplan;     // [ntiles][kpl][nct]
    std::vector<uint16_t> iplan;   // [ntiles][kpl][nct]
    int32_t max_tile_segments = 0;
    int64_t max_tile_elems = 0;
    int64_t sum_tile_elems = 0;
    int64_t sum_tile_cols = 0;     // distinct source columns per tile, summed (the ideal footprint)
};

// Picks (lanes per row, links per lane) for a maximum row length; false if no staged
// configuration can hold it.
bool choose_lanes(int32_t max_row_nnz, int32_t &lpr, int32_t &kpl);

// force_lpr/force_kpl > 0 impose a configuration shared by all levels of a 3-D weight set.
// nct = consumer threads per CTA (256 or 512).
// The natural plan tiles consecutive destination rows.  When that is unusable (scattered
// footprints) a second plan is tried with the rows re-ordered by the mean source address of
// their links, which turns locality-preserving unstructured orderings (HEALPix nested, Morton /
// partition-ordered meshes) into compact per-tile footprints.
// force_lpr == -1 requests the packed-rows layout (see prefer_packed).
// ref_order: place the links for the reference's summation order (see staged_kernel ORD) instead of
// the bank-conflict-minimising free placement of the fast sums.
// subset (ascending row ids): tile only these rows (one part of a split plan).
void build_plan(const HostCsr &csr, int32_t force_lpr, int32_t force_kpl, int32_t nct, bool ref_order, HostPlan &plan,
                const std::vector<int32_t> *subset = nullptr);
void long_rows(const HostCsr &csr, std::vector<int32_t> &long_rows_out, std::vector<int32_t> &short_rows_out);

// Packed-rows layout (one thread owns up to 4 short rows): link slots it would spend on `csr`
// (-1: a row does not fit), and whether to use it.
int64_t packed_slots(const HostCsr &csr);
bool prefer_packed(int64_t slots_packed);

// Consumer threads per CTA for a weight set: 512 (one CTA per SM, tiles twice as long, longer TMA
// segments: +4 % on C4, +5 % on C2) when that still leaves at least one tile per SM, else 256.
// SMM_CONSUMER_THREADS=256|512 overrides.
int32_t default_consumer_threads(int64_t n_dst, int32_t lpr, int32_t sm_count);

// ---- on-disk cache of the operator construction (smm_plan_cache.cpp)
struct PlanCacheKey { uint64_t h[2] = {0, 0}; };
// hash of the link arrays (the used part of every level) and of everything else the plans depend on
PlanCacheKey plan_cache_key(int32_t n_levels, const int64_t *link_length, int64_t nl_max, int64_t n_src,
                            int64_t n_dst, const int32_t *src_address, const int32_t *dst_address,
                            const double *remap_matrix, int32_t num_wgts, int32_t index_base,
                            int32_t summation, int32_t sm_count);
// false = miss (absent, stale or damaged file): build as usual.  ref_order = the summation order of
// the weight set, stored in the file as the handle's own value
bool plan_cache_load(const std::string &dir, const PlanCacheKey &key, int32_t n_levels, int64_t n_src,
                     int64_t n_dst, std::vector<HostCsr> &csrs, std::vector<HostPlan> &plans, bool &ref_order);
bool plan_cache_store(const std::string &dir, const PlanCacheKey &key, std::vector<HostCsr> &csrs,
                      std::vector<HostPlan> &plans, bool ref_order);

}  // namespace smm
