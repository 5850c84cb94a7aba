// smm_common.h -- structures shared by the host plan builder, the kernels and the C ABI.
//
// Vocabulary (follows the reference / CDO SCRIP files): a *link* is one (src_address,
// dst_address, remap_matrix[:,0]) triple; a *level* is one weight matrix of a 3-D
// (mask_dim) weight set; a destination *row* is one dst cell; a *tile* is a run of
// consecutive destination rows whose source *footprint* (the union of the source columns
// they touch, widened to aligned *segments*) is staged in shared memory per batch row.
#pragma once
#include <cstdint>

namespace smm {

// Consumer threads per CTA (threads holding links in registers) are a plan parameter:
// 256 (two CTAs per SM) or 512 (one CTA per SM, tiles twice as long -> longer TMA segments).
// The CTA adds a warpgroup of four TMA producer warps.
constexpr int kMaxConsumerThreads = 512;
constexpr int kMaxStages = 12;
constexpr int kSegAlign = 8;                        // segment bounds: multiples of 8 elements
constexpr int kSegGap = 32;                         // merge segments closer than this
constexpr int kSmemHeader = 256;                    // full[12] + empty[12] mbarriers
constexpr int kMaxJobs = 128;                       // levels per grouped launch (by-value args, 14 KB of the 32 KB parameter space)
constexpr int kGatherThreads = 256;
constexpr int kGatherBT = 4;                        // batch rows register-blocked by the gather kernel

// compact (two-pass) path of scattered-source levels
#ifndef SMM_COMPACT_BC
#define SMM_COMPACT_BC 64
#endif
#ifndef SMM_COMPACT_W
#define SMM_COMPACT_W 256
#endif
constexpr int kCompactBC = SMM_COMPACT_BC;          // batch rows per chunk (lanes handle b and b + 32)
constexpr int kCompactW = SMM_COMPACT_W;            // source columns per pass-1 block

struct Seg {          // one aligned run of source columns, in elements
    uint32_t src;     // first source column
    uint32_t dst;     // offset inside the staged footprint
    uint32_t len;     // number of elements
    uint32_t pad;
};

struct TileDesc {
    int32_t row0;     // first destination row
    int32_t nrows;    // rows in this tile (<= rows_per_tile)
    int32_t seg0;     // first segment in the level's segment array
    int32_t nseg;
    int32_t elems;    // staged footprint, elements (= sum of segment lengths)
    int32_t pad[3];
};

// One level of a (possibly grouped) apply.  Passed by value inside JobBatch.
struct LevelJob {
    const TileDesc *tiles;
    const Seg *segs;
    const double *wplan;      // [ntiles][KPL][NCT] register image of the link weights
    const uint16_t *iplan;    // [ntiles][KPL][NCT] footprint-local element index per link
    const int32_t *rowmap;    // staged: destination row of every tile slot, or null: slot i of tile t is row t*R + i
                              // gather: the rows this job serves (nrows of them), or null: all n_dst rows
    const int32_t *rowptr;    // CSR by destination row, columns ascending (reference order)
    const int32_t *col;
    const double *val;
    const int32_t *imask;     // dst_grid_imask (used when masked)
    const double *frac;       // dst_grid_frac (used when remap_area_min > 0)
    const void *x;            // level base of the source slab
    void *y;                  // level base of the destination slab
    int32_t nblocks;          // tiles (staged) or row blocks (gather) of this level
    int32_t item0;            // first work item of this level in the launch
    int32_t masked;
    int32_t nrows;            // gather: length of the row list (0: every row of the level)
};

struct JobBatch {
    LevelJob jobs[kMaxJobs];
    int32_t njobs;
    int32_t pad;
};

// CF unpacking of 16-bit raw source values (smm_decode; read by the packed element types only).
// Raw r -> NaN if r is one of fill[] (compared on the raw 16 bits; unused slots hold -1, which no
// zero-extended 16-bit value equals), else D(D(v) * scale) + offset with v = r as int16 (sign_xor =
// 0x8000) or uint16 (sign_xor = 0), each operation rounded once in the decoded type D.
struct Decode {
    double scale, offset;       // D = float64
    float scale_f, offset_f;    // D = float32 (exactly the doubles above)
    int32_t fill[4];
    uint32_t sign_xor;
    float bias_f;               // 2^23 + (int16: 2^15 | uint16: 0), see decode16
};

struct ApplyArgs {
    int64_t B;            // batch rows per level
    int64_t x_bstride;    // elements between consecutive batch rows of x
    int64_t y_bstride;
    int64_t n_src, n_dst;
    int64_t chunk;        // batch rows per work item
    int32_t nchunks;
    int32_t nstages;
    uint32_t stage_bytes; // bytes reserved per stage = rows_per_stage * row_bytes
    uint32_t row_bytes;   // bytes one batch row's footprint occupies in a stage (>= largest footprint, 128-aligned)
    int32_t rows_per_stage;   // batch rows staged together (small footprints: amortises barrier + loop overhead)
    uint32_t stage_off;   // byte offset of stage 0 in dynamic shared memory
    double remap_area_min;
    double renorm_min_valid;  // < 0: reference semantics (fill 1e20); >= 0: opt-in renormalising mode
    uint32_t debug_flags; // bit 0: stream only (profiling aid: consumers skip the arithmetic)
    int32_t ord_k;        // ordered_kernel: links per row of the shared-memory image (= the plan's links per lane)
    uint32_t wimg_off, oimg_off;   // ordered_kernel: byte offsets of the weight / offset images in shared memory
    Decode dec;           // packed 16-bit sources only (appended: the offsets of the fields above do not move)
};

}  // namespace smm
