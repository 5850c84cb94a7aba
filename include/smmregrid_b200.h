/*
 * smmregrid_b200.h -- C ABI of the B200-native weight-application operator.
 *
 * Drop-in boundary for the hot path of jhardenberg/smmregrid (v0.1.6).  The reference has
 * no FFI; its seam is the opaque "weights matrix" object that every caller only builds,
 * indexes per level and hands to tensordot.  Each entry point below cites the reference
 * interface it replaces (paths relative to the reference root).  Plain C, no torch types;
 * every function returns an int status (SMM_OK = 0) and never throws across the ABI.
 * smm_last_error() returns a thread-local message for the last non-zero status.
 *
 * Ownership: a handle owns device copies of the operator (CSR, tile plan, dst_grid_imask,
 * dst_grid_frac).  Arrays passed to create/set functions are HOST pointers, copied, never
 * retained.  x / y of smm_apply* are DEVICE pointers owned by the caller (smm_apply_host
 * takes HOST pointers and stages them itself).  A handle is immutable after creation
 * except through smm_set_dst_mask / smm_mask_sum (which must not run concurrently with an
 * apply on the same level); everything that varies per call -- kernel family, the
 * renormalising extension -- is an ARGUMENT of smm_apply* (smm_apply_opts), never handle
 * state, so smm_apply* are re-entrant across threads and streams and one handle can be
 * shared by any number of callers.  There is no CPU fallback: every function fails with
 * SMM_ERR_CUDA when no sm_100 device is usable.
 */
#ifndef SMMREGRID_B200_H
#define SMMREGRID_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMM_OK 0
#define SMM_ERR_INVALID 1   /* bad argument (Python shim: ValueError)                     */
#define SMM_ERR_RANGE 2     /* address outside [index_base, n + index_base) (ValueError)  */
#define SMM_ERR_CUDA 3      /* CUDA runtime failure or no sm_100 device (RuntimeError)    */
#define SMM_ERR_ALLOC 4     /* host or device allocation failure (MemoryError)            */
#define SMM_ERR_DTYPE 5     /* unsupported dtype code (TypeError)                         */

#define SMM_F32 0
#define SMM_F64 1
#define SMM_I16 2           /* x_dtype only (smm_apply*): CF-packed 16-bit integers, decoded inside the */
                            /* kernels as smm_apply_opts.decode says (smm_decode)                       */
#define SMM_F16 3           /* x_dtype only (smm_apply*): IEEE binary16, read as its float32 widening   */
#define SMM_BF16 4          /* x_dtype only (smm_apply*): bfloat16, read as its float32 widening        */

/* Which kernel family serves a level (smm_info.kernel). */
#define SMM_KERNEL_STAGED 1 /* TMA-staged source footprint, register-resident weights     */
#define SMM_KERNEL_GATHER 2 /* direct-gather CSR (scattered sources / oversized rows)     */
#define SMM_KERNEL_COMPACT 3 /* smm_set_kernel only: gather-family levels take the two-pass */
                             /* path (touched columns transposed into a compact buffer,    */
                             /* then applied with lanes over the batch) whatever B is;     */
                             /* by default it is chosen per apply from B and the density   */

/*
 * Summation order of a destination row's links (smm_create_opts.summation, smm_info.summation).
 * The reference's matmul loop (pydata/sparse ndarray . COO, reached from
 * dask.array.tensordot, smmregrid/regrid.py:550) adds a row's products one by one in ascending
 * source order, each product and each sum rounded once.
 *   SMM_SUM_REFERENCE  exactly that order: every value is bit-identical to the reference loop.
 *   SMM_SUM_FAST       lane-split, tree-reduced FMA sums: agree with the reference to rounding
 *                      of sum |w x| (<= 1e-12 relative whenever the products share one sign);
 *                      the `> 1e19` decision is still taken on a reference-order replay.
 *   SMM_SUM_AUTO       REFERENCE when some weight is negative (bicubic, second-order
 *                      conservative: products cancel), else FAST.
 */
#define SMM_SUM_AUTO 0
#define SMM_SUM_FAST 1
#define SMM_SUM_REFERENCE 2

typedef struct smm_handle smm_handle;
typedef void *smm_stream_t; /* cudaStream_t; NULL = legacy default stream */

/* Options of smm_create / smm_create_levels (NULL = all defaults = zero-initialised). */
typedef struct smm_create_opts {
    int32_t summation;          /* SMM_SUM_*                                                  */
    int32_t reserved;
    const char *plan_cache_dir; /* NULL: none.  Directory of an on-disk cache of the operator */
                                /* construction (CSR + tile plan), keyed by a hash of the link */
                                /* arrays: a hit skips the host-side build (C4: 1.6 s -> 0.2 s) */
} smm_create_opts;

/*
 * CF-packed 16-bit source data (x_dtype SMM_I16): the semantics of xarray's CF decoding
 * (CFMaskCoder + CFScaleOffsetCoder, _choose_float_dtype) followed by the reference's apply.
 * For a raw element r:
 *   1. v = r read as int16, or as uint16 when is_unsigned != 0;
 *   2. v equal to one of fill[0 .. n_fill) (_FillValue and every entry of missing_value, given in
 *      the raw type's range; a value outside it matches nothing) -> NaN;
 *   3. else x = D(D(v) * scale_factor) + add_offset: both operations in the decoded dtype D
 *      (`dtype`), each rounded once, no FMA contraction.  Absent attributes: scale_factor = 1.0,
 *      add_offset = -0.0 (x + -0.0 leaves every value, -0.0 included, unchanged, as numpy does
 *      when it skips the addition);
 *   4. then the reference: non-finite (including a decode that overflowed to +-inf) -> 1e20 in D,
 *      float64 products and sums, imask / frac / `> 1e19 -> NaN`.
 * D follows xarray's _choose_float_dtype for 16-bit integers: scale_factor and add_offset of the
 * same type (float32 or float64): that type; only scale_factor: its type; add_offset present and
 * types differ or scale_factor missing: float64; neither (fill values only): float32.  A Python
 * float counts as float64; valid_min / valid_max / valid_range are ignored.
 * smm_apply* return SMM_ERR_INVALID for SMM_I16 without decode, decode with a float x_dtype,
 * n_fill outside [0, 4], a non-finite scale_factor or add_offset, and (dtype SMM_F32) a
 * scale_factor or add_offset float32 cannot hold exactly.  Results are bit-identical to
 * decoding as above on the host and applying the float path (x of dtype D) with reference-order
 * sums (SMM_SUM_REFERENCE, or automatic with a negative weight), or when both calls run the same
 * kernel family.  With fast sums and automatic kernel choice the two may pick different families
 * -- 2-byte rows stage only when n_src % 8 == 0 (float32: n_src % 4 == 0), and the compact
 * path's cost model counts the element size -- and then differ in the last bits of the sums.
 */
typedef struct smm_decode {
    int32_t dtype;              /* SMM_F32 | SMM_F64: the decoded dtype D                       */
    int32_t is_unsigned;        /* != 0: raw values are uint16 (_Unsigned = "true")             */
    double scale_factor;        /* 1.0 when absent                                              */
    double add_offset;          /* -0.0 when absent                                             */
    int32_t n_fill;             /* 0..4                                                         */
    int32_t fill[4];            /* raw values that decode to NaN                                */
} smm_decode;

/* Per-call options of smm_apply* (NULL = all defaults = zero-initialised). */
typedef struct smm_apply_opts {
    int32_t kernel;             /* 0 = automatic, else force SMM_KERNEL_STAGED (fails if the    */
                                /* level has no staged plan), SMM_KERNEL_GATHER (direct gathers) */
                                /* or SMM_KERNEL_COMPACT (two-pass path for gather-family levels) */
    int32_t renormalize;        /* EXTENSION, 0 = off = reference semantics.  != 0: non-finite   */
                                /* source values are EXCLUDED instead of filled with 1e20: a     */
                                /* destination that saw missing sources becomes                  */
                                /*   sum_valid(w x) * sum_all(w) / sum_valid(w)                  */
                                /* if |sum_valid(w)| >= min_valid_fraction * |sum_all(w)|, else  */
                                /* NaN; destinations without missing sources, dst_grid_imask and */
                                /* dst_grid_frac masking are unchanged and the `> 1e19 -> NaN`   */
                                /* rule is not used (the reference has no counterpart: README.md:40) */
    double min_valid_fraction;  /* within [0, 1]; read only when renormalize != 0                */
    const smm_decode *decode;   /* x_dtype SMM_I16 only (required there), else NULL              */
} smm_apply_opts;

typedef struct smm_info {
    int64_t n_src, n_dst, nnz;   /* nnz after duplicate links were summed                 */
    int32_t n_levels;            /* 1 for a 2-D operator                                  */
    int32_t kernel;              /* SMM_KERNEL_* chosen for this level                    */
    int32_t lanes_per_row;       /* staged plan: lanes sharing one destination row        */
    int32_t links_per_lane;      /* staged plan: register-resident links per lane; thread- */
                                 /* per-row reference-order plans (lanes_per_row = 1,      */
                                 /* more than 16 links): the longest row, kept in shared   */
                                 /* memory                                                 */
    int32_t rows_per_tile;       /* staged plan: destination rows per tile                */
    int32_t n_tiles;
    int32_t max_row_nnz;
    int32_t max_tile_segments;
    int32_t consumer_threads;    /* staged plan: link-holding threads per CTA (256 | 512)  */
    int32_t rows_reordered;      /* staged plan tiles rows re-ordered by mean source address */
    int32_t packed_rows;         /* staged plan packs up to 4 short rows per thread (then  */
                                 /* rows_per_tile is the most a tile can hold)             */
    int32_t summation;           /* SMM_SUM_FAST or SMM_SUM_REFERENCE: the order this handle sums in */
    int64_t max_tile_elems;      /* largest staged source footprint of a tile (elements)  */
    int64_t sum_tile_elems;      /* sum of staged footprints: source elements one batch   */
                                 /* row pulls through TMA (>= touched columns)            */
    int64_t touched_src;         /* distinct source columns with >= 1 link                */
    int64_t device_bytes;        /* device memory held for this level                     */
    int32_t plan_cache_hit;      /* 1: CSR + plan came from smm_create_opts.plan_cache_dir */
    int32_t gather_rows;         /* split plan: rows longer than the packed layout's 16 links, served */
                                 /* by the gather kernel next to the staged launch (0: none)          */
} smm_info;

/*
 * compute_weights_matrix (smmregrid/weights.py:25-44).
 * Builds the device operator from CDO link arrays: src_address/dst_address are
 * index_base-based (CDO: 1), remap_matrix is [nnz, num_wgts] row-major and only column 0
 * is used (weights.py:33).  Duplicate (src,dst) links are summed like sparse.COO does.
 */
int smm_create(int64_t n_src, int64_t n_dst, int64_t nnz,
               const int32_t *src_address, const int32_t *dst_address,
               const double *remap_matrix, int32_t num_wgts, int32_t index_base,
               int32_t device, const smm_create_opts *opts, smm_handle **out);

/*
 * compute_weights_matrix3d (smmregrid/weights.py:7-23) on the padded 3-D layout written by
 * CdoGenerate.weightslist_to_3d (smmregrid/cdogenerate.py:310-343): arrays are
 * [n_levels, nl_max] row-major (remap_matrix [n_levels, nl_max, num_wgts]); level i uses
 * links [0, link_length[i]).
 */
int smm_create_levels(int32_t n_levels, const int64_t *link_length, int64_t nl_max,
                      int64_t n_src, int64_t n_dst,
                      const int32_t *src_address, const int32_t *dst_address,
                      const double *remap_matrix, int32_t num_wgts, int32_t index_base,
                      int32_t device, const smm_create_opts *opts, smm_handle **out);

/* The reference drops the matrix object; here the handle is released explicitly. */
int smm_destroy(smm_handle *h);

int smm_get_info(const smm_handle *h, int32_t level, smm_info *out);

/*
 * mask_tensordot (smmregrid/weights.py:47-52) for one level (0 for 2-D):
 *   t[dst] = sum_src src_imask[src] * W[src,dst] (float64, links in ascending-src order),
 *   dst_imask[dst] = t < 0.5 ? 0 : 1.
 * src_imask [n_src] and dst_imask_out [n_dst] are HOST int32 arrays.  The result is also
 * installed as the level's dst_grid_imask, as mask_weights (weights.py:55-84) does.
 * *any_masked_out (optional) = check_mask (weights.py:103-120): 1 if some dst cell is 0.
 */
int smm_mask_sum(smm_handle *h, int32_t level, const int32_t *src_imask,
                 int32_t *dst_imask_out, int32_t *any_masked_out);

/*
 * Install the per-level epilogue vectors read by apply_weights (smmregrid/regrid.py:506-508):
 * dst_grid_imask [n_dst] int32 (NULL keeps the current one) and dst_grid_frac [n_dst]
 * float64 (NULL keeps the current one).  HOST pointers.  Synchronises the device: call it
 * while no apply on this level is in flight.
 */
int smm_set_dst_mask(smm_handle *h, int32_t level, const int32_t *dst_grid_imask,
                     const double *dst_grid_frac);

/*
 * Numeric core of Regridder.apply_weights (smmregrid/regrid.py:536-570) on one level:
 *   x [B, n_src] row-major with row stride ldx (elements), dtype x_dtype (SMM_I16: decoded
 *   to its dtype D first, see smm_decode);
 *   non-finite -> 1e20 (in x's dtype), Y = X.W accumulated in float64,
 *   masked != 0:            Y[:, d] = NaN where dst_grid_imask[d] == 0     (:553-559)
 *   remap_area_min > 0:     Y[:, d] = NaN where dst_grid_frac[d] < min     (:562-565)
 *   Y > 1e19 -> NaN                                                         (:570)
 *   y [B, n_dst] row stride ldy, dtype y_dtype (SMM_F64 = the reference's result_type;
 *   SMM_F32 rounds the float64 result once at the store).
 * x and y are DEVICE pointers; the launch is asynchronous on `stream`.
 *
 * Half-precision sources (x_dtype SMM_F16 / SMM_BF16; y_dtype stays SMM_F32 or SMM_F64, a half
 * y_dtype is SMM_ERR_DTYPE).  The kernels read the 2-byte values and widen each one exactly to
 * float32; from there on the float32 semantics apply unchanged: non-finite -> 1e20 IN FLOAT32
 * (1.00000002004e20 as a float64), float64 products and sums, the masks and the `> 1e19` rule,
 * and the renormalising extension excludes non-finite sources.  Contract: every result of
 * smm_apply, smm_apply_levels, smm_apply_host and smm_apply_levels_host with half data is
 * bit-identical to the same call on the float32 widening of that data (same B, row strides and
 * options; the float32 slab 16-byte aligned), for every summation order and kernel option.  The
 * kernel family is the one float32 data would get; where that family is the staged kernel but the
 * 2-byte rows cannot be staged (x not 16-byte aligned, a row stride or n_src that is not a
 * multiple of 8), the rows are widened into float32 chunks from the handle's stream-ordered pool
 * and applied there (SMM_ERR_ALLOC if the pool cannot provide a chunk).  Forced SMM_KERNEL_GATHER
 * reads the 2-byte data directly, and so does forced SMM_KERNEL_COMPACT on gather-family levels;
 * a level with a staged plan stays staged under SMM_KERNEL_COMPACT, as float32 data does, and so
 * takes the float32 chunks like an automatic call when its 2-byte rows cannot be staged.  The
 * chunks hold up to 256 MB of float32 rows; the pool keeps that memory for later calls (one chunk
 * per stream applying at the same time) until the handle is destroyed.  One exception: when the pool cannot
 * provide the compact path's transposed buffer, the path falls back to direct gathers; that
 * buffer is half the size for 2-byte data, so under memory pressure half and float32 data may land
 * on different sides of that fallback and then differ in the last bits of fast sums.
 */
int smm_apply(const smm_handle *h, int32_t level,
              const void *x, int32_t x_dtype, int64_t B, int64_t ldx,
              void *y, int32_t y_dtype, int64_t ldy,
              int32_t masked, double remap_area_min, const smm_apply_opts *opts,
              smm_stream_t stream);

/*
 * Regridder.regrid3d's level loop (smmregrid/regrid.py:387-410) as ONE grouped launch.
 * For i in [0, n_sel): data level i uses weight level level_index[i] (the caller resolves
 * the nearest-level rule of regrid.py:390-395).  Batch row b of data level i lives at
 *   x + (b * x_batch_stride + i * x_level_stride) elements, and is written to
 *   y + (b * y_batch_stride + i * y_level_stride) elements,
 * which places every level directly at its final [.., L, n_dst] position (the concat +
 * transpose of regrid.py:410-427).  masked[i] is the per-level flag of check_mask.
 */
int smm_apply_levels(const smm_handle *h, int32_t n_sel, const int32_t *level_index,
                     const void *x, int32_t x_dtype, int64_t B,
                     int64_t x_batch_stride, int64_t x_level_stride,
                     void *y, int32_t y_dtype,
                     int64_t y_batch_stride, int64_t y_level_stride,
                     const uint8_t *masked, double remap_area_min, const smm_apply_opts *opts,
                     smm_stream_t stream);

/*
 * smm_apply for HOST buffers: x/y are host pointers (pinned or pageable); the batch axis
 * is cut into chunks of `chunk_rows` (0 = auto) that are copied host->device, applied and
 * copied back on alternating streams so copies overlap the kernel.  Synchronous: returns
 * when y is complete.
 */
int smm_apply_host(const smm_handle *h, int32_t level,
                   const void *x, int32_t x_dtype, int64_t B, int64_t ldx,
                   void *y, int32_t y_dtype, int64_t ldy,
                   int32_t masked, double remap_area_min, const smm_apply_opts *opts,
                   int64_t chunk_rows);


/*
 * smm_apply_levels for HOST buffers in the canonical layout: x [B, n_sel, n_src] and
 * y [B, n_sel, n_dst], both contiguous (data level i uses weight level level_index[i]); same
 * streaming pipeline as smm_apply_host, chunked over B.  Synchronous.
 */
int smm_apply_levels_host(const smm_handle *h, int32_t n_sel, const int32_t *level_index,
                          const void *x, int32_t x_dtype, int64_t B,
                          void *y, int32_t y_dtype,
                          const uint8_t *masked, double remap_area_min, const smm_apply_opts *opts,
                          int64_t chunk_rows);

/*
 * detect_nan_variation_dims (smmregrid/util.py:57-85), one axis per call: the DEVICE array x is
 * viewed as [outer, n_axis, inner] (contiguous); *count_out = number of (outer, inner)
 * positions whose NaN-ness changes somewhere along the axis -- the reference's
 * `isnull().astype("int8").diff(dim).astype(bool).any(dim).sum()`.  A dimension "has NaN
 * variation" (and becomes a mask dimension, regrid.py:630-653) when the count is > 0.
 * NaN only, as isnull: +-inf does not count.  Synchronous on `stream`.  x_dtype SMM_F32 or
 * SMM_F64 only (anything else, SMM_F16 / SMM_BF16 included, is SMM_ERR_DTYPE: widen half data first,
 * which keeps its NaN-ness exactly).
 */
int smm_nan_variation(const void *x, int32_t x_dtype, int64_t outer, int64_t n_axis, int64_t inner,
                      int64_t *count_out, smm_stream_t stream);

/*
 * Host-only introspection of the operator construction (no device needed): builds the
 * same CSR + tile plan smm_create uploads, so the host logic can be verified on a CPU-only
 * machine.  No compute entry point exists on the host side.
 *   smm_host_plan_copy: any output pointer may be NULL.  Sizes: rowptr [n_dst+1], col/val
 *   [nnz], tiles [n_tiles*8] int32 (row0,nrows,seg0,nseg,elems,pad*3), segs [n_segs*4]
 *   uint32 (src,dst,len,pad), wplan/iplan [n_tiles*links_per_lane*consumer_threads].
 */
typedef struct smm_host_plan smm_host_plan;
int smm_host_plan_build(int64_t n_src, int64_t n_dst, int64_t nnz,
                        const int32_t *src_address, const int32_t *dst_address,
                        const double *remap_matrix, int32_t num_wgts, int32_t index_base,
                        const smm_create_opts *opts, smm_host_plan **out);
int smm_host_plan_info(const smm_host_plan *p, smm_info *out, int64_t *n_segs_out);
int smm_host_plan_copy(const smm_host_plan *p, int32_t *rowptr, int32_t *col, double *val,
                       int32_t *tiles, uint32_t *segs, double *wplan, uint16_t *iplan);
/* rowmap [n_dst]: destination row held by every tile slot (only when info.rows_reordered). */
int smm_host_plan_rowmap(const smm_host_plan *p, int32_t *rowmap);
/* rows [info.gather_rows]: the long rows of a split plan, ascending. */
int smm_host_plan_gather_rows(const smm_host_plan *p, int32_t *rows);
/* rowslot [n_tiles*4*consumer_threads] (only when info.packed_rows): destination row whose value
 * starts in sub-row u (link slots 4u..4u+3) of thread t at [tile][u][t]; -1 none, -2 the sub-row
 * continues the row of sub-row u-1. */
int smm_host_plan_rowslot(const smm_host_plan *p, int32_t *rowslot);
/* Two-pass compact plan of the operator (what gather-family levels upload for the compact path):
 * tcols [touched_src] = touched source columns, ascending; blk_ptr [n_blocks + 1] = their range
 * per block of 256 source columns; rcol [nnz] = rank in tcols of every CSR link's column.  Call
 * once with NULL arrays for the sizes. */
int smm_host_plan_compact(const smm_host_plan *p, int64_t *n_touched_out, int64_t *n_blocks_out,
                          int32_t *tcols, int32_t *blk_ptr, int32_t *rcol);
void smm_host_plan_free(smm_host_plan *p);

/*
 * Bare host<->device copy ceiling of this process's device (measurement aid used by bench.py to
 * put the end-to-end figure next to what the PCIe link itself sustains): copies `bytes` from
 * the PINNED host buffer `host` to an internal device buffer (direction 0) or back (1) `reps`
 * times on one stream and returns the average seconds per copy in *seconds_out.
 */
int smm_copy_ceiling(int32_t device, void *host, int64_t bytes, int32_t direction, int32_t reps,
                     double *seconds_out);

/* Kernels launched by this library in the calling process so far (bench.py gpu_launches). */
int64_t smm_launch_count(void);

const char *smm_last_error(void);
const char *smm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SMMREGRID_B200_H */
