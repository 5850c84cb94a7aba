// smm_tuning.h -- the SMM_* environment switches.  They exist for experiments, A/B runs and
// diagnostics; unset, every one gives the tuned default.  smm_tuning.cpp is the only place that
// reads the environment, and the three structs below say when: per operator construction, once per
// process, or per host streaming call.  Each field names its switch, its default and how the value
// is parsed.
#pragma once
#include <cstdint>

namespace smm {

constexpr int kHostSlots = 4;      // device buffer slots of the host pipeline's ring

// Switches that shape the plans of an operator: read once at the start of smm_create_levels and of
// smm_host_plan_build, and passed to every planning decision.  The plan cache key hashes each of
// them except plan_threads, which only spreads the work and does not change the plan.
struct PlanSettings {
    // SMM_FORCE_LANES="lpr,kpl": lanes per row and links per lane, both > 0, else ignored (0, 0).
    // choose_lanes uses them only for rows that fit lpr * kpl links.
    int32_t force_lpr = 0, force_kpl = 0;
    // SMM_CONSUMER_THREADS: atoi; only 256 and 512 are honoured, else 0 (chosen per weight set).
    int32_t consumer_threads = 0;
    // SMM_PACKED: 1 when the first character is '1', else 0 (so an empty value is off); -1 unset
    // (packed rows whenever every row fits).
    int32_t packed = -1;
    // SMM_SPLIT: parsed as SMM_PACKED; -1 unset (split when the long rows are few).  On applies only
    // when some row is long.
    int32_t split = -1;
    // SMM_ORDLONG: atoi != 0 (default on): reference-order sums may use ordered-long plans.
    bool ordlong = true;
    // SMM_ORD_ROWS: atoi (default 0: the tallest tile whose link image fits): rows per ordered-long tile.
    int32_t ord_rows = 0;
    // SMM_SUMMATION: SMM_SUM_FAST when the first character is 'f', SMM_SUM_REFERENCE when it is 'r',
    // else SMM_SUM_AUTO (no override of smm_create_opts.summation).
    int32_t summation = 0;
    // SMM_PLAN_THREADS: atoi (default: the CPUs of the affinity mask); build_plan clamps it to
    // [1, min(16, tiles / 32)] host threads per plan.
    int32_t plan_threads = 1;
};
PlanSettings plan_settings();

// Switches of the launch code: read once per process, at the first launch or host streaming call.
struct LaunchSettings {
    int min_rows_per_item;   // SMM_MIN_ROWS_PER_ITEM: atoi, at least 1 (default 8): fewest batch rows per work item
    int waves;               // SMM_WAVES: atoi (default 0: from the cost model); > 0 fixes the waves per launch
    uint32_t debug_flags;    // SMM_DEBUG_STREAM_ONLY: atoi & 3 (default 0): staged consumers skip bit 0 the
                             // arithmetic, bit 1 the stores (profiling aid: results are meaningless)
    int max_stages;          // SMM_MAX_STAGES: atoi, at least 2 (default kMaxStages): cap on the stage ring
    int rows_per_stage;      // SMM_ROWS_PER_STAGE: atoi (default 0: from the footprint); > 0 fixes batch rows per stage
    int ord_tpr;             // SMM_ORD_TPR: atoi (default 0: 2 when tiles have <= 128 rows); 2 forces two
                             // threads per row of the ordered kernel, any other value one
    bool compact_bulk;       // SMM_COMPACT_BULK: off when the first character is '0' (element copies), else on
    int compact_f64_rows;    // SMM_COMPACT_F64_ROWS: atoi (default 32): batch rows per compact pass for 8-byte
                             // elements with bulk copies; outside (0, kCompactBC) a full kCompactBC
    bool host_trace;         // SMM_HOST_TRACE: atoi != 0 (default off): host pipeline phase times on stderr
    int host_in_streams;     // SMM_HOST_IN_STREAMS: atoi clamped to [1, 2] (default 2): host->device copy streams
    int host_slots;          // SMM_HOST_SLOTS: atoi clamped to [2, kHostSlots] (default kHostSlots): ring depth
};
const LaunchSettings &launch_settings();

// Switches read at every smm_apply_host / smm_apply_levels_host call.
struct HostCallSettings {
    int chunk_mb;            // SMM_HOST_CHUNK_MB: atoi, at least 1; 0 when unset: 128 for pinned x, 64 when staged
    int copy_threads;        // SMM_HOST_COPY_THREADS: atoi (default 12) clamped to [1, CPUs of the affinity mask]:
                             // threads filling the pinned bounce buffers
};
HostCallSettings host_call_settings();

// CPUs in the calling thread's affinity mask (at least 1)
int host_cpus();

}  // namespace smm
