// smm_tuning.cpp -- the only reader of the SMM_* environment switches (see smm_tuning.h).
#include "smm_tuning.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include <sched.h>

#include "../../include/smmregrid_b200.h"
#include "smm_common.h"

namespace smm {

namespace {

int env_int(const char *name, int dflt)
{
    const char *e = std::getenv(name);
    return e ? std::atoi(e) : dflt;
}

// -1 unset, else whether the first character is '1'
int32_t env_flag(const char *name)
{
    const char *e = std::getenv(name);
    return e ? (e[0] == '1' ? 1 : 0) : -1;
}

}  // namespace

int host_cpus()
{
    cpu_set_t set;
    return sched_getaffinity(0, sizeof(set), &set) == 0 ? std::max(1, CPU_COUNT(&set)) : 1;
}

PlanSettings plan_settings()
{
    PlanSettings s;
    if (const char *e = std::getenv("SMM_FORCE_LANES")) {
        int a = 0, b = 0;
        if (std::sscanf(e, "%d,%d", &a, &b) == 2 && a > 0 && b > 0) { s.force_lpr = a; s.force_kpl = b; }
    }
    const int nct = env_int("SMM_CONSUMER_THREADS", 0);
    s.consumer_threads = (nct == 256 || nct == 512) ? nct : 0;
    s.packed = env_flag("SMM_PACKED");
    s.split = env_flag("SMM_SPLIT");
    s.ordlong = env_int("SMM_ORDLONG", 1) != 0;
    s.ord_rows = env_int("SMM_ORD_ROWS", 0);
    if (const char *e = std::getenv("SMM_SUMMATION")) {
        if (e[0] == 'f') s.summation = SMM_SUM_FAST;
        if (e[0] == 'r') s.summation = SMM_SUM_REFERENCE;
    }
    s.plan_threads = env_int("SMM_PLAN_THREADS", host_cpus());
    return s;
}

const LaunchSettings &launch_settings()
{
    static const LaunchSettings s = [] {
        LaunchSettings r;
        r.min_rows_per_item = std::max(1, env_int("SMM_MIN_ROWS_PER_ITEM", 8));
        r.waves = env_int("SMM_WAVES", 0);
        r.debug_flags = static_cast<uint32_t>(env_int("SMM_DEBUG_STREAM_ONLY", 0)) & 3u;
        r.max_stages = std::max(2, env_int("SMM_MAX_STAGES", kMaxStages));
        r.rows_per_stage = env_int("SMM_ROWS_PER_STAGE", 0);
        r.ord_tpr = env_int("SMM_ORD_TPR", 0);
        const char *bulk = std::getenv("SMM_COMPACT_BULK");
        r.compact_bulk = !(bulk && bulk[0] == '0');
        r.compact_f64_rows = env_int("SMM_COMPACT_F64_ROWS", 32);
        r.host_trace = env_int("SMM_HOST_TRACE", 0) != 0;
        r.host_in_streams = std::max(1, std::min(2, env_int("SMM_HOST_IN_STREAMS", 2)));
        r.host_slots = std::max(2, std::min(kHostSlots, env_int("SMM_HOST_SLOTS", kHostSlots)));
        return r;
    }();
    return s;
}

HostCallSettings host_call_settings()
{
    HostCallSettings s;
    const char *mb = std::getenv("SMM_HOST_CHUNK_MB");
    s.chunk_mb = mb ? std::max(1, std::atoi(mb)) : 0;
    s.copy_threads = std::max(1, std::min(host_cpus(), env_int("SMM_HOST_COPY_THREADS", 12)));
    return s;
}

}  // namespace smm
