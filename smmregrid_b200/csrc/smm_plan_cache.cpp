// smm_plan_cache.cpp -- on-disk cache of the operator construction (CSR + tile plans).
//
// Building the device operator from CDO link arrays is host work (sort/merge into CSR, tile
// footprints, link placement: 1.6 s for the 7.1 M links of the 0.1 deg -> 1 deg remapcon set,
// 3.5 s for 75 ocean levels), repeated by every process that opens the same weight file.  The
// cache stores the finished host structures under a key hashed from the link arrays themselves
// (plus everything else the plan depends on), so a second process only reads and uploads them.
// Each writer fills a temporary file of its own (several threads or processes may build the same
// operator at once) and renames it into place, so readers never see a partial file.  The file ends
// with a hash of everything before it: any mismatch (magic, version, sizes, content, truncated file)
// is treated as a miss, so a damaged payload never reaches the device.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>

#include <sys/stat.h>
#include <unistd.h>

#include "smm_plan.h"

namespace smm {

namespace {

constexpr char kMagic[8] = {'S', 'M', 'M', 'P', 'L', 'A', 'N', '7'};

// 4 interleaved 64-bit multiply-xorshift lanes over 8-byte words (a few GB/s on one core)
struct Hasher {
    uint64_t h[4] = {0x9E3779B97F4A7C15ull, 0xC2B2AE3D27D4EB4Full, 0x165667B19E3779F9ull, 0x27D4EB2F165667C5ull};
    uint64_t n = 0;
    static inline uint64_t mix(uint64_t h, uint64_t w)
    {
        h = (h ^ w) * 0xFF51AFD7ED558CCDull;
        return h ^ (h >> 32);
    }
    void bytes(const void *p, size_t len)
    {
        const unsigned char *c = static_cast<const unsigned char *>(p);
        n += len;
        size_t i = 0;
        for (; i + 32 <= len; i += 32) {
            uint64_t w[4];
            std::memcpy(w, c + i, 32);
            h[0] = mix(h[0], w[0]); h[1] = mix(h[1], w[1]); h[2] = mix(h[2], w[2]); h[3] = mix(h[3], w[3]);
        }
        for (int lane = 0; i < len; i += 8, lane = (lane + 1) & 3) {
            uint64_t w = 0;
            std::memcpy(&w, c + i, len - i < 8 ? len - i : 8);
            h[lane] = mix(h[lane], w ^ 0xA5A5A5A5A5A5A5A5ull);
        }
    }
    template <typename T> void pod(const T &v) { bytes(&v, sizeof(T)); }
    void str(const char *s) { const uint64_t l = s ? std::strlen(s) : 0; pod(l); if (l) bytes(s, l); }
    void finish(uint64_t out[2])
    {
        uint64_t a = mix(mix(h[0], h[1]), n), b = mix(mix(h[2], h[3]), ~n);
        out[0] = mix(a, b);
        out[1] = mix(b, a ^ 0x5851F42D4C957F2Dull);
    }
};

struct Writer {
    FILE *f;
    bool ok = true;
    Hasher hs;                      // of every byte written
    void raw(const void *p, size_t n)
    {
        if (ok && n && std::fwrite(p, 1, n, f) != n) ok = false;
        hs.bytes(p, n);
    }
    template <typename T> void pod(const T &v) { raw(&v, sizeof(T)); }
    template <typename T> void vec(const std::vector<T> &v)
    {
        const uint64_t n = v.size();
        pod(n);
        raw(v.data(), n * sizeof(T));
    }
    void str(const std::string &s) { const uint64_t n = s.size(); pod(n); raw(s.data(), n); }
};

struct Reader {
    FILE *f;
    bool ok = true;
    uint64_t left;                  // bytes remaining in the file: bounds every vector length
    Hasher hs;                      // of every byte read
    void raw(void *p, size_t n)
    {
        if (!ok) return;
        if (n > left || (n && std::fread(p, 1, n, f) != n)) { ok = false; return; }
        left -= n;
        hs.bytes(p, n);
    }
    template <typename T> void pod(T &v) { raw(&v, sizeof(T)); }
    template <typename T> void vec(std::vector<T> &v)
    {
        uint64_t n = 0;
        pod(n);
        if (!ok || n > left / sizeof(T)) { ok = false; return; }
        v.resize(n);
        raw(v.data(), n * sizeof(T));
    }
    void str(std::string &s)
    {
        uint64_t n = 0;
        pod(n);
        if (!ok || n > left) { ok = false; return; }
        s.resize(n);
        raw(&s[0], n);
    }
};

template <typename IO> void io_csr(IO &io, HostCsr &c)
{
    io.pod(c.n_src); io.pod(c.n_dst); io.pod(c.max_row_nnz); io.pod(c.touched_src); io.pod(c.has_negative);
    io.vec(c.rowptr); io.vec(c.col); io.vec(c.val);
}

template <typename IO> void io_plan(IO &io, HostPlan &p)
{
    io.pod(p.ok); io.str(p.why);
    io.pod(p.lpr); io.pod(p.kpl); io.pod(p.rows_per_tile); io.pod(p.nct);
    io.pod(p.reordered); io.pod(p.packed); io.pod(p.ref_order); io.pod(p.ordlong);
    io.pod(p.max_tile_segments); io.pod(p.max_tile_elems); io.pod(p.sum_tile_elems); io.pod(p.sum_tile_cols);
    io.vec(p.tiles); io.vec(p.segs); io.vec(p.rowmap); io.vec(p.rowslot); io.vec(p.wplan); io.vec(p.iplan);
    io.pod(p.nrows);
    io.vec(p.gather_rows);
}

std::string cache_file(const std::string &dir, const PlanCacheKey &key)
{
    char name[64];
    std::snprintf(name, sizeof(name), "/smm_%016llx%016llx.plan", static_cast<unsigned long long>(key.h[0]),
                  static_cast<unsigned long long>(key.h[1]));
    return dir + name;
}

}  // namespace

PlanCacheKey plan_cache_key(int32_t n_levels, const int64_t *link_length, int64_t nl_max, int64_t n_src,
                            int64_t n_dst, const int32_t *src_address, const int32_t *dst_address,
                            const double *remap_matrix, int32_t num_wgts, int32_t index_base,
                            int32_t summation, int32_t sm_count)
{
    Hasher hs;
    hs.bytes(kMagic, sizeof(kMagic));
    hs.pod(n_levels); hs.pod(nl_max); hs.pod(n_src); hs.pod(n_dst); hs.pod(num_wgts); hs.pod(index_base);
    hs.pod(summation); hs.pod(sm_count);
    // plan-shaping experiment switches are part of the key
    for (const char *env : {"SMM_CONSUMER_THREADS", "SMM_PACKED", "SMM_FORCE_LANES", "SMM_SPLIT", "SMM_ORDLONG",
                            "SMM_ORD_ROWS", "SMM_SUMMATION"})
        hs.str(std::getenv(env));
    for (int32_t i = 0; i < n_levels; ++i) {
        const int64_t nl = link_length[i], o = static_cast<int64_t>(i) * nl_max;
        hs.pod(nl);
        if (nl <= 0) continue;
        hs.bytes(src_address + o, static_cast<size_t>(nl) * sizeof(int32_t));
        hs.bytes(dst_address + o, static_cast<size_t>(nl) * sizeof(int32_t));
        hs.bytes(remap_matrix + o * num_wgts, static_cast<size_t>(nl) * num_wgts * sizeof(double));
    }
    PlanCacheKey key;
    hs.finish(key.h);
    return key;
}

bool plan_cache_load(const std::string &dir, const PlanCacheKey &key, int32_t n_levels, int64_t n_src,
                     int64_t n_dst, std::vector<HostCsr> &csrs, std::vector<HostPlan> &plans, bool &ref_order)
{
    const std::string path = cache_file(dir, key);
    FILE *f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    struct stat st;
    if (fstat(fileno(f), &st) != 0) { std::fclose(f); return false; }
    Reader rd{f, true, static_cast<uint64_t>(st.st_size)};
    char magic[8] = {0};
    uint64_t k0 = 0, k1 = 0;
    int32_t nl = 0;
    uint8_t ord = 0;
    rd.raw(magic, 8); rd.pod(k0); rd.pod(k1); rd.pod(nl); rd.pod(ord);
    bool good = rd.ok && std::memcmp(magic, kMagic, 8) == 0 && k0 == key.h[0] && k1 == key.h[1] && nl == n_levels;
    if (good) {
        csrs.assign(static_cast<size_t>(n_levels), HostCsr{});
        plans.assign(static_cast<size_t>(n_levels), HostPlan{});
        for (int32_t i = 0; i < n_levels && rd.ok; ++i) {
            io_csr(rd, csrs[i]);
            io_plan(rd, plans[i]);
            // structural sanity: sizes must be those of this operator
            const HostCsr &c = csrs[i];
            const HostPlan &p = plans[i];
            if (!rd.ok || c.n_src != n_src || c.n_dst != n_dst || c.rowptr.size() != static_cast<size_t>(n_dst) + 1 ||
                c.col.size() != c.val.size() || static_cast<size_t>(c.rowptr.back()) != c.col.size() ||
                (p.ok && (p.wplan.size() != p.tiles.size() * static_cast<size_t>(p.kpl) * p.nct ||
                          p.iplan.size() != p.wplan.size())))
                rd.ok = false;
        }
        uint64_t want[2], tail[2] = {0, 0};
        rd.hs.finish(want);
        rd.pod(tail);
        good = rd.ok && rd.left == 0 && tail[0] == want[0] && tail[1] == want[1];
    }
    std::fclose(f);
    if (!good) { csrs.clear(); plans.clear(); }
    else ref_order = ord != 0;
    return good;
}

bool plan_cache_store(const std::string &dir, const PlanCacheKey &key, std::vector<HostCsr> &csrs,
                      std::vector<HostPlan> &plans, bool ref_order)
{
    ::mkdir(dir.c_str(), 0777);            // best effort; an existing directory is fine
    const std::string path = cache_file(dir, key);
    const std::string tmp = path + ".tmp" + std::to_string(static_cast<long long>(getpid())) + "." +
                            std::to_string(std::hash<std::thread::id>{}(std::this_thread::get_id()));
    FILE *f = std::fopen(tmp.c_str(), "wb");
    if (!f) return false;
    Writer wr{f};
    wr.raw(kMagic, 8);
    wr.pod(key.h[0]); wr.pod(key.h[1]);
    const int32_t nl = static_cast<int32_t>(csrs.size());
    const uint8_t ord = ref_order ? 1 : 0;
    wr.pod(nl); wr.pod(ord);
    for (size_t i = 0; i < csrs.size(); ++i) {
        io_csr(wr, csrs[i]);
        io_plan(wr, plans[i]);
    }
    uint64_t tail[2];
    wr.hs.finish(tail);
    wr.pod(tail);
    const bool ok = wr.ok && std::fclose(f) == 0;
    if (!wr.ok) std::fclose(f);
    if (!ok || std::rename(tmp.c_str(), path.c_str()) != 0) { std::remove(tmp.c_str()); return false; }
    return true;
}

}  // namespace smm
