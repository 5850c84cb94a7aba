// smm_plan.cpp -- CDO links -> CSR by destination row -> tile plan of the staged kernel.
//
// Restates, for the device layout, what the reference does when it wraps the CDO arrays in
// sparse.COO (smmregrid/weights.py:25-44): addresses made 0-based, column 0 of
// remap_matrix, duplicate coordinates summed.  The row-major-by-destination order keeps
// each row's links in ascending source order, i.e. the order in which the reference's
// matmul loop visits them.
#include "smm_plan.h"

#include <algorithm>
#include <atomic>
#include <numeric>
#include <thread>

#include "../../include/smmregrid_b200.h"

namespace smm {

int build_csr(int64_t n_src, int64_t n_dst, int64_t nnz, const int32_t *src_address,
              const int32_t *dst_address, const double *remap_matrix, int32_t num_wgts,
              int32_t index_base, HostCsr &out, std::string &err)
{
    if (n_src <= 0 || n_dst <= 0 || nnz < 0 || num_wgts < 1) {
        err = "smm_create: n_src, n_dst must be > 0, nnz >= 0, num_wgts >= 1";
        return SMM_ERR_INVALID;
    }
    if (n_src > INT32_MAX || n_dst >= INT32_MAX || nnz >= INT32_MAX) {
        err = "smm_create: sizes beyond int32 addressing are not supported";
        return SMM_ERR_INVALID;
    }
    if (nnz > 0 && (!src_address || !dst_address || !remap_matrix)) {
        err = "smm_create: null link array";
        return SMM_ERR_INVALID;
    }
    out.n_src = n_src;
    out.n_dst = n_dst;

    std::vector<uint64_t> key(static_cast<size_t>(nnz));
    bool sorted = true;
    for (int64_t k = 0; k < nnz; ++k) {
        const int64_t s = static_cast<int64_t>(src_address[k]) - index_base;
        const int64_t d = static_cast<int64_t>(dst_address[k]) - index_base;
        if (s < 0 || s >= n_src || d < 0 || d >= n_dst) {
            err = "smm_create: link " + std::to_string(k) + " addresses (" +
                  std::to_string(src_address[k]) + "," + std::to_string(dst_address[k]) +
                  ") outside the grids";
            return SMM_ERR_RANGE;
        }
        key[k] = (static_cast<uint64_t>(d) << 32) | static_cast<uint64_t>(s);
        if (k > 0 && key[k] <= key[k - 1]) sorted = false;
    }
    std::vector<int64_t> order;
    if (!sorted) {
        order.resize(static_cast<size_t>(nnz));
        std::iota(order.begin(), order.end(), int64_t{0});
        std::stable_sort(order.begin(), order.end(),
                         [&](int64_t a, int64_t b) { return key[a] < key[b]; });
    }
    out.rowptr.assign(static_cast<size_t>(n_dst) + 1, 0);
    out.col.clear();
    out.val.clear();
    out.col.reserve(static_cast<size_t>(nnz));
    out.val.reserve(static_cast<size_t>(nnz));
    uint64_t prev = ~uint64_t{0};
    for (int64_t i = 0; i < nnz; ++i) {
        const int64_t k = sorted ? i : order[i];
        const double w = remap_matrix[k * static_cast<int64_t>(num_wgts)];
        if (i > 0 && key[k] == prev) {
            out.val.back() += w;   // sum_duplicates, original order
        } else {
            out.col.push_back(static_cast<int32_t>(key[k] & 0xffffffffu));
            out.val.push_back(w);
            out.rowptr[(key[k] >> 32) + 1] += 1;
            prev = key[k];
        }
    }
    out.max_row_nnz = 0;
    for (int64_t r = 0; r < n_dst; ++r) {
        out.max_row_nnz = std::max(out.max_row_nnz, out.rowptr[r + 1]);
        out.rowptr[r + 1] += out.rowptr[r];
    }
    std::vector<uint8_t> seen(static_cast<size_t>(n_src), 0);
    int64_t touched = 0;
    for (int32_t c : out.col)
        if (!seen[c]) { seen[c] = 1; ++touched; }
    out.touched_src = touched;
    out.has_negative = false;
    for (double v : out.val)
        if (v < 0.0) { out.has_negative = true; break; }
    return SMM_OK;
}

bool choose_lanes(const PlanSettings &s, int32_t m, int32_t &lpr, int32_t &kpl)
{
    if (s.force_lpr > 0 && m <= s.force_lpr * s.force_kpl) { lpr = s.force_lpr; kpl = s.force_kpl; return true; }
    // (lanes per row, links per lane): fewest padded slots first -- every slot, padded or not,
    // costs an F2F conversion, and conversion throughput bounds link-dense operators
    if (m <= 4) { lpr = 1; kpl = 4; }
    else if (m <= 8) { lpr = 1; kpl = 8; }
    else if (m <= 12) { lpr = 1; kpl = 12; }
    else if (m <= 16) { lpr = 1; kpl = 16; }
    else if (m <= 24) { lpr = 2; kpl = 12; }
    else if (m <= 28) { lpr = 2; kpl = 14; }
    else if (m <= 32) { lpr = 2; kpl = 16; }
    else if (m <= 48) { lpr = 4; kpl = 12; }
    else if (m <= 64) { lpr = 4; kpl = 16; }
    else if (m <= 96) { lpr = 8; kpl = 12; }
    else if (m <= 112) { lpr = 8; kpl = 14; }
    else if (m <= 128) { lpr = 8; kpl = 16; }
    else if (m <= 256) { lpr = 16; kpl = 16; }
    else if (m <= 512) { lpr = 32; kpl = 16; }
    else return false;
    return true;
}

int32_t default_consumer_threads(const PlanSettings &s, int64_t n_dst, int32_t lpr, int32_t sm_count)
{
    if (s.consumer_threads) return s.consumer_threads;
    if (lpr <= 0) return 256;
    const int64_t tiles512 = (n_dst + 512 / lpr - 1) / (512 / lpr);
    return tiles512 >= sm_count ? 512 : 256;
}

// Packed rows (short-row operators: nn, bilinear, 1:1 conservative, ocean levels): a thread's 16
// link slots are four sub-rows of four; a row takes 1-4 consecutive sub-rows of ONE thread, so a
// thread owns up to four destination rows and a tile up to 4*NCT.  Fewer, fuller consumer
// iterations where the lane-per-row layout would mostly multiply padding.
constexpr int kSubRows = 4, kSubLinks = 4;

static void build_plan_rows(const HostCsr &csr, int32_t force_lpr, int32_t force_kpl, int32_t nct,
                            const std::vector<int32_t> *order, bool packed, bool ref_order, const PlanSettings &s,
                            HostPlan &plan)
{
    plan = HostPlan{};
    plan.ref_order = ref_order;
    if (nct < 32 || nct > 512 || nct % 32 != 0) nct = 256;
    int32_t lpr = force_lpr, kpl = force_kpl;
    int32_t max_row = csr.max_row_nnz;
    if (order) {
        max_row = 0;
        for (int32_t r : *order) max_row = std::max(max_row, csr.rowptr[r + 1] - csr.rowptr[r]);
    }
    if (packed) {
        if (max_row > kSubRows * kSubLinks) { plan.why = "row too long for the packed layout"; return; }
        lpr = 1; kpl = kSubRows * kSubLinks;
    } else if (lpr <= 0 || kpl <= 0) {
        if (!choose_lanes(s, max_row, lpr, kpl)) {
            plan.why = "a destination row has more than 512 links";
            return;
        }
    } else if (max_row > lpr * kpl) {
        plan.why = "row longer than the forced lane configuration";
        return;
    }
    // rows this plan tiles: all of them in natural order, or the given sequence (a re-ordering of
    // all rows, or the subset one part of a split plan covers)
    const int64_t n_dst = order ? static_cast<int64_t>(order->size()) : csr.n_dst, n_src = csr.n_src;
    const int32_t R = packed ? nct * kSubRows : nct / lpr;          // most rows a tile can hold
    auto row_at = [&](int64_t pos) -> int64_t { return order ? (*order)[pos] : pos; };
    // tile boundaries (positions in the row order); packed: also every row's (thread, sub-row)
    std::vector<int64_t> tile_start;
    std::vector<int32_t> row_thread;
    std::vector<int8_t> row_sub;
    if (!packed) {
        for (int64_t r = 0; r < n_dst; r += R) tile_start.push_back(r);
    } else {
        // Rows are dealt round-robin over the 32 lanes of a warp (lane l's j-th row is about
        // row base + 32*j + l): the lanes of a warp read neighbouring source elements and write
        // neighbouring destination cells in every slot, like the lane-per-row layout does.
        row_thread.resize(static_cast<size_t>(n_dst));
        row_sub.resize(static_cast<size_t>(n_dst));
        const int32_t nwarps = nct / 32;
        int32_t wi = 0, next = 0;
        int8_t used[32] = {0};
        tile_start.push_back(0);
        for (int64_t pos = 0; pos < n_dst; ++pos) {
            const int64_t r = row_at(pos);
            const int32_t nnz = csr.rowptr[r + 1] - csr.rowptr[r];
            const int32_t c = std::max(1, (nnz + kSubLinks - 1) / kSubLinks);
            int32_t lane = -1;
            for (int32_t tries = 0; tries < 32 && lane < 0; ++tries) {
                const int32_t l = (next + tries) & 31;
                if (used[l] + c <= kSubRows) lane = l;
            }
            if (lane < 0) {                                // warp full: next warp, maybe next tile
                if (++wi == nwarps) { wi = 0; tile_start.push_back(pos); }
                std::fill(used, used + 32, static_cast<int8_t>(0));
                lane = 0;
            }
            row_thread[pos] = wi * 32 + lane;
            row_sub[pos] = used[lane];
            used[lane] = static_cast<int8_t>(used[lane] + c);
            next = (lane + 1) & 31;
        }
    }
    const int64_t ntiles = static_cast<int64_t>(tile_start.size());
    tile_start.push_back(n_dst);
    if (ntiles > INT32_MAX / 2) { plan.why = "too many tiles"; return; }
    plan.lpr = lpr; plan.kpl = kpl; plan.rows_per_tile = R; plan.nct = nct; plan.packed = packed;
    if (packed) plan.rowslot.assign(static_cast<size_t>(ntiles) * kSubRows * nct, -1);
    plan.tiles.resize(static_cast<size_t>(ntiles));
    plan.wplan.assign(static_cast<size_t>(ntiles) * kpl * nct, 0.0);
    plan.iplan.assign(static_cast<size_t>(ntiles) * kpl * nct, 0);

    // Tiles are independent: a few host threads each build a contiguous range of tiles into
    // their own segment list; the lists are stitched together afterwards.
    struct Part {
        int64_t t0 = 0, t1 = 0;
        std::vector<Seg> segs;
        int64_t sum_cols = 0, sum_blocks = 0, sum_elems = 0, max_elems = 0;
        int32_t max_segs = 0;
        bool too_big = false, failed = false;
    };
    auto work = [&](Part &out) {
    std::vector<int32_t> cols;
    for (int64_t t = out.t0; t < out.t1; ++t) {
        const int64_t r0 = tile_start[t], r1 = tile_start[t + 1];       // positions in the row order
        if (!order) {
            cols.assign(csr.col.begin() + csr.rowptr[r0], csr.col.begin() + csr.rowptr[r1]);
        } else {
            cols.clear();
            for (int64_t pos = r0; pos < r1; ++pos) {
                const int64_t r = row_at(pos);
                cols.insert(cols.end(), csr.col.begin() + csr.rowptr[r], csr.col.begin() + csr.rowptr[r + 1]);
            }
        }
        std::sort(cols.begin(), cols.end());
        cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
        out.sum_cols += static_cast<int64_t>(cols.size());

        TileDesc &td = plan.tiles[t];
        td = TileDesc{};
        td.row0 = static_cast<int32_t>(r0);
        td.nrows = static_cast<int32_t>(r1 - r0);
        td.seg0 = static_cast<int32_t>(out.segs.size());   // index in this part; rebased when stitching
        int64_t cs = -1, ce = -1, last_block = -1;
        uint32_t off = 0;
        auto flush = [&]() {
            if (cs < 0) return;
            Seg sg{static_cast<uint32_t>(cs), off, static_cast<uint32_t>(ce - cs), 0};
            out.segs.push_back(sg);
            off += sg.len;
        };
        for (int32_t c : cols) {
            const int64_t blk = c / kSegAlign;
            if (blk != last_block) { ++out.sum_blocks; last_block = blk; }
            if (cs >= 0 && c < ce) continue;
            const int64_t s_al = blk * kSegAlign;
            const int64_t e_al = std::min<int64_t>((blk + 1) * kSegAlign, n_src);
            if (cs >= 0 && s_al - ce <= kSegGap) {
                ce = e_al;
            } else {
                flush();
                cs = s_al; ce = e_al;
            }
        }
        flush();
        td.nseg = static_cast<int32_t>(out.segs.size()) - td.seg0;
        td.elems = static_cast<int32_t>(off);
        out.max_segs = std::max(out.max_segs, td.nseg);
        out.max_elems = std::max<int64_t>(out.max_elems, off);
        out.sum_elems += off;
        if (off > 65535u) { out.too_big = true; return; }

        // ---- register image of the tile: which (thread, slot) holds which link
        const Seg *sb = out.segs.data() + td.seg0;
        const size_t tbase = static_cast<size_t>(t) * kpl * nct;
        auto local_index = [&](uint32_t c) -> uint32_t {      // footprint-local element of source column c
            int lo = 0, hi = td.nseg - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (sb[mid].src <= c) lo = mid; else hi = mid - 1;
            }
            return sb[lo].dst + (c - sb[lo].src);
        };
        // Link placement for one warp: lane `l` serves row slot l / lpr_ of the warp; the links of a
        // row slot wait in bucket[slot * 32 + bank] (bank = local index % 32 for 4-byte elements).
        // A row's links may sit in any (lane, slot) of its lane group -- the kernel sums them
        // all -- so per link slot a bipartite matching of lanes to banks spreads the warp-wide
        // shared-memory load over distinct banks.  Unplaced slots carry weight 0.
        struct Link { uint16_t li; double w; };
        std::vector<std::vector<Link>> bucket(32 * 32);
        int remaining[32];
        int32_t rep_any[32];                         // some link of the row slot (padding when a slot places nothing)
        auto reset_warp = [&]() {      // (the buckets are empty: a completed placement drains them)
            for (int i = 0; i < 32; ++i) { rep_any[i] = -1; remaining[i] = 0; }
        };
        auto add_link = [&](int slot, uint32_t li, double w) {
            bucket[static_cast<size_t>(slot) * 32 + (li & 31u)].push_back(Link{static_cast<uint16_t>(li), w});
            rep_any[slot] = static_cast<int32_t>(li);
            ++remaining[slot];
        };
        std::vector<Link> pool[32];                  // a row slot's links in ascending-src order
        // [nslots][32] candidate placements: in order / bank-matched / bank-matched + co-scheduled
        std::vector<uint16_t> s_li, m_li, c_li;
        std::vector<double> s_w, m_w, c_w;
        std::vector<uint8_t> s_have, m_have, c_have;
        // shared-memory wavefronts of a placement: per slot, the fullest bank counted in DISTINCT
        // addresses (lanes reading the same word are served by one broadcast)
        auto wavefronts = [&](const std::vector<uint16_t> &li, int nslots) -> int {
            int total = 0;
            for (int k = 0; k < nslots; ++k) {
                uint16_t a[32];
                std::copy(li.begin() + k * 32, li.begin() + k * 32 + 32, a);
                std::sort(a, a + 32);
                int cnt[32] = {0}, worst = 0;
                for (int i = 0; i < 32; ++i)
                    if (i == 0 || a[i] != a[i - 1]) worst = std::max(worst, ++cnt[a[i] & 31]);
                total += worst;
            }
            return total;
        };
        auto place_warp = [&](int lpr_, int nslots, int slot0, int thread0) -> bool {
            const int rows_in_warp = 32 / lpr_;
            const size_t cells = static_cast<size_t>(nslots) * 32;
            s_li.assign(cells, 0); m_li.assign(cells, 0); c_li.assign(cells, 0);
            s_w.assign(cells, 0.0); m_w.assign(cells, 0.0); c_w.assign(cells, 0.0);
            s_have.assign(cells, 0); m_have.assign(cells, 0); c_have.assign(cells, 0);
            if (ref_order) {
                // reference-order plans: no freedom -- lane l of a row holds links [l*nslots, (l+1)*nslots)
                // of the row's ascending-source list, slot k the k-th of them (the kernel chains them
                // in exactly that order); the free placements below are for the fast sums only
                for (int jr = 0; jr < rows_in_warp; ++jr) {
                    pool[jr].clear();
                    for (int b = 0; b < 32; ++b) {
                        auto &bk = bucket[static_cast<size_t>(jr) * 32 + b];
                        for (const Link &l : bk) pool[jr].push_back(l);
                        bk.clear();
                    }
                    std::sort(pool[jr].begin(), pool[jr].end(), [](const Link &x, const Link &y) { return x.li < y.li; });
                    for (size_t j = 0; j < pool[jr].size(); ++j) {
                        const size_t at = (j % nslots) * 32 + static_cast<size_t>(jr) * lpr_ + j / nslots;
                        s_li[at] = pool[jr][j].li; s_w[at] = pool[jr][j].w; s_have[at] = 1;
                    }
                }
                for (int k = 0; k < nslots; ++k) {
                    int32_t pad = -1;
                    for (int lane = 0; lane < 32 && pad < 0; ++lane)
                        if (s_have[k * 32 + lane]) pad = s_li[k * 32 + lane];
                    for (int lane = 0; lane < 32 && pad < 0; ++lane)
                        if (rep_any[lane / lpr_] >= 0) pad = rep_any[lane / lpr_];
                    if (pad < 0) pad = 0;
                    for (int lane = 0; lane < 32; ++lane) {
                        const size_t at = tbase + static_cast<size_t>(slot0 + k) * nct + thread0 + lane;
                        plan.wplan[at] = s_have[k * 32 + lane] ? s_w[k * 32 + lane] : 0.0;
                        plan.iplan[at] = s_have[k * 32 + lane] ? s_li[k * 32 + lane] : static_cast<uint16_t>(pad);
                    }
                }
                return true;
            }
            // in-order alternative: link j of a row slot -> (lane j % lpr_, slot j / lpr_).  It keeps
            // equal addresses of neighbouring rows in the same slot (up-sampling: broadcasts), which
            // the bank matching below cannot see
            for (int jr = 0; jr < rows_in_warp; ++jr) {
                pool[jr].clear();
                for (int b = 0; b < 32; ++b)
                    for (const Link &l : bucket[static_cast<size_t>(jr) * 32 + b]) pool[jr].push_back(l);
                std::sort(pool[jr].begin(), pool[jr].end(), [](const Link &x, const Link &y) { return x.li < y.li; });
                for (size_t j = 0; j < pool[jr].size(); ++j) {
                    const size_t at = (j / lpr_) * 32 + static_cast<size_t>(jr) * lpr_ + j % lpr_;
                    s_li[at] = pool[jr][j].li; s_w[at] = pool[jr][j].w; s_have[at] = 1;
                }
            }
            auto run_matching = [&](bool cosched, std::vector<uint16_t> &o_li, std::vector<double> &o_w,
                                    std::vector<uint8_t> &o_have) -> bool {
            // (re)fill the per-bank buckets from the row pools; descending, so pop_back ascends
            for (int jr = 0; jr < rows_in_warp; ++jr)
                for (const Link &l : pool[jr]) bucket[static_cast<size_t>(jr) * 32 + (l.li & 31u)].clear();
            for (int jr = 0; jr < rows_in_warp; ++jr) {
                remaining[jr] = static_cast<int>(pool[jr].size());
                for (size_t j = pool[jr].size(); j-- > 0;)
                    bucket[static_cast<size_t>(jr) * 32 + (pool[jr][j].li & 31u)].push_back(pool[jr][j]);
            }
            for (int k = 0; k < nslots; ++k) {
                uint32_t cand[32], rowmask[32];
                int order[32], ncand[32];
                for (int jr = 0; jr < rows_in_warp; ++jr) {      // banks in which the row still has links
                    uint32_t m = 0;
                    for (const Link &l : pool[jr])
                        if (!bucket[static_cast<size_t>(jr) * 32 + (l.li & 31u)].empty()) m |= 1u << (l.li & 31u);
                    rowmask[jr] = m;
                }
                for (int lane = 0; lane < 32; ++lane) {
                    cand[lane] = rowmask[lane / lpr_];
                    ncand[lane] = __builtin_popcount(cand[lane]);
                    order[lane] = lane;
                }
                std::stable_sort(order, order + 32, [&](int x, int y) { return ncand[x] < ncand[y]; });
                int owner[32];
                int lane_bank[32];
                for (int b = 0; b < 32; ++b) { owner[b] = -1; lane_bank[b] = -1; }
                // a lane may only be matched while its row still has links left for this slot:
                // a row with fewer remaining links than lanes matches only that many lanes
                int quota[32];
                for (int jr = 0; jr < rows_in_warp; ++jr) quota[jr] = remaining[jr];
                // banks are tried fullest first, so a row drains its banks evenly and the later
                // slots still have a choice
                uint8_t pref[32][32], npref[32];          // a row's non-empty banks: fullest first, then by bank
                for (int jr = 0; jr < rows_in_warp; ++jr) {
                    uint8_t *pr = pref[jr];
                    const size_t base = static_cast<size_t>(jr) * 32;
                    int n = 0;
                    for (uint32_t m = rowmask[jr]; m; m &= m - 1) {
                        const int b = __builtin_ctz(m);
                        const size_t sz = bucket[base + b].size();
                        int at = n++;
                        while (at > 0 && bucket[base + pr[at - 1]].size() < sz) { pr[at] = pr[at - 1]; --at; }
                        pr[at] = static_cast<uint8_t>(b);
                    }
                    npref[jr] = static_cast<uint8_t>(n);
                }
                auto augment = [&](auto &&self, int lane, uint32_t &seen) -> bool {
                    const uint8_t *pr = pref[lane / lpr_];
                    const int n = npref[lane / lpr_];
                    for (int i = 0; i < n; ++i) {
                        const int b = pr[i];
                        if ((seen >> b) & 1u) continue;
                        seen |= 1u << b;
                        if (owner[b] < 0 || self(self, owner[b], seen)) { owner[b] = lane; return true; }
                    }
                    return false;
                };
                bool matched[32] = {false};
                for (int oi = 0; oi < 32; ++oi) {
                    const int lane = order[oi];
                    const int jr = lane / lpr_;
                    if (quota[jr] <= 0 || cand[lane] == 0) continue;
                    uint32_t seen = 0;
                    if (augment(augment, lane, seen)) { matched[lane] = true; --quota[jr]; }
                }
                for (int b = 0; b < 32; ++b) if (owner[b] >= 0) lane_bank[owner[b]] = b;
                // a bucket holds links of one bank: two lanes of a row matched to the same row's
                // buckets always differ in bank, so each pops its own link
                int load[32] = {0};
                Link chosen[32];
                bool have[32] = {false};
                for (int lane = 0; lane < 32; ++lane) {
                    if (!matched[lane] || lane_bank[lane] < 0) continue;
                    const int jr = lane / lpr_;
                    auto &bk = bucket[static_cast<size_t>(jr) * 32 + lane_bank[lane]];
                    if (bk.empty()) continue;            // bank taken by a same-row lane in a previous augmentation
                    chosen[lane] = bk.back(); bk.pop_back(); have[lane] = true;
                    --remaining[jr]; ++load[lane_bank[lane]];
                }
                for (int lane = 0; lane < 32; ++lane) {
                    if (have[lane]) continue;
                    const int jr = lane / lpr_;
                    if (remaining[jr] <= 0) continue;
                    int best = -1;
                    for (int b = 0; b < 32; ++b)
                        if (!bucket[static_cast<size_t>(jr) * 32 + b].empty() && (best < 0 || load[b] < load[best])) best = b;
                    auto &bk = bucket[static_cast<size_t>(jr) * 32 + best];
                    chosen[lane] = bk.back(); bk.pop_back(); have[lane] = true;
                    --remaining[jr]; ++load[best];
                }
                // Co-scheduling: neighbouring rows often link the SAME source element (the shared
                // boundary column of two conservative cells, the common corner of bilinear cells).
                // Lanes reading one address are served by one broadcast, but only if they read it
                // in the same slot -- so whenever a lane takes an address that another row of the
                // warp also has, a lane of that row takes it now as well (its previous pick goes
                // back to its bucket).  Without this the twins are consumed at different times and
                // pile up in a few banks in the last slots.
                bool locked[32] = {false};
                for (int lane = 0; cosched && lane < 32; ++lane) {
                    if (!have[lane] || locked[lane]) continue;
                    const uint16_t a = chosen[lane].li;
                    const int b = a & 31, jr0 = lane / lpr_;
                    for (int jr = 0; jr < rows_in_warp; ++jr) {
                        if (jr == jr0) continue;
                        auto &bk = bucket[static_cast<size_t>(jr) * 32 + b];
                        size_t at = bk.size();
                        for (size_t i = 0; i < bk.size(); ++i)
                            if (bk[i].li == a) { at = i; break; }
                        if (at == bk.size()) continue;
                        int pick = -1;
                        for (int l2 = jr * lpr_; l2 < (jr + 1) * lpr_ && pick < 0; ++l2)
                            if (!have[l2]) pick = l2;
                        for (int l2 = jr * lpr_; l2 < (jr + 1) * lpr_ && pick < 0; ++l2)
                            if (!locked[l2]) pick = l2;
                        if (pick < 0) continue;
                        const Link twin = bk[at];
                        bk.erase(bk.begin() + static_cast<std::ptrdiff_t>(at));
                        --remaining[jr];
                        if (have[pick]) {
                            bucket[static_cast<size_t>(jr) * 32 + (chosen[pick].li & 31)].push_back(chosen[pick]);
                            ++remaining[jr];
                        }
                        chosen[pick] = twin; have[pick] = true;
                        locked[pick] = locked[lane] = true;
                    }
                }
                for (int lane = 0; lane < 32; ++lane)
                    if (have[lane]) {
                        o_li[k * 32 + lane] = chosen[lane].li; o_w[k * 32 + lane] = chosen[lane].w; o_have[k * 32 + lane] = 1;
                    }
            }
            for (int jr = 0; jr < rows_in_warp; ++jr)
                if (remaining[jr] != 0) return false;
            return true;
            };
            if (!run_matching(false, m_li, m_w, m_have) || !run_matching(true, c_li, c_w, c_have)) return false;
            // padding (weight 0) broadcasts an address the warp reads in this slot anyway: no
            // extra wavefront, and the value belongs to a row of this warp, whose non-finite
            // vote is warp-wide -- a padded slot never drags in a NaN the warp does not own
            auto pad_out = [&](std::vector<uint16_t> &li, const std::vector<uint8_t> &hv) {
                for (int k = 0; k < nslots; ++k) {
                    int32_t pad = -1;
                    for (int lane = 0; lane < 32 && pad < 0; ++lane)
                        if (hv[k * 32 + lane]) pad = li[k * 32 + lane];
                    for (int lane = 0; lane < 32 && pad < 0; ++lane)
                        if (rep_any[lane / lpr_] >= 0) pad = rep_any[lane / lpr_];
                    if (pad < 0) pad = 0;
                    for (int lane = 0; lane < 32; ++lane)
                        if (!hv[k * 32 + lane]) li[k * 32 + lane] = static_cast<uint16_t>(pad);
                }
            };
            pad_out(m_li, m_have);
            pad_out(c_li, c_have);
            pad_out(s_li, s_have);
            const int cost_s = wavefronts(s_li, nslots), cost_m = wavefronts(m_li, nslots), cost_c = wavefronts(c_li, nslots);
            const int pick = (cost_s <= cost_m && cost_s <= cost_c) ? 0 : (cost_m <= cost_c ? 1 : 2);
            const std::vector<uint16_t> &li = pick == 0 ? s_li : pick == 1 ? m_li : c_li;
            const std::vector<double> &w = pick == 0 ? s_w : pick == 1 ? m_w : c_w;
            for (int k = 0; k < nslots; ++k)
                for (int lane = 0; lane < 32; ++lane) {
                    const size_t at = tbase + static_cast<size_t>(slot0 + k) * nct + thread0 + lane;
                    plan.wplan[at] = w[k * 32 + lane];
                    plan.iplan[at] = li[k * 32 + lane];
                }
            return true;
        };

        if (packed) {
            // links j of a row go to its sub-row u0 + j / 4 (any slot of that sub-row)
            const size_t sbase = static_cast<size_t>(t) * kSubRows * nct;
            const int nwarps = nct / 32;
            int64_t pos = r0;
            for (int wi = 0; wi < nwarps; ++wi) {
                const int64_t pos0 = pos;
                while (pos < r1 && row_thread[pos] / 32 == wi) ++pos;
                int32_t thread_first[32];
                for (int32_t &v : thread_first) v = -1;
                for (int64_t q = pos0; q < pos; ++q) {
                    const int64_t r = row_at(q);
                    const int32_t thread = row_thread[q], u0 = row_sub[q];
                    const int32_t a = csr.rowptr[r], b = csr.rowptr[r + 1];
                    const int32_t c = std::max(1, (b - a + kSubLinks - 1) / kSubLinks);
                    plan.rowslot[sbase + static_cast<size_t>(u0) * nct + thread] = static_cast<int32_t>(r);
                    for (int32_t u = 1; u < c; ++u) plan.rowslot[sbase + static_cast<size_t>(u0 + u) * nct + thread] = -2;
                    if (b > a && thread_first[thread & 31] < 0)
                        thread_first[thread & 31] = static_cast<int32_t>(local_index(static_cast<uint32_t>(csr.col[a])));
                }
                for (int u = 0; u < kSubRows; ++u) {
                    reset_warp();
                    for (int lane = 0; lane < 32; ++lane) rep_any[lane] = thread_first[lane];
                    for (int64_t q = pos0; q < pos; ++q) {
                        const int32_t lane = row_thread[q] & 31, u0 = row_sub[q];
                        const int64_t r = row_at(q);
                        const int32_t a = csr.rowptr[r], b = csr.rowptr[r + 1];
                        const int32_t j0 = a + (u - u0) * kSubLinks;
                        if (u < u0 || j0 >= b) continue;
                        for (int32_t j = std::min(b, j0 + kSubLinks) - 1; j >= j0; --j)
                            add_link(lane, local_index(static_cast<uint32_t>(csr.col[j])), csr.val[j]);
                    }
                    if (!place_warp(1, kSubLinks, u * kSubLinks, wi * 32)) { out.failed = true; return; }
                }
            }
            continue;
        }
        const int rows_per_warp = 32 / lpr;
        const int nwarps = nct / 32;
        for (int wi = 0; wi < nwarps; ++wi) {
            reset_warp();
            for (int jr = 0; jr < rows_per_warp; ++jr) {
                const int64_t pos = r0 + static_cast<int64_t>(wi) * rows_per_warp + jr;
                if (pos >= r1) continue;
                const int64_t r = row_at(pos);
                const int32_t a = csr.rowptr[r], b = csr.rowptr[r + 1];
                for (int32_t j = b - 1; j >= a; --j)            // pushed in reverse: popped ascending
                    add_link(jr, local_index(static_cast<uint32_t>(csr.col[j])), csr.val[j]);
            }
            if (!place_warp(lpr, kpl, 0, wi * 32)) { out.failed = true; return; }
        }
    }
    };

    const int nthreads = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>({s.plan_threads, 16, ntiles / 32})));
    std::vector<Part> parts(static_cast<size_t>(nthreads));
    for (int i = 0; i < nthreads; ++i) {
        parts[i].t0 = ntiles * i / nthreads;
        parts[i].t1 = ntiles * (i + 1) / nthreads;
    }
    parallel_for(nthreads, nthreads, [&](int64_t i) { work(parts[i]); });
    int64_t sum_blocks = 0;
    for (Part &pt : parts) {
        if (pt.too_big) { plan.why = "tile footprint exceeds 16-bit local indices"; return; }
        if (pt.failed) { plan.why = "internal: link placement failed"; return; }
        const int32_t base = static_cast<int32_t>(plan.segs.size());
        for (int64_t t = pt.t0; t < pt.t1; ++t) plan.tiles[t].seg0 += base;
        plan.segs.insert(plan.segs.end(), pt.segs.begin(), pt.segs.end());
        plan.sum_tile_cols += pt.sum_cols;
        plan.sum_tile_elems += pt.sum_elems;
        plan.max_tile_elems = std::max(plan.max_tile_elems, pt.max_elems);
        plan.max_tile_segments = std::max(plan.max_tile_segments, pt.max_segs);
        sum_blocks += pt.sum_blocks;
    }
    // Staging pays when footprints are compact runs; otherwise the gather kernel is used.
    const double avg_seg = plan.segs.empty() ? 0.0
                                             : static_cast<double>(plan.sum_tile_elems) / plan.segs.size();
    if (plan.max_tile_elems > 25600) { plan.why = "tile footprint too large for two f32 stages"; return; }
    if (!plan.segs.empty() && avg_seg < 16.0) { plan.why = "source footprint is scattered (short segments)"; return; }
    if (plan.sum_tile_elems > 2 * sum_blocks * kSegAlign + 1024) {
        plan.why = "staged footprint over-reads the touched sectors";
        return;
    }
    if (order && !packed) plan.rowmap = *order;      // packed plans carry row ids in rowslot
    plan.reordered = order != nullptr;
    plan.nrows = n_dst;
    plan.ok = true;
}

// staged cost of one batch row in element-equivalents: bytes moved + ~64 elements per bulk copy
static double plan_cost(const HostPlan &p)
{
    return static_cast<double>(p.sum_tile_elems) + 64.0 * static_cast<double>(p.segs.size());
}

// Link slots the packed layout spends on this operator (4*ceil(nnz/4) per row, at least one
// sub-row), or -1 when a row does not fit a thread.
int64_t packed_slots(const HostCsr &csr)
{
    if (csr.max_row_nnz > kSubRows * kSubLinks) return -1;
    int64_t slots = 0;
    for (int64_t r = 0; r < csr.n_dst; ++r) {
        const int32_t nnz = csr.rowptr[r + 1] - csr.rowptr[r];
        slots += kSubLinks * std::max(1, (nnz + kSubLinks - 1) / kSubLinks);
    }
    return slots;
}

// Every operator whose rows fit (<= 16 links) packs: such operators are dominated by the
// destination side, and four rows per thread amortise the per-row loop / barrier / epilogue
// instructions that bound the lane-per-row layout there (measured on B200: bilinear
// 1440x721 -> 3600x1800 2841 -> 5141 GB/s, 1:1 conservative 3845 -> 6096, 75 ocean levels
// 2665 -> 5490; bilinear down-sampling within 2 %).
bool prefer_packed(const PlanSettings &s, int64_t slots_packed)
{
    return slots_packed >= 0 && s.packed != 0;
}

void build_plan(const HostCsr &csr, int32_t force_lpr, int32_t force_kpl, int32_t nct, bool ref_order,
                const PlanSettings &s, HostPlan &plan, const std::vector<int32_t> *subset)
{
    const bool packed = force_lpr == -1;       // -1: packed layout requested (see smm_create_levels)
    if (packed) { force_lpr = 0; force_kpl = 0; }
    build_plan_rows(csr, force_lpr, force_kpl, nct, subset, packed, ref_order, s, plan);
    if (plan.lpr == 0 || csr.col.empty() || (subset && subset->empty())) return;
    // natural order good enough: footprints within 30 % of the columns actually touched
    if (plan.ok && plan_cost(plan) <= 1.3 * static_cast<double>(plan.sum_tile_cols)) return;
    // otherwise try rows sorted by the mean source address of their links
    const int64_t n_rows = subset ? static_cast<int64_t>(subset->size()) : csr.n_dst;
    std::vector<int32_t> order(static_cast<size_t>(n_rows));
    if (subset) order = *subset; else std::iota(order.begin(), order.end(), 0);
    std::vector<double> key(static_cast<size_t>(csr.n_dst), 1e300);
    for (int32_t r : order) {
        const int32_t a = csr.rowptr[r], b = csr.rowptr[r + 1];
        double sum = 0.0;
        for (int32_t j = a; j < b; ++j) sum += csr.col[j];
        key[r] = b > a ? sum / (b - a) : 1e300;          // empty rows last
    }
    std::stable_sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return key[x] < key[y]; });
    HostPlan alt;
    build_plan_rows(csr, force_lpr, force_kpl, nct, &order, packed, ref_order, s, alt);
    if (alt.ok && (!plan.ok || plan_cost(alt) < 0.8 * plan_cost(plan))) plan = std::move(alt);
}

// Rows above the packed layout's 16 links, in ascending order.
void long_rows(const HostCsr &csr, std::vector<int32_t> &long_rows_out, std::vector<int32_t> &short_rows_out)
{
    long_rows_out.clear();
    short_rows_out.clear();
    for (int64_t r = 0; r < csr.n_dst; ++r)
        (csr.rowptr[r + 1] - csr.rowptr[r] > kSubRows * kSubLinks ? long_rows_out : short_rows_out).push_back(static_cast<int32_t>(r));
}

void parallel_for(int threads, int64_t n, const std::function<void(int64_t)> &fn)
{
    if (threads <= 1) {
        for (int64_t i = 0; i < n; ++i) fn(i);
        return;
    }
    std::atomic<int64_t> next{0};
    std::vector<std::thread> pool;
    for (int t = 0; t < threads; ++t)
        pool.emplace_back([&]() { for (int64_t i = next.fetch_add(1); i < n; i = next.fetch_add(1)) fn(i); });
    for (auto &th : pool) th.join();
}

void build_compact(const HostCsr &csr, int32_t block_cols, CompactPlan &out)
{
    out = CompactPlan{};
    std::vector<int32_t> rank(static_cast<size_t>(csr.n_src), -1);
    for (int32_t c : csr.col) rank[c] = 0;
    const int64_t nblk = (csr.n_src + block_cols - 1) / block_cols;
    out.blk_ptr.assign(static_cast<size_t>(nblk) + 1, 0);
    for (int64_t c = 0; c < csr.n_src; ++c) {
        if (rank[c] < 0) continue;
        rank[c] = static_cast<int32_t>(out.tcols.size());
        out.tcols.push_back(static_cast<int32_t>(c));
        ++out.blk_ptr[c / block_cols + 1];
    }
    for (int64_t i = 0; i < nblk; ++i) out.blk_ptr[i + 1] += out.blk_ptr[i];
    out.rcol.resize(csr.col.size());
    for (size_t j = 0; j < csr.col.size(); ++j) out.rcol[j] = rank[csr.col[j]];
}

}  // namespace smm
