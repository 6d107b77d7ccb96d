#include "plan.h"

#include <algorithm>
#include <cstdlib>
#include <exception>
#include <mutex>
#include <numeric>

namespace bsg {

void resolve_regions(const BamFile& bam, int64_t R, const char* const* seq_levels, int32_t n_levels,
                     const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                     Regions* out) {
    if (R < 0 || (R > 0 && (!seq_idx || !loc || !width || !strand || !seq_levels))) fail(BSG_EARG, "invalid region arrays");
    std::vector<int> level_rid(size_t(std::max(n_levels, 0)), -2);
    out->R = R;
    out->rid.resize(R); out->loc.assign(loc, loc + R); out->width.assign(width, width + R); out->strand.assign(strand, strand + R);
    for (int64_t i = 0; i < R; ++i) {
        const int lv = seq_idx[i];
        if (lv < 0 || lv >= n_levels) fail(BSG_EARG, "region refers to a seqlevel index out of range");
        if (level_rid[lv] == -2) {
            level_rid[lv] = bam.name2id(seq_levels[lv]);                                      // getRefId, :26-28
            if (level_rid[lv] < 0)
                fail(BSG_ENOCHROM, std::string("chromosome ") + seq_levels[lv] + " not present in the bam file");   // :119
        }
        if (width[i] < 0) fail(BSG_EARG, "negative region width");
        out->rid[i] = level_rid[lv];
    }
}

const std::vector<int64_t>& Regions::sorted_order() const {
    if (int64_t(order.size()) == R) return order;
    order.resize(R);
    std::iota(order.begin(), order.end(), int64_t(0));
    bool sorted = true;
    for (int64_t i = 1; i < R && sorted; ++i)
        sorted = rid[i - 1] < rid[i] || (rid[i - 1] == rid[i] && loc[i - 1] <= loc[i]);
    if (!sorted) {
        // Stable LSD radix sort of packed keys (rid, loc) with the index as payload: 11-bit digits over the bits that
        // are actually used (the span of loc + what the largest rid needs: 3 passes on a human genome), so 100 k regions take about a millisecond
        // instead of the 7 ms of a comparison sort.  Ties keep input order, like the (rid, loc, index) key did.
        struct KV { uint64_t key; int64_t idx; };
        std::vector<KV> a(R), b(R);
        int32_t lo = loc[0], hi = loc[0];
        for (int64_t i = 1; i < R; ++i) { lo = std::min(lo, loc[i]); hi = std::max(hi, loc[i]); }
        int lbits = 0;                                   // loc - lo needs lbits bits, the rid sits right above them
        while (lbits < 32 && ((uint64_t(int64_t(hi) - lo)) >> lbits) != 0) ++lbits;
        uint64_t all = 0;
        for (int64_t i = 0; i < R; ++i) {
            a[i] = KV{uint64_t(uint32_t(rid[i])) << lbits | uint64_t(int64_t(loc[i]) - lo), i};
            all |= a[i].key;
        }
        int bits = 0;
        while (bits < 64 && (all >> bits) != 0) ++bits;
        constexpr int kDigit = 11;
        std::vector<int64_t> cnt(size_t(1) << kDigit);
        for (int sh = 0; sh < bits; sh += kDigit) {
            std::fill(cnt.begin(), cnt.end(), 0);
            for (int64_t i = 0; i < R; ++i) ++cnt[(a[i].key >> sh) & ((1u << kDigit) - 1)];
            int64_t run = 0;
            for (auto& c : cnt) { const int64_t t = c; c = run; run += t; }
            for (int64_t i = 0; i < R; ++i) b[cnt[(a[i].key >> sh) & ((1u << kDigit) - 1)]++] = a[i];
            a.swap(b);
        }
        for (int64_t i = 0; i < R; ++i) order[i] = a[i].idx;
    }
    return order;
}

void make_tiles(const Regions& rg, Mode mode, int32_t binsize, int ss, const int64_t* out_offsets, int tile_ints,
                HostTiles* t) {
    const int64_t R = rg.R;
    const int mult = ss ? 2 : 1;
    const std::vector<int64_t>& order = rg.sorted_order();
    int64_t cur_region = 0;
    t->rid.reserve(R); t->loc.reserve(R); t->len.reserve(R); t->strand.reserve(R);
    t->out_off.reserve(R); t->region.reserve(R); t->ints.reserve(R);
    auto push = [&](int32_t rid, int64_t loc, int64_t len, int32_t strand, int64_t off, int64_t ints) {
        t->rid.push_back(rid); t->loc.push_back(int32_t(loc)); t->len.push_back(int32_t(len));
        t->strand.push_back(strand); t->out_off.push_back(off);
        t->region.push_back(cur_region); t->ints.push_back(int32_t(ints));
        t->max_tile_ints = std::max<int64_t>(t->max_tile_ints, ints);
    };
    for (int64_t oi = 0; oi < R; ++oi) {
        const int64_t i = order[oi];
        cur_region = i;
        const int64_t loc = rg.loc[i], width = rg.width[i], base = out_offsets[i];
        const int32_t strand = rg.strand[i];
        if (mode == MODE_COUNT) { push(rg.rid[i], loc, width, strand, base, mult); continue; }
        if (width == 0) continue;
        const int64_t bs = mode == MODE_COVERAGE ? 1 : binsize;
        const int64_t nb = (width + bs - 1) / bs;
        const int64_t tb = std::max<int64_t>(1, tile_ints / mult);          // bins per tile
        for (int64_t k = 0; k * tb < nb; ++k) {
            const int64_t rel_lo = k * tb * bs, rel_hi = std::min(width, (k + 1) * tb * bs);
            const int64_t tloc = strand < 0 ? loc + width - rel_hi : loc + rel_lo;
            const int64_t bins = (rel_hi - rel_lo + bs - 1) / bs;
            push(rg.rid[i], tloc, rel_hi - rel_lo, strand, base + mult * k * tb, mult * bins);
        }
    }
}

namespace {

// The BGZF header chain of one segment, one block per step(): the next header's place is only known once this one has
// been read, and every hop is a cache miss into the page cache - so a worker advances several segments in turn and
// asks for each one's next header line (and the trailer that sits right in front of it) before moving on.
struct SegmentScan {
    const BamFile* bamp;
    Segment* s;
    uint64_t c, cend, uoff_end;
    bool closed = false;
    SegmentScan(const BamFile& b, Segment* seg) : bamp(&b), s(seg), c(seg->vbeg >> 16), cend(seg->vend >> 16), uoff_end(seg->vend & 0xffff) {
        s->ubeg = s->vbeg & 0xffff;
        s->usize = 0; s->csize = 0;
        touch();
    }
    void touch() const {
        const BamFile& bam = *bamp;
        if (c + 64 < bam.size()) { __builtin_prefetch(bam.data() + (c >= 8 ? c - 8 : 0)); __builtin_prefetch(bam.data() + c + 17); }
    }
    bool step() {                                   // false when the segment is finished
        const BamFile& bam = *bamp;
        if (c == cend && uoff_end == 0) { s->uend = s->usize; closed = true; return finish(); }
        if (c > cend) return finish();
        BlockInfo b;
        if (!bam.block_at(c, &b)) return finish();
        s->blocks.push_back(b);
        s->usize += b.isize; s->csize += b.csize;
        if (c == cend) {
            if (uoff_end > b.isize) fail(BSG_EFORMAT, "index offset beyond its BGZF block in " + bam.path());
            s->uend = s->usize - b.isize + uoff_end; closed = true; return finish();
        }
        c += b.csize;
        touch();
        return true;
    }
    bool finish() {
        const BamFile& bam = *bamp;
        if (!closed) fail(BSG_EFORMAT, "BAM index does not match the BGZF block structure of " + bam.path());
        if (!s->blocks.empty() && s->ubeg > s->blocks[0].isize) fail(BSG_EFORMAT, "index offset beyond its BGZF block in " + bam.path());
        if (s->blocks.empty()) { s->ubeg = s->uend = 0; }
        if (s->ubeg > s->uend) fail(BSG_EFORMAT, "inconsistent index offsets in " + bam.path());
        return false;
    }
};

void scan_segments(const BamFile& bam, Segment* segs, int64_t a, int64_t b) {
    constexpr int kLanes = 8;
    std::vector<SegmentScan> lane;
    lane.reserve(kLanes);
    int64_t next = a;
    while (next < b && int(lane.size()) < kLanes) lane.emplace_back(bam, &segs[next++]);
    while (!lane.empty())
        for (size_t i = 0; i < lane.size();) {
            if (lane[i].step()) { ++i; continue; }
            if (next < b) lane[i++] = SegmentScan(bam, &segs[next++]);
            else { lane[i] = lane.back(); lane.pop_back(); }
        }
}

}  // namespace

void plan_fetch(const BamFile& bam, const Regions& rg, int64_t ext, uint64_t seg_cbytes, Pool& pool,
                std::vector<Segment>* segs, std::vector<QueryInterval>* queries) {
    const bool dbg = getenv("BSG_DEBUG") != nullptr;
    double t0 = now_ms();
    auto lap = [&](const char* what) { if (dbg) { const double t = now_ms(); fprintf(stderr, "[bsg]   plan: %s %.1f ms\n", what, t - t0); t0 = t; } };
    using Q = QueryInterval;
    std::vector<Q> qs;
    qs.reserve(rg.R);
    for (int64_t i : rg.sorted_order()) {                        // (rid, loc) order == (rid, beg) order: ext is constant
        if (rg.width[i] == 0) continue;
        const int64_t b = std::max<int64_t>(0, int64_t(rg.loc[i]) - ext), e = int64_t(rg.loc[i]) + rg.width[i] + ext;
        if (e > b) qs.push_back(Q{rg.rid[i], b, e});
    }
    lap("sort regions");
    std::vector<VRange> ranges;
    for (size_t i = 0; i < qs.size();) {
        Q cur = qs[i];
        size_t j = i + 1;
        // queries closer than a linear-index window read the same records: ask the index once
        const int64_t gap = 16384;
        for (; j < qs.size() && qs[j].rid == cur.rid && qs[j].beg <= cur.end + gap; ++j) cur.end = std::max(cur.end, qs[j].end);
        bam.query(cur.rid, cur.beg, cur.end, &ranges);
        if (queries) queries->push_back(cur);
        i = j;
    }
    lap("index queries");
    // queries were asked in (rid, beg) order, so on a coordinate-sorted file the ranges usually come out sorted already
    const auto by_beg = [](const VRange& a, const VRange& b) { return a.beg < b.beg; };
    if (!std::is_sorted(ranges.begin(), ranges.end(), by_beg)) std::sort(ranges.begin(), ranges.end(), by_beg);
    std::vector<VRange> merged;
    for (const VRange& r : ranges) {
        if (r.end <= r.beg) continue;
        // Ranges that touch the same or neighbouring BGZF blocks are fused: fetching is block-granular, so a gap
        // shorter than a block would only make both neighbours inflate the shared blocks twice.
        if (!merged.empty() && (r.beg >> 16) <= (merged.back().end >> 16))
            merged.back().end = std::max(merged.back().end, r.end);
        else merged.push_back(r);
    }
    const std::vector<uint64_t>& ent = bam.entry_points();
    segs->reserve(segs->size() + merged.size());
    auto it = ent.begin();
    for (const VRange& r : merged) {
        uint64_t cur = r.beg;
        // only a range longer than a segment can be split: the others (most of a region-list query) never touch the
        // entry-point table; merged ranges ascend, so the search for the next long one starts where the last one ended
        if ((r.end >> 16) - (cur >> 16) >= seg_cbytes) {
            it = std::upper_bound(it, ent.end(), cur);
            for (; it != ent.end() && *it < r.end; ++it)
                if ((*it >> 16) - (cur >> 16) >= seg_cbytes) {
                    Segment s; s.vbeg = cur; s.vend = *it; segs->push_back(std::move(s));
                    cur = *it;
                }
        }
        Segment s; s.vbeg = cur; s.vend = r.end; segs->push_back(std::move(s));
    }
    lap("merge + split");
    std::mutex em; Error first{0, ""};
    const int64_t grain = std::max<int64_t>(1, int64_t(segs->size()) / (int64_t(pool.size()) * 8));
    pool.parallel_for(int64_t(segs->size()), grain, [&](int64_t a, int64_t b, int) {
        try { scan_segments(bam, segs->data(), a, b); }
        catch (Error& e) { std::lock_guard<std::mutex> g(em); if (!first.code) first = e; }
        catch (std::exception& e) {          // nothing may escape a pool thread
            std::lock_guard<std::mutex> g(em);
            if (!first.code) first = Error{BSG_ENOMEM, std::string("block scan failed: ") + e.what()};
        }
    });
    lap("block scan");
    if (first.code) throw first;
}

}  // namespace bsg
