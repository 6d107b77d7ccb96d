// Host-side planning: regions -> counting tiles, regions -> BGZF fetch segments.
#pragma once
#include <cstdint>
#include <vector>

#include "bamio.h"
#include "pool.h"

namespace bsg {

enum Mode { MODE_COUNT = 0, MODE_PROFILE = 1, MODE_COVERAGE = 2 };

struct Regions {            // parseRegions' result (src/bamsignals.cpp:92-135) with chromosome names resolved
    int64_t R = 0;
    std::vector<int32_t> rid, loc, width;
    std::vector<int8_t> strand;
    // indices in (rid, loc) order — the std::sort of src/bamsignals.cpp:246; computed once (sorted_order()) and shared
    // by the tile builder and the fetch planner
    mutable std::vector<int64_t> order;
    const std::vector<int64_t>& sorted_order() const;
};

struct HostTiles {          // one row per counting tile, in (rid, loc) order
    std::vector<int32_t> rid, loc, len, strand;
    std::vector<int64_t> out_off;      // offset of the tile's ints in the CALLER's flat layout (bsg_output_layout order)
    std::vector<int64_t> region;       // index of the region the tile belongs to
    std::vector<int32_t> ints;         // output ints the tile owns
    int max_tile_ints = 0;  // largest number of output ints any tile owns
    int64_t size() const { return int64_t(rid.size()); }
};

// Resolve seqlevel names against the BAM header; throws BSG_ENOCHROM with the reference's message (:119).
void resolve_regions(const BamFile& bam, int64_t R, const char* const* seq_levels, int32_t n_levels,
                     const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                     Regions* out);

// Cut regions into tiles of at most tile_ints output ints.  A profile tile is a bin-aligned sub-interval counted from
// the region's 5' end (loc for +/*, end for -, because of src/bamsignals.cpp:357); a coverage tile is any
// sub-interval (the clamp at :424/:432 makes its prefix sum self-contained); bamCount regions are never cut.  With ss a
// bin (a base for coverage) owns two output ints, sense and antisense.
void make_tiles(const Regions& rg, Mode mode, int32_t binsize, int ss, const int64_t* out_offsets, int tile_ints,
                HostTiles* tiles);

struct Segment {            // an independently inflatable + walkable piece of the file
    uint64_t vbeg = 0, vend = 0;       // record-aligned virtual offsets
    std::vector<BlockInfo> blocks;     // consecutive BGZF blocks covering [vbeg, vend)
    uint64_t usize = 0;                // sum of isize over blocks
    uint64_t ubeg = 0, uend = 0;       // first record starts at ubeg, walk ends at uend (offsets in the concatenation)
    uint64_t csize = 0;                // compressed bytes
};

struct QueryInterval {      // one index query of the planner, after the merge: [beg, end) on contig rid
    int32_t rid;
    int64_t beg, end;
};

// Regions (+/- ext) -> merged index queries -> record-aligned virtual-offset ranges -> segments of roughly
// seg_cbytes compressed bytes, cut at index entry points; BGZF block headers are scanned on the pool.
// queries (optional) receives the merged index queries in (rid, beg) order: every record that overlaps one of them
// is inside the planned segments.
void plan_fetch(const BamFile& bam, const Regions& rg, int64_t ext, uint64_t seg_cbytes, Pool& pool,
                std::vector<Segment>* segs, std::vector<QueryInterval>* queries = nullptr);

}  // namespace bsg
