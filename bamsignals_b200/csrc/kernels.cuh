// Device-side data layout and kernel launchers of the counting path (sm_100a).
//
// HBM layout (all arrays cudaMalloc-aligned, SoA so that every kernel's loads and stores are coalesced):
//   raw batch      uint8  raw[]         uncompressed BAM record bytes of one staged batch (+16 B slack)
//                  uint32 offs[n+1]     byte offset of every record's block_size field; offs[n] = end of last record
//   read table     int32  tid[N] pos[N]  (8 B / read) the join key: rows are in file order = sorted by (tid, pos)
//                  int32  c0[N] c1[N]    (8 B / read) pileup: c0 = 5'/midpoint coordinate, c1 = 0 '+', 1 '-', -1 dropped
//                                       coverage: [c0,c1] = inclusive interval, dropped reads get c0 > c1 sentinels;
//                                       strand-specific coverage: c1 = ~end for reverse reads, dropped reads c0 = INT_MAX
//                                       (end, tlen, flag and mapq never leave the decode kernel's registers)
//   tiles          int32  rid loc len strand, int64 out_off, int64 cand_lo cand_hi   one row per region tile
//   result         int32  out[]         flat, bsg_output_layout() order; every element written exactly once
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bsg {

struct ReadTable {
    int32_t* tid;
    int32_t* pos;
    int32_t* c0;
    int32_t* c1;
};

struct TileTable {
    const int32_t* rid;
    const int32_t* loc;
    const int32_t* len;
    const int32_t* strand;
    const int64_t* out_off;
    int64_t* cand_lo;
    int64_t* cand_hi;
};

struct FilterParams {   // Pileupper / Coverager fields, src/bamsignals.cpp:296-303, :369-373
    int32_t mapqual;
    uint32_t required;
    uint32_t filtered;
    int32_t have_tlen, tmin, tmax;
    int32_t midpoint, shift;   // pileup
    int32_t tspan;             // coverage
};

// Device scalars shared by the kernels of one call.
struct DeviceScalars {
    int32_t halo_lo;     // pileup: max(c0 - pos) over kept reads; coverage: max(c1 - pos)
    int32_t halo_hi;     // pileup: max(pos - c0);                coverage: max(pos - c0)
    uint32_t status;     // bit 0: unsorted input, bit 1: corrupt record
    uint32_t pad;
    unsigned long long candidates;
    unsigned long long pad2[13];           // the counters below start on a 128-byte line
    unsigned long long kept[32 * 16];      // partial counts of reads that passed the filter: CTA i adds to slot i % 32,
};                                         // slots are 128 bytes apart (one L2 line each); the host sums them
constexpr int kKeptSlots = 32, kKeptStride = 16;
enum : uint32_t { STATUS_UNSORTED = 1u, STATUS_CORRUPT = 2u, STATUS_BAD_DEFLATE = 4u, STATUS_BAD_CRC = 8u };

constexpr int kTileInts = 8192;   // int32 per counting tile (32 KiB of shared memory)

// One staged batch of raw records for K1.
struct DecodeBatch {
    const uint8_t* raw;     // uncompressed record bytes (16-byte aligned, >= 64 bytes of slack behind the data)
    const uint32_t* offs;   // n + 1 byte offsets into raw
    int64_t row0;           // first read-table row of this batch
    int32_t n;              // records
    int32_t chunk0;         // first 256-record chunk of this batch in a multi-batch launch
};
#ifndef BSG_DECODE_THREADS
#define BSG_DECODE_THREADS 128
#endif
constexpr int kDecodeChunk = BSG_DECODE_THREADS;     // records per K1 CTA (one thread per record)

// K1 (decode + filter, fused): raw record bytes -> read table rows [row0, row0 + n).  Replaces bam_read1's field
// extraction, bam_endpos (src/bamsignals.cpp:16-18) and setRead (:326-346 pileup, :392-415 coverage).
// launch_decode: one batch (streaming path); launch_decode_table: every resident batch of a staged session in ONE
// launch (d_table lives in device memory).
// ss (coverage only): strand-specific coverage, reverse reads store ~c1 (DESIGN.md §12).
void launch_decode(const DecodeBatch& one, ReadTable t, bool coverage, bool ss, const FilterParams& p, DeviceScalars* sc, cudaStream_t s);
void launch_decode_table(const DecodeBatch* d_table, int n_batches, int total_chunks, ReadTable t, bool coverage, bool ss,
                         const FilterParams& p, DeviceScalars* sc, cudaStream_t s);

// Staged sessions (DESIGN.md §13): the resident record index, built once by launch_resident_index, and the fused pileup
// step that decodes only the rows near each tile.  A key is uint64: tid as uint32 in the high half, pos ^ 0x80000000 in
// the low half, so that unsigned order is lower_bound_tp's (tid as uint32, then pos as a signed number).
constexpr int kIndexStride = 32;    // one sampled key per 32 rows
constexpr int kSpanBuckets = 32;    // span bucket b = floor(log2(span))
struct IndexScalars {
    uint32_t status;                    // STATUS_UNSORTED / STATUS_CORRUPT as K1 detects them
    uint32_t n_long;                    // pass 1: rows appended to the long list
    long long reach;                    // max(0, max over rows of pos + span), a signed maximum
    uint32_t bucket_n[kSpanBuckets];    // rows per span bucket
    uint32_t bucket_max[kSpanBuckets];  // largest span per bucket
};
struct ResidentView {
    const DecodeBatch* batches;         // the session's batch table (device)
    int n_batches;
    int64_t n;                          // resident rows
    const unsigned long long* keys;     // keys[j] = key of row kIndexStride * j
    int64_t n_keys;
    const unsigned long long* long_key; // rows with span > long_span, in key order ...
    const int2* long_row;               // ... and where they are: (batch, record of the batch)
    int64_t n_long;
    uint32_t long_span;
};
// Key ranges around a tile [loc, loc + len): short rows with pos in [loc - s_lo, loc + len + s_hi), long rows likewise.
struct FusedHalos { int64_t s_lo, s_hi, l_lo, l_hi; };
// pass 0: keys[], status, reach, span buckets (isc zeroed before); pass 1: the long list, unsorted (isc->n_long zeroed)
void launch_resident_index(const DecodeBatch* d_table, int n_batches, int total_chunks, int pass, uint32_t long_span,
                           unsigned long long* keys, unsigned long long* long_key, int2* long_row, IndexScalars* isc, cudaStream_t s);
// K3f: tiles.cand_lo/hi = short row range, long_lo/hi = long list range; sc->candidates += rows examined
void launch_join_fused(const ResidentView& v, TileTable tiles, int64_t* long_lo, int64_t* long_hi, int64_t n_tiles,
                       const FusedHalos& h, DeviceScalars* sc, cudaStream_t s);
// K4f: bamProfile (binsize >= 1) or bamCount (binsize <= 0, one tile per region) straight from the raw records
void launch_pileup_fused(const ResidentView& v, TileTable tiles, const int64_t* long_lo, const int64_t* long_hi, int64_t n_tiles,
                         int ss, int32_t binsize, int max_tile_ints, const FilterParams& p, int32_t* out, cudaStream_t s);

// K0 (gpu_inflate): one BGZF block = one raw-DEFLATE stream of at most 64 KiB.
struct InflateBlock {
    uint32_t in_off;    // byte offset of the DEFLATE payload in the batch's compressed buffer
    uint32_t in_len;    // payload bytes (block size - header - 8)
    uint32_t out_off;   // byte offset in the batch's raw buffer
    uint32_t out_len;   // ISIZE
};
// d_spec (inflate_spec_words(n_blocks) uint32 of device memory, or null): per block, the record chain that starts at the
// block's first byte, followed while the block passes through shared memory: [n_blocks] record counts (0xffffffff = no
// usable chain), [n_blocks] where the chain lands, [n_blocks][1824] the records' offsets.  launch_walk links them.
void launch_inflate(const InflateBlock* d_blocks, int n_blocks, const uint8_t* d_comp, uint8_t* d_raw, uint32_t* d_spec, DeviceScalars* sc,
                    cudaStream_t s);
size_t inflate_spec_words(int n_blocks);
// BGZF blocks one launch keeps in flight on a device with n_sm SMs: batches that are a multiple of this leave no partly
// filled last generation.
int inflate_wave_blocks(int n_sm);
// CRC32 of every inflated block against the BGZF trailer (d_crc[i] belongs to d_blocks[i]).
void launch_crc32(const InflateBlock* d_blocks, const uint32_t* d_crc, int n_blocks, const uint8_t* d_raw, DeviceScalars* sc,
                  cudaStream_t s);
// Record-boundary walk between index entry points: walkers[w] = (begin, end) byte positions in d_raw, both record
// boundaries, each inside one run of consecutive blocks (d_blocks[0..n_blocks) in out_off order).  scheme 1 (or d_spec
// null): every span's chain is followed through global memory, twice; otherwise the spans are linked through the
// per-block chains the inflate kernel left in d_spec (launch_inflate) and only what those cannot cover is walked.
// Fills d_offs[0..total] (+ end sentinel) and *d_total; d_scratch: walk_scratch_words() uint32 of device memory.
void launch_walk(const uint8_t* d_raw, const uint2* d_walkers, int n_walkers, int scheme, const InflateBlock* d_blocks, int n_blocks,
                 const uint32_t* d_spec, uint32_t* d_scratch, uint32_t* d_counts, uint32_t* d_base, uint32_t* d_total, uint32_t* d_offs,
                 uint32_t end_pos, DeviceScalars* sc, cudaStream_t s);
size_t walk_scratch_words(int n_blocks, int n_walkers);

// dst[0] = *d_a, dst[1] = *d_b by a one-thread kernel; dst may be pinned host memory.  (Control values of the streaming
// pipeline - a batch's record count, the (tid, pos) frontier - must not travel as cudaMemcpy: a 4-byte copy queues behind
// the 32 MiB result copies on the device-to-host copy engine.)
void launch_publish_pair(const int32_t* d_a, const int32_t* d_b, int32_t* dst, cudaStream_t s);

// Result narrowing for the trip over PCIe: dst[i] = min(src[i], 255) for i < n, and every element outside 0..254 also
// goes, as (i, value), into ovf[0..cap) - which may be pinned host memory - through the counter *cnt (device memory,
// zero before the launch; it keeps counting past cap, entries beyond cap are dropped).  launch_publish_reset then copies the
// counter to *host_cnt (pinned host memory) and zeroes it.
void launch_pack_u8(const int32_t* d_src, int64_t n, uint8_t* d_dst, uint2* ovf, uint32_t cap, uint32_t* d_cnt, cudaStream_t s);
void launch_publish_reset(uint32_t* d_cnt, uint32_t* host_cnt, cudaStream_t s);

// K3: per tile, binary-search the (tid,pos)-sorted table for the candidate row range (the job of the sort + chunk
// + sweep in overlapAndPileup, src/bamsignals.cpp:246-285).
void launch_join(ReadTable t, int64_t n, TileTable tiles, int64_t n_tiles, const DeviceScalars* sc, cudaStream_t s);

// K4: bamCount (one or two counters per region; Pileupper::pileup with every read in bin 0, :349-363, :162-167)
void launch_count(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t* out,
                  DeviceScalars* sc, cudaStream_t s);
// K4: bamProfile (shared-memory bin histogram per tile; Pileupper::pileup, :349-363)
void launch_profile(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                    int max_tile_ints, int32_t* out, DeviceScalars* sc, cudaStream_t s);
// K5: bamCoverage (shared-memory difference array + block scan; Coverager::pileup + cumsum, :418-438, :464-470);
// ss: sense and antisense rows interleaved like a binsize-1 strand-specific profile (DESIGN.md §12)
void launch_coverage(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                     int32_t* out, DeviceScalars* sc, cudaStream_t s);

// K5r: bamCoverage as runs (DESIGN.md §10).  Per-tile arrays in tile order; region / rel come from the host, the rest is
// written by the kernels.  rfirst / rlast ([R], zeroed before the launch): tile-order run index of a region's first run
// and one past its last.
struct RunTiles {
    const int32_t* region;   // the caller's index of the tile's region
    const int32_t* rel;      // the tile's first output element, relative to its region (region orientation)
    int32_t* nnz;            // d[j] != 0 for j in [1, len)
    int32_t* first;          // coverage at the tile's first element
    int32_t* last;           // coverage at its last element
    int64_t* toff;           // tile-order index of the tile's first run start
    int64_t* rfirst;
    int64_t* rlast;
};
// With ss, rt, vt and the lists are those of a strand-specific profile (K4r below): row a of region i is list 2i + a.
// count pass + scans: run_off[0..lists] (device) = every list's span of runs in the caller's region order
void launch_coverage_runs(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                          RunTiles rt, const int32_t* vt, int64_t lists, int64_t* run_off, cudaStream_t s);
// write pass: values[k] and lengths[k] for k in [0, run_off[lists]); lengths must be zero before the launch
void launch_coverage_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                                RunTiles rt, const int32_t* vt, const int64_t* run_off, int32_t* lengths, int32_t* values,
                                cudaStream_t s);

// K4r: bamProfile as runs (DESIGN.md §11), over VIRTUAL tiles: row a (sense / antisense with ss) of the j-th of region
// i's n_i tiles, T_i its first tile, is virtual tile v = mult * T_i + a * n_i + j in list mult * i + a (mult = ss ? 2 : 1).
// rt is indexed by virtual tile and list (region = the list, rel = the tile's first bin relative to the region);
// vt[a * n_tiles + t] = v of row a of tile t, or NULL for the identity (no ss).  The same histogram as launch_profile
// with the same binsize; rfirst / rlast ([lists], zeroed before the launch) as for coverage.
// count pass + scans: run_off[0..lists] (device) = every list's span of runs, lists in the caller's region order
void launch_profile_runs(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                         int max_tile_ints, RunTiles rt, const int32_t* vt, int64_t lists, int64_t* run_off, cudaStream_t s);
// write pass: values[k] and lengths[k] for k in [0, run_off[lists]); lengths must be zero before the launch
void launch_profile_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                               int max_tile_ints, RunTiles rt, const int32_t* vt, const int64_t* run_off, int32_t* lengths,
                               int32_t* values, cudaStream_t s);

}  // namespace bsg
