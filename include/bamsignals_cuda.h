/* bamsignals_cuda.h — C ABI of libbamsignals_cuda.so, the B200-native counting path of bamsignals.
 *
 * This is the drop-in boundary: the two entry points below are what the reference's R/Rcpp glue binds instead of its
 * own per-region htslib loops.  Citations are relative to the reference tree (lamortenera/bamsignals):
 *
 *   bsg_pileup    replaces  overlapAndPileup<Pileupper>  called from pileup_core    src/bamsignals.cpp:444-461
 *                           (.Call symbol bamsignals_pileup_core, src/RcppExports.cpp:34-52, src/bamsignals_init.c:15)
 *   bsg_coverage  replaces  overlapAndPileup<Coverager> + cumsum in coverage_core   src/bamsignals.cpp:474-494
 *                           (.Call symbol bamsignals_coverage_core, src/RcppExports.cpp:55-70, src/bamsignals_init.c:16)
 *
 * Plain C types only; nothing here depends on R, Rcpp, torch or htslib.  The caller (the R shim in rshim/, or the
 * Python mirror bamsignals_b200/api.py) keeps doing what touches its own objects — parseRegions (S4 slots ->
 * arrays, src/bamsignals.cpp:92-135) and allocateList (result vectors, :139-192) — and hands flat arrays over.
 *
 * Regions are parallel arrays of length R in the caller's order:
 *   seq_levels[n_levels]  chromosome names (the factor levels of seqnames(gr)); looked up in the BAM header by NAME
 *   seq_idx[i]            index into seq_levels
 *   loc[i]                0-based start (= start(gr)[i] - 1, src/bamsignals.cpp:131)
 *   width[i]              number of bases
 *   strand[i]             +1 '+', -1 '-', 0 '*'
 * tlen_filter is NULL (no TLEN filter; R passes integer()) or two ints {min,max} (src/bamsignals.cpp:330-332).
 *
 * Output: the library OVERWRITES every output element (no reliance on zero-fill).  Two ways to receive it:
 *   out + out_offsets : one flat int32 buffer; region i occupies [out_offsets[i], out_offsets[i+1]) with
 *                       bsg_output_layout()'s layout: bamCount (binsize <= 0): mult ints per region, i.e. the R
 *                       IntegerVector(R) / column-major IntegerMatrix(2,R) (:148-169); otherwise mult*ceil(width/binsize)
 *                       ints, interleaved [sense_0, antisense_0, sense_1, ...] when ss (:172-191).  mult = ss ? 2 : 1.
 *   out_ptrs          : R pointers, out_ptrs[i] receives region i's slice (the R shim passes INTEGER(sig_i));
 *                       used when `out` is NULL.  out_offsets is still required (it carries the sizes).
 * The *_device variants below write the same flat layout into the caller's DEVICE memory instead ("results on the GPU").
 *
 * Errors: functions return 0 or a negative BSG_E* code; bsg_last_error() returns the message (thread-local).  The
 * messages for BSG_EOPEN / BSG_ENOINDEX / BSG_ENOCHROM are the reference's own Rcpp::stop strings
 * (src/bamsignals.cpp:204, :209, :119) so the shim can re-raise them verbatim.  Nothing throws across the boundary,
 * nothing calls back into the caller, all helper threads are joined before return.
 *
 * There is NO CPU fallback: without a CUDA device every compute entry point returns BSG_ECUDA.
 */
#ifndef BAMSIGNALS_CUDA_H
#define BAMSIGNALS_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BSG_OK         0
#define BSG_EOPEN     -1   /* "Fail to open BAM file <path>" */
#define BSG_ENOINDEX  -2   /* "BAM indexing file is not available for file <path>" */
#define BSG_ENOCHROM  -3   /* "chromosome <name> not present in the bam file" */
#define BSG_EFORMAT   -4   /* corrupt BGZF / BAM / BAI (bad magic, CRC, ISIZE, truncated record) */
#define BSG_EUNSORTED -5   /* records not coordinate-sorted */
#define BSG_ECUDA     -6   /* no device, launch or runtime failure */
#define BSG_ENOMEM    -7   /* host or device allocation failed */
#define BSG_EARG      -8   /* invalid argument ("negative 'ext' values don't make sense", :243, ...) */

/* Execution options; none of them changes results.  Zero-initialise, set struct_size = sizeof(bsg_opts): every field's
 * zero value is its default.  A library built against a longer or shorter version of the struct takes the first
 * struct_size bytes and defaults for the rest; struct_size < 4 is BSG_EARG.  opts == NULL means all defaults. */
typedef struct bsg_opts {
    int32_t struct_size;
    int32_t n_devices;        /* 0 = device 0 only; 1..16 = devices[0..n): regions (wide ones cut into bin-aligned pieces)
                                 are sharded over the devices inside the call, balanced by the compressed bytes between
                                 their index positions; one host thread + pipeline per device, no collective */
    int32_t devices[16];
    int32_t inflate_threads;  /* host inflate / record-walk workers; 0 = all hardware threads */
    int64_t batch_bytes;      /* uncompressed bytes per staged batch; 0 = default (1 GiB device inflate with a first batch
                                 of a quarter of that, 64 MiB host) */
    int32_t verify_crc;       /* BGZF CRC32 of every inflated block is checked, as htslib does: 0 (default) or 1 = on,
                                 -1 = off */
    int32_t use_cache;        /* reserved, must be 0 (open BAM handles and buffers are always reused across calls;
                                 record data is never cached: every call reads, inflates and decodes the file again) */
    int32_t gpu_inflate;      /* 1: inflate BGZF blocks + verify CRC32 + walk record boundaries on the device (the host
                                 only ships compressed bytes); -1: host zlib worker pool; 0 (default): on the device
                                 unless the job inflates to less than 16 MiB, which the worker pool finishes sooner than
                                 one device launch */
    int32_t stream_min_ints;  /* result ints that must be final before a portion is counted + shipped while later
                                 batches are still inflating; 0 = default (4 Mi), -1 = never (one pass at the end) */
    int32_t result_pack;      /* how a large result crosses PCIe: 0 (default) = one byte per element plus a list of
                                 (index, value) pairs for the elements above 254, widened to int32 by the host while it
                                 scatters them into the caller's buffers (a portion with too many such elements travels
                                 as int32); -1 = always int32; N > 0 = as 0 with room for one pair per N elements
                                 (default 64) */
    int32_t walk_scheme;      /* device record walk between index entry points: 1 = every span's record chain is followed
                                 through device memory (count, scan, write); 2 = spans are linked through per-block
                                 chains that the inflate kernel follows while the blocks are L2-resident, and only what
                                 those cannot cover is walked; 0 (default) = 1 when no span of the batch exceeds 96 KiB,
                                 else 2 */
    int32_t resident_scheme;  /* staged bamProfile / bamCount calls (bsg_pileup_staged*): 1 = decode every resident record
                                 (K1) and join against the read table; 2 = fused: find each tile's rows in the session's
                                 record index and decode only those, inside the counting kernel; 0 (default) = 2 when the
                                 fused join would examine at most 0.3 of the resident records, else 1.  Same results. */
    int32_t reserved[4];
} bsg_opts;

/* Counters and timings of the last call on this thread (milliseconds; kernel times from CUDA events on the
 * launching stream, summed over launches and max over devices). */
typedef struct bsg_timings {
    int64_t records;          /* records of the fetched ranges the call answers for */
    int64_t records_kept;     /* records that passed the mapq/flag/tlen filter; -1 for a staged call on the fused path
                                 (opts.resident_scheme), which filters only the rows it examines */
    int64_t bytes_compressed; /* BGZF bytes read */
    int64_t bytes_inflated;   /* uncompressed bytes produced */
    int64_t candidates;       /* (read, tile) pairs examined by the counting kernels (fused path: rows the join hands them) */
    int64_t out_elems;        /* int32 written to the result */
    int64_t n_tiles;
    int64_t n_batches;
    int64_t n_launches;       /* kernels launched by this library during the call */
    int32_t n_devices;
    int32_t upload_mode;      /* device inflate: 1 = compressed bytes DMA'd straight from the page-locked file mapping,
                                 0 = staged through pinned chunks by the worker pool (or host inflate) */
    double ms_total, ms_plan, ms_fetch, ms_h2d, ms_d2h;
    double ms_decode, ms_filter, ms_join, ms_count, ms_inflate_gpu, ms_kernels;   /* bsg_stage_open: ms_decode is the pass
                                 that builds the session's record index; a fused staged call has no decode span */
    double ms_device;         /* first to last device event of the call on the compute stream (kernels + gaps) */
    double bytes_d2h;         /* result bytes that crossed PCIe device -> host (packed bytes + (index, value) pairs, or int32) */
    double reserved[6];
} bsg_timings;

/* bamCount (binsize <= 0) and bamProfile (binsize >= 1).  Argument order follows pileup_core
 * (src/bamsignals.cpp:444-446); maxgap is accepted for signature parity and ignored (it only prunes I/O). */
int bsg_pileup(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
               const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
               const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss,
               int32_t requiredF, int32_t filteredF, int32_t pe_mid, int32_t maxgap,
               int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs, const bsg_opts* opts);

/* bamCoverage.  Argument order follows coverage_core (src/bamsignals.cpp:474-476). */
int bsg_coverage(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                 const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                 const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                 int32_t maxgap, int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs,
                 const bsg_opts* opts);

/* ---- results on the GPU: count into device memory the caller owns ------------------------------------------------
 * bsg_pileup_device / bsg_coverage_device take the arguments of bsg_pileup / bsg_coverage up to maxgap and write the
 * result into d_out instead of host memory, for callers that consume it on the device (a torch / CuPy tensor, ...).
 *   Layout   d_out receives exactly bsg_output_layout()'s layout, as the host `out` does; out_offsets stays in host
 *            memory and is validated the same way.  Every element of [0, out_offsets[R]) is written exactly once,
 *            nothing outside it is touched.  d_out may be NULL only when out_offsets[R] == 0.
 *   Device   the call runs on the device that owns d_out (cudaPointerGetAttributes).  BSG_EARG, before any write, for:
 *            device or managed memory on another device than opts->devices[0] (opts with n_devices == 1);
 *            n_devices > 1; host memory of any kind (page-locked, registered or not); a pointer that is not 4-byte
 *            aligned.  Without a device: BSG_ECUDA ("no CUDA device").
 *   Stream   `stream` is a cudaStream_t of that device (0 = the legacy default stream).  The library's writes to d_out
 *            are ordered after everything queued on `stream` when the call begins (e.g. a kernel still using memory the
 *            caller's allocator has just handed out again).  The call is synchronous like the others: when it returns,
 *            every write to d_out is complete and the buffer may be used on any stream.
 *   Transfer nothing of the result crosses PCIe: no pinned staging, no host scatter, opts->result_pack is ignored;
 *            bsg_timings.bytes_d2h counts only the control scalars.  opts->stream_min_ints still decides when finished
 *            tiles are counted while later batches are still inflating.
 * Multi-device calls, out_ptrs and output types other than int32 have no device variant. */
int bsg_pileup_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                      const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                      const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss,
                      int32_t requiredF, int32_t filteredF, int32_t pe_mid, int32_t maxgap,
                      int32_t* d_out, const int64_t* out_offsets, void* stream, const bsg_opts* opts);
int bsg_coverage_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                        const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                        const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                        int32_t maxgap, int32_t* d_out, const int64_t* out_offsets, void* stream, const bsg_opts* opts);

/* allocateList's sizes (src/bamsignals.cpp:139-192): fills offsets[0..R], returns the total element count. */
int64_t bsg_output_layout(int64_t R, const int32_t* width, int32_t binsize, int32_t ss, int64_t* offsets);

/* ---- resident sessions: stage once, count many times -------------------------------------------------------------
 * bsg_stage() fetches, inflates and uploads the byte ranges a region set needs and keeps the RAW record bytes and
 * record offsets resident in HBM.  bsg_pileup_staged()/bsg_coverage_staged() then run the device path only
 * (decode -> filter -> join -> count) and leave the result on the device unless `out` is given.  This is how the
 * kernel-only throughput is measured.  bsg_pileup_staged_device()/bsg_coverage_staged_device() write the result into
 * the caller's device memory with the contract of bsg_pileup_device (d_out must be on the session's device): this is
 * how an application amortises inflate over many parameter settings and keeps every result on the GPU.
 * ext_hint is the halo fetched around every region, the `ext` of src/bamsignals.cpp:457,487: a staged call needs
 * |shift| (+ tlen_filter[1] when pe_mid) for pileups and tlen_filter[1] when tspan for coverage; a call that needs
 * more than the session was staged with is refused with BSG_EARG instead of silently missing reads.
 * A session owns its resident device memory (returned by bsg_stage_close); several sessions may be open on one device
 * and may be interleaved with each other and with bsg_pileup / bsg_coverage calls.  bsg_shutdown() ends every open
 * session: later calls on its handle return BSG_EARG, bsg_stage_close() on it stays valid.
 * out_offsets of every call must be the layout bsg_output_layout() gives for that call's binsize / ss (BSG_EARG
 * otherwise): the result scatter trusts it. */
typedef struct bsg_stage bsg_stage;
int bsg_stage_open(bsg_stage** st, const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                   const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                   int32_t ext_hint, const bsg_opts* opts);
int bsg_pileup_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                      int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid,
                      int32_t* out, const int64_t* out_offsets);
int bsg_coverage_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                        int32_t filteredF, int32_t tspan, int32_t* out, const int64_t* out_offsets);
int bsg_pileup_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                             int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid,
                             int32_t* d_out, const int64_t* out_offsets, void* stream);
int bsg_coverage_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                               int32_t filteredF, int32_t tspan, int32_t* d_out, const int64_t* out_offsets, void* stream);
void bsg_stage_close(bsg_stage* st);

/* ---- region views of a staged session: count another region set against the same resident records ----------------
 * bsg_stage_view() binds the region set (the region arrays of bsg_stage_open) to the records `st` already holds on the
 * device.  It reads no BAM or index bytes and launches nothing: names are looked up in the BAM header the session
 * holds (BSG_ENOCHROM with the reference's message for an unknown name, BSG_EARG for malformed region arrays).  *view
 * is a bsg_stage handle: every bsg_*_staged* entry point accepts it as it accepts the session it came from, with the
 * session's options and device.  `st` may itself be a view; its view counts the same resident records.
 * Coverage rule.  The session records the index queries its open sent (each region +/- ext_hint, clamped at 0, with
 * queries less than 16 kb apart merged into one): every record overlapping such a query is resident.  A view region
 * with width > 0 needs a halo a >= 0 such that [max(0, loc - a), loc + width + a) lies inside one query; a view with a
 * region that has none is refused with BSG_EARG, naming the 1-based region.  The view's halo is the smallest a over its
 * regions (unbounded without non-empty regions), and a staged call on the view that needs more (the ext of
 * bsg_stage_open's ext_hint rule: |shift| + tlen_filter[1] with pe_mid for pileups, tlen_filter[1] with tspan for
 * coverage) is BSG_EARG instead of silently missing reads.
 * Lifetime.  A session and its views share the resident records: bsg_stage_close() on any handle frees that handle's own
 * tables, and the resident device memory goes with the last handle, in whatever order they are closed.
 * bsg_shutdown() ends views as it ends sessions (later calls BSG_EARG, bsg_stage_close stays valid).
 * Cost.  A view owns only its tile table and per-call scratch on the device; its calls report the session's
 * bytes_compressed, bytes_inflated and n_batches.  bsg_stage_view itself reports only ms_total. */
int bsg_stage_view(bsg_stage** view, const bsg_stage* st, int64_t R, const char* const* seq_levels, int32_t n_levels,
                   const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand);

/* ---- bamCoverage as runs: run-length (length, value) pairs counted on the GPU ------------------------------------------
 * Coverage is piecewise constant; these calls return it as runs instead of one int32 per base, without ever holding the
 * dense result.  Region i's coverage, in region orientation (a '-' region's runs describe the reversed vector), is
 * runs [run_offsets[i], run_offsets[i+1]): expanding them gives exactly what bsg_coverage writes for that region.
 * Adjacent runs of a region have different values, every length is >= 1, a region's lengths sum to its width, a
 * zero-width region has no runs, and runs never merge across regions (even regions that touch).
 *   bsg_coverage_runs          the arguments of bsg_coverage up to maxgap; run_offsets is host memory of R + 1 int64
 *                              (the total may pass 2^31).  *runs receives the result, which stays in device memory on
 *                              the device the call ran on until bsg_runs_free.
 *   bsg_coverage_runs_staged   the same on a staged session (its device).
 *   bsg_runs_read              copies all run_offsets[R] lengths and values into the caller's arrays, any number of
 *                              times.  Each destination is host memory, or 4-byte aligned device / managed memory on the
 *                              result's device; device copies follow the contract of bsg_pileup_device: ordered after
 *                              what `stream` (0 = the legacy default stream) has queued, complete on return.
 *                              NULL destinations are accepted only for an empty result.
 *   bsg_runs_free              releases a result (NULL is a no-op).  bsg_shutdown() frees every live result's device
 *                              memory: bsg_runs_read on it is then BSG_EARG, bsg_runs_free on it stays valid.
 * BSG_EARG before any work: runs == NULL, opts->n_devices > 1 (no multi-device variant), a bsg_runs_read destination
 * that is misaligned or on another device.  Without a device: BSG_ECUDA.
 * Timings (bsg_get_timings): out_elems is 2 x runs; bytes_d2h counts only what crosses PCIe - the control scalars and
 * run_offsets - nothing of the runs themselves.  bsg_runs_read does not change the timings.
 * The runs are counted when every batch has been decoded: opts->stream_min_ints does not apply. */
typedef struct bsg_runs bsg_runs;      /* a finished run-length result (coverage or profile), held in device memory */
int bsg_coverage_runs(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                      const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                      const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                      int32_t maxgap, int64_t* run_offsets, bsg_runs** runs, const bsg_opts* opts);
int bsg_coverage_runs_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                             int32_t filteredF, int32_t tspan, int64_t* run_offsets, bsg_runs** runs);
int bsg_runs_read(const bsg_runs* runs, int32_t* lengths, int32_t* values, void* stream);
void bsg_runs_free(bsg_runs* runs);

/* ---- bamProfile as runs: run-length (length, value) pairs of read-end profiles counted on the GPU -----------------------
 * The same result as bsg_pileup with binsize >= 1, as runs over output elements (bins) instead of one int32 per bin,
 * without ever holding the dense result.  A result has L = (ss ? 2 : 1) x R lists, in the caller's region order:
 *   without ss, list i is region i's profile;
 *   with ss, list 2i is region i's sense row and list 2i+1 its antisense row.
 * List k is runs [run_offsets[k], run_offsets[k+1]), in region orientation, exactly as bsg_pileup lays the bins out (a
 * partial last bin is one element): expanding list i, or interleaving the expansions of lists 2i and 2i+1, gives
 * exactly region i's slice of bsg_pileup's result with the same arguments.  Every length is >= 1, a list's lengths sum
 * to its bin count, adjacent runs of a list have different values, a zero-width region has no runs, and runs never merge
 * across lists.  bamCount (binsize <= 0) has no runs form.
 *   bsg_profile_runs           the arguments of bsg_pileup up to maxgap; run_offsets is host memory of L + 1 int64.
 *                              *runs receives the result, which stays in device memory on the device the call ran on.
 *   bsg_profile_runs_staged    the same on a staged session (its device).
 * bsg_runs_read, bsg_runs_free and the bsg_shutdown() rules of coverage runs apply unchanged.
 * BSG_EARG before any work: runs or run_offsets NULL, binsize < 1, opts->n_devices > 1, pe_mid without tlen_filter, a
 * staged call that needs more halo than the session was staged with.  Without a device: BSG_ECUDA.
 * Timings, and opts->stream_min_ints: as for coverage runs (out_elems is 2 x runs; bytes_d2h counts only the control
 * scalars and run_offsets). */
int bsg_profile_runs(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                     const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                     const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift, int32_t ss,
                     int32_t requiredF, int32_t filteredF, int32_t pe_mid, int32_t maxgap,
                     int64_t* run_offsets /* (ss ? 2R : R) + 1 */, bsg_runs** runs, const bsg_opts* opts);
int bsg_profile_runs_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t binsize, int32_t shift,
                            int32_t ss, int32_t requiredF, int32_t filteredF, int32_t pe_mid,
                            int64_t* run_offsets, bsg_runs** runs);

/* ---- strand-specific bamCoverage: sense and antisense coverage in one pass ---------------------------------------------
 * Each call takes the arguments of its counterpart without _ss, with `ss` inserted right after tspan (nonzero = on).
 * With ss == 0 it is its counterpart, exactly.  With ss:
 *   Strand   a read's strand is its own flag bit 0x10.  Sense and antisense are relative to the region, as for
 *            bsg_pileup: on '+' and '*' regions forward reads are sense; on '-' regions reverse reads are sense and both
 *            rows are mirrored, as unstranded coverage of a '-' region is.  With tspan (paired_end = "extend",
 *            requiredF 66) only first mates count, and the whole fragment goes to the first mate's strand.
 *   Layout   bsg_output_layout(R, width, 1, 1, offsets): region i is 2 x width[i] int32, interleaved
 *            [sense_0, antisense_0, sense_1, ...] in region orientation (R's IntegerMatrix(2, w)); a zero-width region is
 *            empty.  Runs: 2R lists as for bsg_profile_runs with ss, list 2i the sense and list 2i+1 the antisense row of
 *            region i, run_offsets of 2R + 1 int64.
 *   Identity with cov(F) = bsg_coverage with requiredF = F and every other argument the same: on '+' and '*' regions
 *            antisense = cov(requiredF | 16) and sense = cov(requiredF) - cov(requiredF | 16); on '-' regions sense =
 *            cov(requiredF | 16) and antisense = cov(requiredF) - cov(requiredF | 16).  So sense + antisense = cov(requiredF).
 *   BSG_EARG before any work, besides the counterpart's refusals: an out_offsets that is not the stranded layout, and a
 *            region that starts before position 1.  Multi-device calls (opts->n_devices > 1) exist for bsg_coverage_ss
 *            only, as for the counterparts. */
int bsg_coverage_ss(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                    const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                    const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                    int32_t ss, int32_t maxgap, int32_t* out, const int64_t* out_offsets, int32_t* const* out_ptrs,
                    const bsg_opts* opts);
int bsg_coverage_ss_device(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                           const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                           const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                           int32_t ss, int32_t maxgap, int32_t* d_out, const int64_t* out_offsets, void* stream,
                           const bsg_opts* opts);
int bsg_coverage_ss_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                           int32_t filteredF, int32_t tspan, int32_t ss, int32_t* out, const int64_t* out_offsets);
int bsg_coverage_ss_staged_device(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                                  int32_t filteredF, int32_t tspan, int32_t ss, int32_t* d_out, const int64_t* out_offsets,
                                  void* stream);
int bsg_coverage_runs_ss(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                         const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                         const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF, int32_t filteredF, int32_t tspan,
                         int32_t ss, int32_t maxgap, int64_t* run_offsets /* (ss ? 2R : R) + 1 */, bsg_runs** runs,
                         const bsg_opts* opts);
int bsg_coverage_runs_ss_staged(bsg_stage* st, const int32_t* tlen_filter, int32_t mapqual, int32_t requiredF,
                                int32_t filteredF, int32_t tspan, int32_t ss, int64_t* run_offsets, bsg_runs** runs);

/*
 * writeSamAsBamAndIndex (src/bamsignals.cpp:496-534, .Call symbol bamsignals_writeSamAsBamAndIndex,
 * src/bamsignals_init.c:17): SAM text -> <bampath> (BGZF/BAM) + <bampath>.bai.  Host-only (no device needed).  The
 * reference goes through htslib's sam_read1 / bam_write1 / bam_index_build and ignores their return values; here
 * malformed lines are BSG_EFORMAT and input that is not coordinate-sorted is BSG_EUNSORTED (an index over unsorted
 * records would be wrong).  Positions beyond 2^29 cannot be indexed by a .bai (BSG_EFORMAT); .csi indexes are read
 * by the counting path but not written here.
 */
int bsg_write_sam_as_bam_and_index(const char* sampath, const char* bampath);

/*
 * Diagnostic, host-only (no device needed): runs the fetch planner for the regions with halo `ext` (index queries,
 * range fusion, segment split, BGZF header scan - what replaces bam_itr_queryi, src/bamsignals.cpp:267) and reports
 * what it decided: segment count, compressed / inflated bytes, and the (refID, pos) of every record inside the planned
 * ranges (inflated with zlib and walked on the CPU; at most `cap` are written, all are counted).  It counts nothing:
 * the CPU test-suite uses it to check the index logic (.bai vs .csi, halos, pruning) without a GPU.
 * Returns the number of records inside the planned ranges, or a negative BSG_E* code.
 */
int64_t bsg_debug_plan(const char* bampath, int64_t R, const char* const* seq_levels, int32_t n_levels,
                       const int32_t* seq_idx, const int32_t* loc, const int32_t* width, const int8_t* strand,
                       int64_t ext, int64_t* n_segments, int64_t* bytes_compressed, int64_t* bytes_inflated,
                       int32_t* tid_out, int32_t* pos_out, int64_t cap);

const char* bsg_last_error(void);          /* valid until the next call on this thread */
int  bsg_get_timings(bsg_timings* t);      /* of the last call on this thread */
int  bsg_device_count(void);               /* CUDA devices visible (0 if none) */
void bsg_shutdown(void);                   /* release cached device / pinned memory, worker threads, cached BAM handles,
                                              open staged sessions and run-length results
                                              (the mmap of up to four recently used BAM files + their parsed indexes are
                                              kept between calls while size and mtime are unchanged: do not truncate or
                                              rewrite a BAM in place while a call on it is running) */
const char* bsg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BAMSIGNALS_CUDA_H */
