// Hand-written sm_100a kernels of the counting path.  Integer / byte work bounded by HBM bandwidth and shared-memory
// atomics: no tensor cores by design (nothing here is a dense contraction).  See kernels.cuh for the data layout and
// DESIGN.md for the per-kernel algorithmic bytes.
#include "kernels.cuh"

#include <climits>
#include <type_traits>

namespace bsg {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int kThreads = 256;

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------------------------
// K1 decode + filter.  One CTA per chunk of 256 consecutive records, one thread per record.
//
// Records start at arbitrary byte offsets, so a per-thread gather from global memory makes every load instruction
// touch a dozen 128-byte lines (measured: 15 % of HBM peak).  Instead the CTA's records are one CONTIGUOUS byte span
// [offs[i0], offs[i0+256]) of the batch: thread 0 issues a single TMA bulk copy (cp.async.bulk, completion on an
// mbarrier) of that span into shared memory, so DRAM is read in full lines exactly once, and the threads then pick
// their fields out of shared memory with aligned 32-bit loads + funnel shifts.  Eight CTAs are resident per SM, so
// the copy of one chunk overlaps the decode and the coalesced SoA stores of the others.  Spans that do not fit the
// shared buffer (records with long SEQ/QUAL: only ~60 of their bytes are needed) take the direct global-load path.
//
// Fixed part of a record (offsets from the block_size field): refID +4, pos +8, l_read_name +12, mapq +13,
// bin +14, n_cigar_op +16, flag +18, l_seq +20, next_refID +24, next_pos +28, tlen +32, read_name +36, cigar after.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kDecThreads = kDecodeChunk;
constexpr int kSpanCap = 96 * kDecThreads;   // bytes of shared staging per CTA (average record <= 96 B)

struct GlobalLd {
    const uint8_t* raw;
    __device__ __forceinline__ uint32_t operator()(uint32_t aligned_off) const {
        return __ldg(reinterpret_cast<const uint32_t*>(raw + aligned_off));
    }
};
struct SharedLd {
    const uint8_t* sm;
    uint32_t lo;
    __device__ __forceinline__ uint32_t operator()(uint32_t aligned_off) const {
        return *reinterpret_cast<const uint32_t*>(sm + (aligned_off - lo));
    }
};

struct Decoded {
    int32_t tid, pos, end, tlen;
    uint32_t flagmq, bad;
};

template <class LD>
__device__ __forceinline__ Decoded decode_one(const LD& ld, uint32_t o, uint32_t rec_end) {
    Decoded d;
    const uint32_t a = o + 4, b = a & ~3u, sh = (a & 3u) * 8;
    const uint32_t w0 = ld(b), w1 = ld(b + 4), w2 = ld(b + 8), w3 = ld(b + 12), w4 = ld(b + 16);
    const uint32_t w7 = ld(b + 28), w8 = ld(b + 32);
    d.tid = int32_t(__funnelshift_r(w0, w1, sh));
    d.pos = int32_t(__funnelshift_r(w1, w2, sh));
    const uint32_t nm = __funnelshift_r(w2, w3, sh);   // l_read_name | mapq << 8 | bin << 16
    const uint32_t cf = __funnelshift_r(w3, w4, sh);   // n_cigar_op | flag << 16
    d.tlen = int32_t(__funnelshift_r(w7, w8, sh));
    const uint32_t l_name = nm & 0xffu, mapq = (nm >> 8) & 0xffu;
    const uint32_t n_cigar = cf & 0xffffu, flag = cf >> 16;
    const uint32_t c = o + 36 + l_name;
    uint32_t rlen = 0;
    d.bad = 0;
    if (c + 4u * n_cigar > rec_end) {
        d.bad = STATUS_CORRUPT;
    } else if (!(flag & 0x4u) && n_cigar) {             // bam_endpos: unmapped reads have no reference length
        // nine reads in ten have a one-operation CIGAR: that case is straight-line code; the rest take a plain loop
        // (unrolled by eight, the loop's remainder ladder cost a one-op read 45 instructions)
        const uint32_t cb = c & ~3u, csh = (c & 3u) * 8;
        uint32_t lo = ld(cb), hi = ld(cb + 4);
        uint32_t op = __funnelshift_r(lo, hi, csh);
        rlen = ((0x18Du >> (op & 0xfu)) & 1u) ? op >> 4 : 0u;    // M, D, N, =, X consume the reference
#pragma unroll 1
        for (uint32_t k = 1; k < n_cigar; ++k) {
            lo = hi;
            hi = ld(cb + 4 * k + 4);
            op = __funnelshift_r(lo, hi, csh);
            if ((0x18Du >> (op & 0xfu)) & 1u) rlen += op >> 4;
        }
    }
    if (rlen == 0) rlen = 1;
    d.end = int32_t(uint32_t(d.pos) + rlen - 1u);
    d.flagmq = flag | (mapq << 16);
    return d;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

// (tid, pos) of the record at the start of raw + o
__device__ __forceinline__ int2 record_key(const uint8_t* raw, uint32_t o) {
    const GlobalLd ld{raw};
    const uint32_t a = o + 4, b = a & ~3u, sh = (a & 3u) * 8;
    const uint32_t w0 = ld(b), w1 = ld(b + 4), w2 = ld(b + 8);
    return make_int2(int32_t(__funnelshift_r(w0, w1, sh)), int32_t(__funnelshift_r(w1, w2, sh)));
}

// Bring raw[lo, lo + bytes) into shared memory with one bulk copy that completes on the mbarrier at bar_a (thread 0).
__device__ __forceinline__ void bulk_to_shared(uint32_t bar_a, void* dst, const uint8_t* src, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(bar_a) : "memory");
}
__device__ __forceinline__ void wait_parity(uint32_t bar_a, uint32_t parity) {
    uint32_t done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar_a), "r"(parity) : "memory");
}

// K1's chunks of a multi-batch launch (and the resident index's, which are the same): the batch that chunk blk belongs to
__device__ __forceinline__ int chunk_batch(const DecodeBatch* __restrict__ table, int n_batches, int blk) {
    int lo = 0, hi = n_batches - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (blk >= table[mid].chunk0) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Coordinate-sortedness, K1 and the resident index: the (tid, pos) of the record before record i of resident batch bi,
// from the raw bytes - record i - 1 of the batch, or for i == 0 the last record of batch bi - 1 (callers ensure that
// one exists)
__device__ __forceinline__ int2 key_before(const DecodeBatch* __restrict__ table, int bi, const DecodeBatch& B, int i) {
    if (i > 0) return record_key(B.raw, __ldg(B.offs + i - 1));
    const DecodeBatch& P = table[bi - 1];
    return record_key(P.raw, __ldg(P.offs + P.n - 1));
}
__device__ __forceinline__ bool before_key(uint32_t tid, int32_t pos, uint32_t ptid, int32_t ppos) {
    return tid < ptid || (tid == ptid && pos < ppos);
}


// setRead's filter (src/bamsignals.cpp:328-333, :394-399)
__device__ __forceinline__ bool keep_read(const FilterParams& p, uint32_t fm, int32_t tlen, int32_t* abs_tlen) {
    const uint32_t flag = fm & 0xffffu, mapq = fm >> 16;
    const int32_t a = tlen < 0 ? -tlen : tlen;   // abs() as the reference computes it (INT_MIN stays negative)
    *abs_tlen = a;
    bool keep = int32_t(mapq) >= p.mapqual;
    keep = keep && !(p.required & ~flag);          // every required bit present   (src/bamsignals.cpp:21-23, :328)
    keep = keep && (p.filtered & ~flag);           // not all filtered bits present (:329); filtered == 0 drops all
    keep = keep && (!p.have_tlen || (a >= p.tmin && a <= p.tmax));
    return keep;
}

// setRead's pileup coordinate (src/bamsignals.cpp:339-344): the read's 5' end, or with `midpoint` its fragment's
// midpoint, moved `shift` bases downstream.  Shared by K1 and the fused resident kernel.
__device__ __forceinline__ int32_t pileup_coord(const FilterParams& p, const Decoded& d, int32_t abs_tlen, bool neg) {
    const int32_t offset = p.midpoint ? abs_tlen / 2 + p.shift : p.shift;                 // :339
    return neg ? d.end - offset : d.pos + offset;                                         // :340-344
}

// K1+K2 fused: the filter and the pileup / coverage coordinate (setRead, :326-346 and :392-415) are applied to the
// decoded fields while they are still in registers, so a read costs its raw bytes in and 16 bytes out
// (tid, pos for the join; c0, c1 for the counting kernels) instead of a 20-byte table row written, read again and
// turned into 8 more bytes by a second kernel.
// SS (strand-specific coverage, DESIGN.md §12): a reverse read stores ~e in c1, so c1 < 0 marks the strand (e >= pos >= 0
// for every read that can overlap a region; a kept read with e < 0 overlaps none and is stored dropped).
template <bool COVERAGE, bool SS>
__device__ __forceinline__ void decode_chunk(DecodeBatch single, const DecodeBatch* __restrict__ table, int n_batches,
                                             ReadTable t, const FilterParams& p, DeviceScalars* sc) {
    extern __shared__ __align__(128) uint8_t sm_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t s_lo, s_bytes;
    __shared__ int s_hlo, s_hhi, s_ghlo, s_ghhi;
    __shared__ int2 s_last[kDecThreads / 32];         // (tid, pos) of every warp's last record
    // which batch does this chunk belong to?
    DecodeBatch B = single;
    int bi = 0;
    if (table) {
        bi = chunk_batch(table, n_batches, int(blockIdx.x));
        B = table[bi];
    }
    const int i0 = (int(blockIdx.x) - B.chunk0) * kDecThreads;
    const int i = i0 + threadIdx.x;
    const bool active = i < B.n;
    if (threadIdx.x == 0) {
        const int i1 = min(i0 + kDecThreads, B.n);
        const uint32_t o_lo = B.offs[i0], o_hi = B.offs[i1];
        const uint32_t lo = o_lo & ~15u;
        const uint32_t bytes = (o_hi - lo + 15u) & ~15u;
        if (bytes <= uint32_t(kSpanCap)) {
            const uint32_t bar_a = smem_u32(&bar);
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            bulk_to_shared(bar_a, sm_raw, B.raw + lo, bytes);
            s_lo = lo; s_bytes = bytes;
        } else {
            s_lo = 0; s_bytes = 0;
        }
        s_hlo = INT_MIN; s_hhi = INT_MIN;
        // the running halo maxima, read ONCE per CTA (L2, in flight during the copy) and handed to the warps through
        // shared memory: a warp whose own maxima do not beat them has nothing to publish, and a stale value only costs
        // a redundant atomicMax.  (Every warp reading them itself put 3.6 M loads on one L2 line: +0.35 ms.)
        const int2 g = __ldcg(reinterpret_cast<const int2*>(&sc->halo_lo));
        s_ghlo = g.x; s_ghhi = g.y;
    }
    uint32_t o = 0, rec_end = 0;
    if (active) { o = __ldg(B.offs + i); rec_end = __ldg(B.offs + i + 1); }   // in flight while the bulk copy lands
    const int lane = threadIdx.x & 31;
    __syncthreads();
    const bool staged = s_bytes != 0;
    if (staged) wait_parity(smem_u32(&bar), 0);
    Decoded d;
    d.tid = -1; d.pos = -1; d.end = -1; d.tlen = 0; d.flagmq = 0; d.bad = 0;
    const SharedLd sld{sm_raw, s_lo};
    const GlobalLd gld{B.raw};
    int hlo = INT_MIN, hhi = INT_MIN;
    bool keep = false;
    if (active) {
        d = staged ? decode_one(sld, o, rec_end) : decode_one(gld, o, rec_end);
        int32_t a;
        keep = keep_read(p, d.flagmq, d.tlen, &a);
        const bool neg = (d.flagmq & 0x10u) != 0;
        int32_t o0, o1;
        if (!COVERAGE) {
            const int32_t pos5 = pileup_coord(p, d, a, neg);
            o0 = pos5;
            o1 = keep ? int32_t(neg) : -1;
            if (keep) { hlo = pos5 - d.pos; hhi = d.pos - pos5; }
        } else {
            int32_t s = d.pos, e = d.end;                                                 // :401-403
            if (p.tspan) {
                if (neg && d.tlen < 0) s = e + d.tlen + 1;                                // :408-409
                else if (!neg && d.tlen > 0) e = s + d.tlen - 1;                          // :410-411
            }
            o0 = keep ? s : INT_MAX;
            o1 = keep ? e : INT_MIN;
            if (keep) { hlo = e - d.pos; hhi = d.pos - s; }
            if (SS) {
                if (e < 0) o0 = INT_MAX;
                if (keep && neg) o1 = ~e;
            }
        }
        const int64_t row = B.row0 + i;
        t.tid[row] = d.tid;
        t.pos[row] = d.pos;
        t.c0[row] = o0;
        t.c1[row] = o1;
    }
    // One barrier serves the cross-warp sortedness check and the CTA-wide statistics: before it, every warp leaves the
    // key of its last record and its halo maxima in shared memory; the barrier itself counts the kept reads.
    const int wid = threadIdx.x >> 5;
    hlo = __reduce_max_sync(FULL, hlo);
    hhi = __reduce_max_sync(FULL, hhi);
    if (lane == 31) s_last[wid] = make_int2(d.tid, d.pos);
    if (lane == 0 && hlo != INT_MIN) { atomicMax(&s_hlo, hlo); atomicMax(&s_hhi, hhi); }
    uint32_t ptid = __shfl_up_sync(FULL, uint32_t(d.tid), 1);
    int32_t ppos = __shfl_up_sync(FULL, d.pos, 1);
    const int kept_cta = __syncthreads_count(keep);
    // coordinate-sortedness: compare with the previous record (previous lane; lane 0 takes the previous warp's last
    // record; thread 0 re-reads the record before the chunk)
    bool have_prev = active;
    if (lane == 0 && active) {
        if (threadIdx.x > 0) {
            const int2 l = s_last[wid - 1];
            ptid = uint32_t(l.x); ppos = l.y;
        } else if (i > 0) {
            const int2 k = record_key(B.raw, __ldg(B.offs + i - 1));
            ptid = uint32_t(k.x); ppos = k.y;
        } else if (table && bi > 0) {
            // first record of a resident batch: the record before it is the last one of the batch before, which this
            // same launch decodes (its table row may not be written yet): read it from the raw bytes
            const int2 k = key_before(table, bi, B, 0);
            ptid = uint32_t(k.x); ppos = k.y;
        } else if (B.row0 > 0) {          // streaming path: the row was written by an earlier launch on this stream
            ptid = uint32_t(t.tid[B.row0 - 1]);
            ppos = t.pos[B.row0 - 1];
        } else {
            have_prev = false;
        }
    }
    uint32_t bad = d.bad;
    if (have_prev && before_key(uint32_t(d.tid), d.pos, ptid, ppos)) bad |= STATUS_UNSORTED;
    if (bad) atomicOr(&sc->status, bad);
    // halo maxima and the kept-read count: published once per CTA, the maxima only when they beat the value read at the
    // start, the count into one of kKeptSlots counters that sit on different 128-byte lines (atomics on one line
    // serialise in its L2 slice: 1.8 M same-line atomics cost this kernel 3.7 ms)
    if (threadIdx.x == 0 && kept_cta) {
        if (s_hlo > s_ghlo) atomicMax(&sc->halo_lo, s_hlo);
        if (s_hhi > s_ghhi) atomicMax(&sc->halo_hi, s_hhi);
        atomicAdd(&sc->kept[(blockIdx.x & (kKeptSlots - 1)) * kKeptStride], (unsigned long long)kept_cta);
    }
}

template <bool COVERAGE>
__global__ void __launch_bounds__(kDecThreads) k_decode(DecodeBatch single, const DecodeBatch* __restrict__ table,
                                                     int n_batches, ReadTable t, FilterParams p, DeviceScalars* sc) {
    decode_chunk<COVERAGE, false>(single, table, n_batches, t, p, sc);
}

__global__ void __launch_bounds__(kDecThreads) k_decode_coverage_ss(DecodeBatch single, const DecodeBatch* __restrict__ table,
                                                                 int n_batches, ReadTable t, FilterParams p, DeviceScalars* sc) {
    decode_chunk<true, true>(single, table, n_batches, t, p, sc);
}

// ---------------------------------------------------------------------------------------------------------------
// K3 region join: two binary searches per tile over the (tid,pos)-sorted table.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int64_t lower_bound_tp(const int32_t* __restrict__ tid, const int32_t* __restrict__ pos,
                                                  int64_t n, uint32_t ktid, int64_t kpos) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const uint32_t t = uint32_t(__ldg(tid + mid));
        const int64_t p = __ldg(pos + mid);
        const bool less = t < ktid || (t == ktid && p < kpos);
        if (less) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kThreads) k_join(ReadTable t, int64_t n, TileTable tiles, int64_t n_tiles,
                                                   const DeviceScalars* sc_in, DeviceScalars* sc) {
    const int64_t i = int64_t(blockIdx.x) * kThreads + threadIdx.x;
    long long cand = 0;
    if (i < n_tiles) {
        const int64_t halo_lo = sc_in->halo_lo, halo_hi = sc_in->halo_hi;
        const uint32_t rid = uint32_t(tiles.rid[i]);
        const int64_t loc = tiles.loc[i], len = tiles.len[i];
        const int64_t lo = lower_bound_tp(t.tid, t.pos, n, rid, loc - halo_lo);
        const int64_t hi = lower_bound_tp(t.tid, t.pos, n, rid, loc + len + halo_hi);
        tiles.cand_lo[i] = lo;
        tiles.cand_hi[i] = hi > lo ? hi : lo;
        cand = hi > lo ? hi - lo : 0;
    }
    // block reduce the candidate count (diagnostic: C in the 8*C + 4*B algorithmic-byte formula)
    __shared__ long long s_c[kThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand += __shfl_xor_sync(FULL, cand, o);
    if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = cand;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long tot = 0;
        for (int k = 0; k < kThreads / 32; ++k) tot += s_c[k];
        if (tot) atomicAdd(&sc->candidates, (unsigned long long)tot);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K4 bamCount: one warp per region, per-lane counters, no atomics.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_count(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                    const int32_t* __restrict__ c1, int ss, int32_t* __restrict__ out) {
    const int64_t w = (int64_t(blockIdx.x) * kThreads + threadIdx.x) >> 5;
    if (w >= n_tiles) return;
    const int lane = threadIdx.x & 31;
    const int64_t lo = tiles.cand_lo[w], hi = tiles.cand_hi[w];
    const int32_t loc = tiles.loc[w];
    const uint32_t len = uint32_t(tiles.len[w]);
    const int flip = tiles.strand[w] < 0 ? 1 : 0;
    int sense = 0, anti = 0;
    for (int64_t i = lo + lane; i < hi; i += 32) {
        const int32_t p5 = __ldg(c0 + i), ng = __ldg(c1 + i);
        const bool ok = ng >= 0 && uint32_t(p5 - loc) < len;                 // src/bamsignals.cpp:351-353
        const int a = (ng ^ flip) & 1;                                        // :355-359
        sense += ok && !a;
        anti += ok && a;
    }
    sense = warp_sum(sense);
    anti = warp_sum(anti);
    if (lane == 0) {
        const int64_t off = tiles.out_off[w];
        if (ss) { out[off] = sense; out[off + 1] = anti; } else { out[off] = sense + anti; }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// shared -> global write-out of one tile.  `sm` was placed so that sm and dst have the same phase modulo four
// ints, which lets the body move as 128-bit shared loads + 128-bit streaming stores.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void copy_out(int32_t* __restrict__ dst, const int32_t* sm, int n) {
    const int head = min(n, int((4 - ((reinterpret_cast<uintptr_t>(dst) >> 2) & 3)) & 3));
    if (int(threadIdx.x) < head) __stcs(dst + threadIdx.x, sm[threadIdx.x]);
    const int body = (n - head) >> 2;
    int4* d4 = reinterpret_cast<int4*>(dst + head);
    const int4* s4 = reinterpret_cast<const int4*>(sm + head);
    for (int k = threadIdx.x; k < body; k += blockDim.x) __stcs(d4 + k, s4[k]);
    for (int k = head + 4 * body + threadIdx.x; k < n; k += blockDim.x) __stcs(dst + k, sm[k]);
}

// Position of an int32 destination inside its 16-byte line.  Taken from the ADDRESS, not from the offset: the base of a
// caller's buffer (bsg_*_device) is only 4-byte aligned, e.g. a tensor slice big[1:].
__device__ __forceinline__ int out_phase(const int32_t* dst) {
    return int((reinterpret_cast<uintptr_t>(dst) >> 2) & 3);
}

// exact floor(n / d) for 0 <= n < 2^31 with a precomputed multiplier (host: magic_for())
__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint64_t magic, uint32_t shift) {
    return uint32_t((uint64_t(n) * magic) >> shift);
}

// ---------------------------------------------------------------------------------------------------------------
// K4 bamProfile: one CTA per tile (<= kTileInts output ints), shared-memory histogram.
// k_profile: one read per lane and one shared atomic per counted read (binsize 1..3: neighbouring reads fall into
// different bins anyway).
// The histograms are built by __device__ helpers shared with the run-length kernels (K4r), so that both count every
// tile through the same code: hist[0, nout) zeroed before, the caller's barrier after.
// ---------------------------------------------------------------------------------------------------------------
// One read of a tile (Pileupper::pileup, :349-363): its histogram slot, or -1 when the tile does not count it.
// p5 = pileup coordinate, ng = 0 '+', 1 '-', -1 dropped by the filter.  BIN: 0 = binsize 1, 1 = floor(rel / binsize)
// by the 64-bit multiplier (fast_div), 2 = one bin per tile (bamCount: tiles are whole regions).
enum : int { kBin1 = 0, kBinDiv = 1, kBinOne = 2 };
template <bool SS, int BIN>
__device__ __forceinline__ int32_t profile_slot(int32_t p5, int32_t ng, int32_t loc, int32_t len, int flip, uint64_t magic,
                                                uint32_t mshift) {
    int32_t rel = p5 - loc;
    if (ng < 0 || uint32_t(rel) >= uint32_t(len)) return -1;                       // src/bamsignals.cpp:351-353
    const int a = (ng ^ flip) & 1;
    if (flip) rel = len - 1 - rel;                                                 // :356-359
    const int32_t bin = BIN == kBin1 ? rel : (BIN == kBinOne ? 0 : int32_t(fast_div(uint32_t(rel), magic, mshift)));
    return SS ? 2 * bin + a : bin;                                                 // :361-362
}

template <bool SS, bool BIN1>
__device__ __forceinline__ void scatter_profile(int32_t* hist, int32_t loc, int32_t len, int flip, int64_t lo, int64_t hi,
                                                const int32_t* __restrict__ c0, const int32_t* __restrict__ c1,
                                                uint64_t magic, uint32_t mshift) {
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
        const int32_t p5 = __ldg(c0 + i), ng = __ldg(c1 + i);
        const int32_t k = profile_slot<SS, BIN1 ? kBin1 : kBinDiv>(p5, ng, loc, len, flip, magic, mshift);
        if (k < 0) continue;
        atomicAdd(&hist[k], 1);
    }
}

template <bool SS, bool BIN1>
__global__ void __launch_bounds__(kThreads) k_profile(TileTable tiles, const int32_t* __restrict__ c0,
                                                      const int32_t* __restrict__ c1, int32_t binsize, uint64_t magic,
                                                      uint32_t mshift, int32_t* __restrict__ out) {
    extern __shared__ __align__(16) int32_t smem[];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const int flip = tiles.strand[tix] < 0 ? 1 : 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    const int64_t off = tiles.out_off[tix];
    const int nbins = BIN1 ? len : int((uint32_t(len) + uint32_t(binsize) - 1u) / uint32_t(binsize));
    const int nout = SS ? 2 * nbins : nbins;
    int32_t* hist = smem + out_phase(out + off);           // same 16-byte phase as the destination
    for (int k = threadIdx.x; k < nout; k += kThreads) hist[k] = 0;
    __syncthreads();
    scatter_profile<SS, BIN1>(hist, loc, len, flip, lo, hi, c0, c1, magic, mshift);
    __syncthreads();
    copy_out(out + off, hist, nout);
}

// k_profile_agg (binsize >= 4): the table is coordinate-sorted, so the reads a warp looks at fall into very few
// bins (C4: 128 consecutive reads span ~400 bp of 200 bp bins).  Every lane takes FOUR consecutive reads (128-bit
// loads) and folds them into one (key, count) pair; the warp then peels off its smallest key with redux.sync
// (min over keys, add over the matching counts) and lane 0 issues ONE shared atomic per distinct key.  Three rounds
// cover the common case (<= 3 distinct keys per warp); what is left goes out as one atomic per lane.
// Division by binsize: exact for 0 <= n < 2^31 with a 32-bit multiplier m = ceil(2^(31+L) / d), L = ceil(log2 d):
// n / d = umulhi(n, m) >> (L - 1).
template <bool SS>
__device__ __forceinline__ void scatter_profile_agg(int32_t* hist, int32_t loc, int32_t len, bool flip, int64_t lo, int64_t hi,
                                                    const int32_t* __restrict__ c0, const int32_t* __restrict__ c1,
                                                    uint32_t magic, uint32_t mshift) {
    const int lane = threadIdx.x & 31;
    const int4* c0q = reinterpret_cast<const int4*>(c0);
    const int4* c1q = reinterpret_cast<const int4*>(c1);
    const int64_t q_lo = lo >> 2, q_hi = (hi + 3) >> 2;                            // quads of rows
    for (int64_t qb = q_lo + (threadIdx.x & ~31); qb < q_hi; qb += kThreads) {     // whole warps iterate together
        const int64_t q = qb + lane;
        int key = INT_MAX, cnt = 0;
        if (q < q_hi) {
            const int4 P = __ldg(c0q + q);
            int4 N = __ldg(c1q + q);
            if (4 * q < lo || 4 * q + 4 > hi) {                                    // first / last quad of the range
                const int64_t r0 = 4 * q;
                if (r0 < lo || r0 >= hi) N.x = -1;
                if (r0 + 1 < lo || r0 + 1 >= hi) N.y = -1;
                if (r0 + 2 < lo || r0 + 2 >= hi) N.z = -1;
                if (r0 + 3 < lo || r0 + 3 >= hi) N.w = -1;
            }
            const int32_t ps[4] = {P.x, P.y, P.z, P.w}, ns[4] = {N.x, N.y, N.z, N.w};
            int k[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int32_t r = ps[j] - loc;
                const bool ok = ns[j] >= 0 && uint32_t(r) < uint32_t(len);         // src/bamsignals.cpp:351-353
                const int32_t rel = flip ? len - 1 - r : r;                        // :356-359
                const int32_t bin = int32_t(__umulhi(uint32_t(rel), magic) >> mshift);
                const int kk = SS ? 2 * bin + ((ns[j] ^ int(flip)) & 1) : bin;     // :361-362
                k[j] = ok ? kk : INT_MAX;
            }
            key = min(min(k[0], k[1]), min(k[2], k[3]));
            cnt = int(k[0] == key) + int(k[1] == key) + int(k[2] == key) + int(k[3] == key);
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (k[j] != key && k[j] != INT_MAX) atomicAdd(&hist[k[j]], 1);
        }
#pragma unroll 1
        for (int r = 0; r < 3; ++r) {
            const int kmin = __reduce_min_sync(FULL, key);
            if (kmin == INT_MAX) break;                                            // warp-uniform
            const bool mine = key == kmin;
            const int tot = __reduce_add_sync(FULL, mine ? cnt : 0);
            if (lane == 0) atomicAdd(&hist[kmin], tot);
            if (mine) key = INT_MAX;
        }
        if (key != INT_MAX) atomicAdd(&hist[key], cnt);
    }
}

template <bool SS>
__global__ void __launch_bounds__(kThreads) k_profile_agg(TileTable tiles, const int32_t* __restrict__ c0,
                                                          const int32_t* __restrict__ c1, int32_t binsize, uint32_t magic,
                                                          uint32_t mshift, int32_t* __restrict__ out) {
    extern __shared__ __align__(16) int32_t smem[];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const bool flip = tiles.strand[tix] < 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    const int64_t off = tiles.out_off[tix];
    const int nbins = int((uint32_t(len) + uint32_t(binsize) - 1u) / uint32_t(binsize));
    const int nout = SS ? 2 * nbins : nbins;
    int32_t* hist = smem + out_phase(out + off);
    for (int k = threadIdx.x; k < nout; k += kThreads) hist[k] = 0;
    __syncthreads();
    scatter_profile_agg<SS>(hist, loc, len, flip, lo, hi, c0, c1, magic, mshift);
    __syncthreads();
    copy_out(out + off, hist, nout);
}

// ---------------------------------------------------------------------------------------------------------------
// K5 bamCoverage: one CTA per tile; +1/-1 into a shared difference array, then a block-wide inclusive scan fused with
// the coalesced write-out.  A tile is treated as its own region: the clamp max(start - loc, 0) makes every tile's scan
// self-contained.
// The scan: every WARP owns one contiguous eighth of the tile and runs through it 128 ints at a time (one int4 per
// lane, warp shuffles, its own running carry in a register), leaving its total in shared memory; after ONE barrier every
// warp adds the totals of the warps before it while it streams its own part out.  (Round 1 scanned 1024-int chunks
// across the whole CTA with three barriers per chunk: ncu showed the kernel issue-bound - 66 % of the issue slots, 2.5 TB/s
// of DRAM traffic - on ~6 k warp instructions per tile, half of them the scan.)
// ---------------------------------------------------------------------------------------------------------------
// The tile's difference array d[0, len): +1 where a read's interval begins (a start before the tile is clamped into
// d[0]), -1 behind where it ends (an end past the tile is dropped).  Shared by k_coverage and the run-length kernels.
// SS (c1 from k_decode_coverage_ss): the tile holds two rows interleaved, d[2j + a], a = read strand XOR region strand
// (0 sense, 1 antisense), in region orientation like the unstranded array.
template <bool SS = false>
__device__ __forceinline__ void scatter_coverage(int32_t* d, int32_t loc, int32_t len, bool neg_region, int64_t lo, int64_t hi,
                                                 const int32_t* __restrict__ c0, const int32_t* __restrict__ c1) {
    const int32_t rend = loc + len;                          // region end, exclusive
    for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
        const int32_t s = __ldg(c0 + i);
        int32_t e = __ldg(c1 + i);
        int a = 0;
        if (SS) { a = int(e < 0) ^ int(neg_region); e = e < 0 ? ~e : e; }
        if (s >= rend || e < loc) continue;                  // src/bamsignals.cpp:420 (dropped reads: s = INT_MAX)
        int32_t up, down;
        if (!neg_region) { up = s - loc; down = e + 1 - loc; }          // :423-428
        else { up = rend - 1 - e; down = rend - s; }                    // :431-436
        if (SS) {
            atomicAdd(&d[2 * (up > 0 ? up : 0) + a], 1);
            if (down < len) atomicAdd(&d[2 * down + a], -1);
        } else {
            atomicAdd(&d[up > 0 ? up : 0], 1);
            if (down < len) atomicAdd(&d[down], -1);
        }
    }
}

__global__ void __launch_bounds__(kThreads) k_coverage(TileTable tiles, const int32_t* __restrict__ c0,
                                                       const int32_t* __restrict__ c1, int32_t* __restrict__ out) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_warp[kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const bool neg_region = tiles.strand[tix] < 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    const int64_t off = tiles.out_off[tix];
    // d[j] <-> out[off + j]; d sits `ph` ints into the 16-byte aligned buffer so that shared and global addresses
    // have the same phase; the ph leading ints are zeros and simply take part in the scan.
    const int ph = out_phase(out + off);
    int32_t* d = smem + ph;
    const int total = ph + len;
    const int nquads = (total + 3) >> 2;
    int4* s4 = reinterpret_cast<int4*>(smem);
    for (int k = threadIdx.x; k < nquads; k += kThreads) s4[k] = make_int4(0, 0, 0, 0);
    __syncthreads();
    scatter_coverage(d, loc, len, neg_region, lo, hi, c0, c1);
    __syncthreads();
    // pass 1: every warp scans its own contiguous part in place (cumsum, src/bamsignals.cpp:464-470)
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int kWarps = kThreads / 32;
    const int qpw = ((nquads + kWarps - 1) / kWarps + 31) & ~31;          // quads per warp, whole warp steps
    const int q_lo = wid * qpw, q_hi = min(nquads, q_lo + qpw);
    int carry = 0;
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {                            // warp-uniform
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        v.y += v.x; v.z += v.y; v.w += v.z;
        int incl = v.w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        const int prefix = carry + incl - v.w;
        if (q < q_hi) { v.x += prefix; v.y += prefix; v.z += prefix; v.w += prefix; s4[q] = v; }
        carry += __shfl_sync(FULL, incl, 31);
    }
    if (lane == 0) s_warp[wid] = carry;
    __syncthreads();
    // pass 2: add the totals of the warps in front and stream the warp's own part out (128-bit streaming stores; the
    // first and the last quad of the tile may be partial)
    int before = 0;
    for (int k = 0; k < wid; ++k) before += s_warp[k];
    int32_t* dst = out + off - ph;                           // dst[j] <-> smem[j]; 16-byte aligned by construction
    for (int q = q_lo + lane; q < q_hi; q += 32) {
        int4 v = s4[q];
        v.x += before; v.y += before; v.z += before; v.w += before;
        const int j = 4 * q;
        if (j >= ph && j + 4 <= total) {
            __stcs(reinterpret_cast<int4*>(dst + j), v);
        } else {
            if (j >= ph && j < total) __stcs(dst + j, v.x);
            if (j + 1 >= ph && j + 1 < total) __stcs(dst + j + 1, v.y);
            if (j + 2 >= ph && j + 2 < total) __stcs(dst + j + 2, v.z);
            if (j + 3 >= ph && j + 3 < total) __stcs(dst + j + 3, v.w);
        }
    }
}

// K5 with SS (DESIGN.md §12): the same tile, two rows interleaved as in the output, d[2j + a].  A quad of shared memory is
// (row r, row r^1, row r, row r^1) with r fixed by the 16-byte phase, so the per-warp scan adds within the quad x -> z and
// y -> w and carries two running sums (an int2 shuffle scan); the write-out is k_coverage's.
__global__ void __launch_bounds__(kThreads) k_coverage_ss(TileTable tiles, const int32_t* __restrict__ c0,
                                                          const int32_t* __restrict__ c1, int32_t* __restrict__ out) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int2 s_warp[kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const bool neg_region = tiles.strand[tix] < 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    int32_t* const tile_out = out + tiles.out_off[tix];
    const int ph = out_phase(tile_out);                    // as in k_coverage: d[k] <-> tile_out[k], over 2 len ints
    int32_t* d = smem + ph;
    const int total = ph + 2 * len;
    const int nquads = (total + 3) >> 2;
    int4* s4 = reinterpret_cast<int4*>(smem);
    for (int k = threadIdx.x; k < nquads; k += kThreads) s4[k] = make_int4(0, 0, 0, 0);
    __syncthreads();
    scatter_coverage<true>(d, loc, len, neg_region, lo, hi, c0, c1);
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int kWarps = kThreads / 32;
    const int qpw = ((nquads + kWarps - 1) / kWarps + 31) & ~31;
    const int q_lo = wid * qpw, q_hi = min(nquads, q_lo + qpw);
    int2 carry = make_int2(0, 0);
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {                            // warp-uniform
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        v.z += v.x; v.w += v.y;
        int2 incl = make_int2(v.z, v.w);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int ux = __shfl_up_sync(FULL, incl.x, o), uy = __shfl_up_sync(FULL, incl.y, o);
            if (lane >= o) { incl.x += ux; incl.y += uy; }
        }
        const int px = carry.x + incl.x - v.z, py = carry.y + incl.y - v.w;
        if (q < q_hi) { v.x += px; v.y += py; v.z += px; v.w += py; s4[q] = v; }
        carry.x += __shfl_sync(FULL, incl.x, 31);
        carry.y += __shfl_sync(FULL, incl.y, 31);
    }
    if (lane == 0) s_warp[wid] = carry;
    __syncthreads();
    int bx = 0, by = 0;
    for (int k = 0; k < wid; ++k) { bx += s_warp[k].x; by += s_warp[k].y; }
    int32_t* dst = tile_out - ph;
    for (int q = q_lo + lane; q < q_hi; q += 32) {
        int4 v = s4[q];
        v.x += bx; v.y += by; v.z += bx; v.w += by;
        const int j = 4 * q;
        if (j >= ph && j + 4 <= total) {
            __stcs(reinterpret_cast<int4*>(dst + j), v);
        } else {
            if (j >= ph && j < total) __stcs(dst + j, v.x);
            if (j + 1 >= ph && j + 1 < total) __stcs(dst + j + 1, v.y);
            if (j + 2 >= ph && j + 2 < total) __stcs(dst + j + 2, v.z);
            if (j + 3 >= ph && j + 3 < total) __stcs(dst + j + 3, v.w);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K5r bamCoverage as runs (DESIGN.md §10).  Inside a tile the coverage v[j] changes exactly where d[j] != 0 (j >= 1), its
// first value is d[0] and its last value the sum of d: a tile's runs follow from the difference array without a scan.
//   k_runs_count  per tile: nnz = #{j in [1, len): d[j] != 0}, first = d[0], last = sum(d)
//   k_runs_scan   tile t holds runs(t) = nnz(t) + (t opens its region || first(t) != last(t-1)) run starts; one CTA
//                 scans them over the tiles, then over the regions (caller order) -> run_off[R + 1]
//   k_runs_write  scatter + scan again, write every run start's value at its index; lengths are end - start, added up
//                 with atomics from the two places that know them (the run's own start, and the next run's start or
//                 the region's end), into a zeroed buffer
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_runs_count(TileTable tiles, const int32_t* __restrict__ c0,
                                                         const int32_t* __restrict__ c1, RunTiles rt) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_nz[kThreads / 32], s_sum[kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    for (int k = threadIdx.x; k < len; k += kThreads) smem[k] = 0;
    __syncthreads();
    scatter_coverage(smem, loc, len, tiles.strand[tix] < 0, tiles.cand_lo[tix], tiles.cand_hi[tix], c0, c1);
    __syncthreads();
    int nz = 0, sum = 0;
    for (int j = threadIdx.x; j < len; j += kThreads) {
        const int32_t v = smem[j];
        sum += v;
        nz += int(j > 0 && v != 0);
    }
    nz = __reduce_add_sync(FULL, nz);
    sum = __reduce_add_sync(FULL, sum);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) { s_nz[wid] = nz; s_sum[wid] = sum; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int tn = 0, ts = 0;
        for (int k = 0; k < kThreads / 32; ++k) { tn += s_nz[k]; ts += s_sum[k]; }
        rt.nnz[tix] = tn;
        rt.first[tix] = smem[0];
        rt.last[tix] = ts;
    }
}

// Exclusive prefix of v over the CTA (1024 threads, blockDim.x == kScanThreads); *total receives the sum.
constexpr int kScanThreads = 1024;
__device__ __forceinline__ long long block_exclusive_scan(long long v, long long* total) {
    __shared__ long long s_w[kScanThreads / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    if (lane == 31) s_w[wid] = incl;
    __syncthreads();
    long long before = 0, all = 0;
    for (int k = 0; k < kScanThreads / 32; ++k) {
        const long long w = s_w[k];
        if (k < wid) before += w;
        all += w;
    }
    __syncthreads();                                        // s_w may be reused by the next call
    *total = all;
    return before + incl - v;
}

__device__ __forceinline__ int64_t tile_runs(const RunTiles& rt, int64_t t) {
    const bool head = t == 0 || rt.region[t - 1] != rt.region[t];
    return int64_t(rt.nnz[t]) + int64_t(head || rt.first[t] != rt.last[t - 1]);
}

// One CTA.  Every thread walks a contiguous chunk of tiles, then of regions (a few hundred thousand of either take
// tens of microseconds: not worth a multi-CTA scan).
__global__ void __launch_bounds__(kScanThreads) k_runs_scan(RunTiles rt, int64_t n_tiles, int64_t R, int64_t* __restrict__ run_off) {
    long long total = 0;
    {
        const int64_t per = (n_tiles + kScanThreads - 1) / kScanThreads;
        const int64_t t0 = min(n_tiles, per * int64_t(threadIdx.x)), t1 = min(n_tiles, t0 + per);
        long long mine = 0;
        for (int64_t t = t0; t < t1; ++t) mine += tile_runs(rt, t);
        long long run = block_exclusive_scan(mine, &total);
        for (int64_t t = t0; t < t1; ++t) {
            const int32_t reg = rt.region[t];
            if (t == 0 || rt.region[t - 1] != reg) rt.rfirst[reg] = run;
            rt.toff[t] = run;
            run += tile_runs(rt, t);
            if (t + 1 == n_tiles || rt.region[t + 1] != reg) rt.rlast[reg] = run;
        }
    }
    __syncthreads();                                        // rfirst / rlast of every region are written
    const int64_t per = (R + kScanThreads - 1) / kScanThreads;
    const int64_t i0 = min(R, per * int64_t(threadIdx.x)), i1 = min(R, i0 + per);
    long long mine = 0;
    for (int64_t i = i0; i < i1; ++i) mine += rt.rlast[i] - rt.rfirst[i];
    long long run = block_exclusive_scan(mine, &total);
    for (int64_t i = i0; i < i1; ++i) { run_off[i] = run; run += rt.rlast[i] - rt.rfirst[i]; }
    if (threadIdx.x == 0) run_off[R] = total;
}

__global__ void __launch_bounds__(kThreads) k_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                         const int32_t* __restrict__ c1, RunTiles rt,
                                                         const int64_t* __restrict__ run_off, int32_t* __restrict__ lengths,
                                                         int32_t* __restrict__ values) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_sum[kThreads / 32], s_cnt[kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const int32_t reg = rt.region[tix], rel = rt.rel[tix];
    const bool head = tix == 0 || rt.region[tix - 1] != reg;
    const bool tail = tix + 1 == n_tiles || rt.region[tix + 1] != reg;
    const bool start0 = head || rt.first[tix] != rt.last[tix - 1];      // a run starts at the tile's first base
    const int64_t kbeg = run_off[reg], kend = run_off[reg + 1];
    const int64_t k0 = kbeg + (rt.toff[tix] - rt.rfirst[reg]);        // index of the tile's first run start
    const int nquads = (len + 3) >> 2;
    int4* s4 = reinterpret_cast<int4*>(smem);
    for (int k = threadIdx.x; k < nquads; k += kThreads) s4[k] = make_int4(0, 0, 0, 0);
    __syncthreads();
    scatter_coverage(smem, loc, len, tiles.strand[tix] < 0, tiles.cand_lo[tix], tiles.cand_hi[tix], c0, c1);
    __syncthreads();
    // every warp owns a contiguous part of the tile (as in k_coverage): pass 1 sums its d and counts its run starts,
    // pass 2 adds what the warps in front of it have and writes the runs
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int kWarps = kThreads / 32;
    const int qpw = ((nquads + kWarps - 1) / kWarps + 31) & ~31;
    const int q_lo = wid * qpw, q_hi = min(nquads, q_lo + qpw);
    auto flags = [&](int q, const int4& v) {                // bit e: a run starts at 4q + e
        const int j = 4 * q;
        return (j < len && (j == 0 ? start0 : v.x != 0) ? 1u : 0u) | (j + 1 < len && v.y != 0 ? 2u : 0u) |
               (j + 2 < len && v.z != 0 ? 4u : 0u) | (j + 3 < len && v.w != 0 ? 8u : 0u);
    };
    int wsum = 0, wcnt = 0;
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        wsum += __reduce_add_sync(FULL, v.x + v.y + v.z + v.w);
        wcnt += __reduce_add_sync(FULL, q < q_hi ? __popc(flags(q, v)) : 0);
    }
    if (lane == 0) { s_sum[wid] = wsum; s_cnt[wid] = wcnt; }
    __syncthreads();
    int val = 0, cnt = 0;
    for (int k = 0; k < wid; ++k) { val += s_sum[k]; cnt += s_cnt[k]; }
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        const unsigned f = q < q_hi ? flags(q, v) : 0u;
        int isum = v.x + v.y + v.z + v.w, icnt = __popc(f);
        const int qs = isum, qc = icnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int us = __shfl_up_sync(FULL, isum, o), uc = __shfl_up_sync(FULL, icnt, o);
            if (lane >= o) { isum += us; icnt += uc; }
        }
        int x = val + isum - qs;                            // coverage just before 4q
        int64_t k = k0 + cnt + icnt - qc;                   // index of the next run start
        const int e4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            x += e4[e];
            if (f >> e & 1u) {
                const int32_t p = rel + 4 * q + e;          // run start, relative to the region in its orientation
                values[k] = x;
                atomicAdd(&lengths[k], -p);
                if (k > kbeg) atomicAdd(&lengths[k - 1], p);
                ++k;
            }
        }
        val += __shfl_sync(FULL, isum, 31);
        cnt += __shfl_sync(FULL, icnt, 31);
    }
    if (tail && threadIdx.x == 0 && kend > kbeg) atomicAdd(&lengths[kend - 1], rel + len);     // the region's last run ends at its width
}

// K5r with SS (DESIGN.md §12): the interleaved array of k_coverage_ss, at smem[0].  Row a of a tile is a virtual tile of
// list 2i + a, vt[a * n_tiles + t] = v, as for strand-specific profile runs (K4r below); k_runs_scan runs unchanged over
// the 2 * n_tiles virtual tiles and 2R lists.
__global__ void __launch_bounds__(kThreads) k_runs_count_ss(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                            const int32_t* __restrict__ c1, RunTiles rt,
                                                            const int32_t* __restrict__ vt) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_nz[2][kThreads / 32], s_sum[2][kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    for (int k = threadIdx.x; k < 2 * len; k += kThreads) smem[k] = 0;
    __syncthreads();
    scatter_coverage<true>(smem, loc, len, tiles.strand[tix] < 0, tiles.cand_lo[tix], tiles.cand_hi[tix], c0, c1);
    __syncthreads();
    // element k = 2j + a: kThreads is even, so a thread only ever sees row a = threadIdx.x & 1
    int nz = 0, sum = 0;
    for (int k = threadIdx.x; k < 2 * len; k += kThreads) {
        const int32_t v = smem[k];
        sum += v;
        nz += int(k >= 2 && v != 0);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const bool mine = int(threadIdx.x & 1) == a;
        const int n = __reduce_add_sync(FULL, mine ? nz : 0), t = __reduce_add_sync(FULL, mine ? sum : 0);
        if (lane == 0) { s_nz[a][wid] = n; s_sum[a][wid] = t; }
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        const int a = threadIdx.x;
        int tn = 0, ts = 0;
        for (int k = 0; k < kThreads / 32; ++k) { tn += s_nz[a][k]; ts += s_sum[a][k]; }
        const int32_t v = vt[a * n_tiles + tix];
        rt.nnz[v] = tn;
        rt.first[v] = smem[a];
        rt.last[v] = ts;
    }
}

// k_runs_write per row: a quad of shared memory holds bases 2q and 2q + 1 of both rows, (s, a, s, a).
__global__ void __launch_bounds__(kThreads) k_runs_write_ss(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                            const int32_t* __restrict__ c1, RunTiles rt,
                                                            const int32_t* __restrict__ vt, const int64_t* __restrict__ run_off,
                                                            int32_t* __restrict__ lengths, int32_t* __restrict__ values) {
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int2 s_sum[kThreads / 32], s_cnt[kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const int64_t n_virtual = 2 * n_tiles;
    int32_t rel[2];
    int64_t kbeg[2], k0[2];
    bool start0[2];
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int64_t v = vt[a * n_tiles + tix];
        const int32_t list = rt.region[v];
        rel[a] = rt.rel[v];
        start0[a] = v == 0 || rt.region[v - 1] != list || rt.first[v] != rt.last[v - 1];    // a run starts at base 0
        kbeg[a] = run_off[list];
        k0[a] = kbeg[a] + (rt.toff[v] - rt.rfirst[list]);                                 // the row's first run start
    }
    const int nquads = (len + 1) >> 1;
    int4* s4 = reinterpret_cast<int4*>(smem);
    for (int k = threadIdx.x; k < nquads; k += kThreads) s4[k] = make_int4(0, 0, 0, 0);
    __syncthreads();
    scatter_coverage<true>(smem, loc, len, tiles.strand[tix] < 0, tiles.cand_lo[tix], tiles.cand_hi[tix], c0, c1);
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int kWarps = kThreads / 32;
    const int qpw = ((nquads + kWarps - 1) / kWarps + 31) & ~31;
    const int q_lo = wid * qpw, q_hi = min(nquads, q_lo + qpw);
    auto flags = [&](int q, int d0, int d1, int a) {        // bit e: row a has a run start at base 2q + e
        const int j = 2 * q;
        return (j < len && (j == 0 ? start0[a] : d0 != 0) ? 1u : 0u) | (j + 1 < len && d1 != 0 ? 2u : 0u);
    };
    int2 wsum = make_int2(0, 0), wcnt = make_int2(0, 0);
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        wsum.x += __reduce_add_sync(FULL, v.x + v.z);
        wsum.y += __reduce_add_sync(FULL, v.y + v.w);
        wcnt.x += __reduce_add_sync(FULL, q < q_hi ? __popc(flags(q, v.x, v.z, 0)) : 0);
        wcnt.y += __reduce_add_sync(FULL, q < q_hi ? __popc(flags(q, v.y, v.w, 1)) : 0);
    }
    if (lane == 0) { s_sum[wid] = wsum; s_cnt[wid] = wcnt; }
    __syncthreads();
    int val[2] = {0, 0}, cnt[2] = {0, 0};
    for (int k = 0; k < wid; ++k) { val[0] += s_sum[k].x; val[1] += s_sum[k].y; cnt[0] += s_cnt[k].x; cnt[1] += s_cnt[k].y; }
    for (int q0 = q_lo; q0 < q_hi; q0 += 32) {
        const int q = q0 + lane;
        int4 v = make_int4(0, 0, 0, 0);
        if (q < q_hi) v = s4[q];
        const int d[2][2] = {{v.x, v.z}, {v.y, v.w}};
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const unsigned f = q < q_hi ? flags(q, d[a][0], d[a][1], a) : 0u;
            int isum = d[a][0] + d[a][1], icnt = __popc(f);
            const int qs = isum, qc = icnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int us = __shfl_up_sync(FULL, isum, o), uc = __shfl_up_sync(FULL, icnt, o);
                if (lane >= o) { isum += us; icnt += uc; }
            }
            int x = val[a] + isum - qs;                     // the row's coverage just before base 2q
            int64_t k = k0[a] + cnt[a] + icnt - qc;         // index of the row's next run start
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                x += d[a][e];
                if (f >> e & 1u) {
                    const int32_t p = rel[a] + 2 * q + e;   // run start, relative to the region in its orientation
                    values[k] = x;
                    atomicAdd(&lengths[k], -p);
                    if (k > kbeg[a]) atomicAdd(&lengths[k - 1], p);
                    ++k;
                }
            }
            val[a] += __shfl_sync(FULL, isum, 31);
            cnt[a] += __shfl_sync(FULL, icnt, 31);
        }
    }
    if (threadIdx.x == 0) {
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const int64_t v = vt[a * n_tiles + tix];
            const int32_t list = rt.region[v];
            const int64_t kend = run_off[list + 1];
            const bool tail = v + 1 == n_virtual || rt.region[v + 1] != list;
            if (tail && kend > kbeg[a]) atomicAdd(&lengths[kend - 1], rel[a] + len);   // the row's last run ends at the width
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// K4r bamProfile as runs (DESIGN.md §11).  A profile has no running sum: inside a tile, strand row a's histogram
// h[j] = hist[mult * j + a] changes exactly where h[j] != h[j-1].  Row a of the j-th of region i's n_i tiles (T_i its
// first) is the virtual tile v = mult * T_i + a * n_i + j, in list mult * i + a; vt[a * n_tiles + t] holds v for tile t.
// A list's pieces are consecutive virtual tiles, so k_runs_scan runs unchanged over the virtual tiles.
//   k_profile_runs_count  per tile and row: nnz = #{j in [1, nbins): h[j] != h[j-1]}, first = h[0], last = h[nbins-1]
//   k_profile_runs_write  the histogram again; every run start writes h[j] at its index, and the lengths are added up
//                         with atomics as in k_runs_write
// KIND: 0 = k_profile<SS, true>'s histogram (binsize 1), 1 = k_profile<SS, false>'s, 2 = k_profile_agg<SS>'s
// (binsize >= 4): the same helpers give the same histogram as the dense call.  The histogram sits at smem[0].
// ---------------------------------------------------------------------------------------------------------------
template <bool SS, int KIND>
__device__ __forceinline__ int profile_runs_hist(int32_t* hist, const TileTable& tiles, int64_t tix, const int32_t* __restrict__ c0,
                                                 const int32_t* __restrict__ c1, int32_t binsize, uint64_t magic, uint32_t mshift) {
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const bool flip = tiles.strand[tix] < 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    const int nbins = KIND == 0 ? len : int((uint32_t(len) + uint32_t(binsize) - 1u) / uint32_t(binsize));
    const int nout = SS ? 2 * nbins : nbins;
    for (int k = threadIdx.x; k < nout; k += kThreads) hist[k] = 0;
    __syncthreads();
    if constexpr (KIND == 2) scatter_profile_agg<SS>(hist, loc, len, flip, lo, hi, c0, c1, uint32_t(magic), mshift);
    else scatter_profile<SS, KIND == 0>(hist, loc, len, flip ? 1 : 0, lo, hi, c0, c1, magic, mshift);
    __syncthreads();
    return nbins;
}

template <bool SS, int KIND>
__global__ void __launch_bounds__(kThreads) k_profile_runs_count(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                                 const int32_t* __restrict__ c1, int32_t binsize, uint64_t magic,
                                                                 uint32_t mshift, RunTiles rt, const int32_t* __restrict__ vt) {
    constexpr int M = SS ? 2 : 1;
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_nz[M][kThreads / 32];
    const int64_t tix = blockIdx.x;
    const int nbins = profile_runs_hist<SS, KIND>(smem, tiles, tix, c0, c1, binsize, magic, mshift);
    // element k = M j + a compares with k - M; kThreads is even, so a thread only ever sees one row (a = k & 1)
    int nz = 0;
    for (int k = threadIdx.x + M; k < M * nbins; k += kThreads) nz += int(smem[k] != smem[k - M]);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < M; ++a) {
        const int n = __reduce_add_sync(FULL, (threadIdx.x & (M - 1)) == a ? nz : 0);
        if (lane == 0) s_nz[a][wid] = n;
    }
    __syncthreads();
    if (threadIdx.x < M) {
        const int a = threadIdx.x;
        int tn = 0;
        for (int k = 0; k < kThreads / 32; ++k) tn += s_nz[a][k];
        const int32_t v = vt ? vt[a * n_tiles + tix] : int32_t(tix);
        rt.nnz[v] = tn;
        rt.first[v] = smem[a];
        rt.last[v] = smem[M * (nbins - 1) + a];
    }
}

template <bool SS, int KIND>
__global__ void __launch_bounds__(kThreads) k_profile_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* __restrict__ c0,
                                                                 const int32_t* __restrict__ c1, int32_t binsize, uint64_t magic,
                                                                 uint32_t mshift, RunTiles rt, const int32_t* __restrict__ vt,
                                                                 const int64_t* __restrict__ run_off, int32_t* __restrict__ lengths,
                                                                 int32_t* __restrict__ values) {
    constexpr int M = SS ? 2 : 1;
    constexpr int kWarps = kThreads / 32;
    extern __shared__ __align__(16) int32_t smem[];
    __shared__ int32_t s_cnt[M][kWarps];
    const int64_t tix = blockIdx.x;
    const int nbins = profile_runs_hist<SS, KIND>(smem, tiles, tix, c0, c1, binsize, magic, mshift);
    const int64_t n_virtual = M * n_tiles;
    // every warp owns a contiguous part of the tile's bins (as in k_runs_write): pass 1 counts its run starts per row,
    // pass 2 adds what the warps in front of it have and writes the runs
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int bpw = ((nbins + kWarps - 1) / kWarps + 31) & ~31;
    const int j_lo = wid * bpw, j_hi = min(nbins, j_lo + bpw);
    bool start0[M];
    int cnt[M];
#pragma unroll
    for (int a = 0; a < M; ++a) {
        const int64_t v = vt ? vt[a * n_tiles + tix] : tix;
        const int32_t list = rt.region[v];
        start0[a] = v == 0 || rt.region[v - 1] != list || rt.first[v] != rt.last[v - 1];     // a run starts at bin 0
        cnt[a] = 0;
    }
    auto flag = [&](int j, int a) {
        return j < j_hi && (j == 0 ? start0[a] : smem[M * j + a] != smem[M * (j - 1) + a]);
    };
    for (int j0 = j_lo; j0 < j_hi; j0 += 32) {                                      // warp-uniform
#pragma unroll
        for (int a = 0; a < M; ++a) cnt[a] += __popc(__ballot_sync(FULL, flag(j0 + lane, a)));
    }
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < M; ++a) s_cnt[a][wid] = cnt[a];
    }
    __syncthreads();
    const unsigned below = (1u << lane) - 1u;
#pragma unroll
    for (int a = 0; a < M; ++a) {
        const int64_t v = vt ? vt[a * n_tiles + tix] : tix;
        const int32_t list = rt.region[v], rel = rt.rel[v];
        const int64_t kbeg = run_off[list], kend = run_off[list + 1];
        int64_t k0 = kbeg + (rt.toff[v] - rt.rfirst[list]);                      // index of the tile's first run start
        for (int w = 0; w < wid; ++w) k0 += s_cnt[a][w];
        for (int j0 = j_lo; j0 < j_hi; j0 += 32) {
            const int j = j0 + lane;
            const bool f = flag(j, a);
            const unsigned b = __ballot_sync(FULL, f);
            if (f) {
                const int64_t k = k0 + __popc(b & below);
                const int32_t p = rel + j;                                         // run start, relative to the list
                values[k] = smem[M * j + a];
                atomicAdd(&lengths[k], -p);
                if (k > kbeg) atomicAdd(&lengths[k - 1], p);
            }
            k0 += __popc(b);
        }
        const bool tail = v + 1 == n_virtual || rt.region[v + 1] != list;
        if (tail && threadIdx.x == 0 && kend > kbeg) atomicAdd(&lengths[kend - 1], rel + nbins);    // the list's last run ends at its bin count
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Staged sessions: the resident record index (K0i, once per session) and the fused pileup step (K3f join, K4f count).
// K1 decodes every resident record on every call, but the fetch planner works in whole BGZF blocks and 16 kb index
// windows, so most of them lie far from every region (C2: 57.8 M resident records, ~7 M near a region).  The fused
// step finds each tile's rows from a sampled key index and decodes only those, inside the counting CTA.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_key(int32_t tid, int32_t pos) {
    return (unsigned long long)uint32_t(tid) << 32 | (uint32_t(pos) ^ 0x80000000u);
}
// key < (qt, qp) in lower_bound_tp's order: tid as uint32, then pos as a signed number (qp may lie outside int32)
__device__ __forceinline__ bool key_less(unsigned long long k, uint32_t qt, int64_t qp) {
    const uint32_t t = uint32_t(k >> 32);
    const int64_t p = int32_t(uint32_t(k) ^ 0x80000000u);
    return t < qt || (t == qt && p < qp);
}

// the resident batch that holds row r (the table has one entry per non-empty batch, rows contiguous)
__device__ __forceinline__ int batch_of_row(const ResidentView& v, int64_t r) {
    int lo = 0, hi = v.n_batches - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (r >= __ldg(&v.batches[mid].row0)) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// K0i: one pass over every resident record (K1's chunking, bulk copy and decode_one).  PASS 0: sampled keys, the
// unsorted / corrupt status bits (K1's checks, across batch boundaries too), reach = max(pos + span) and the span
// buckets the host picks the long-span threshold from.  PASS 1: appends every row with span > long_span to the long
// list, in no particular order (the host sorts it).
template <int PASS>
__global__ void __launch_bounds__(kDecThreads) k_resident_index(const DecodeBatch* __restrict__ table, int n_batches,
                                                                uint32_t long_span, unsigned long long* __restrict__ keys,
                                                                unsigned long long* __restrict__ long_key, int2* __restrict__ long_row,
                                                                IndexScalars* isc) {
    extern __shared__ __align__(128) uint8_t sm_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t s_lo, s_bytes, s_nl, s_base;
    __shared__ int2 s_key[kDecThreads];
    __shared__ uint32_t s_bn[kSpanBuckets], s_bm[kSpanBuckets];
    __shared__ long long s_reach;
    const int bi = chunk_batch(table, n_batches, int(blockIdx.x));
    const DecodeBatch B = table[bi];
    const int i0 = (int(blockIdx.x) - B.chunk0) * kDecThreads;
    const int i = i0 + threadIdx.x;
    const bool active = i < B.n;
    if (threadIdx.x < kSpanBuckets) { s_bn[threadIdx.x] = 0; s_bm[threadIdx.x] = 0; }
    if (threadIdx.x == 0) {
        const int i1 = min(i0 + kDecThreads, B.n);
        const uint32_t lo = B.offs[i0] & ~15u;
        const uint32_t bytes = (B.offs[i1] - lo + 15u) & ~15u;
        s_lo = lo; s_bytes = 0; s_nl = 0; s_reach = 0;
        if (bytes <= uint32_t(kSpanCap)) {
            const uint32_t bar_a = smem_u32(&bar);
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            bulk_to_shared(bar_a, sm_raw, B.raw + lo, bytes);
            s_bytes = bytes;
        }
    }
    uint32_t o = 0, rec_end = 0;
    if (active) { o = __ldg(B.offs + i); rec_end = __ldg(B.offs + i + 1); }
    __syncthreads();
    const bool staged = s_bytes != 0;
    if (staged) wait_parity(smem_u32(&bar), 0);
    Decoded d;
    d.tid = -1; d.pos = -1; d.end = -1; d.tlen = 0; d.flagmq = 0; d.bad = 0;
    uint32_t span = 0;
    if (active) {
        d = staged ? decode_one(SharedLd{sm_raw, s_lo}, o, rec_end) : decode_one(GlobalLd{B.raw}, o, rec_end);
        span = uint32_t(d.end) - uint32_t(d.pos) + 1u;                 // decode_one's reference length (>= 1)
    }
    const int64_t row = B.row0 + i;
    if (PASS == 0) {
        s_key[threadIdx.x] = make_int2(d.tid, d.pos);
        if (active) {
            const int bk = 31 - __clz(span);
            atomicAdd(&s_bn[bk], 1u);
            atomicMax(&s_bm[bk], span);
            atomicMax(&s_reach, (long long)(int64_t(d.pos) + int64_t(span)));   // signed: a malformed pos < -1 cannot win
            if ((row & (kIndexStride - 1)) == 0) keys[row / kIndexStride] = pack_key(d.tid, d.pos);
        }
        __syncthreads();
        uint32_t bad = d.bad;
        if (active) {
            const bool have_prev = threadIdx.x > 0 || i > 0 || bi > 0;
            const int2 prev = threadIdx.x > 0 ? s_key[threadIdx.x - 1] : (have_prev ? key_before(table, bi, B, i) : make_int2(0, 0));
            if (have_prev && before_key(uint32_t(d.tid), d.pos, uint32_t(prev.x), prev.y)) bad |= STATUS_UNSORTED;
        }
        if (bad) atomicOr(&isc->status, bad);
        if (threadIdx.x < kSpanBuckets && s_bn[threadIdx.x]) {
            atomicAdd(&isc->bucket_n[threadIdx.x], s_bn[threadIdx.x]);
            atomicMax(&isc->bucket_max[threadIdx.x], s_bm[threadIdx.x]);
        }
        if (threadIdx.x == 0) atomicMax(&isc->reach, s_reach);
    } else {
        const bool is_long = active && span > long_span;
        const uint32_t slot = is_long ? atomicAdd(&s_nl, 1u) : 0u;
        __syncthreads();
        if (threadIdx.x == 0 && s_nl) s_base = atomicAdd(&isc->n_long, s_nl);
        __syncthreads();
        if (is_long) {
            long_key[s_base + slot] = pack_key(d.tid, d.pos);
            long_row[s_base + slot] = make_int2(bi, i);
        }
    }
}

// K3f: per tile, the short-span rows with key in [loc - s_lo, loc + len + s_hi) and the long-list entries with key in
// [loc - l_lo, loc + len + l_hi).  A short range is found in the sampled keys first (every 32nd row; they stay in L2),
// then among the <= 31 rows between two samples through offs[] and the raw bytes.
__device__ __forceinline__ int64_t lower_bound_rows(const ResidentView& v, uint32_t qt, int64_t qp) {
    int64_t lo = 0, hi = v.n_keys;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key_less(__ldg(v.keys + mid), qt, qp)) lo = mid + 1; else hi = mid;
    }
    if (lo == 0) return 0;                                   // row 0 is not below the key
    int64_t a = (lo - 1) * kIndexStride + 1, b = min(lo * kIndexStride, v.n);   // row a-1 is below, row b is not (or n)
    while (a < b) {
        const int64_t mid = (a + b) >> 1;
        const DecodeBatch& B = v.batches[batch_of_row(v, mid)];
        const int2 k = record_key(B.raw, __ldg(B.offs + (mid - B.row0)));
        if (key_less(pack_key(k.x, k.y), qt, qp)) a = mid + 1; else b = mid;
    }
    return a;
}
__device__ __forceinline__ int64_t lower_bound_long(const ResidentView& v, uint32_t qt, int64_t qp) {
    int64_t lo = 0, hi = v.n_long;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key_less(__ldg(v.long_key + mid), qt, qp)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(kThreads) k_join_fused(ResidentView v, TileTable tiles, int64_t* __restrict__ long_lo,
                                                         int64_t* __restrict__ long_hi, int64_t n_tiles, FusedHalos h,
                                                         DeviceScalars* sc) {
    const int64_t i = int64_t(blockIdx.x) * kThreads + threadIdx.x;
    long long cand = 0;
    if (i < n_tiles) {
        const uint32_t rid = uint32_t(tiles.rid[i]);
        const int64_t loc = tiles.loc[i], len = tiles.len[i];
        const int64_t lo = lower_bound_rows(v, rid, loc - h.s_lo);
        const int64_t hi = max(lo, lower_bound_rows(v, rid, loc + len + h.s_hi));
        const int64_t llo = lower_bound_long(v, rid, loc - h.l_lo);
        const int64_t lhi = max(llo, lower_bound_long(v, rid, loc + len + h.l_hi));
        tiles.cand_lo[i] = lo; tiles.cand_hi[i] = hi;
        long_lo[i] = llo; long_hi[i] = lhi;
        cand = (hi - lo) + (lhi - llo);
    }
    __shared__ long long s_c[kThreads / 32];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cand += __shfl_xor_sync(FULL, cand, o);
    if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = cand;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long tot = 0;
        for (int k = 0; k < kThreads / 32; ++k) tot += s_c[k];
        if (tot) atomicAdd(&sc->candidates, (unsigned long long)tot);
    }
}

// K4f: one CTA per tile.  The tile's short range goes through shared memory in chunks of <= kThreads rows that stay
// inside one resident batch, one bulk copy per chunk (a chunk whose bytes exceed kFusedCap is halved until it fits; a
// single record that does not fit takes the global-load path); one thread per record: decode_one, keep_read,
// pileup_coord, profile_slot - K1's and K4's code.  Rows with span > long_span are left to the long list, which is read
// with global loads.  Then copy_out, as k_profile.
constexpr int kFusedCap = 12288;          // staging bytes per CTA: 256 records of <= 48 B, or fewer larger ones
template <bool SS, int BIN>
__global__ void __launch_bounds__(kThreads) k_pileup_fused(ResidentView v, TileTable tiles, const int64_t* __restrict__ long_lo,
                                                           const int64_t* __restrict__ long_hi, FilterParams p, int32_t binsize,
                                                           uint64_t magic, uint32_t mshift, int32_t* __restrict__ out) {
    extern __shared__ __align__(128) uint8_t smem_f[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t s_lo, s_bytes;
    __shared__ int s_b;
    __shared__ long long s_r1;
    const int64_t tix = blockIdx.x;
    const int32_t loc = tiles.loc[tix], len = tiles.len[tix];
    const int flip = tiles.strand[tix] < 0 ? 1 : 0;
    const int64_t lo = tiles.cand_lo[tix], hi = tiles.cand_hi[tix];
    const int64_t off = tiles.out_off[tix];
    const int nbins = BIN == kBinOne ? 1 : (BIN == kBin1 ? len : int((uint32_t(len) + uint32_t(binsize) - 1u) / uint32_t(binsize)));
    const int nout = SS ? 2 * nbins : nbins;
    int32_t* const dst = out + off;
    int32_t* hist = reinterpret_cast<int32_t*>(smem_f + kFusedCap) + out_phase(dst);     // same 16-byte phase as dst
    const uint32_t bar_a = smem_u32(&bar);
    // thread 0 stages the chunk of rows that starts at r0: <= kThreads rows inside one resident batch, halved until
    // their bytes fit the staging buffer (s_bytes = 0: one record too large, the chunk takes the global-load path)
    auto stage_chunk = [&](int64_t r0) {
        const int b = batch_of_row(v, r0);
        const DecodeBatch B = v.batches[b];
        int64_t r1 = min(hi, min(r0 + kThreads, B.row0 + B.n));
        const uint32_t o_lo = B.offs[r0 - B.row0] & ~15u;
        uint32_t bytes = (B.offs[r1 - B.row0] - o_lo + 15u) & ~15u;
        while (bytes > uint32_t(kFusedCap) && r1 - r0 > 1) {
            r1 = r0 + (r1 - r0) / 2;
            bytes = (B.offs[r1 - B.row0] - o_lo + 15u) & ~15u;
        }
        s_bytes = 0;
        if (bytes <= uint32_t(kFusedCap)) { bulk_to_shared(bar_a, smem_f, B.raw + o_lo, bytes); s_bytes = bytes; }
        s_lo = o_lo; s_b = b; s_r1 = r1;
    };
    // the first chunk's copy is in flight while the histogram is zeroed and the long-list rows are counted
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (lo < hi) stage_chunk(lo);
    }
    {
        int4* h4 = reinterpret_cast<int4*>(smem_f + kFusedCap);
        const int nq = (int(hist - reinterpret_cast<int32_t*>(h4)) + nout + 3) >> 2;
        for (int k = threadIdx.x; k < nq; k += kThreads) h4[k] = make_int4(0, 0, 0, 0);
    }
    __syncthreads();
    auto count = [&](const Decoded& d) {
        int32_t a;
        const bool keep = keep_read(p, d.flagmq, d.tlen, &a);
        const bool neg = (d.flagmq & 0x10u) != 0;
        const int32_t k = profile_slot<SS, BIN>(pileup_coord(p, d, a, neg), keep ? int32_t(neg) : -1, loc, len, flip, magic, mshift);
        if (k >= 0) atomicAdd(&hist[k], 1);
    };
    for (int64_t e = long_lo[tix] + threadIdx.x; e < long_hi[tix]; e += kThreads) {
        const int2 br = __ldg(v.long_row + e);
        const DecodeBatch& B = v.batches[br.x];
        count(decode_one(GlobalLd{B.raw}, __ldg(B.offs + br.y), __ldg(B.offs + br.y + 1)));
    }
    uint32_t phase = 0;
    for (int64_t r0 = lo; r0 < hi;) {                                             // block-uniform
        const int64_t r1 = s_r1;
        const DecodeBatch& B = v.batches[s_b];
        const int64_t r = r0 + threadIdx.x;
        uint32_t o = 0, rec_end = 0;
        if (r < r1) { o = __ldg(B.offs + (r - B.row0)); rec_end = __ldg(B.offs + (r - B.row0) + 1); }
        const bool staged = s_bytes != 0;
        if (staged) { wait_parity(bar_a, phase); phase ^= 1u; }
        if (r < r1) {
            const Decoded d = staged ? decode_one(SharedLd{smem_f, s_lo}, o, rec_end) : decode_one(GlobalLd{B.raw}, o, rec_end);
            if (uint32_t(d.end) - uint32_t(d.pos) + 1u <= v.long_span) count(d);  // a longer read is the long list's
        }
        __syncthreads();                                                          // staging buffer and s_* free again
        r0 = r1;
        if (r0 < hi) {
            if (threadIdx.x == 0) stage_chunk(r0);
            __syncthreads();
        }
    }
    __syncthreads();
    copy_out(dst, hist, nout);
}

// ---------------------------------------------------------------------------------------------------------------
// Result narrowing (see kernels.cuh): four elements per thread, one 32-bit store; src is only 4-byte aligned.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_u8(const int32_t* __restrict__ src, int64_t n, uint8_t* __restrict__ dst, uint2* ovf,
                                                 uint32_t cap, uint32_t* cnt) {
    const int64_t i0 = (int64_t(blockIdx.x) * 256 + threadIdx.x) * 4;
    if (i0 >= n) return;
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int64_t i = i0 + k;
        if (i < n) {
            const int32_t v = __ldcs(src + i);
            uint32_t b = uint32_t(v);
            if (uint32_t(v) > 254u) {                  // also negative values (none are produced; they would be kept exactly)
                b = 255u;
                const uint32_t slot = atomicAdd(cnt, 1u);
                if (slot < cap) ovf[slot] = make_uint2(uint32_t(i), uint32_t(v));
            }
            word |= b << (8 * k);
        }
    }
    if (i0 + 3 < n) *reinterpret_cast<uint32_t*>(dst + i0) = word;
    else for (int k = 0; k < 4 && i0 + k < n; ++k) dst[i0 + k] = uint8_t(word >> (8 * k));
}
__global__ void k_publish_reset(uint32_t* cnt, uint32_t* host_cnt) {
    *host_cnt = *cnt;
    *cnt = 0u;
    __threadfence_system();
}

void magic_for(int32_t d, uint64_t* magic, uint32_t* shift) {
    uint32_t L = 0;
    while ((1ull << L) < uint64_t(d)) ++L;
    *shift = 32 + L;
    const unsigned __int128 num = (unsigned __int128)1 << (32 + L);
    *magic = uint64_t((num + uint64_t(d) - 1) / uint64_t(d));
}
// k_profile_agg's 32-bit multiplier and shift (see there)
void agg_magic_for(int32_t d, uint32_t* magic, uint32_t* shift) {
    uint32_t L = 0;
    while ((1ull << L) < uint64_t(d)) ++L;
    *magic = uint32_t(((1ull << (31 + L)) + uint64_t(d) - 1) / uint64_t(d));
    *shift = L - 1;
}

// The runs kernels' instantiation for (ss, binsize), with the divisor of the dense kernel that binsize selects:
// f(std::bool_constant<SS>, std::integral_constant<int, KIND>, magic, mshift).
template <class F>
void with_profile_kind(int ss, int32_t binsize, F&& f) {
    using K0 = std::integral_constant<int, 0>;
    using K1 = std::integral_constant<int, 1>;
    using K2 = std::integral_constant<int, 2>;
    if (binsize >= 4) {
        uint32_t magic, mshift;
        agg_magic_for(binsize, &magic, &mshift);
        if (ss) f(std::true_type{}, K2{}, uint64_t(magic), mshift); else f(std::false_type{}, K2{}, uint64_t(magic), mshift);
        return;
    }
    uint64_t magic; uint32_t mshift;
    magic_for(binsize, &magic, &mshift);
    if (binsize == 1) { if (ss) f(std::true_type{}, K0{}, magic, mshift); else f(std::false_type{}, K0{}, magic, mshift); }
    else              { if (ss) f(std::true_type{}, K1{}, magic, mshift); else f(std::false_type{}, K1{}, magic, mshift); }
}

}  // namespace

void launch_decode(const DecodeBatch& one, ReadTable t, bool coverage, bool ss, const FilterParams& p, DeviceScalars* sc, cudaStream_t s) {
    if (one.n <= 0) return;
    const int grid = (one.n + kDecThreads - 1) / kDecThreads;
    DecodeBatch b = one;
    b.chunk0 = 0;
    if (coverage && ss) k_decode_coverage_ss<<<unsigned(grid), kDecThreads, kSpanCap + 32, s>>>(b, nullptr, 1, t, p, sc);
    else if (coverage) k_decode<true><<<unsigned(grid), kDecThreads, kSpanCap + 32, s>>>(b, nullptr, 1, t, p, sc);
    else k_decode<false><<<unsigned(grid), kDecThreads, kSpanCap + 32, s>>>(b, nullptr, 1, t, p, sc);
}

void launch_decode_table(const DecodeBatch* d_table, int n_batches, int total_chunks, ReadTable t, bool coverage, bool ss,
                         const FilterParams& p, DeviceScalars* sc, cudaStream_t s) {
    if (n_batches <= 0 || total_chunks <= 0) return;
    const unsigned grid = unsigned(total_chunks);
    if (coverage && ss) k_decode_coverage_ss<<<grid, kDecThreads, kSpanCap + 32, s>>>(DecodeBatch{}, d_table, n_batches, t, p, sc);
    else if (coverage) k_decode<true><<<grid, kDecThreads, kSpanCap + 32, s>>>(DecodeBatch{}, d_table, n_batches, t, p, sc);
    else k_decode<false><<<grid, kDecThreads, kSpanCap + 32, s>>>(DecodeBatch{}, d_table, n_batches, t, p, sc);
}

void launch_join(ReadTable t, int64_t n, TileTable tiles, int64_t n_tiles, const DeviceScalars* sc, cudaStream_t s) {
    if (n_tiles <= 0) return;
    const int64_t grid = (n_tiles + kThreads - 1) / kThreads;
    k_join<<<unsigned(grid), kThreads, 0, s>>>(t, n, tiles, n_tiles, sc, const_cast<DeviceScalars*>(sc));
}

void launch_count(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t* out,
                  DeviceScalars*, cudaStream_t s) {
    if (n_tiles <= 0) return;
    const int64_t grid = (n_tiles * 32 + kThreads - 1) / kThreads;
    k_count<<<unsigned(grid), kThreads, 0, s>>>(tiles, n_tiles, c0, c1, ss, out);
}

void launch_profile(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                    int max_tile_ints, int32_t* out, DeviceScalars*, cudaStream_t s) {
    if (n_tiles <= 0) return;
    const size_t smem = size_t(max_tile_ints + 4) * sizeof(int32_t);
    const unsigned grid = unsigned(n_tiles);
    if (binsize >= 4) {
        uint32_t magic, mshift;
        agg_magic_for(binsize, &magic, &mshift);
        if (ss) k_profile_agg<true><<<grid, kThreads, smem, s>>>(tiles, c0, c1, binsize, magic, mshift, out);
        else k_profile_agg<false><<<grid, kThreads, smem, s>>>(tiles, c0, c1, binsize, magic, mshift, out);
        return;
    }
    uint64_t magic; uint32_t mshift;
    magic_for(binsize, &magic, &mshift);
#define BSG_LAUNCH_PROFILE(SS, B1) k_profile<SS, B1><<<grid, kThreads, smem, s>>>(tiles, c0, c1, binsize, magic, mshift, out)
    if (binsize == 1) { if (ss) BSG_LAUNCH_PROFILE(true, true); else BSG_LAUNCH_PROFILE(false, true); }
    else              { if (ss) BSG_LAUNCH_PROFILE(true, false); else BSG_LAUNCH_PROFILE(false, false); }
#undef BSG_LAUNCH_PROFILE
}

void launch_coverage(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                     int32_t* out, DeviceScalars*, cudaStream_t s) {
    if (n_tiles <= 0) return;
    const size_t smem = size_t(max_tile_ints + 8) * sizeof(int32_t);
    if (ss) k_coverage_ss<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, c0, c1, out);
    else k_coverage<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, c0, c1, out);
}

void launch_coverage_runs(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                          RunTiles rt, const int32_t* vt, int64_t lists, int64_t* run_off, cudaStream_t s) {
    const size_t smem = size_t(max_tile_ints) * sizeof(int32_t);
    if (n_tiles > 0) {
        if (ss) k_runs_count_ss<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, n_tiles, c0, c1, rt, vt);
        else k_runs_count<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, c0, c1, rt);
    }
    k_runs_scan<<<1, kScanThreads, 0, s>>>(rt, (ss ? 2 : 1) * n_tiles, lists, run_off);
}

void launch_coverage_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int max_tile_ints,
                                RunTiles rt, const int32_t* vt, const int64_t* run_off, int32_t* lengths, int32_t* values,
                                cudaStream_t s) {
    if (n_tiles <= 0) return;
    const size_t smem = size_t(max_tile_ints + 4) * sizeof(int32_t);
    if (ss) k_runs_write_ss<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, n_tiles, c0, c1, rt, vt, run_off, lengths, values);
    else k_runs_write<<<unsigned(n_tiles), kThreads, smem, s>>>(tiles, n_tiles, c0, c1, rt, run_off, lengths, values);
}

void launch_profile_runs(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                         int max_tile_ints, RunTiles rt, const int32_t* vt, int64_t lists, int64_t* run_off, cudaStream_t s) {
    if (n_tiles > 0)
        with_profile_kind(ss, binsize, [&](auto SS, auto KIND, uint64_t magic, uint32_t mshift) {
            k_profile_runs_count<SS(), KIND()><<<unsigned(n_tiles), kThreads, size_t(max_tile_ints) * sizeof(int32_t), s>>>(
                tiles, n_tiles, c0, c1, binsize, magic, mshift, rt, vt);
        });
    k_runs_scan<<<1, kScanThreads, 0, s>>>(rt, (ss ? 2 : 1) * n_tiles, lists, run_off);
}

void launch_profile_runs_write(TileTable tiles, int64_t n_tiles, const int32_t* c0, const int32_t* c1, int ss, int32_t binsize,
                               int max_tile_ints, RunTiles rt, const int32_t* vt, const int64_t* run_off, int32_t* lengths,
                               int32_t* values, cudaStream_t s) {
    if (n_tiles <= 0) return;
    with_profile_kind(ss, binsize, [&](auto SS, auto KIND, uint64_t magic, uint32_t mshift) {
        k_profile_runs_write<SS(), KIND()><<<unsigned(n_tiles), kThreads, size_t(max_tile_ints) * sizeof(int32_t), s>>>(
            tiles, n_tiles, c0, c1, binsize, magic, mshift, rt, vt, run_off, lengths, values);
    });
}

void launch_resident_index(const DecodeBatch* d_table, int n_batches, int total_chunks, int pass, uint32_t long_span,
                           unsigned long long* keys, unsigned long long* long_key, int2* long_row, IndexScalars* isc, cudaStream_t s) {
    if (n_batches <= 0 || total_chunks <= 0) return;
    if (pass == 0) k_resident_index<0><<<unsigned(total_chunks), kDecThreads, kSpanCap + 32, s>>>(d_table, n_batches, long_span, keys, long_key, long_row, isc);
    else k_resident_index<1><<<unsigned(total_chunks), kDecThreads, kSpanCap + 32, s>>>(d_table, n_batches, long_span, keys, long_key, long_row, isc);
}

void launch_join_fused(const ResidentView& v, TileTable tiles, int64_t* long_lo, int64_t* long_hi, int64_t n_tiles,
                       const FusedHalos& h, DeviceScalars* sc, cudaStream_t s) {
    if (n_tiles <= 0) return;
    k_join_fused<<<unsigned((n_tiles + kThreads - 1) / kThreads), kThreads, 0, s>>>(v, tiles, long_lo, long_hi, n_tiles, h, sc);
}

void launch_pileup_fused(const ResidentView& v, TileTable tiles, const int64_t* long_lo, const int64_t* long_hi, int64_t n_tiles,
                         int ss, int32_t binsize, int max_tile_ints, const FilterParams& p, int32_t* out, cudaStream_t s) {
    if (n_tiles <= 0) return;
    const size_t smem = kFusedCap + size_t(max_tile_ints + 8) * sizeof(int32_t);
    uint64_t magic = 0; uint32_t mshift = 0;
    if (binsize > 1) magic_for(binsize, &magic, &mshift);
    const unsigned grid = unsigned(n_tiles);
#define BSG_LAUNCH_FUSED(SS, BIN) k_pileup_fused<SS, BIN><<<grid, kThreads, smem, s>>>(v, tiles, long_lo, long_hi, p, binsize, magic, mshift, out)
    if (binsize <= 0)      { if (ss) BSG_LAUNCH_FUSED(true, kBinOne); else BSG_LAUNCH_FUSED(false, kBinOne); }
    else if (binsize == 1) { if (ss) BSG_LAUNCH_FUSED(true, kBin1);   else BSG_LAUNCH_FUSED(false, kBin1); }
    else                   { if (ss) BSG_LAUNCH_FUSED(true, kBinDiv); else BSG_LAUNCH_FUSED(false, kBinDiv); }
#undef BSG_LAUNCH_FUSED
}

void launch_pack_u8(const int32_t* d_src, int64_t n, uint8_t* d_dst, uint2* ovf, uint32_t cap, uint32_t* d_cnt, cudaStream_t s) {
    if (n <= 0) return;
    k_pack_u8<<<unsigned((n + 1023) / 1024), 256, 0, s>>>(d_src, n, d_dst, ovf, cap, d_cnt);
}
void launch_publish_reset(uint32_t* d_cnt, uint32_t* host_cnt, cudaStream_t s) { k_publish_reset<<<1, 1, 0, s>>>(d_cnt, host_cnt); }

}  // namespace bsg
