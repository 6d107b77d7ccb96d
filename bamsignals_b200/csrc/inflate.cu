// GPU-side BGZF inflate, CRC32 check and record-boundary walk (SURVEY.md 8f ranks 1 and 2): the host only reads the
// file and ships COMPRESSED bytes; raw-DEFLATE decoding of every BGZF block, its integrity check and the block_size
// chain walk run on the device.
//
// k_inflate_ws: warp-specialised.  One persistent CTA per SM holds 64 BGZF blocks (RFC 1951 streams, <= 64 KiB out each)
//   at a time: the 64 lanes of warps 0-1 each decode the Huffman symbols of ONE stream into a shared-memory token queue
//   (32 tokens per round); warps 2-17 turn the queues of the previous round into bytes, byte-parallel, in 256-byte
//   chunks built on a shared-memory stage (materialise()); warp 18 follows the RECORD chain of every block right behind
//   them (SpecOut).  The halves overlap through double-buffered queues and ONE CTA barrier per round.  The CTA leaves
//   2 KB of the SM's shared memory free: kernels without shared memory (the ones below) run next to it.
// k_crc32: one warp per block: 32 slicing-by-4 pieces folded with carry-less multiplies; tables in global memory.
// k_walk_*: record boundaries between index entry points (BAI linear-index offsets and chunk bounds are record-aligned).
//   k_walk_span: every span's chain followed through device memory (count, scan, write) - for short spans.
//   k_walk_link / k_walk_write: spans linked through the per-block chains the inflate kernel left, O(1) per block; only
//   what those cannot cover (a record straddling into a block) is walked.  A scan of the per-span counts gives every span
//   its slice of the offsets array (no atomics, deterministic order).
//
// Designs measured and dropped (C2, B200; see DESIGN.md): round 1: per-symbol warp round trip (150 ms), D = 4/8/16
// lock-step streams per warp with group copies (142-282 ms), one stream per lane doing its own copies (235 ms), one warp
// per TWO streams alternating between a decode phase on lanes 0/16 and a warp-wide copy phase (73.7 ms; one stream 82.8,
// four 99.2; next-line prefetch of the compressed input and loads-first match copies: no gain,
// profiles/r2_ab_inflate_variants_c2.json).  ncu on that kernel: 70 warp instructions per token with 1.6 active lanes in
// the decode phase - the lanes were the wasted resource, hence one stream per LANE here.
#include "kernels.cuh"

#include <algorithm>

#include "inflate_core.cuh"

namespace bsg {
namespace {

constexpr unsigned FULL = 0xffffffffu;

// ---------------------------------------------------------------------------------------------------------------
// k_inflate_ws
// ---------------------------------------------------------------------------------------------------------------
constexpr int kWsDecWarps = 2;                       // warps whose 32 lanes decode one stream each
constexpr int kWsStreams = kWsDecWarps * 32;         // streams resident per CTA (= per SM)
constexpr int kWsCopyWarps = 16;                     // warps that materialise the token queues, four streams each
constexpr int kWsChainWarp = kWsDecWarps + kWsCopyWarps;      // the warp that follows the record chains (SpecOut)
constexpr int kWsThreads = (kWsDecWarps + kWsCopyWarps + 1) * 32;

struct WsStream {
    inflate_core::Tables T;
    uint32_t q[2][inflate_core::kQueue];             // token queues of the round being decoded / being materialised
};
struct WsCtl {
    uint8_t qn[2][kWsStreams];                       // tokens in q[buf] of every stream (<= 32)
    uint32_t pos[kWsStreams];                        // bytes materialised so far (owned by the stream's copy warp)
    uint32_t out_off[kWsStreams];
    uint32_t produced[2][kWsDecWarps];               // did the decode warp hand over anything in round buf, or has it a
                                                     // stream that is not finished?
    alignas(8) uint8_t stage[kWsCopyWarps][256];     // a copy warp's chunk of output being built (also its bitmap scratch)
};
constexpr size_t kWsSmem = sizeof(WsStream) * kWsStreams + sizeof(WsCtl);
static_assert(sizeof(WsStream) % 4 == 0 && (sizeof(WsStream) * kWsStreams) % 8 == 0, "stream slots keep queues and stage aligned");
// One CTA per SM, and 2 KB less than the SM has (228 KB - 1 KB reserved per resident CTA): a CTA of a kernel WITHOUT shared
// memory (record walk, CRC32, the one-thread publishers) then fits next to it, so those kernels of the batch before run
// in the shadow of this one instead of between two launches (the launch is persistent and would otherwise own every SM
// until it ends).
static_assert(kWsSmem <= 226 * 1024, "leave room for a co-resident CTA without shared memory");
static_assert(kWsCopyWarps * 4 == kWsStreams, "every copy warp owns four streams");

// fill_queue's table lookups and queue stores through explicit shared-space addresses (kept in registers)
struct SmemAccess {
    uint32_t lit_a, dist_a, q_a;
    __device__ __forceinline__ uint32_t lit(uint32_t byte_off) const {
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(lit_a + byte_off) : "memory");
        return r;
    }
    __device__ __forceinline__ uint32_t dist(uint32_t byte_off) const {
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(dist_a + byte_off) : "memory");
        return r;
    }
    __device__ __forceinline__ void put(uint32_t byte_off, uint32_t v) const {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(q_a + byte_off), "r"(v) : "memory");
    }
    __device__ __forceinline__ uint32_t sub_if(bool take, uint32_t byte_off, uint32_t otherwise) const {     // predicated
        constexpr uint32_t off = offsetof(inflate_core::Tables, lit_sub);
        uint32_t r = otherwise;
        asm volatile("{ .reg .pred p; setp.ne.u32 p, %2, 0; @p ld.shared.u16 %0, [%1]; }"
                     : "+r"(r) : "r"(lit_a + off + byte_off), "r"(uint32_t(take)) : "memory");
        return r;
    }
    __device__ __forceinline__ uint32_t count(uint32_t len) const {
        constexpr uint32_t off = offsetof(inflate_core::Tables, dist_count);
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(lit_a + off + 2u * len) : "memory");
        return r;
    }
    __device__ __forceinline__ uint32_t first() const {
        constexpr uint32_t off = offsetof(inflate_core::Tables, dist_first);
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(lit_a + off) : "memory");
        return r;
    }
    __device__ __forceinline__ uint32_t index() const {
        constexpr uint32_t off = offsetof(inflate_core::Tables, dist_index);
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(lit_a + off) : "memory");
        return r;
    }
    __device__ __forceinline__ uint32_t sorted(uint32_t i) const {
        constexpr uint32_t off = offsetof(inflate_core::Tables, dist_sorted);
        uint32_t r;
        asm volatile("ld.shared.u16 %0, [%1];" : "=r"(r) : "r"(lit_a + off + 2u * i) : "memory");
        return r;
    }
};

// Copy side: a queue (<= 32 tokens, one token per lane) -> bytes, by one warp.
//
// Byte-parallel: every lane produces ONE byte of 32 consecutive output bytes per step.  The lane finds the token that owns
// its byte - a bitmap of token start positions (one 32-bit word per step, 1024 bytes per window) plus a prefix pop-count,
// moved between lanes with shuffles - and then where the byte comes from: the token's literal, or `dist` bytes back (a
// match that overlaps itself, dist < len, jumps in front of its own start with one modulo; a source inside the step's own
// 32 bytes, distance < 32: rare, is chased through its owner token).
// The output is built in CHUNKS of 256 bytes (eight steps) in a shared-memory stage owned by the warp:
//   pass 1  resolves the eight bytes of every lane; a source in front of the chunk is finished output in global memory
//           and its load is ISSUED (eight independent loads per lane in flight); a source inside the chunk is noted;
//   pass 2  goes through the steps in order: bytes with a source inside the chunk read it from the stage (written by an
//           earlier step: ~30 cycles instead of a trip to L2), every byte is put on the stage;
//   pass 3  writes the chunk out with one 8-byte store per lane (the partial first / last word byte by byte).
// So the warp waits for memory once per 256 bytes - for loads that were all issued before the first one is needed - and
// what it waits for is usually a record several back, not the previous step's stores.
// History (ncu, C2): token-per-lane copies in waves of matches that read each other's output: the copy warps sat on
// dependent L2 round trips (22 % of all samples on one line) while the decode warps waited at the barrier, 10.0 ms per
// wave of 9472 blocks; four bytes per lane chased through the whole window: ~10 rounds of shuffles per step, 10.7 ms;
// chased through the 128 bytes of the step only: 5.5 rounds, 8.7 ms; one byte per lane, load -> store -> next step, four
// queues interleaved per warp: 6.6 ms, then 5.5 ms with the faster decode side, the copy warps the bottleneck again
// (half of the L2 reads miss: the 32 KiB windows of 9472 streams are 2.5x the L2, so every step waited for DRAM).
constexpr int kQpw = 4;                              // queues (streams) per copy warp, one after the other (taking them
                                                     // dynamically, one atomic per queue: measured, 8.69 vs 8.50 ms - dropped;
                                                     // so was a second-level table for long DISTANCE codes: 8.55 vs 8.50)
constexpr int kChunk = 256;                          // bytes staged per chunk
constexpr int kSteps = kChunk / 32;

// One more warp of the CTA, the CHAIN warp, follows every resident block's RECORD chain (block_size -> next record) right
// behind the copy warps, one or two streams per lane: the bytes are a round old and L2-resident (~235 ns per step,
// profiles/r2_chain_probe.txt; the same chain costs up to 500 ns per step once the batch has left the L2), a round
// brings ~4 records per stream, and the warp has the whole round (~14 us) for them.  The record walk gets, per block, the
// offsets of the chain that starts at the block's first byte - a speculation (a record may straddle into the block),
// verified and linked by k_walk_link.  (Following the chain from lane 0 of the copy warps while a chunk is on the stage
// was measured first: 8.5 -> 12.2 ms per two waves, 31 idle lanes per step.)
struct SpecOut {
    uint32_t* offs;        // [n_blocks][kSpecStride] absolute offsets (into the batch's raw buffer) of the chain's records
    uint32_t* cnt;         // [n_blocks] records on the chain; kSpecNone = no usable chain (implausible record, stored block ...)
    uint32_t* end;         // [n_blocks] where the chain first reaches or passes the block's end (absolute)
};
constexpr uint32_t kSpecStride = 1824;               // a record takes >= 36 bytes: at most 1821 start in a 64 KiB block
constexpr uint32_t kSpecNone = 0xffffffffu;

// One queue -> bytes at first_byte; stage = kChunk bytes of shared memory owned by the warp (8-byte aligned).
// Returns the number of bytes.
__device__ __forceinline__ uint32_t materialise(const uint32_t* q, int nq, uint8_t* first_byte, int lane, uint8_t* stage) {
    const bool valid = lane < nq;
    const uint32_t t = valid ? q[lane] : 0u;
    const uint32_t len = (t >> 31) ? (t & 0x1ffu) : (valid ? 1u : 0u);
    uint32_t incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t up = __shfl_up_sync(FULL, incl, o);
        if (lane >= o) incl += up;
    }
    const uint32_t total = __shfl_sync(FULL, incl, 31);
    if (total == 0) return 0;
    // u coordinates: byte u lives at al[u]; al is the 8-byte aligned address at or before the first byte
    const int32_t a0 = int32_t(reinterpret_cast<uintptr_t>(first_byte) & 7u);
    uint8_t* al = first_byte - a0;
    const int32_t s = int32_t(incl - len) + a0, e = s + int32_t(len), end_u = a0 + int32_t(total);
    uint32_t* bm_s = reinterpret_cast<uint32_t*>(stage);          // the first 128 bytes double as the bitmap scratch
    for (int32_t wb = 0; wb < end_u; wb += 1024) {                 // warp-uniform
        // bitmap of token starts in the window + prefix counts: tokens that end at or before the window come first; then
        // bit (start - wb) for every token in the window (one that began before it and reaches into it owns bit 0)
        const int32_t wend = min(end_u, wb + 1024);
        const uint32_t firstk = uint32_t(__popc(__ballot_sync(FULL, valid && e <= wb)));
        bm_s[lane] = 0u;
        __syncwarp();
        if (valid && e > wb && s < wend) {
            const uint32_t r = uint32_t(max(s, wb) - wb);
            atomicOr(&bm_s[r >> 5], 1u << (r & 31u));
        }
        __syncwarp();
        const uint32_t bm = bm_s[lane];
        __syncwarp();
        uint32_t pre;
        {
            const uint32_t pc = uint32_t(__popc(bm));
            uint32_t inc = pc;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t up = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += up;
            }
            pre = inc - pc;
        }
        for (int32_t cb = wb; cb < wend; cb += kChunk) {           // warp-uniform
            const int32_t clim = min(wend, cb + kChunk);
            const int32_t front = max(cb, a0);                     // sources below this are finished output in global memory
            uint32_t val[kSteps];
            uint32_t near_mask = 0u, far_mask = 0u;                // bit i: val[i] is a position on the stage / in front of it, not a byte
            // ---- pass 1: resolve ... -------------------------------------------------------------------------------------
#pragma unroll
            for (int i = 0; i < kSteps; ++i) {
                const int32_t base = cb + 32 * i;
                val[i] = 0u;
                if (base < clim) {                                 // warp-uniform
                    const int32_t x = base + lane;
                    const int32_t lim = max(base, a0);             // first byte of the step inside the queue
                    const uint32_t m = __shfl_sync(FULL, bm, (base - wb) >> 5), p = __shfl_sync(FULL, pre, (base - wb) >> 5);
                    int k = int((firstk + p + uint32_t(__popc(m & ((2u << lane) - 1u))) - 1u) & 31u);
                    uint32_t tk = __shfl_sync(FULL, t, k);
                    int32_t sk = __shfl_sync(FULL, s, k);
                    const bool mine = x >= a0 && x < end_u;
                    const bool is_lit = !(tk >> 31);
                    const int32_t d0 = int32_t(((tk >> 16) & 0x7fffu) + 1u);
                    const int32_t y0 = x - d0;
                    // the common case without a branch: a literal, or a match whose source lies in front of the step and of
                    // the match itself
                    const bool slow = mine && !is_lit && y0 >= min(sk, lim);
                    val[i] = is_lit ? (tk & 0xffu) : uint32_t(y0 - cb);
                    const uint32_t bit = (mine && !is_lit && !slow) ? (1u << i) : 0u;
                    far_mask |= y0 < front ? bit : 0u;
                    near_mask |= y0 < front ? 0u : bit;
                    if (__any_sync(FULL, slow)) {
                        // rare: the match overlaps itself (dist < len: same phase, in front of it), or its source lies inside
                        // this step's 32 bytes and is chased through its own owner token
                        int32_t xx = x;
                        bool need = slow;
                        for (;;) {
                            if (need) {
                                if (!(tk >> 31)) { val[i] = tk & 0xffu; need = false; }
                                else {
                                    const int32_t d = int32_t(((tk >> 16) & 0x7fffu) + 1u);
                                    int32_t y = xx - d;
                                    if (y >= sk) y = sk - d + (xx - sk) % d;
                                    if (y < lim) {
                                        val[i] = uint32_t(y - cb);
                                        if (y < front) far_mask |= 1u << i; else near_mask |= 1u << i;
                                        need = false;
                                    } else xx = y;
                                }
                            }
                            if (!__any_sync(FULL, need)) break;
                            const uint32_t r = uint32_t((need ? xx : lim) - wb);
                            const uint32_t m2 = __shfl_sync(FULL, bm, int(r >> 5)), p2 = __shfl_sync(FULL, pre, int(r >> 5));
                            k = int((firstk + p2 + uint32_t(__popc(m2 & ((2u << (r & 31u)) - 1u))) - 1u) & 31u);
                            tk = __shfl_sync(FULL, t, k);
                            sk = __shfl_sync(FULL, s, k);
                        }
                    }
                }
            }
            // ... and issue the loads of the sources in front of the chunk, back to back (no control flow between them: a
            // load inside the resolve loop was waited for at the next step's first branch)
#pragma unroll
            for (int i = 0; i < kSteps; ++i)
                if ((far_mask >> i) & 1u) val[i] = __ldcg(al + cb + int32_t(val[i]));     // L2 only: L1 stays with the decode lanes
            // ---- pass 2: in order through the stage ------------------------------------------------------------------------
#pragma unroll
            for (int i = 0; i < kSteps; ++i) {
                const int32_t base = cb + 32 * i;
                if (base < clim) {                                 // warp-uniform
                    const int32_t x = base + lane;
                    uint32_t v = val[i];
                    if ((near_mask >> i) & 1u) v = stage[v];
                    if (x >= a0 && x < end_u) stage[x - cb] = uint8_t(v);
                    __syncwarp();
                }
            }
            // ---- pass 3: the chunk goes out: whole 8-byte words one per lane, the partial first / last word of the queue
            // byte by byte on lanes 0-7 / 8-15 -----------------------------------------------------------------------------------
            {
                const int32_t lo = cb + 8 * lane;
                if (lo >= front && lo + 8 <= clim) *reinterpret_cast<uint2*>(al + lo) = *reinterpret_cast<const uint2*>(stage + 8 * lane);
                const int32_t hw = front & ~7, tw = clim & ~7;
                const int32_t u = lane < 8 ? hw + lane : tw + (lane - 8);
                const int32_t w = u & ~7;
                if (lane < 16 && (lane < 8 || tw != hw) && u >= front && u < clim && !(w >= front && w + 8 <= clim)) al[u] = stage[u - cb];
            }
            __syncwarp();                                          // the stage is reused; the stores are visible to the next loads
        }
    }
    return total;
}

__global__ void __launch_bounds__(kWsThreads, 1) k_inflate_ws(const InflateBlock* __restrict__ blocks, int n_blocks,
                                                              const uint8_t* __restrict__ comp, uint8_t* raw, SpecOut spec, DeviceScalars* sc) {
    using namespace inflate_core;
    extern __shared__ __align__(16) uint8_t ws_smem[];
    WsStream* S = reinterpret_cast<WsStream*>(ws_smem);
    WsCtl& ctl = *reinterpret_cast<WsCtl*>(ws_smem + sizeof(WsStream) * kWsStreams);
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool is_dec = wid < kWsDecWarps;
    const int s = threadIdx.x;                               // decode lanes: threads 0..63 own streams 0..63
    // Generations: the CTA takes 64 consecutive blocks at a time; all 64 streams of a generation start together, so that
    // the (serial, per-lane) block-header parse and table build run in all lanes at once.
    for (int gen = 0;; ++gen) {
        const int b0 = (gen * int(gridDim.x) + int(blockIdx.x)) * kWsStreams;
        if (b0 >= n_blocks) break;
        bool fin = true;
        InflateBlock blk{0u, 0u, 0u, 0u};
        BitReader br;
        br.base = reinterpret_cast<const uint64_t*>(comp);  // cudaMalloc'ed: aligned
        br.wi = br.a0 = br.a1 = br.b0 = br.b1 = br.p0 = br.p1 = br.bo = 0;
        SmemAccess acc{0u, 0u, 0u};
        if (is_dec) {
            fin = b0 + s >= n_blocks;
            if (!fin) { blk = blocks[b0 + s]; br.init(br.base, blk.in_off); }
            ctl.out_off[s] = blk.out_off; ctl.pos[s] = 0;
            ctl.qn[0][s] = 0; ctl.qn[1][s] = 0;
            acc.lit_a = uint32_t(__cvta_generic_to_shared(S[s].T.lit));
            // identity shuffle: ptxas cannot re-derive the value from %tid inside the decode loop (it otherwise rebuilds
            // the address with several instructions per token); dist and the queues are fixed offsets from it
            acc.lit_a = __shfl_sync(FULL, acc.lit_a, lane);
            acc.dist_a = acc.lit_a + uint32_t(sizeof(uint16_t) << kLitBits);
        }
        const uint32_t out_len = blk.out_len;
        // chain warp: lane l follows the chains of streams l and l + 32 of this generation
        uint32_t c_rp[2] = {0u, 0u}, c_rn[2] = {0u, 0u}, c_len[2] = {0u, 0u}, c_off[2] = {0u, 0u};
        if (wid == kWsChainWarp && spec.offs) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int bi = b0 + lane + 32 * h;
                if (bi < n_blocks) { c_len[h] = blocks[bi].out_len; c_off[h] = blocks[bi].out_off; } else c_rn[h] = kSpecNone;
            }
        }
        // Follow both chains as far as the bytes are known to be written (all = true: to the end of the blocks).  The warp
        // learns how far that is without reading anything another warp writes in the same round: in round r the copy
        // warps turn the queues of round r - 1 into bytes, so the chain warp adds up the token lengths of those queues
        // (read-only in this round) and may, one round later, read that many bytes more.
        uint32_t c_avail[2] = {0u, 0u}, c_pend[2] = {0u, 0u};
        auto chain_follow = [&](bool all, int pb, bool have_q) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int k = lane + 32 * h;
                if (!all) {
                    c_avail[h] += c_pend[h];
                    uint32_t sum = 0;
                    if (have_q) {
                        const int nq = int(ctl.qn[pb][k]);
                        const uint32_t* q = S[k].q[pb];
                        if (nq == 2 && !(q[0] >> 31) && (q[0] & kTokSkip)) sum = q[0] & 0xffffu;
                        else for (int i = 0; i < nq; ++i) { const uint32_t t = q[i]; sum += (t >> 31) ? (t & 0x1ffu) : 1u; }
                    }
                    c_pend[h] = sum;
                }
                const uint32_t avail = all ? c_len[h] : c_avail[h];
                if (c_rn[h] == kSpecNone) continue;
                uint32_t* row = spec.offs + size_t(b0 + k) * kSpecStride;
                uint32_t rp = c_rp[h], rn = c_rn[h];
                while (rp < c_len[h] && rp + 4u <= avail) {
                    const uint32_t a = c_off[h] + rp;                                              // raw itself is aligned, blocks are not
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(raw + (a & ~3u));
                    const uint32_t sh = (a & 3u) * 8u;
                    const uint32_t lo = __ldcg(w), hi = sh ? __ldcg(w + 1) : 0u;                  // L2: L1 may hold the line as it was a round ago
                    const uint32_t bs = __funnelshift_r(lo, hi, sh);
                    if (bs < 32u || bs > 0x00ffffffu || rn >= kSpecStride) { rn = kSpecNone; break; }
                    row[rn++] = c_off[h] + rp;
                    rp += 4u + bs;
                }
                c_rp[h] = rp; c_rn[h] = rn;
            }
        };
        const uint64_t end_bit = (uint64_t(blk.in_off) + blk.in_len) * 8u;
        uint32_t op_dec = 0;
        int phase = 0, last = 0;
        __syncthreads();
        for (int r = 0;; ++r) {
            const int buf = r & 1;
            if (is_dec) {
                // ---- one round of one stream per lane: <= kQueue tokens into q[buf] ------------------------------------
                int nq = 0, state = 0;               // state: 0 = go on, 1 = stream finished, 2 = error
                if (!fin) {
                    uint32_t* q = S[s].q[buf];
                    acc.q_a = acc.lit_a + uint32_t(sizeof(Tables)) + uint32_t(buf) * uint32_t(sizeof(uint32_t) * kQueue);
                    if (phase == 0) {
                        const int h = read_block_header(br, S[s].T, reinterpret_cast<uint8_t*>(q), &last);
                        if (h == 2) state = 2;
                        else if (h == 1) {           // stored block: LEN, NLEN, then LEN bytes that a copy warp moves
                            br.consume((0u - br.bo) & 7u);
                            const uint32_t v = br.peek();
                            br.consume(32);
                            const uint32_t len = v & 0xffffu, nlen = v >> 16;
                            const uint32_t src_off = br.byte_pos();
                            if ((len ^ nlen) != 0xffffu || op_dec + len > out_len || (uint64_t(src_off) + len) * 8u > end_bit) state = 2;
                            else {
                                op_dec += len;
                                br.init(br.base, src_off + len);
                                q[0] = kTokSkip | len;
                                q[1] = src_off;
                                nq = 2;
                                if (last) state = 1;
                            }
                        } else phase = 1;
                    }
                    if (phase == 1 && nq == 0 && state == 0) {
                        int eob = 0, bad = 0;
                        nq = fill_queue(br, acc, &op_dec, &eob, &bad);
                        if (eob) { phase = 0; if (last) state = 1; }
                        if (bad || op_dec > out_len || br.bit_pos() > end_bit) state = 2;
                    }
                    if (state == 2) nq = 0;          // a broken round is discarded; the status flag reports it
                    if (state != 0) {
                        if (state == 2 || op_dec != out_len) atomicOr(&sc->status, STATUS_BAD_DEFLATE);
                        fin = true;
                    }
                }
                ctl.qn[buf][s] = uint8_t(nq);
                // a stream that is not finished keeps the generation going even when it handed over nothing this round (a
                // non-final block that is empty, or whose end-of-block code starts the round); it consumes header bits or
                // meets the end_bit check every round, so the loop stays finite on corrupt input
                const bool any = __any_sync(FULL, nq > 0 || !fin);
                if (lane == 0) ctl.produced[buf][wid] = any ? 1u : 0u;
            } else if (wid == kWsChainWarp) {
                if (spec.offs) chain_follow(false, buf ^ 1, r > 0);
            } else if (r > 0) {
                // ---- the queues of the previous round -> bytes: this warp's four streams, one after the other -----------------
                const int pb = buf ^ 1;
                const int cw = wid - kWsDecWarps;
                uint8_t* stage = ctl.stage[cw];
                for (int j = 0; j < kQpw; ++j) {
                    const int k = cw * kQpw + j;
                    int nq = int(ctl.qn[pb][k]);
                    const uint32_t* q = S[k].q[pb];
                    uint8_t* out = raw + ctl.out_off[k];
                    const uint32_t pos = ctl.pos[k];
                    if (nq == 2 && !(q[0] >> 31) && (q[0] & kTokSkip)) {          // stored block: copy from the compressed buffer
                        const uint32_t len = q[0] & 0xffffu;
                        const uint8_t* src = comp + q[1];
                        for (uint32_t i = lane; i < len; i += 32) out[pos + i] = src[i];
                        __syncwarp();
                        if (lane == 0) ctl.pos[k] = pos + len;
                        nq = 0;
                    }
                    if (nq > 0) {                                                  // warp-uniform
                        const uint32_t total = materialise(q, nq, out + pos, lane, stage);
                        if (lane == 0) ctl.pos[k] = pos + total;
                    }
                }
            }
            __syncthreads();
            bool more = false;
#pragma unroll
            for (int w = 0; w < kWsDecWarps; ++w) more = more || ctl.produced[buf][w] != 0;
            if (!more) break;                        // every stream finished and nothing was handed over in round r: round r - 1
                                                     // was the last one with tokens
        }
        // every stream must have produced exactly ISIZE bytes
        if (threadIdx.x < kWsStreams && b0 + s < n_blocks && ctl.pos[s] != out_len) atomicOr(&sc->status, STATUS_BAD_DEFLATE);
        if (spec.offs && wid == kWsChainWarp) {                 // the rest of the chains, then what the record walk needs of them
            chain_follow(true, 0, false);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int bi = b0 + lane + 32 * h;
                if (bi < n_blocks) {
                    // a chain that stopped short of the block's end (its next size field straddles the end), or whose block
                    // came out short (reported above), is no chain
                    const bool ok = c_rn[h] != kSpecNone && c_rp[h] >= c_len[h] && ctl.pos[lane + 32 * h] == c_len[h];
                    spec.cnt[bi] = ok ? c_rn[h] : kSpecNone;
                    spec.end[bi] = c_off[h] + c_rp[h];
                }
            }
        }
        __syncthreads();                             // the next generation re-initialises the control block
    }
}

// ---------------------------------------------------------------------------------------------------------------
// k_crc32: BGZF integrity check on the device (htslib verifies the CRC32 of every inflated block; so do we).
// One WARP per block: the block is cut into 32 pieces (lane 0 takes the remainder, the other 31 pieces are equally
// long), every lane runs slicing-by-4 over its piece, and the 32 registers are folded in a five-level tree:
// CRC(A || B) = CRC(A) * x^(8 |B|) mod P  xor  CRC(B), where the multiplication is a 32-step carry-less multiply and
// x^(8 |B|) doubles from level to level.  (One THREAD per block, the first version, walked 64 KiB serially with a
// 60-cycle dependent chain per word: 2.4 ms for 0.9 GB, 14-20 % of the end-to-end GPU time; this one is ~25x shorter.)
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t kCrcPoly = 0xEDB88320u;

// a * b mod P in the reflected representation (bit 31 = x^0), as zlib's multmodp
__device__ __forceinline__ uint32_t crc_mul(uint32_t a, uint32_t b) {
    uint32_t p = 0;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
        p ^= (a & 0x80000000u) ? b : 0u;
        a <<= 1;
        b = (b >> 1) ^ ((b & 1u) ? kCrcPoly : 0u);
    }
    return p;
}

constexpr int kCrcWarps = 4;
// x^(2^k) mod P for k = 0..19, reflected (x^1 = 0x40000000; each entry is the square of the one before)
__constant__ uint32_t c_x2n[20] = {0x40000000u, 0x20000000u, 0x08000000u, 0x00800000u, 0x00008000u, 0xedb88320u, 0xb1e6b092u,
                                   0xa06a2517u, 0xed627daeu, 0x88d14467u, 0xd7bbfe6au, 0xec447f11u, 0x8e7ea170u, 0x6427800eu,
                                   0x4d47bae0u, 0x09fe548fu, 0x83852d0fu, 0x30362f1au, 0x7b5a9cc3u, 0x31fec169u};

// slicing-by-4 tables in GLOBAL memory (4 KB, L1-resident): the kernel uses no shared memory, so that its CTAs fit next to
// the persistent inflate CTA of the following batch
__device__ uint32_t g_crc_tab[4][256];
__global__ void k_crc_init() {
    const int i = threadIdx.x;
    uint32_t c = uint32_t(i);
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? kCrcPoly ^ (c >> 1) : c >> 1;
    g_crc_tab[0][i] = c;
    __syncthreads();
    for (int t = 1; t < 4; ++t) { c = g_crc_tab[0][c & 0xffu] ^ (c >> 8); g_crc_tab[t][i] = c; }
}

__global__ void __launch_bounds__(kCrcWarps * 32) k_crc32(const InflateBlock* __restrict__ blocks, const uint32_t* __restrict__ want, int n_blocks,
                                                          const uint8_t* __restrict__ raw, DeviceScalars* sc) {
    const uint32_t (*tab)[256] = g_crc_tab;
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * kCrcWarps + (threadIdx.x >> 5);
    if (b >= n_blocks) return;
    const InflateBlock blk = blocks[b];
    const uint32_t len = blk.out_len;
    const uint32_t seg = (len / 32u) & ~3u;      // lanes 1..31: seg bytes each; lane 0: the remaining head
    const uint32_t head = len - 31u * seg;
    const uint32_t beg = lane == 0 ? 0u : head + uint32_t(lane - 1) * seg;
    uint32_t n = lane == 0 ? head : seg;
    const uint8_t* p = raw + blk.out_off + beg;
    uint32_t crc = lane == 0 ? 0xffffffffu : 0u;
    while (n && (reinterpret_cast<uintptr_t>(p) & 3)) { crc = __ldg(&tab[0][(crc ^ *p++) & 0xffu]) ^ (crc >> 8); --n; }
    const uint32_t* w = reinterpret_cast<const uint32_t*>(p);
    for (; n >= 4; n -= 4) {
        crc ^= *w++;
        crc = __ldg(&tab[3][crc & 0xffu]) ^ __ldg(&tab[2][(crc >> 8) & 0xffu]) ^ __ldg(&tab[1][(crc >> 16) & 0xffu]) ^ __ldg(&tab[0][crc >> 24]);
    }
    p = reinterpret_cast<const uint8_t*>(w);
    while (n--) crc = __ldg(&tab[0][(crc ^ *p++) & 0xffu]) ^ (crc >> 8);
    // fold: at level l the left partner is followed by 2^l pieces of seg bytes
    uint32_t X = 0x80000000u;                    // x^0
    for (uint32_t bits = 8u * seg, k = 0; bits; bits >>= 1, ++k)
        if (bits & 1u) X = crc_mul(c_x2n[k], X);   // x^(8 seg); 8 * seg < 2^20
#pragma unroll
    for (int l = 0; l < 5; ++l) {
        const uint32_t other = __shfl_down_sync(FULL, crc, 1u << l);
        if ((lane & ((2 << l) - 1)) == 0) crc = crc_mul(crc, X) ^ other;
        X = crc_mul(X, X);
    }
    if (lane == 0 && ~crc != want[b]) atomicOr(&sc->status, STATUS_BAD_CRC);
}

// ---------------------------------------------------------------------------------------------------------------
// record-boundary walk
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_u32_any(const uint8_t* raw, uint32_t off) {
    const uint32_t* w = reinterpret_cast<const uint32_t*>(raw + (off & ~3u));
    const uint32_t sh = (off & 3u) * 8;
    const uint32_t lo = w[0];
    const uint32_t hi = sh ? w[1] : 0u;
    return __funnelshift_r(lo, hi, sh);
}

// The walk, block-parallel.  A walker is the span between two index entry points; its record chain is serial, and on deep
// data a span holds tens of thousands of records (C4: 10.8 ms per batch for the longest chains, 2 of 32 lanes busy, the
// bottleneck of the whole call) - and a step of such a chain through global memory costs 235-500 ns.  BAM writers start
// nearly every BGZF block on a record boundary, and the inflate kernel has followed, for every block, the chain that
// starts at the block's first byte while the block went through shared memory (SpecOut).  That chain is a speculation
// - a record may straddle into the block - but an entry point IS a record boundary: from an entry point that lies on the
// block's chain onwards, that chain is the true one.  So:
//   k_walk_link   one thread per WALKER counts its records block by block in O(1) per block (binary searches in the
//                 blocks' chains): first block = (block's count - rank of the span's begin), blocks inside the span =
//                 their count if the true chain enters them at their first byte, last block = rank of the span's end.
//                 Where speculation does not apply (a record straddling into a block, an entry point off the block's
//                 chain, a block without a chain) it walks that piece itself.
//   k_scan_counts bases of the walkers in the offsets array.
//   k_walk_write  one thread per block copies the offsets of its chain: records from an on-chain entry point j onwards go
//                 to base[j] + (rank - rank of j), those before the first entry point continue the walker in front if the
//                 chain truly entered the block at its first byte; one thread per walker writes the pieces it walked itself.
// On htslib-written files no thread follows a chain through global memory at all.
struct WalkScratch {       // per batch; n_blocks / n_walkers entries each
    const uint32_t* spec_cnt;   // block: records on its speculative chain (kSpecNone: no usable chain); from the inflate kernel
    const uint32_t* spec_end;   // block: where that chain first reaches or passes the block's end
    const uint32_t* spec_offs;  // block: [kSpecStride] the chain's record offsets
    uint32_t* entry;       // block inside a span: where the true chain enters it; with owner / first set by k_walk_link
    uint32_t* first;       // ... how many records of its walker come before it
    uint32_t* owner;       // ... and the walker (kNoOwner: not inside one span)
    uint32_t* entry_true;  // block: 1 = the true chain enters it exactly at its first byte
    uint32_t* rank;        // walker: rank of its begin on its block's speculative chain (kSpecNone = not on it)
    uint32_t* self_first;  // walker: 1 = it walked (and writes) its piece of its first block itself
    uint32_t* last_entry;  // walker: entry + records before of a last, partial block it walked itself (kNoOwner = none)
    uint32_t* last_first;
};
constexpr uint32_t kNoOwner = 0xffffffffu;

// A chain only moves forward, one dependent load per record, ~50 bytes further on every time - and caches fill by 32-byte
// SECTOR, so unassisted every step is a trip to DRAM of its own (the bytes were inflated a moment ago, a batch is several
// times the L2): measured 0.7 us per record, a 64 KiB block 0.85 ms.  (prefetch.global hints on the next LINES changed
// nothing: they fetch one sector of the line, not the one the next record starts in.)  Whenever the chain enters a new
// kilobyte it asks L2 for the whole kilobyte two ahead with ONE bulk prefetch (no registers, no shared memory).
// (tools/probes/chain_probe.cu: a dependent step costs ~500 ns cold, ~420 ns with this or with four per-sector prefetches
// per line, ~235 ns when everything is L2-resident: the floor of a chain through global memory on this GPU.)
__device__ __forceinline__ void walk_prefetch(const uint8_t* raw, uint32_t from, uint32_t to, uint32_t lim) {
    if ((to >> 10) != (from >> 10)) {
        const uint32_t a = (to & ~1023u) + 2048u;
        if (a + 16u <= lim) {
            const uint32_t n = min(1024u, lim - a) & ~15u;
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(raw + a), "r"(n) : "memory");
        }
    }
}
// the first three kilobytes of a chain that starts at p
__device__ __forceinline__ void walk_prefetch_start(const uint8_t* raw, uint32_t p, uint32_t lim) {
    const uint32_t a = p & ~15u;
    if (a + 16u <= lim) {
        const uint32_t n = min(3072u + (p & 1023u), lim - a) & ~15u;
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(raw + a), "r"(n) : "memory");
    }
}
__device__ __forceinline__ bool walk_step(const uint8_t* raw, uint32_t& p, uint32_t lim) {
    if (p + 4 > lim) return false;
    const uint32_t bs = ld_u32_any(raw, p);
    if (bs < 32u || bs > 0x7fffffffu || uint64_t(p) + 4 + bs > lim) return false;
    walk_prefetch(raw, p, p + 4 + bs, lim);
    p += 4 + bs;
    return true;
}

// The simple scheme (opts.walk_scheme = 1, or no chains from the inflate kernel): one thread per walker counts its
// records, a scan, the same walk again writes the offsets: two chains through global memory per span.
template <bool WRITE>
__global__ void __launch_bounds__(128) k_walk_span(const uint8_t* __restrict__ raw, const uint2* __restrict__ walkers, int n_walkers,
                                                   uint32_t* __restrict__ counts, const uint32_t* __restrict__ base,
                                                   uint32_t* __restrict__ offs, DeviceScalars* sc) {
    const int w = blockIdx.x * 128 + threadIdx.x;
    if (w >= n_walkers) return;
    const uint32_t e = walkers[w].y;
    uint32_t p = walkers[w].x, n = 0;
    uint32_t* o = WRITE ? offs + base[w] : nullptr;
    bool bad = false;
    walk_prefetch_start(raw, p, e);
    while (p < e) {
        if (WRITE) o[n] = p;
        if (!walk_step(raw, p, e)) { bad = true; break; }
        ++n;
    }
    if (!WRITE) {
        counts[w] = n;
        if (bad || p != e) atomicOr(&sc->status, STATUS_CORRUPT);
    }
}

// index of the first walker whose begin is >= pos
__device__ __forceinline__ int first_walker_at_or_after(const uint2* __restrict__ walkers, int n_walkers, uint32_t pos) {
    int lo = 0, hi = n_walkers;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (walkers[mid].x < pos) lo = mid + 1; else hi = mid;
    }
    return lo;
}
// index of the block that holds pos: the last one that starts at or before it
__device__ __forceinline__ int block_of(const InflateBlock* __restrict__ blocks, int n_blocks, uint32_t pos) {
    int lo = 0, hi = n_blocks - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (blocks[mid].out_off <= pos) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(128) k_walk_init(int n_blocks, WalkScratch ws) {
    const int b = blockIdx.x * 128 + threadIdx.x;
    if (b < n_blocks) { ws.owner[b] = kNoOwner; ws.entry_true[b] = 0u; }
}

// rank of position x on block b's speculative chain (kSpecNone = not on it)
__device__ __forceinline__ uint32_t rank_on_chain(const WalkScratch& ws, int b, uint32_t x) {
    const uint32_t n = ws.spec_cnt[b];
    if (n == kSpecNone) return kSpecNone;
    const uint32_t* o = ws.spec_offs + size_t(b) * kSpecStride;
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (o[mid] < x) lo = mid + 1; else hi = mid;
    }
    return (lo < n && o[lo] == x) ? lo : kSpecNone;
}

__global__ void __launch_bounds__(128) k_walk_link(const uint8_t* __restrict__ raw, const uint2* __restrict__ walkers, int n_walkers,
                                                   const InflateBlock* __restrict__ blocks, int n_blocks, uint32_t* __restrict__ counts,
                                                   WalkScratch ws, DeviceScalars* sc) {
    const int w = blockIdx.x * 128 + threadIdx.x;
    if (w >= n_walkers) return;
    const uint32_t wb = walkers[w].x, we = walkers[w].y;
    int b = block_of(blocks, n_blocks, wb);
    uint32_t p = wb, n = 0;
    bool bad = false;
    ws.last_entry[w] = kNoOwner;
    ws.self_first[w] = 0u;
    ws.rank[w] = kSpecNone;
    // rank of the span's END on the chain of the block that holds it (the next walker's begin, when the spans touch):
    // looked up only where it is needed
    const bool end_is_entry = w + 1 < n_walkers && walkers[w + 1].x == we;
    if (p < we && p != blocks[b].out_off) {
        // the span begins inside a block
        const uint32_t e0 = blocks[b].out_off + blocks[b].out_len;
        const uint32_t r0 = rank_on_chain(ws, b, wb);
        ws.rank[w] = r0;
        uint32_t r1 = kSpecNone;
        if (r0 != kSpecNone && e0 > we && end_is_entry) r1 = rank_on_chain(ws, b, we);
        if (r0 != kSpecNone && e0 <= we) { n = ws.spec_cnt[b] - r0; p = ws.spec_end[b]; }
        else if (r1 != kSpecNone) { n = r1 - r0; p = we; }
        else {
            ws.self_first[w] = 1u;
            const uint32_t stop = min(e0, we);
            walk_prefetch_start(raw, p, we);
            while (p < stop) {
                if (!walk_step(raw, p, we)) { bad = true; break; }
                ++n;
            }
        }
    } else if (p < we) ws.rank[w] = ws.spec_cnt[b] != kSpecNone ? 0u : kSpecNone;      // begins at a block's first byte
    while (p < we && !bad) {
        while (b + 1 < n_blocks && blocks[b + 1].out_off <= p) ++b;
        const uint32_t s0 = blocks[b].out_off, e0 = s0 + blocks[b].out_len;
        if (p >= e0) { bad = true; break; }     // padding between two segments of the batch: no span crosses it
        if (p == s0) ws.entry_true[b] = 1u;
        const bool spec_ok = p == s0 && ws.spec_cnt[b] != kSpecNone;
        if (e0 <= we) {                         // the block lies inside the span
            ws.entry[b] = p; ws.first[b] = n; ws.owner[b] = uint32_t(w);
            if (spec_ok) { n += ws.spec_cnt[b]; p = ws.spec_end[b]; continue; }
        } else {                                // the span ends inside this block
            const uint32_t r1 = (spec_ok && end_is_entry) ? rank_on_chain(ws, b, we) : kSpecNone;
            if (r1 != kSpecNone) { n += r1; p = we; continue; }
            ws.last_entry[w] = p; ws.last_first[w] = n;
        }
        const uint32_t stop = min(e0, we);
        walk_prefetch_start(raw, p, we);
        while (p < stop) {
            if (!walk_step(raw, p, we)) { bad = true; break; }
            ++n;
        }
    }
    if (p != we) bad = true;                    // the chain must land exactly on the next entry point
    counts[w] = n;
    if (bad) atomicOr(&sc->status, STATUS_CORRUPT);
}

// BLOCK: one thread per block; !BLOCK: one thread per walker, the pieces it walked itself in k_walk_link
template <bool BLOCK>
__global__ void __launch_bounds__(128) k_walk_write(const uint8_t* __restrict__ raw, const uint2* __restrict__ walkers, int n_walkers,
                                                    const InflateBlock* __restrict__ blocks, int n_blocks, const uint32_t* __restrict__ base,
                                                    WalkScratch ws, uint32_t* __restrict__ offs) {
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (BLOCK) {
        if (i >= n_blocks) return;
        const uint32_t s0 = blocks[i].out_off, e0 = s0 + blocks[i].out_len;
        const uint32_t cnt = ws.spec_cnt[i];
        const uint32_t* so = ws.spec_offs + size_t(i) * kSpecStride;
        if (ws.owner[i] != kNoOwner) {                  // inside one span
            const uint32_t w = ws.owner[i], lim = walkers[w].y;
            uint32_t* o = offs + base[w] + ws.first[i];
            uint32_t p = ws.entry[i];
            if (p == s0 && cnt != kSpecNone) {           // its chain is the true one: a copy
                for (uint32_t r = 0; r < cnt; ++r) o[r] = so[r];
                return;
            }
            walk_prefetch_start(raw, p, lim);           // entered behind its first byte: from where the true chain enters it
            while (p < e0) {
                *o++ = p;
                if (!walk_step(raw, p, lim)) break;     // (validated by k_walk_link; never taken)
            }
            return;
        }
        // a block with entry points inside: its speculative chain, attributed walker by walker
        if (cnt == kSpecNone) return;
        int j = first_walker_at_or_after(walkers, n_walkers, s0);
        if (j >= n_walkers || walkers[j].x >= e0) return;
        uint32_t next = walkers[j].x;
        // records in front of the first entry point continue the walker before it - if the chain truly entered at s0
        bool live = ws.entry_true[i] != 0u && ws.rank[j] != kSpecNone && j > 0 && walkers[j - 1].y == next;
        uint32_t idx0 = live ? base[j] - ws.rank[j] : 0u, lim = next;      // offs index of the chain's record 0; end of the current walker
        for (uint32_t n0 = 0; n0 < cnt; n0 += 8) {      // eight offsets per step: their loads are independent (one by one, every
            uint32_t pv[8];                              // record cost an L2 round trip, as if the chain were being chased)
#pragma unroll
            for (int u = 0; u < 8; ++u) pv[u] = n0 + u < cnt ? so[n0 + u] : 0xffffffffu;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const uint32_t n = n0 + u, p = pv[u];
                if (n < cnt) {
                    while (next <= p) {
                        if (next == p && ws.rank[j] == n) { live = true; idx0 = base[j] - n; lim = walkers[j].y; }
                        else live = false;              // an entry point off the chain: what follows is not verified
                        ++j;
                        next = (j < n_walkers && walkers[j].x < e0) ? walkers[j].x : 0xffffffffu;
                    }
                    if (live && p >= lim) live = false; // behind the last walker of a segment
                    if (live) offs[idx0 + n] = p;
                }
            }
        }
    } else {
        if (i >= n_walkers) return;
        const uint32_t wb = walkers[i].x, we = walkers[i].y;
        if (wb >= we) return;
        if (ws.self_first[i]) {                         // [wb, min(end of its block, we))
            const int b = block_of(blocks, n_blocks, wb);
            const uint32_t stop = min(blocks[b].out_off + blocks[b].out_len, we);
            uint32_t p = wb;
            uint32_t* o = offs + base[i];
            walk_prefetch_start(raw, p, we);
            while (p < stop) {
                *o++ = p;
                if (!walk_step(raw, p, we)) break;
            }
        }
        if (ws.last_entry[i] != kNoOwner) {             // the last block, entered by the chain at last_entry
            uint32_t p = ws.last_entry[i];
            uint32_t* o = offs + base[i] + ws.last_first[i];
            walk_prefetch_start(raw, p, we);
            while (p < we) {
                *o++ = p;
                if (!walk_step(raw, p, we)) break;
            }
        }
    }
}

// exclusive scan of counts[0..n) into base[0..n), total into *total and (when offs != null) the end sentinel.
// ONE warp, shuffles only: no shared memory and 32 threads, so that it fits next to a resident inflate CTA.  Sixteen counts
// per lane and step, their four loads issued together (one load per step left the warp waiting for memory 100 times over).
__global__ void __launch_bounds__(32) k_scan_counts(const uint32_t* __restrict__ counts, int n, uint32_t* __restrict__ base,
                                                    uint32_t* total, uint32_t* __restrict__ offs, uint32_t end_pos) {
    const int lane = threadIdx.x;
    uint32_t carry = 0;
    for (int i0 = 0; i0 < n; i0 += 512) {
        const int i = i0 + 16 * lane;
        uint32_t v[16];
        if (i + 15 < n) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint4 q = *reinterpret_cast<const uint4*>(counts + i + 4 * k);
                v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = i + k < n ? counts[i + k] : 0u;
        }
        uint32_t sum = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) { const uint32_t t = v[k]; v[k] = sum; sum += t; }      // exclusive within the lane
        uint32_t incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += up;
        }
        const uint32_t pre = carry + incl - sum;
        if (i + 15 < n) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                *reinterpret_cast<uint4*>(base + i + 4 * k) = make_uint4(pre + v[4 * k], pre + v[4 * k + 1], pre + v[4 * k + 2], pre + v[4 * k + 3]);
        } else {
#pragma unroll
            for (int k = 0; k < 16; ++k) if (i + k < n) base[i + k] = pre + v[k];
        }
        carry += __shfl_sync(FULL, incl, 31);
    }
    if (lane == 0) {
        if (offs) offs[carry] = end_pos;
        *total = carry;                   // may be pinned host memory (the streaming pipeline reads it after an event)
        __threadfence_system();
    }
}

}  // namespace

void launch_inflate(const InflateBlock* d_blocks, int n_blocks, const uint8_t* d_comp, uint8_t* d_raw, uint32_t* d_spec, DeviceScalars* sc,
                    cudaStream_t s) {
    if (n_blocks <= 0) return;
    static thread_local int sms[16] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 16 && sms[dev] == 0) {
        cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
        cudaFuncSetAttribute(k_inflate_ws, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kWsSmem));
    }
    const int n_sm = (dev >= 0 && dev < 16 && sms[dev] > 0) ? sms[dev] : 148;
    const int grid = std::min(n_sm, (n_blocks + kWsStreams - 1) / kWsStreams);     // persistent: one CTA per SM
    SpecOut spec{nullptr, nullptr, nullptr};
    if (d_spec) { spec.cnt = d_spec; spec.end = d_spec + n_blocks; spec.offs = d_spec + 2 * size_t(n_blocks); }
    k_inflate_ws<<<grid, kWsThreads, kWsSmem, s>>>(d_blocks, n_blocks, d_comp, d_raw, spec, sc);
}
size_t inflate_spec_words(int n_blocks) { return size_t(n_blocks) * (2 + kSpecStride) + 16; }

int inflate_wave_blocks(int n_sm) { return n_sm * kWsStreams; }

namespace {
__global__ void k_publish_pair(const int32_t* __restrict__ a, const int32_t* __restrict__ b, int32_t* dst) {
    dst[0] = *a;
    dst[1] = *b;
    __threadfence_system();
}
}  // namespace
void launch_publish_pair(const int32_t* d_a, const int32_t* d_b, int32_t* dst, cudaStream_t s) { k_publish_pair<<<1, 1, 0, s>>>(d_a, d_b, dst); }

void launch_crc32(const InflateBlock* d_blocks, const uint32_t* d_crc, int n_blocks, const uint8_t* d_raw, DeviceScalars* sc,
                  cudaStream_t s) {
    if (n_blocks <= 0) return;
    static thread_local bool have_tab[16] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16 || !have_tab[dev]) {
        k_crc_init<<<1, 256, 0, s>>>();
        if (dev >= 0 && dev < 16) have_tab[dev] = true;
    }
    k_crc32<<<(n_blocks + kCrcWarps - 1) / kCrcWarps, kCrcWarps * 32, 0, s>>>(d_blocks, d_crc, n_blocks, d_raw, sc);
}

void launch_walk(const uint8_t* d_raw, const uint2* d_walkers, int n_walkers, int scheme, const InflateBlock* d_blocks, int n_blocks,
                 const uint32_t* d_spec, uint32_t* d_scratch, uint32_t* d_counts, uint32_t* d_base, uint32_t* d_total, uint32_t* d_offs,
                 uint32_t end_pos, DeviceScalars* sc, cudaStream_t s) {
    if (n_walkers <= 0 || n_blocks <= 0) {
        k_scan_counts<<<1, 32, 0, s>>>(d_counts, 0, d_base, d_total, d_offs, end_pos);
        return;
    }
    const int gb = (n_blocks + 127) / 128, gw = (n_walkers + 127) / 128;
    if (scheme == 1 || !d_spec) {
        k_walk_span<false><<<gw, 128, 0, s>>>(d_raw, d_walkers, n_walkers, d_counts, nullptr, nullptr, sc);
        k_scan_counts<<<1, 32, 0, s>>>(d_counts, n_walkers, d_base, d_total, d_offs, end_pos);
        k_walk_span<true><<<gw, 128, 0, s>>>(d_raw, d_walkers, n_walkers, nullptr, d_base, d_offs, sc);
        return;
    }
    WalkScratch ws;
    ws.spec_cnt = d_spec; ws.spec_end = d_spec + n_blocks; ws.spec_offs = d_spec + 2 * size_t(n_blocks);
    ws.owner = d_scratch; ws.entry_true = ws.owner + n_blocks; ws.entry = ws.entry_true + n_blocks; ws.first = ws.entry + n_blocks;
    ws.rank = ws.first + n_blocks; ws.self_first = ws.rank + n_walkers; ws.last_entry = ws.self_first + n_walkers;
    ws.last_first = ws.last_entry + n_walkers;
    k_walk_init<<<gb, 128, 0, s>>>(n_blocks, ws);       // (a kernel, not cudaMemsetAsync: that may queue behind the bulk copies of a copy engine)
    k_walk_link<<<gw, 128, 0, s>>>(d_raw, d_walkers, n_walkers, d_blocks, n_blocks, d_counts, ws, sc);
    k_scan_counts<<<1, 32, 0, s>>>(d_counts, n_walkers, d_base, d_total, d_offs, end_pos);
    k_walk_write<true><<<gb, 128, 0, s>>>(d_raw, d_walkers, n_walkers, d_blocks, n_blocks, d_base, ws, d_offs);
    k_walk_write<false><<<gw, 128, 0, s>>>(d_raw, d_walkers, n_walkers, d_blocks, n_blocks, d_base, ws, d_offs);
}
size_t walk_scratch_words(int n_blocks, int n_walkers) { return size_t(n_blocks) * 4 + size_t(n_walkers) * 4 + 16; }

}  // namespace bsg
