// Single-lane DEFLATE decode core shared by the GPU inflate kernel and its host-side unit harness
// (tests/host_inflate_harness.cpp compiles this header with a plain C++ compiler).  Everything here is executed by ONE
// thread per BGZF block: bit reader, decode-table construction, and Huffman symbols -> token queue.
//
// Shared-memory budget: 3284 bytes of tables per stream (16-bit entries; the distance table doubles as the code-length
// scratch while a block header is parsed) + two 32-token queues = 3540 bytes, so that 64 streams and the copy warps'
// stages fit one SM with 2 KB to spare (inflate.cu: a small kernel without shared memory can run next to the CTA).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define BSG_HD __host__ __device__ __forceinline__
#else
#define BSG_HD inline
#endif

namespace bsg {
namespace inflate_core {

#ifndef BSG_LIT_BITS
#define BSG_LIT_BITS 10
#endif
constexpr int kLitBits = BSG_LIT_BITS, kDistBits = 8;
constexpr int kQueue = 32;           // tokens a stream hands over per round

// token: literal = byte ; match = 1 << 31 | (dist - 1) << 16 | len ; skip (stored bytes already in place) = 1 << 30 | len
constexpr uint32_t kTokMatch = 0x80000000u, kTokSkip = 0x40000000u;

// 16-bit decode-table entries.
//   literal/length code:  [3:0] code length, [4] 0 = literal / 1 = anything else,
//                         literal: [15:8] the byte;  otherwise [7:5] class: 0..5 = length symbol with that many extra
//                         bits and [15:8] = base length - 3;  7 = end of block;  6 = not decodable from this entry:
//                         [3:0] = 0: no such code (or symbol 286/287): the stream is corrupt;
//                         [3:0] = b > 0 (primary table only): the code is longer than the primary table - its remaining
//                         bits index a second-level table of 2^b entries at lit_sub[2 * [15:8]] (entries of the same
//                         format, [3:0] = the code's full length)
//   distance code:        [3:0] code length (0 = slow path), [7:4] extra bits, [9:8] mantissa m: base = (m << extra) + 1,
//                         [10] invalid symbol (30/31)
// One test of bit 4 separates literals from everything else; one test of the class separates lengths from the rare rest.
constexpr uint32_t kNonLit = 0x10u, kClsShift = 5, kClsEob = 7u, kClsOther = 6u;
constexpr uint32_t kLitUnset = kNonLit | (kClsOther << kClsShift);      // class 6, length 0: corrupt stream
// Second-level entries for literal/length codes of 11-15 bits.  Codes are canonical, so the long codes of a block are
// sorted by length and share consecutive 10-bit prefixes: every prefix whose codes all have one length needs exactly as
// many entries as it has codes, and only the (at most four) prefixes in which the length changes waste any - zlib's
// `enough 288 10 15` gives 1334 entries for both levels, i.e. 310 here.  An overflow is reported as a corrupt block.
constexpr int kLitSub = 310;
constexpr uint32_t kDistBad = 0x400u;

BSG_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    sh &= 31;
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}
BSG_HD uint32_t rev_bits(uint32_t code, uint32_t len) {
#if defined(__CUDA_ARCH__)
    return __brev(code) >> (32 - len);
#else
    uint32_t r = 0;
    for (uint32_t i = 0; i < len; ++i) r |= ((code >> i) & 1u) << (len - 1 - i);
    return r;
#endif
}

// Bit reader over aligned 64-bit units: A = (a1:a0) and B = (b1:b0) are the 128-bit window, bo < 64 is the bit offset
// into it (so at least 64 valid bits: a token needs at most 52), P = (p1:p0) is the unit in flight.  A token consumes at
// most 48 bits, so there is at most ONE refill per token, written without a branch (selects + a predicated load), and
// the load issued at one refill is first touched at the NEXT refill of that lane (B = P), 64 consumed bits later.
// Why it is built this way: 32 lanes decode 32 streams in lock step, so some lane refills in nearly every step.  With a
// window of 32-bit words a token could need two refills; the second one was a (rare) branch, and at its join the compiler
// copied the register of the load in flight - every step then waited for a global load (ncu: a third of the decode
// warps' time on that one MOV).
struct BitReader {
    const uint64_t* base;  // the buffer (uniform for all blocks of a launch; 8-byte aligned)
    uint32_t wi;           // index of the next 64-bit unit to load
    uint32_t a0, a1, b0, b1, p0, p1, bo;
    BSG_HD static void ld2(const uint64_t* p, uint32_t& lo, uint32_t& hi) { const uint64_t v = *p; lo = uint32_t(v); hi = uint32_t(v >> 32); }
    BSG_HD void init(const void* buf, uint32_t byte_off) {
        base = static_cast<const uint64_t*>(buf);
        wi = byte_off >> 3;
        bo = (byte_off & 7u) * 8u;
        ld2(base + wi, a0, a1); ld2(base + wi + 1, b0, b1); ld2(base + wi + 2, p0, p1);
        wi += 3;
#if defined(__CUDA_ARCH__)
        // the batch has just arrived over PCIe: ask L2 for the lines ahead (one more whenever the reader enters a line)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + wi + 16u));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(base + wi + 32u));
#endif
    }
    BSG_HD uint32_t peek() const {                                            // next 32 bits
        const bool h = bo >= 32u;
        return funnel_r(h ? a1 : a0, h ? b0 : a1, bo);
    }
    BSG_HD uint32_t peek_hi() const {                                         // the 32 bits after those
        const bool h = bo >= 32u;
        return funnel_r(h ? b0 : a1, h ? b1 : b0, bo);
    }
    BSG_HD void consume(uint32_t n) {                                         // n <= 64
        bo += n;
        const bool rf = bo >= 64u;
        bo = rf ? bo - 64u : bo;
        a0 = rf ? b0 : a0; a1 = rf ? b1 : a1;
        b0 = rf ? p0 : b0; b1 = rf ? p1 : b1;
#if defined(__CUDA_ARCH__)
        asm volatile("{ .reg .pred p, q; .reg .b32 t; setp.ne.u32 p, %3, 0; @p ld.global.v2.u32 {%0, %1}, [%2];\n\t"
                     "and.b32 t, %4, 15; setp.eq.and.u32 q, t, 0, p; @q prefetch.global.L2 [%2 + 256]; }"
                     : "+r"(p0), "+r"(p1) : "l"(base + wi), "r"(uint32_t(rf)), "r"(wi) : "memory");
        // (measured and dropped: also asking L1 for the sector 64 bytes ahead - 8.56 vs 8.52 ms, no gain)
#else
        if (rf) ld2(base + wi, p0, p1);
#endif
        wi += rf ? 1u : 0u;
    }
    BSG_HD void consume_short(uint32_t n) { consume(n); }
    BSG_HD uint64_t bit_pos() const { return uint64_t(wi - 3u) * 64u + bo; }  // bits from the start of the buffer
    BSG_HD uint32_t byte_pos() const { return (wi - 3u) * 8u + (bo >> 3); }   // only valid when bo is a multiple of 8
};

struct Tables {
    uint16_t lit[1 << kLitBits];
    uint16_t dist[1 << kDistBits];
    uint16_t lit_sub[kLitSub];
    uint16_t dist_sorted[32];
    uint16_t dist_count[16];
    // canonical-decode state after the code lengths the primary distance table covers (see slow_entry)
    uint16_t dist_first, dist_index, pad0, pad1;
};
constexpr int kLensBytes = 320;     // code lengths of one block header: 288 literal/length + 32 distance symbols
static_assert(sizeof(uint16_t) << kDistBits >= kLensBytes, "the distance table doubles as the code-length scratch");
static_assert(kQueue * 4 >= 32, "the (empty) token queue holds the 32 distance code lengths while the tables are built");

BSG_HD uint32_t lit_entry(int sym, int len) {
    if (sym < 256) return uint32_t(len) | (uint32_t(sym) << 8);
    if (sym == 256) return uint32_t(len) | kNonLit | (kClsEob << kClsShift);
    if (sym > 285) return kLitUnset;
    uint32_t eb, base;
    if (sym < 265) { eb = 0; base = uint32_t(sym - 254); }
    else if (sym == 285) { eb = 0; base = 258; }
    else { eb = uint32_t(sym - 261) >> 2; base = ((4u + (uint32_t(sym - 265) & 3u)) << eb) + 3u; }
    return uint32_t(len) | kNonLit | (eb << kClsShift) | ((base - 3u) << 8);
}
BSG_HD uint32_t dist_entry(int sym, int len) {
    if (sym > 29) return uint32_t(len) | kDistBad;
    uint32_t eb, mant;
    if (sym < 4) { eb = 0; mant = uint32_t(sym); }
    else { eb = (uint32_t(sym) >> 1) - 1u; mant = 2u + (uint32_t(sym) & 1u); }
    return uint32_t(len) | (eb << 4) | (mant << 8);
}

// Table / queue access of fill_queue.  The host harness (and any generic caller) uses plain arrays; the kernel
// passes shared-memory byte addresses and ld.shared / st.shared so that the addresses stay in registers.
struct ArrayAccess {
    const Tables* T;
    uint32_t* q;
    BSG_HD uint32_t lit(uint32_t byte_off) const { return T->lit[byte_off >> 1]; }
    BSG_HD uint32_t sub(uint32_t byte_off) const { return T->lit_sub[byte_off >> 1]; }
    BSG_HD uint32_t dist(uint32_t byte_off) const { return T->dist[byte_off >> 1]; }
    BSG_HD void put(uint32_t byte_off, uint32_t v) const { q[byte_off >> 2] = v; }
    BSG_HD uint32_t count(uint32_t len) const { return T->dist_count[len]; }
    BSG_HD uint32_t sorted(uint32_t i) const { return T->dist_sorted[i]; }
    BSG_HD uint32_t first() const { return T->dist_first; }
    BSG_HD uint32_t index() const { return T->dist_index; }
};

// Canonical decode of a DISTANCE code longer than the primary table (RFC 1951 3.2.2) from the 32 peeked bits: returns
// the table entry the symbol would have had (with its real code length), or an "invalid" entry.  The primary lookup has
// already ruled out every code of up to kDistBits bits, so the search starts behind them: the (first, index) pair of the
// canonical walk at that point depends only on the code-length counts and is stored with the tables.  Fewer than one
// match in a hundred comes here (literal/length codes, one token in twenty, have their second-level table instead).
// Deliberately NOT inlined into the hot loop on the device.
template <class A>
#if defined(__CUDA_ARCH__)
__device__ __noinline__
#else
inline
#endif
uint32_t slow_entry(uint32_t v, const A& acc) {
    constexpr int kBits = kDistBits;
#if defined(BSG_SLOW_COUNTER) && !defined(__CUDA_ARCH__)
    ++BSG_SLOW_COUNTER[1];                        // host-side statistics only (tools / tests)
#endif
    int code = int(rev_bits(v & ((1u << kBits) - 1u), kBits)) << 1;       // the first kBits bits, MSB first
    int first = int(acc.first()), index = int(acc.index());
    v >>= kBits;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int len = kBits + 1; len <= 15; ++len) {
        code |= int(v & 1u);
        v >>= 1;
        const int c = int(acc.count(uint32_t(len)));
        if (code - c < first) {
            const int sym = int(acc.sorted(uint32_t(index + (code - first))));
            return dist_entry(sym, len);
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return 15u | kDistBad;
}

// Which literal/length and distance codes a block may use, as zlib (inftrees.c) decides it: not over-subscribed, and
// complete - except a code whose codes all have length 1, i.e. a single code of one bit (or, for distances, no code at
// all).  `left` is the unused code space after lengths 1..15, `nlong` the number of codes longer than one bit.
BSG_HD bool code_accepted(int left, int nlong) { return left == 0 || nlong == 0; }

// Serial table construction by the owning thread.  is_dist selects the entry format.  Returns false when the code
// is over-subscribed or incomplete (code_accepted).
BSG_HD bool build_table(const uint8_t* lens, int n, uint16_t* primary, int bits, uint16_t* count, uint16_t* sorted, bool is_dist,
                        uint16_t* first_out, uint16_t* index_out) {
    const uint16_t unset = is_dist ? uint16_t(0) : uint16_t(kLitUnset);      // code length 0 = not in the primary table
    for (int i = 0; i < (1 << bits); ++i) primary[i] = unset;
    int cnt[16];
    for (int l = 0; l < 16; ++l) cnt[l] = 0;
    for (int s = 0; s < n; ++s) cnt[lens[s] & 15]++;
    cnt[0] = 0;
    int left = 1, ok = 1, nlong = 0;
    for (int l = 1; l <= 15; ++l) {
        left = left * 2 - cnt[l];
        if (left < 0) { ok = 0; left = 0; }                                  // over-subscribed
        nlong += l > 1 ? cnt[l] : 0;
    }
    ok = ok && code_accepted(left, nlong);
    int next[16], offs[16];
    next[0] = 0; offs[0] = 0; next[1] = 0; offs[1] = 0;
    for (int l = 1; l < 15; ++l) { next[l + 1] = (next[l] + cnt[l]) << 1; offs[l + 1] = offs[l] + cnt[l]; }
    for (int l = 0; l < 16; ++l) count[l] = uint16_t(cnt[l]);
    {   // state of the canonical walk after lengths 1..bits (an over-subscribed code may overflow 16 bits: flagged by ok)
        int first = 0, index = 0;
        for (int l = 1; l <= bits; ++l) { index += cnt[l]; first += cnt[l]; first <<= 1; }
        *first_out = uint16_t(first); *index_out = uint16_t(index);
    }
    for (int s = 0; s < n; ++s) {
        const int l = lens[s] & 15;
        if (!l) continue;
        const uint32_t code = uint32_t(next[l]++);
        sorted[offs[l]++] = uint16_t(s);
        if (l <= bits) {
            const uint16_t e = uint16_t(is_dist ? dist_entry(s, l) : lit_entry(s, l));
            for (int k = int(rev_bits(code, uint32_t(l))); k < (1 << bits); k += (1 << l)) primary[k] = e;
        }
    }
    return ok != 0;
}

// Literal/length tables of one block: 10-bit primary table + second-level tables for the longer codes.
// Returns false when the code is over-subscribed or incomplete (code_accepted) or (corrupt input only) the second
// level overflows.
BSG_HD bool build_lit_table(const uint8_t* lens, Tables& T) {
    constexpr int n = 288, kRoot = kLitBits;
    for (int i = 0; i < (1 << kRoot); ++i) T.lit[i] = uint16_t(kLitUnset);
    int cnt[16];
    for (int l = 0; l < 16; ++l) cnt[l] = 0;
    for (int s = 0; s < n; ++s) cnt[lens[s] & 15]++;
    cnt[0] = 0;
    int left = 1, ok = 1, nlong = 0;
    for (int l = 1; l <= 15; ++l) {
        left = left * 2 - cnt[l];
        if (left < 0) { ok = 0; left = 0; }                                  // over-subscribed
        nlong += l > 1 ? cnt[l] : 0;
    }
    ok = ok && code_accepted(left, nlong);
    if (!ok) return false;
    int first_code[16], next[16];
    first_code[0] = 0; first_code[1] = 0;
    for (int l = 1; l < 15; ++l) first_code[l + 1] = (first_code[l] + cnt[l]) << 1;
    for (int l = 0; l < 16; ++l) next[l] = first_code[l];
    // pass 1: short codes fill the primary table; a long code leaves the number of second-level bits its prefix needs
    int pmin = 1 << kRoot;
    for (int s = 0; s < n; ++s) {
        const int l = lens[s] & 15;
        if (!l) continue;
        const uint32_t code = uint32_t(next[l]++);
        if (l <= kRoot) {
            const uint16_t e = uint16_t(lit_entry(s, l));
            for (int k = int(rev_bits(code, uint32_t(l))); k < (1 << kRoot); k += (1 << l)) T.lit[k] = e;
        } else {
            const int pre = int(code >> (l - kRoot));                 // the code's first 10 bits, MSB first
            uint16_t& slot = T.lit[rev_bits(uint32_t(pre), kRoot)];
            if (uint32_t(l - kRoot) > (slot & 15u)) slot = uint16_t(kLitUnset | uint32_t(l - kRoot));
            if (pre < pmin) pmin = pre;
        }
    }
    // (no early return for "no long codes" and none inside the loops below: 32 lanes build 32 tables in lock step, and a
    // loop with a second exit has no reconvergence point behind it - the lanes ran everything after it, pass 3 included,
    // one lane after the other: ncu showed 1.5 active lanes and half of all instructions of the block-header phase there)
    // pass 2: long codes own the top of the code space: give every prefix from pmin up its second-level table
    int off = 0;
    bool fits = true;
    for (int pre = pmin; pre < (1 << kRoot); ++pre) {
        uint16_t& slot = T.lit[rev_bits(uint32_t(pre), kRoot)];
        const uint32_t e = slot;
        if ((e & (kNonLit | (7u << kClsShift))) == kLitUnset && (e & 15u)) {              // neither a short code nor nothing at all
            const int bits = int(e & 15u), size = 1 << bits;
            if (off + size > kLitSub) fits = false;
            else {
                slot = uint16_t(kLitUnset | uint32_t(bits) | (uint32_t(off >> 1) << 8));
                for (int j = 0; j < size; ++j) T.lit_sub[off + j] = uint16_t(kLitUnset);
                off += size;
            }
        }
    }
    // pass 3: the long codes themselves (a prefix whose table did not fit keeps [15:8] = 0 and [3:0] = its bits: the
    // writes below then stay inside lit_sub, and the block is refused)
    for (int l = 0; l < 16; ++l) next[l] = first_code[l];
    for (int s = 0; s < n; ++s) {
        const int l = lens[s] & 15;
        const uint32_t code = uint32_t(next[l]++);                     // next[0] is never used for a code
        if (l > kRoot) {
            const int rest = l - kRoot;
            const uint32_t link = T.lit[rev_bits(code >> rest, kRoot)];
            const int bits = int(link & 15u), base = int(link >> 8) * 2;
            const uint16_t e = uint16_t(lit_entry(s, l));
            if (fits)
                for (int k = int(rev_bits(code & ((1u << rest) - 1u), uint32_t(rest))); k < (1 << bits); k += (1 << rest)) T.lit_sub[base + k] = e;
        }
    }
    if (!fits) return false;
    return true;
}

// Block header: reads BFINAL/BTYPE and, for Huffman blocks, the code lengths, then builds the tables.
// The code lengths are collected in the (not yet built) distance table; `dlens` is 32 bytes of scratch for the distance
// code lengths while the distance table is written (the kernel lends the empty token queue).
// Returns 0 = Huffman block ready, 1 = stored block (caller handles LEN/NLEN), 2 = error.
template <class BR>
BSG_HD int read_block_header(BR& br, Tables& T, uint8_t* dlens, int* last) {
    uint8_t* lens = reinterpret_cast<uint8_t*>(T.dist);
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    uint32_t v = br.peek();
    *last = int(v & 1u);
    const int btype = int((v >> 1) & 3u);
    br.consume(3);
    if (btype == 0) return 1;
    if (btype == 3) return 2;
    int nlit = 288, ndist = 32;
    if (btype == 1) {
        for (int s = 0; s < 288; ++s) lens[s] = uint8_t(s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8)));
        for (int s = 0; s < 32; ++s) lens[288 + s] = 5;
    } else {
        uint8_t* cl = reinterpret_cast<uint8_t*>(T.lit);      // code-length table borrows the (not yet built) lit table
        v = br.peek();
        nlit = int(v & 31u) + 257;
        ndist = int((v >> 5) & 31u) + 1;
        const int ncl = int((v >> 10) & 15u) + 4;
        br.consume(14);
        uint8_t cll[19];
        for (int i = 0; i < 19; ++i) cll[i] = 0;
        for (int i = 0; i < ncl; ++i) { cll[order[i]] = uint8_t(br.peek() & 7u); br.consume(3); }
        int cnt[8] = {0, 0, 0, 0, 0, 0, 0, 0}, next[8];
        for (int i = 0; i < 19; ++i) cnt[cll[i]]++;
        cnt[0] = 0;
        next[1] = 0;
        // the code-length code must be complete (zlib refuses an incomplete one, even a single code): once the unused
        // code space goes negative (over-subscribed) it stays negative
        int cl_left = 1;
        for (int l = 1; l <= 7; ++l) cl_left = cl_left * 2 - cnt[l];
        for (int l = 1; l < 7; ++l) next[l + 1] = (next[l] + cnt[l]) << 1;
        for (int i = 0; i < 128; ++i) cl[i] = 0;
        for (int s = 0; s < 19; ++s) {
            const int l = cll[s];
            if (!l) continue;
            const uint32_t r = rev_bits(uint32_t(next[l]++), uint32_t(l));
            for (uint32_t k = r; k < 128; k += (1u << l)) cl[k] = uint8_t(s | (l << 5));
        }
        if (nlit > 286 || ndist > 30 || cl_left != 0) return 2;
        const int total = nlit + ndist;
        int i = 0;
        while (i < total) {
            v = br.peek();
            const uint32_t e = cl[v & 127u];
            const int l = int(e >> 5), s = int(e & 31u);
            if (!l) return 2;
            if (s < 16) { lens[i++] = uint8_t(s); br.consume(uint32_t(l)); continue; }
            int rep, val = 0;
            uint32_t used = uint32_t(l);
            if (s == 16) { if (i == 0) return 2; val = lens[i - 1]; rep = 3 + int((v >> l) & 3u); used += 2; }
            else if (s == 17) { rep = 3 + int((v >> l) & 7u); used += 3; }
            else { rep = 11 + int((v >> l) & 127u); used += 7; }
            br.consume(used);
            if (i + rep > total) return 2;
            while (rep--) lens[i++] = uint8_t(val);
        }
        if (lens[256] == 0) return 2;
        for (int k = ndist - 1; k >= 0; --k) lens[288 + k] = lens[nlit + k];
        for (int k = nlit; k < 288; ++k) lens[k] = 0;
    }
    for (int k = 0; k < 32; ++k) dlens[k] = lens[288 + k];
    bool ok = build_lit_table(lens, T);
    ok = build_table(dlens, ndist, T.dist, kDistBits, T.dist_count, T.dist_sorted, true, &T.dist_first, &T.dist_index) && ok;
    return ok ? 0 : 2;
}

// Decode symbols into the queue until it holds kQueue tokens or the block ends.
// *op_dec = bytes decoded so far (updated).  Returns the number of tokens; *eob is set at end-of-block; *bad is
// sticky (errors do not stop the loop: every access stays in bounds, the caller discards the round).
// A match is decoded from ONE 64-bit look-ahead (length code + extra bits <= 20 bits, distance code + extra bits
// <= 28 bits) and consumed once.
// Literals and matches run through ONE instruction sequence (a literal is a "match" with no extra bits whose distance
// lookup is thrown away): on the device 32 lanes decode 32 streams in lock step, and a warp that branched on
// literal / match would execute both sides one after the other in nearly every step.  Only the rare cases branch: codes
// longer than the primary table (second-level lookup), distance codes longer than theirs, end of block, garbage.
template <class BR, class A>
BSG_HD int fill_queue(BR& br, const A& acc, uint32_t* op_dec, int* eob, int* bad) {
    constexpr uint32_t kLitMask2 = ((1u << kLitBits) - 1u) << 1, kDistMask2 = ((1u << kDistBits) - 1u) << 1;
    constexpr uint32_t kClassMask = kNonLit | (7u << kClsShift);
    uint32_t qo = 0;                  // byte offset of the next queue slot
    uint32_t op = *op_dec;
    int err = 0;
    *eob = 0;
#if defined(__CUDA_ARCH__)
    do {
        const uint32_t v = br.peek();
        uint32_t e = acc.lit((v << 1) & kLitMask2);
        {   // a code longer than the primary table: second-level lookup, predicated (some lane needs it in most steps)
            const bool lng = (e & kClassMask) == kLitUnset;
            const uint32_t sb = e & 15u;
            err |= int(lng & (sb == 0u));                                      // no such code
            e = acc.sub_if(lng, (e >> 8) * 4u + (((v >> kLitBits) & ~(~0u << sb)) << 1), e);
        }
        const bool is_lit = !(e & kNonLit);
        const uint32_t cls = (e >> kClsShift) & 7u;
        if (!is_lit & (cls >= kClsOther)) {           // end of block, or garbage
            if (cls == kClsEob) { br.consume_short(e & 15u); *eob = 1; } else err = 1;
            break;
        }
        const uint32_t len = e & 15u, eb = is_lit ? 0u : cls, used = len + eb;      // eb = number of extra bits
        const uint32_t mlen = (e >> 8) + 3u + ((v >> len) & ~(~0u << eb));
        const uint32_t v2 = funnel_r(v, br.peek_hi(), used);      // used <= 20
        uint32_t d = acc.dist((v2 << 1) & kDistMask2);
        if (!is_lit & !(d & 15u)) d = slow_entry(v2, acc);
        const uint32_t dl = d & 15u, deb = (d >> 4) & 15u;
        uint32_t mdist = (((d >> 8) & 3u) << deb) + 1u + ((v2 >> dl) & ~(~0u << deb));
        br.consume(is_lit ? len : used + dl + deb);                // <= 48
        const bool badm = !is_lit & (((d & kDistBad) != 0u) | (mdist > op));
        err |= int(badm);
        mdist = badm ? 1u : mdist;
        acc.put(qo, is_lit ? (e >> 8) : (kTokMatch | ((mdist - 1u) << 16) | mlen));
        qo += 4; op += is_lit ? 1u : mlen;
    } while (qo < uint32_t(kQueue) * 4u);
#else
    do {
        const uint32_t v = br.peek();
        uint32_t e = acc.lit((v << 1) & kLitMask2);
        if ((e & kClassMask) == kLitUnset) {          // a code longer than the primary table, or no code at all
            const uint32_t sb = e & 15u;
            if (!sb) { err = 1; break; }
            e = acc.sub((e >> 8) * 4u + (((v >> kLitBits) & ~(~0u << sb)) << 1));      // second level: one more lookup
        }
        const bool is_lit = !(e & kNonLit);
        const uint32_t cls = (e >> kClsShift) & 7u;
        if (!is_lit && cls >= kClsOther) {            // end of block, or garbage
            if (cls == kClsEob) { br.consume_short(e & 15u); *eob = 1; } else err = 1;
            break;
        }
        const uint32_t len = e & 15u, eb = is_lit ? 0u : cls, used = len + eb;      // eb = number of extra bits
        const uint32_t mlen = (e >> 8) + 3u + ((v >> len) & ~(~0u << eb));
        const uint32_t v2 = funnel_r(v, br.peek_hi(), used);      // used <= 20
        uint32_t d = acc.dist((v2 << 1) & kDistMask2);
        if (!is_lit && !(d & 15u)) d = slow_entry(v2, acc);
        const uint32_t dl = d & 15u, deb = (d >> 4) & 15u;
        uint32_t mdist = (((d >> 8) & 3u) << deb) + 1u + ((v2 >> dl) & ~(~0u << deb));
        br.consume(is_lit ? len : used + dl + deb);                // <= 48
        if (!is_lit && ((d & kDistBad) != 0u || mdist > op)) { err = 1; mdist = 1; }
        acc.put(qo, is_lit ? (e >> 8) : (kTokMatch | ((mdist - 1u) << 16) | mlen));
        qo += 4; op += is_lit ? 1u : mlen;
    } while (qo < uint32_t(kQueue) * 4u);
#endif
    *op_dec = op;
    *bad |= err;
    return int(qo >> 2);
}

}  // namespace inflate_core
}  // namespace bsg
