"""A DEFLATE forge (RFC 1951) for conformance tests of the inflate paths (test infrastructure, pure Python).

zlib's encoder is what wrote every other stream the tests feed the decoders, and it never writes much of what the format
allows and other encoders (libdeflate, igzip) do write: distances up to 32768, many blocks of mixed types in one stream,
empty blocks, single-code or literal-only distance trees, 15-bit codes, length 258 as code 284 plus 31.  The forge writes
such streams bit by bit from explicit block types, code lengths and tokens, and also streams no encoder should write (the
refusal cases).  The reference for every stream is zlib's decoder, asked at run time (zlib_verdict).

Tokens: an int 0..255 is a literal; (length, dist) is a match; (258, dist, True) writes length 258 as code 284 + 31
extra bits; ("sym", s) writes literal/length symbol s alone; ("dsym", lsym, dsym) writes length symbol lsym and distance
symbol dsym with zero extra bits (for symbols that do not exist)."""
import random
import struct
import zlib
from dataclasses import dataclass

LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258]
LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097,
             6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13]
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
FIXED_LIT = [8] * 144 + [9] * 112 + [7] * 24 + [8] * 8
FIXED_DIST = [5] * 32
WINDOW = 32768


class BitWriter:
    """LSB-first bit packing, as DEFLATE stores everything but Huffman codes."""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def bits(self, value, n):
        self.acc |= (value & ((1 << n) - 1)) << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 0xFF)
            self.acc >>= 8
            self.n -= 8

    def code(self, code, length):
        """A Huffman code: its bits go out most significant first.  A symbol without a code (None) writes nothing."""
        if code is None:
            return
        code &= (1 << length) - 1             # (an over-subscribed code's last codes do not fit: a lenient reader's view)
        self.bits(int(format(code, f"0{length}b")[::-1], 2) if length else 0, length)

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def getvalue(self):
        return bytes(self.out) + (bytes([self.acc]) if self.n else b"")


def canonical(lengths):
    """Canonical codes (RFC 1951 3.2.2) for the given code lengths; None where the length is 0.  Works for incomplete and
    over-subscribed lengths too (the codes are then what a lenient decoder would read)."""
    count = [0] * 16
    for ln in lengths:
        count[ln] += 1
    count[0] = 0
    nxt, code = [0] * 16, 0
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    out = []
    for ln in lengths:
        if ln:
            out.append(nxt[ln])
            nxt[ln] += 1
        else:
            out.append(None)
    return out


def huffman_lengths(freqs, limit, complete=True):
    """Length-limited Huffman code lengths (package-merge).  A single used symbol gets length 1; with complete=True a
    second symbol is added so that the code is complete (zlib refuses an incomplete code-length code)."""
    syms = [s for s, f in enumerate(freqs) if f > 0]
    lens = [0] * len(freqs)
    if not syms:
        return lens
    if len(syms) == 1:
        lens[syms[0]] = 1
        if complete:
            lens[1 if syms[0] == 0 else 0] = 1
        return lens
    leaves = sorted(((freqs[s], (s,)) for s in syms), key=lambda x: x[0])
    cur = list(leaves)
    for _ in range(limit - 1):
        paired = [(cur[i][0] + cur[i + 1][0], cur[i][1] + cur[i + 1][1]) for i in range(0, len(cur) - 1, 2)]
        cur = sorted(leaves + paired, key=lambda x: x[0])
    for _, ss in cur[:2 * len(syms) - 2]:
        for s in ss:
            lens[s] += 1
    return lens


def len_symbol(length, as284=False):
    """(symbol, extra value, extra bits) of a match length."""
    if length == 258 and as284:
        return 284, 31, 5
    for i in range(len(LEN_BASE) - 1, -1, -1):
        if LEN_BASE[i] <= length:
            return 257 + i, length - LEN_BASE[i], LEN_EXTRA[i]
    raise ValueError(length)


def dist_symbol(dist):
    for i in range(len(DIST_BASE) - 1, -1, -1):
        if DIST_BASE[i] <= dist:
            return i, dist - DIST_BASE[i], DIST_EXTRA[i]
    raise ValueError(dist)


def token_symbols(tokens):
    """Frequencies of literal/length and distance symbols (EOB counted once)."""
    lf, df = [0] * 286, [0] * 30
    for t in tokens:
        if isinstance(t, int):
            lf[t] += 1
        elif t[0] == "sym" or t[0] == "dsym":
            pass
        else:
            lf[len_symbol(t[0], len(t) > 2 and t[2])[0]] += 1
            df[dist_symbol(t[1])[0]] += 1
    lf[256] += 1
    return lf, df


def write_tokens(bw, tokens, lit_lens, dist_lens, eob=True):
    lc, dc = canonical(lit_lens), canonical(dist_lens)
    for t in tokens:
        if isinstance(t, int):
            bw.code(lc[t], lit_lens[t])
        elif t[0] == "sym":
            bw.code(lc[t[1]], lit_lens[t[1]])
        elif t[0] == "dsym":
            bw.code(lc[t[1]], lit_lens[t[1]])
            bw.bits(0, LEN_EXTRA[t[1] - 257] if t[1] < 286 else 0)
            bw.code(dc[t[2]], dist_lens[t[2]])
        else:
            s, ev, eb = len_symbol(t[0], len(t) > 2 and t[2])
            bw.code(lc[s], lit_lens[s])
            bw.bits(ev, eb)
            s, ev, eb = dist_symbol(t[1])
            bw.code(dc[s], dist_lens[s])
            bw.bits(ev, eb)
    if eob:
        bw.code(lc[256], lit_lens[256])


def stored_block(bw, data, final, nlen=None):
    bw.bits(int(final), 1)
    bw.bits(0, 2)
    bw.align()
    bw.bits(len(data), 16)
    bw.bits((~len(data) & 0xFFFF) if nlen is None else nlen, 16)
    for b in data:
        bw.bits(b, 8)


def fixed_block(bw, tokens, final, eob=True):
    bw.bits(int(final), 1)
    bw.bits(1, 2)
    write_tokens(bw, tokens, FIXED_LIT, FIXED_DIST, eob)


def rle_lengths(lens):
    """Code lengths -> code-length symbols [(sym, extra value)], runs with 16/17/18 (a run may cross from the literal
    lengths into the distance lengths: the caller passes both as one list)."""
    out, i = [], 0
    while i < len(lens):
        v, j = lens[i], i
        while j < len(lens) and lens[j] == v:
            j += 1
        run = j - i
        if v == 0:
            while run >= 11:
                r = min(run, 138)
                out.append((18, r - 11))
                run -= r
            if run >= 3:
                out.append((17, run - 3))
                run = 0
            out += [(0, 0)] * run
        else:
            out.append((v, 0))
            run -= 1
            while run >= 3:
                r = min(run, 6)
                out.append((16, r - 3))
                run -= r
            out += [(v, 0)] * run
        i = j
    return out


def dynamic_block(bw, tokens, final, lit_lens, dist_lens, cl_lens=None, rle=None, hclen=None, hlit=None, hdist=None,
                  eob=True):
    """A dynamic-Huffman block.  lit_lens: HLIT + 257 entries (>= 257), dist_lens: HDIST + 1 entries (>= 1).  cl_lens (19
    entries by symbol), rle ([(sym, extra)]), hclen/hlit/hdist (the raw header fields) override what the block would
    otherwise be given."""
    rle = rle_lengths(list(lit_lens) + list(dist_lens)) if rle is None else rle
    if cl_lens is None:
        f = [0] * 19
        for s, _ in rle:
            f[s] += 1
        cl_lens = huffman_lengths(f, 7)
    if hclen is None:
        n = 19
        while n > 4 and cl_lens[CL_ORDER[n - 1]] == 0:
            n -= 1
        hclen = n - 4
    bw.bits(int(final), 1)
    bw.bits(2, 2)
    bw.bits(len(lit_lens) - 257 if hlit is None else hlit, 5)
    bw.bits(len(dist_lens) - 1 if hdist is None else hdist, 5)
    bw.bits(hclen, 4)
    for k in range(hclen + 4):
        bw.bits(cl_lens[CL_ORDER[k]], 3)
    cc = canonical(cl_lens)
    for s, ev in rle:
        bw.code(cc[s], cl_lens[s])
        if s == 16:
            bw.bits(ev, 2)
        elif s == 17:
            bw.bits(ev, 3)
        elif s == 18:
            bw.bits(ev, 7)
    full_lit = list(lit_lens) + [0] * (288 - len(lit_lens))
    write_tokens(bw, tokens, full_lit, list(dist_lens) + [0] * (32 - len(dist_lens)), eob)


def auto_dynamic(bw, tokens, final, limit=15, hlit=None):
    """A dynamic block with Huffman codes built for the tokens."""
    lf, df = token_symbols(tokens)
    ll = huffman_lengths(lf, limit, complete=False)
    dl = huffman_lengths(df, limit, complete=False)
    nl = max(257, max(i for i, x in enumerate(ll) if x) + 1) if hlit is None else hlit
    nd = max([1] + [i + 1 for i, x in enumerate(dl) if x])
    dynamic_block(bw, tokens, final, ll[:nl] + [0] * (nl - len(ll[:nl])), dl[:nd])


def apply_tokens(tokens, out=None):
    """The bytes the tokens stand for, appended to out (the history)."""
    out = bytearray() if out is None else out
    for t in tokens:
        if isinstance(t, int):
            out.append(t)
        elif t[0] in ("sym", "dsym"):
            raise ValueError("a raw symbol has no meaning")
        else:
            ln, d = t[0], t[1]
            if d > len(out):
                raise ValueError("distance too far back")
            for _ in range(ln):
                out.append(out[-d])
    return out


def lz77(data, max_chain=16, rng=None):
    """Greedy LZ77 over a 32 KiB window, distances up to 32768 (zlib stops at 32768 - 262)."""
    toks, heads, i, n = [], {}, 0, len(data)
    while i < n:
        best_l, best_d = 0, 0
        if i + 3 <= n:
            key = data[i:i + 3]
            cands = heads.get(key, [])
            for c in reversed(cands[-max_chain:]):
                d = i - c
                if d > WINDOW:
                    break
                ln = 3
                lim = min(258, n - i)
                while ln < lim and data[c + ln] == data[i + ln]:
                    ln += 1
                if ln > best_l:
                    best_l, best_d = ln, d
                    if ln == lim:
                        break
        step = best_l if best_l >= 3 else 1
        for k in range(i, min(i + step, n - 2)):
            heads.setdefault(data[k:k + 3], []).append(k)
        if best_l >= 3:
            toks.append((best_l, best_d, True) if best_l == 258 and rng is not None and rng.random() < 0.5 else (best_l, best_d))
            i += best_l
        else:
            toks.append(data[i])
            i += 1
    return toks


def foreign_deflate(data, seed, max_block_tokens=400, empty_blocks=True):
    """A stream as other encoders write them: LZ77 with the whole 32 KiB window, cut into many blocks of random type
    (stored, fixed, dynamic), with empty blocks in between when empty_blocks is set."""
    rng = random.Random(seed)
    toks = lz77(data, rng=rng)
    bw, pos, out = BitWriter(), 0, bytearray()
    while True:
        if empty_blocks and rng.random() < 0.15:
            kind = rng.randrange(3)
            if kind == 0:
                stored_block(bw, b"", False)
            elif kind == 1:
                fixed_block(bw, [], False)
            else:
                dynamic_block(bw, [], False, [0] * 256 + [1], [0])
        n = rng.randint(1, max_block_tokens)
        seg = toks[pos:pos + n]
        pos += len(seg)
        final = pos >= len(toks)
        start = len(out)
        apply_tokens(seg, out)
        kind = rng.randrange(3)
        if kind == 0 and len(out) - start <= 65535:
            stored_block(bw, bytes(out[start:]), final)
        elif kind == 1:
            fixed_block(bw, seg, final)
        else:
            auto_dynamic(bw, seg, final)
        if final:
            break
    assert bytes(out) == data
    return bw.getvalue()


def bgzf_wrap(stream, isize, crc):
    """One BGZF block around a raw DEFLATE stream, with the given trailer (for a stream zlib refuses: the CRC32 and ISIZE
    of what a lenient decoder would produce, so that only the decoder's own checks can refuse it)."""
    hdr = b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(stream) + 25)
    assert len(stream) + 26 <= 65536, "a BGZF block holds at most 64 KiB"
    return hdr + stream + struct.pack("<II", crc & 0xFFFFFFFF, isize)


def reencode_bam(src, dst, deflate=None, empty_before=()):
    """Write the BAM src (with its .bai) again as dst: every block with data recompressed by deflate(data) -> raw DEFLATE
    stream (None: the block is copied as it is), and an ISIZE-0 BGZF block in front of every block whose index in src is
    in empty_before, as concatenated BAMs have them.  The .bai's virtual offsets follow the blocks (past the inserted
    empty blocks)."""
    d = open(src, "rb").read()
    out, moved, off = bytearray(), {}, 0
    while off < len(d):
        bs = struct.unpack_from("<H", d, off + 16)[0] + 1
        blk = d[off:off + bs]
        if len(moved) in empty_before:
            out += bgzf_wrap(b"\x03\x00", 0, 0)
        moved[off] = len(out)
        isize = struct.unpack_from("<I", blk, bs - 4)[0]
        if deflate is None or isize == 0:
            out += blk
        else:
            data = zlib.decompress(blk[18:bs - 8], -15)
            out += bgzf_wrap(deflate(data), len(data), zlib.crc32(data))
        off += bs
    moved[off] = len(out)
    open(dst, "wb").write(out)

    def mv(v):
        return moved[v >> 16] << 16 | (v & 0xFFFF) if v else 0
    bai = open(src + ".bai", "rb").read()
    new = bytearray(bai[:8])
    o = 8
    for _ in range(struct.unpack_from("<i", bai, 4)[0]):
        n_bin = struct.unpack_from("<i", bai, o)[0]
        new += bai[o:o + 4]
        o += 4
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", bai, o)
            new += bai[o:o + 8]
            o += 8
            for k in range(n_chunk):
                u, v = struct.unpack_from("<QQ", bai, o)
                # the pseudo-bin's second pair holds the mapped / unmapped read counts, not offsets
                new += struct.pack("<QQ", u, v) if b == 37450 and k == 1 else struct.pack("<QQ", mv(u), mv(v))
                o += 16
        n_intv = struct.unpack_from("<i", bai, o)[0]
        new += bai[o:o + 4]
        o += 4
        for _ in range(n_intv):
            new += struct.pack("<Q", mv(struct.unpack_from("<Q", bai, o)[0]))
            o += 8
    new += bai[o:]
    open(dst + ".bai", "wb").write(new)


def zlib_verdict(stream, isize, crc):
    """What zlib makes of a stream with this trailer: (accepted, output, trailing bytes).  Accepted means the stream ends
    with a final block and the output matches ISIZE and CRC32."""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(stream)
    except zlib.error:
        return False, None, b""
    ok = d.eof and len(out) == isize and (zlib.crc32(out) & 0xFFFFFFFF) == (crc & 0xFFFFFFFF)
    return ok, out, d.unused_data


# ---------------------------------------------------------------------------------------------------------------------
# the corpus
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    stream: bytes
    data: bytes          # valid: the bytes the stream stands for; refusal: what a lenient decoder would produce
    valid: bool          # zlib accepts the stream with this trailer
    isize: int
    crc: int
    code_check: bool = False      # refused only because a Huffman code is incomplete or over-subscribed
    records: bool = False         # the payload is whole BAM records


def _case(name, bw_or_stream, data, valid=True, isize=None, code_check=False, records=False):
    stream = bw_or_stream.getvalue() if isinstance(bw_or_stream, BitWriter) else bytes(bw_or_stream)
    data = bytes(data)
    return Case(name, stream, data, valid, len(data) if isize is None else isize, zlib.crc32(data) & 0xFFFFFFFF,
                code_check, records)


def _rand_bytes(rng, n, alphabet=256):
    return bytes(rng.randrange(alphabet) for _ in range(n))


def _text(rng, n):
    words = [_rand_bytes(rng, rng.randint(2, 9), 26) for _ in range(40)]
    out = bytearray()
    while len(out) < n:
        out += bytes(c + 97 for c in rng.choice(words)) + b" "
    return bytes(out[:n])


def valid_cases():
    rng = random.Random(1951)
    C = []
    # ---- block types
    bw = BitWriter(); stored_block(bw, b"", True)
    C.append(_case("stored_len0_final", bw, b""))
    d = _text(rng, 500)
    bw = BitWriter(); stored_block(bw, b"", False); fixed_block(bw, lz77(d), True)
    C.append(_case("stored_len0_nonfinal", bw, d))
    d = _rand_bytes(rng, 65535)       # the largest stored block (16 bits of LEN) - more than a BGZF block can hold
    bw = BitWriter(); stored_block(bw, d, True)
    C.append(_case("stored_len65535", bw, d))
    d1, d2 = _text(rng, 700), _rand_bytes(rng, 333)
    bw = BitWriter(); auto_dynamic(bw, lz77(d1), False); stored_block(bw, d2, True)
    C.append(_case("stored_ends_at_in_len", bw, d1 + d2))
    for k in range(8):                # a stored block after a fixed block at every bit offset
        lits = [200 + j for j in range(k)]            # 9-bit literals: 3 + 9k + 7 bits before the stored header
        d2 = _rand_bytes(rng, 40 + k)
        bw = BitWriter(); fixed_block(bw, lits, False); stored_block(bw, d2, False)
        fixed_block(bw, [(20, 40 + k), 7], True)
        C.append(_case(f"stored_after_fixed_bitoff{(3 + 9 * k + 7) % 8}", bw, apply_tokens([(20, 40 + k), 7], bytearray(bytes(lits) + d2))))
    d = _text(rng, 3000)
    t = lz77(d)
    h = len(t) // 2
    for where in ("start", "middle", "end"):
        for kind in ("fixed", "dynamic", "stored"):
            bw = BitWriter()

            def empty():
                if kind == "fixed":
                    fixed_block(bw, [], False)
                elif kind == "dynamic":
                    dynamic_block(bw, [], False, [0] * 256 + [1], [0])
                else:
                    stored_block(bw, b"", False)
            if where == "start":
                empty(); auto_dynamic(bw, t, True)
            elif where == "middle":
                auto_dynamic(bw, t[:h], False); empty(); fixed_block(bw, t[h:], True)
            else:
                auto_dynamic(bw, t, False); empty()
                if kind == "fixed":
                    fixed_block(bw, [], True)
                elif kind == "dynamic":
                    dynamic_block(bw, [], True, [0] * 256 + [1], [0])
                else:
                    stored_block(bw, b"", True)
            C.append(_case(f"empty_{kind}_{where}", bw, d))
    d = _text(rng, 2000)
    t = lz77(d)
    bw, i, r2 = BitWriter(), 0, random.Random(7)
    out = bytearray()
    while i < len(t):                  # hundreds of tiny blocks
        n = r2.randint(1, 5)
        seg = t[i:i + n]
        i += len(seg)
        s0 = len(out)
        apply_tokens(seg, out)
        k = r2.randrange(3)
        if k == 0 and len(out) - s0 <= 65535:
            stored_block(bw, bytes(out[s0:]), i >= len(t))
        elif k == 1:
            fixed_block(bw, seg, i >= len(t))
        else:
            auto_dynamic(bw, seg, i >= len(t))
    C.append(_case("hundreds_of_tiny_blocks", bw, d))
    C.append(_case("isize0", b"\x03\x00", b""))
    # a block of exactly 32 / 64 tokens (one / two whole rounds of the kernel): its end-of-block code starts a round
    for n in (32, 64):
        d = _rand_bytes(rng, n)
        bw = BitWriter(); fixed_block(bw, list(d), False); fixed_block(bw, [(10, 7), 1], True)
        C.append(_case(f"block_of_{n}_tokens_then_more", bw, apply_tokens([(10, 7), 1], bytearray(d))))
    # ---- dynamic headers
    d = bytes(range(255)) * 3
    ll = [8] * 255 + [0, 8]                  # 256 codes of 8 bits: only code-length symbols 8 and 0 are needed
    bw = BitWriter(); dynamic_block(bw, list(d), True, ll, [0])
    C.append(_case("hclen5_literal_only", bw, d))
    d = _text(rng, 1500)
    t = lz77(d)
    lf, df = token_symbols(t)
    ll, dl = huffman_lengths(lf, 15, False), huffman_lengths(df, 15, False)
    bw = BitWriter(); dynamic_block(bw, t, True, ll[:286], dl[:30], hclen=15)
    C.append(_case("hclen19_hlit286_hdist30", bw, d))
    bw = BitWriter(); dynamic_block(bw, [b for b in d[:400]], True, huffman_lengths(token_symbols(list(d[:400]))[0], 15, False)[:257], [0])
    C.append(_case("hlit257_hdist1_literal_only", bw, d[:400]))
    # a single distance code of one bit: every match of the block uses distance symbol 5 (distances 7..8)
    toks, out = [], bytearray()
    for j in range(300):
        if len(out) >= 8 and j % 3 == 0:
            toks.append((rng.randint(3, 258), rng.choice((7, 8))))
        else:
            toks.append(rng.randrange(256))
        apply_tokens(toks[-1:], out)
    lf, _ = token_symbols(toks)
    bw = BitWriter(); dynamic_block(bw, toks, True, huffman_lengths(lf, 15, False)[:286], [0] * 5 + [1])
    C.append(_case("single_distance_code_1bit", bw, out))
    bw = BitWriter(); dynamic_block(bw, [], True, [0] * 256 + [1], [0])
    C.append(_case("eob_only_single_code", bw, b""))
    # distance codes of 9..15 bits: lengths 1, 2, ..., 14, 15, 15 (complete) on distance symbols in scrambled order
    dsyms = list(range(16))
    rng.shuffle(dsyms)
    dl = [0] * 30
    for k, s in enumerate(dsyms):
        dl[s] = min(k + 1, 15)
    toks, out = [], bytearray(_rand_bytes(rng, 300))
    toks = list(out)
    for s in sorted(dsyms, key=lambda s: -dl[s]) * 3:
        dist = DIST_BASE[s] + rng.randrange(1 << DIST_EXTRA[s])
        if dist <= len(out):
            toks.append((rng.randint(3, 40), dist))
            apply_tokens(toks[-1:], out)
    lf, _ = token_symbols(toks)
    bw = BitWriter(); dynamic_block(bw, toks, True, huffman_lengths(lf, 15, False)[:286], dl[:max(dsyms) + 1])
    C.append(_case("distance_codes_9_to_15_bits", bw, out))
    # literal/length codes up to 15 bits, the most second-level entries a complete code of <= 286 symbols can need
    # (306 of the kernel's kLitSub = 310): 1..6 one code each, 11 x 11 bits, 9 x 12, 1 x 13, 1 x 14, 258 x 15
    counts = {1: 1, 2: 1, 3: 1, 4: 1, 5: 1, 6: 1, 11: 11, 12: 9, 13: 1, 14: 1, 15: 258}
    order = list(range(286))
    rng.shuffle(order)
    ll, k = [0] * 286, 0
    for ln in sorted(counts):
        for _ in range(counts[ln]):
            ll[order[k]] = ln
            k += 1
    assert sum(2 ** (15 - x) for x in ll if x) == 2 ** 15 and ll[256]
    toks, out = [], bytearray(_rand_bytes(rng, 64))
    toks = list(out)
    for s in sorted(range(286), key=lambda s: -ll[s]):       # every symbol once, longest codes first
        if s < 256:
            toks.append(s)
        elif s > 256:
            ln = LEN_BASE[s - 257] + rng.randrange(1 << LEN_EXTRA[s - 257])
            toks.append((ln, rng.randint(1, len(out))))
        apply_tokens(toks[-1:], out) if s != 256 else None
    _, df = token_symbols(toks)
    bw = BitWriter(); dynamic_block(bw, toks, True, ll, huffman_lengths(df, 15, False)[:30])
    C.append(_case("lit_codes_15_bits_worst_second_level", bw, out))
    # ---- matches
    d = _rand_bytes(rng, 32768)
    toks = [(258, 32768), (258, 32768, True), (3, 32768), (100, 32767), (50, 32507), (258, 32600)]
    bw = BitWriter(); stored_block(bw, d, False); fixed_block(bw, toks, True)
    C.append(_case("distance_32768_to_byte_0", bw, apply_tokens(toks, bytearray(d))))
    toks, out = [], bytearray(_rand_bytes(rng, 40))
    toks = list(out)
    for dist in range(1, 32):
        for ln in sorted({3, dist, dist + 1, 2 * dist + 5, 31, 32, 33, 258}):
            if ln >= 3:
                toks.append((min(ln, 258), dist))
        toks.append(rng.randrange(256))
    apply_tokens(toks[40:], out)
    bw = BitWriter(); auto_dynamic(bw, toks, True)
    C.append(_case("distances_1_to_31_overlaps", bw, out))
    out = bytearray(_rand_bytes(rng, 300))
    toks = list(out) + [(258, rng.choice((1, 258, 300, 7)), rng.random() < 0.5) for _ in range(40)] + [5]
    apply_tokens(toks[300:], out)
    bw = BitWriter(); fixed_block(bw, toks, True)
    C.append(_case("rounds_of_32_length_258_matches", bw, out))
    out = bytearray(_rand_bytes(rng, 1100))
    toks = list(out)
    for dist in (256, 257, 255, 512, 511, 1024, 1023, 1025, 768, 32, 33, 64):
        toks += [rng.randrange(256)] * rng.randint(0, 3) + [(258, dist), (rng.randint(3, 258), dist)]
    apply_tokens(toks[1100:], out)
    bw = BitWriter(); auto_dynamic(bw, toks, True)
    C.append(_case("sources_at_chunk_fronts", bw, out))
    # ---- streams of the foreign encoder and of zlib's own flush modes
    for seed in range(4):
        r3 = random.Random(seed)
        d = _text(r3, r3.randint(20000, 60000)) if seed % 2 else bytes(r3.choice(b"ACGT") for _ in range(40000))
        C.append(_case(f"foreign_encoder_{seed}", foreign_deflate(d, seed), d))
    d = _text(rng, 30000)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    s = co.compress(d[:10000]) + co.flush(zlib.Z_PARTIAL_FLUSH) + co.compress(d[10000:]) + co.flush(zlib.Z_SYNC_FLUSH) + \
        co.flush(zlib.Z_FULL_FLUSH) + co.flush()
    C.append(_case("zlib_partial_sync_full_flush", s, d))
    d = _text(rng, 900)
    C.append(_case("trailing_bytes_after_final_block", zlib.compress(d, 6, )[2:-4] + b"\xde\xad\xbe\xef", d))
    return C


def refusal_cases():
    rng = random.Random(1952)
    C = []
    d = _text(rng, 300)
    bw = BitWriter(); bw.bits(1, 1); bw.bits(3, 2); bw.bits(0, 32)
    C.append(_case("btype3", bw, b"", valid=False))
    bw = BitWriter(); stored_block(bw, d[:50], True, nlen=0x1234)
    C.append(_case("stored_len_nlen_mismatch", bw, d[:50], valid=False))
    t = lz77(d)
    lf, df = token_symbols(t)
    ll, dl = huffman_lengths(lf, 15, False)[:286], huffman_lengths(df, 15, False)[:30]
    bw = BitWriter(); dynamic_block(bw, t, True, ll + [0], dl)
    C.append(_case("hlit_287", bw, d, valid=False))
    bw = BitWriter(); dynamic_block(bw, t, True, ll, dl + [0])
    C.append(_case("hdist_31", bw, d, valid=False))
    rle = rle_lengths(ll + dl)
    bw = BitWriter(); dynamic_block(bw, t, True, ll, dl, rle=[(16, 0)] + rle)
    C.append(_case("repeat_16_first", bw, d, valid=False))
    bw = BitWriter(); dynamic_block(bw, [], True, [0] * 257, [0], hclen=0, cl_lens=[2] + [0] * 15 + [2, 2, 2],
                                    rle=[(18, 127), (18, 109)], eob=False)
    C.append(_case("hclen4_no_length_symbols", bw, b"", valid=False))
    bw = BitWriter(); fixed_block(bw, t, True, eob=False)
    C.append(_case("missing_end_of_block", bw, d, valid=False))
    for s in (286, 287):
        bw = BitWriter(); fixed_block(bw, list(d[:20]) + [("sym", s)] + list(d[20:40]), True)
        C.append(_case(f"fixed_symbol_{s}", bw, d[:40], valid=False))
    for s in (30, 31):
        bw = BitWriter(); fixed_block(bw, list(d[:20]) + [("dsym", 260, s)] + list(d[20:40]), True)
        C.append(_case(f"fixed_distance_symbol_{s}", bw, d[:40], valid=False))
    bw = BitWriter(); fixed_block(bw, [1, 2, 3, (10, 4)], True)
    C.append(_case("distance_too_far_back", bw, b"\1\2\3" + b"\0" * 10, valid=False))
    bw = BitWriter(); stored_block(bw, d[:100], False); fixed_block(bw, [(5, 101)], True)
    C.append(_case("distance_too_far_back_after_stored", bw, d[:100] + b"\0" * 5, valid=False))
    bw = BitWriter(); dynamic_block(bw, [1, 2, 3, 4, (5, 2)], True, [0] + [3] * 6 + [0] * 249 + [3, 0, 0, 3], [0])
    C.append(_case("match_without_distance_codes", bw, b"\1\2\3\4" + b"\3\4\3\4\3", valid=False))
    # Huffman codes zlib refuses: over-subscribed and incomplete, for all three kinds of code
    ll = [0] * 257
    ll[65], ll[66], ll[256] = 1, 2, 3     # zlib: "invalid literal/lengths set"
    bw = BitWriter(); dynamic_block(bw, [65, 66, 65, 65, 66], True, ll, [0])
    C.append(_case("incomplete_literal_code", bw, b"ABAAB", valid=False, code_check=True))
    ll = [0] * 257
    ll[65], ll[66], ll[256] = 1, 1, 1
    bw = BitWriter(); dynamic_block(bw, [65, 66], True, ll, [0])
    C.append(_case("oversubscribed_literal_code", bw, b"AB", valid=False, code_check=True))
    ll = [0] * 257
    ll[65], ll[256] = 2, 2                 # two codes of two bits: the single-code exception does not cover it
    bw = BitWriter(); dynamic_block(bw, [65, 65], True, ll, [0])
    C.append(_case("incomplete_literal_code_two_bits", bw, b"AA", valid=False, code_check=True))
    ll = [0] * 258
    ll[7], ll[8], ll[9], ll[256], ll[257] = 2, 2, 3, 3, 2
    bw = BitWriter(); dynamic_block(bw, [7, 8, 9, (3, 1), (3, 2)], True, ll, [1, 2, 0])
    C.append(_case("incomplete_distance_code", bw, apply_tokens([7, 8, 9, (3, 1), (3, 2)]), valid=False, code_check=True))
    bw = BitWriter(); dynamic_block(bw, [7, 8, 9, (3, 1), (3, 2)], True, ll, [1, 1, 1])
    C.append(_case("oversubscribed_distance_code", bw, apply_tokens([7, 8, 9, (3, 1), (3, 2)]), valid=False, code_check=True))
    bw = BitWriter(); dynamic_block(bw, [7, 8, 9, (3, 2)], True, ll, [0, 2])
    C.append(_case("incomplete_distance_code_single_2bit", bw, apply_tokens([7, 8, 9, (3, 2)]), valid=False, code_check=True))
    d2 = _text(rng, 200)
    t2 = lz77(d2)
    lf, df = token_symbols(t2)
    ll2, dl2 = huffman_lengths(lf, 15, False)[:286], huffman_lengths(df, 15, False)[:30]
    ll2 = ll2[:max(257, max(i for i, x in enumerate(ll2) if x) + 1)]
    dl2 = dl2[:max([1] + [i + 1 for i, x in enumerate(dl2) if x])]
    cl = [4] * 19
    for s in range(19):
        if s not in {x for x, _ in rle_lengths(ll2 + dl2)} and cl.count(4) > 15:
            cl[s] = 0
    assert cl.count(4) == 15
    bw = BitWriter(); dynamic_block(bw, t2, True, ll2, dl2, cl_lens=cl)
    C.append(_case("incomplete_code_length_code", bw, d2, valid=False, code_check=True))
    cl = [3] * 19                              # 19 codes of three bits: over-subscribed
    bw = BitWriter(); dynamic_block(bw, t2, True, ll2, dl2, cl_lens=cl)
    C.append(_case("oversubscribed_code_length_code", bw, d2, valid=False, code_check=True))
    # ISIZE and length
    d3 = _text(rng, 2000)
    s3 = zlib.compress(d3, 6)[2:-4]
    C.append(_case("output_longer_than_isize", s3, d3[:1999], valid=False))
    C.append(Case("output_shorter_than_isize", s3, d3, False, 2001, zlib.crc32(d3) & 0xFFFFFFFF))
    C.append(_case("truncated_input", s3[:len(s3) // 2], d3, valid=False))
    C.append(_case("truncated_by_one_byte", s3[:-1], d3, valid=False))
    return C


def corpus():
    return valid_cases() + refusal_cases()


def write_corpus(path, cases):
    """The harnesses' input: per case <u32 in_len><u32 isize><u32 crc><in_len bytes>."""
    with open(path, "wb") as f:
        for c in cases:
            f.write(struct.pack("<III", len(c.stream), c.isize, c.crc) + c.stream)
