"""DEFLATE conformance of the device inflate kernel (k_inflate_ws + k_crc32), byte for byte against zlib, on the forge's
streams (deflate_forge.py) and on batch layouts the engine produces without choosing them: every byte phase of the
compressed and raw offsets, blocks packed back to back, block counts around a generation (64 streams per CTA) and a wave
(64 x SMs), one long stream among short ones, empty non-final blocks in the last stream still running, ISIZE-0 blocks.
tests/gpu_inflate_harness.cu runs each batch with and without SpecOut (the record chains the record walk links); the
chains are compared with a restatement in Python.  Then whole BAMs written by other encoders go through the C ABI."""
import os
import random
import struct
import subprocess
import zlib

import numpy as np
import pytest

import bamsignals_b200 as B
import bamwriter as W
import deflate_forge as F
import edge_cases as E
import oracle_api as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATUS_BAD_DEFLATE, STATUS_BAD_CRC = 4, 8
SPEC_NONE, SPEC_STRIDE = 0xFFFFFFFF, 1824
GUARD = 0xA5


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    from __graft_entry__ import NVCC_FLAGS, _nvcc
    exe = str(tmp_path_factory.mktemp("gpu_harness") / "gpu_inflate_harness")
    subprocess.check_call([_nvcc()] + NVCC_FLAGS + ["-o", exe, os.path.join(ROOT, "tests", "gpu_inflate_harness.cu")])
    return exe


@pytest.fixture(scope="module")
def n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def corpus():
    print(f"zlib {zlib.ZLIB_RUNTIME_VERSION}")
    return F.corpus()


class Batch:
    """One launch: cases laid out in a compressed and a raw buffer.  in_phase(i) / out_phase(i): byte phase of block i's
    payload (mod 8) and output (mod 16); packed: BGZF-like 18 + 8 bytes around every payload and outputs back to back,
    as the engine lays a batch out."""

    def __init__(self, cases, in_phase=lambda i: 0, out_phase=lambda i: 0, packed=False, seed=0):
        rng = random.Random(seed)
        comp, raw_off = bytearray(), 64
        self.cases, self.blocks = cases, []
        for i, c in enumerate(cases):
            if packed:
                comp += bytes(rng.randrange(256) for _ in range(18))
            else:
                comp += bytes((in_phase(i) - len(comp)) % 8 + 8)
            in_off = len(comp)
            comp += c.stream
            if packed:
                comp += bytes(rng.randrange(256) for _ in range(8))
                out_off = raw_off
            else:
                out_off = raw_off + 16 + (out_phase(i) - raw_off) % 16
            self.blocks.append((in_off, len(c.stream), out_off, c.isize))
            raw_off = out_off + c.isize
        self.comp, self.raw_bytes = bytes(comp), raw_off + 64

    def write(self, path):
        with open(path, "wb") as f:
            f.write(struct.pack("<IIII", len(self.blocks), len(self.comp), self.raw_bytes, 0))
            f.write(b"".join(struct.pack("<IIII", *b) for b in self.blocks))
            f.write(b"".join(struct.pack("<I", c.crc) for c in self.cases))
            f.write(self.comp)


class Result:
    """The harness's output for one batch: both statuses, the raw buffer, and per block (cnt, end, record offsets)."""

    def __init__(self, path, n, raw_bytes):
        d = open(path, "rb").read()
        self.status_plain, self.status_spec, self.same = struct.unpack_from("<III", d, 0)
        self.raw = np.frombuffer(d, np.uint8, raw_bytes, 12)
        o, self.spec = 12 + raw_bytes, []
        for _ in range(n):
            cnt, end = struct.unpack_from("<II", d, o)
            o += 8
            offs = []
            if cnt != SPEC_NONE:
                offs = list(struct.unpack_from(f"<{cnt}I", d, o))
                o += 4 * cnt
            self.spec.append((cnt, end, offs))
        assert o == len(d)


def run(harness, tmp_path, batches):
    args = []
    for k, b in enumerate(batches):
        p = str(tmp_path / f"b{k}.in")
        b.write(p)
        args += [p, str(tmp_path / f"b{k}.out")]
    r = subprocess.run([harness] + args, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return [Result(str(tmp_path / f"b{k}.out"), len(b.blocks), b.raw_bytes) for k, b in enumerate(batches)]


def spec_restated(data, off):
    """The chain warp's SpecOut for one block: the record chain (block_size fields) from the block's first byte, with
    block_size in [32, 0xffffff] and at most 1824 records, until it reaches or passes the block's end."""
    rp, offs = 0, []
    while rp < len(data) and rp + 4 <= len(data):
        bs = struct.unpack_from("<I", data, rp)[0]
        if bs < 32 or bs > 0xFFFFFF or len(offs) >= SPEC_STRIDE:
            return SPEC_NONE, None, None
        offs.append(off + rp)
        rp += 4 + bs
    if rp < len(data):
        return SPEC_NONE, None, None
    return len(offs), off + rp, offs


def check_valid(batch, res, what):
    assert res.status_plain == 0 and res.status_spec == 0, (what, res.status_plain, res.status_spec)
    assert res.same == 1, what
    covered = np.zeros(batch.raw_bytes, bool)
    for i, (c, (_, _, out_off, isize)) in enumerate(zip(batch.cases, batch.blocks)):
        got = res.raw[out_off:out_off + isize].tobytes()
        assert got == c.data, (what, i, c.name)
        covered[out_off:out_off + isize] = True
        cnt, end, offs = spec_restated(c.data, out_off)
        gc, ge, go = res.spec[i]
        assert gc == cnt, (what, i, c.name, gc, cnt)
        if cnt != SPEC_NONE:
            assert ge == end and go == offs, (what, i, c.name)
    assert np.all(res.raw[~covered] == GUARD), what


def check_guard(batch, res, what):
    covered = np.zeros(batch.raw_bytes, bool)
    for _, _, out_off, isize in batch.blocks:
        covered[out_off:out_off + isize] = True
    assert np.all(res.raw[~covered] == GUARD), what


def tiny_case(k):
    """A stream of one round: a fixed block of a few literals and one match."""
    bw = F.BitWriter()
    toks = [65 + k % 26, 66, 67, (5, 3)]
    F.fixed_block(bw, toks, True)
    return F._case(f"tiny_{k}", bw, F.apply_tokens(toks))


def long_with_empty_block_near_end(seed):
    """A long dynamic block, then an empty non-final fixed block, then a final block of two literals: the stream is still
    running after every short neighbour has finished when it reaches the empty block."""
    rng = random.Random(seed)
    d = F._text(rng, 60000)
    t = F.lz77(d)
    bw = F.BitWriter()
    F.auto_dynamic(bw, t, False)
    F.fixed_block(bw, [], False)
    F.fixed_block(bw, [1, 2], True)
    return F._case(f"long_empty_near_end_{seed}", bw, d + b"\1\2")


def test_valid_all_phases_and_packed(harness, corpus, tmp_path):
    valid = [c for c in corpus if c.valid]
    batches = [Batch(valid, in_phase=lambda i, k=k: (i + k) % 8, out_phase=lambda i, k=k: (5 * i + 3 * k) % 16) for k in range(8)]
    batches += [Batch(valid, in_phase=lambda i, k=k: (i + k) % 8, out_phase=lambda i, k=k: (5 * i + 3 * k + 8) % 16) for k in range(8)]
    batches.append(Batch(valid, packed=True, seed=1))
    batches.append(Batch(valid[::-1], packed=True, seed=2))
    for k, (b, r) in enumerate(zip(batches, run(harness, tmp_path, batches))):
        check_valid(b, r, f"layout {k}")


def test_block_counts(harness, corpus, tmp_path, n_sm):
    """1, 63, 64, 65, 64 x SMs, 64 x SMs + 1, 2 x 64 x SMs + 1 blocks: partial generations, several generations per CTA"""
    small = [c for c in corpus if c.valid and c.isize <= 8192] + [tiny_case(k) for k in range(5)]
    big = [c for c in corpus if c.valid and c.isize > 8192]
    batches = []
    for n in (1, 63, 64, 65, 64 * n_sm, 64 * n_sm + 1, 2 * 64 * n_sm + 1):
        cases = [big[(i // 97) % len(big)] if i % 97 == 96 else small[i % len(small)] for i in range(n)]
        batches.append(Batch(cases, in_phase=lambda i: (3 * i) % 8, out_phase=lambda i: (7 * i) % 16, packed=n % 2 == 1, seed=n))
    for b, r in zip(batches, run(harness, tmp_path, batches)):
        check_valid(b, r, f"{len(b.blocks)} blocks")


def test_long_stream_among_short_ones(harness, corpus, tmp_path):
    """One long stream among 63 one-round streams, at several places; the long one with an empty non-final block near
    its end, alone and in the last slot of a generation"""
    longs = [c for c in corpus if c.name.startswith("foreign_encoder")] + [long_with_empty_block_near_end(s) for s in range(2)]
    batches = []
    for j, lc in enumerate(longs):
        for pos in (0, 37, 63):
            cases = [tiny_case(k) for k in range(64)]
            cases[pos] = lc
            batches.append(Batch(cases, in_phase=lambda i, j=j: (i + j) % 8, out_phase=lambda i: i % 16))
        batches.append(Batch([lc]))
        batches.append(Batch([tiny_case(k) for k in range(64)] + [lc]))      # alone in a CTA of its own
    for b, r in zip(batches, run(harness, tmp_path, batches)):
        check_valid(b, r, [c.name for c in b.cases if not c.name.startswith("tiny")])


def test_empty_block_in_last_active_stream(harness, corpus, tmp_path):
    """A batch whose only data block hands over nothing in some round and is not finished (an empty non-final block, or
    the end-of-block code of a block of exactly 32 / 64 tokens at the start of a round): the generation must go on."""
    by = {c.name: c for c in corpus}
    names = [n for n in by if n.startswith(("empty_fixed_", "empty_dynamic_", "empty_stored_", "block_of_"))]
    names += ["zlib_partial_sync_full_flush", "stored_len0_nonfinal", "hundreds_of_tiny_blocks"]
    batches = [Batch([by[n]]) for n in names]
    batches += [Batch([tiny_case(1), by[n]]) for n in names]
    for n, b, r in zip(names * 2, batches, run(harness, tmp_path, batches)):
        check_valid(b, r, n)


def test_isize0_blocks_between_data_blocks(harness, corpus, tmp_path):
    by = {c.name: c for c in corpus}
    zero = [by["isize0"], by["stored_len0_final"], by["eob_only_single_code"], F._case("isize0_stored", b"\x01\x00\x00\xff\xff", b"")]
    data = [c for c in corpus if c.valid and c.isize > 0]
    cases = []
    for i, c in enumerate(data):
        cases += [c, zero[i % len(zero)]]
    batches = [Batch(cases, in_phase=lambda i: i % 8, out_phase=lambda i: (3 * i) % 16), Batch(cases, packed=True, seed=5),
               Batch(zero * 20)]
    for b, r in zip(batches, run(harness, tmp_path, batches)):
        check_valid(b, r, "isize0")


def test_refusals(harness, corpus, tmp_path):
    """Every refusal case alone in a launch and between valid blocks: the status must report it - for a Huffman code
    zlib refuses, as a DEFLATE error (the trailer matches the lenient decode, so the CRC32 cannot catch it).  Nothing
    outside the blocks' outputs may be written."""
    bad = [c for c in corpus if not c.valid]
    good = [c for c in corpus if c.valid and c.isize <= 8192]
    batches, kinds = [], []
    for c in bad:
        batches.append(Batch([c]))
        kinds.append(c)
        batches.append(Batch(good[:20] + [c] + good[20:40], in_phase=lambda i: i % 8, out_phase=lambda i: (5 * i) % 16))
        kinds.append(c)
    wrong = []
    for c, b, r in zip(kinds, batches, run(harness, tmp_path, batches)):
        for st in (r.status_plain, r.status_spec):
            want = STATUS_BAD_DEFLATE if c.code_check else STATUS_BAD_DEFLATE | STATUS_BAD_CRC
            if not st & want:
                wrong.append((c.name, len(b.blocks), st))
        check_guard(b, r, c.name)
    assert not wrong, wrong


def record_cases():
    """Blocks whose payloads are BAM records (the chain warp's SpecOut is what the record walk links), in the foreign
    encoder's streams, stored blocks and fixed blocks; one cut mid-record."""
    rng = random.Random(11)
    stream = bytearray()
    for i, r in enumerate(E.variety_reads(n=400)):
        b, _ = W.record_bytes(r["tid"], r["pos"], r["flag"], r["mapq"], r.get("cigar"), r.get("tlen", 0), f"q{i}")
        stream += b
    cases, a = [], 0
    while a < len(stream):
        n = rng.randint(2000, 30000)
        b = a
        while b < len(stream) and b - a < n:
            b += 4 + struct.unpack_from("<i", stream, b)[0]
        d = bytes(stream[a:b])
        k = len(cases) % 3
        if k == 0:
            s = F.foreign_deflate(d, len(cases))
        elif k == 1:
            bw = F.BitWriter(); F.stored_block(bw, d[:len(d) // 2], False); F.stored_block(bw, d[len(d) // 2:], True)
            s = bw.getvalue()
        else:
            bw = F.BitWriter(); F.fixed_block(bw, F.lz77(d), True)
            s = bw.getvalue()
        cases.append(F._case(f"records_{len(cases)}", s, d, records=True))
        a = b
    d = bytes(stream[5:9000])                  # starts inside a record
    cases.append(F._case("records_mid_record", F.foreign_deflate(d, 99), d, records=True))
    return cases


def test_spec_out_on_record_blocks(harness, tmp_path):
    cases = record_cases()
    batches = [Batch(cases, in_phase=lambda i: i % 8, out_phase=lambda i: (3 * i) % 16), Batch(cases, packed=True, seed=3)]
    for b, r in zip(batches, run(harness, tmp_path, batches)):
        check_valid(b, r, "records")
        assert sum(cnt != SPEC_NONE for cnt, _, _ in r.spec) >= len(cases) - 1


# ---- whole BAMs through the C ABI ---------------------------------------------------------------------------------


def partial_flush(d):
    """zlib with a Z_PARTIAL_FLUSH (an empty fixed block, not final) two thirds into the block"""
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    k = 2 * len(d) // 3
    return co.compress(d[:k]) + co.flush(zlib.Z_PARTIAL_FLUSH) + co.compress(d[k:]) + co.flush()


def foreign(seed):
    counter = [seed]

    def enc(d):
        counter[0] += 1
        return F.foreign_deflate(d, counter[0])
    return enc


BAMS = {          # write_bam arguments, then the re-encoding (empty_before: indices of the BGZF blocks, 0 = the header)
    "foreign_encoder": (dict(n=1500, block_payload=30000), dict(deflate=foreign(0))),
    "foreign_encoder_empty_blocks": (dict(n=1500, block_payload=20000), dict(deflate=foreign(100), empty_before={1, 3, 4, 8})),
    "zlib_partial_flush_one_block": (dict(n=150, block_payload=0xFF00), dict(deflate=partial_flush)),
    "zlib_partial_flush": (dict(n=1500, block_payload=0xFF00), dict(deflate=partial_flush)),
    "zlib_empty_blocks": (dict(n=1500, block_payload=15000), dict(empty_before={2, 3, 6, 10})),
}


@pytest.mark.parametrize("name", sorted(BAMS))
def test_bams_of_other_encoders(tmp_path, name):
    kw, rk = BAMS[name]
    kw = dict(kw)
    n = kw.pop("n")
    src, p = str(tmp_path / "zlib.bam"), str(tmp_path / f"{name}.bam")
    W.write_bam(src, E.REFS, E.variety_reads(n=n), **kw)
    F.reencode_bam(src, p, **rk)
    gr = E.variety_regions()
    for fn, args in (("bamCount", dict(ss=True)), ("bamProfile", dict(binsize=7, ss=True, shift=30)),
                     ("bamCoverage", dict(paired_end="extend"))):
        want = getattr(O, fn)(p, gr, **args)
        for gi in (1, -1):
            got = getattr(B, fn)(p, gr, opts=B.default_opts(gpu_inflate=gi), **args)
            if fn == "bamCount":
                assert np.array_equal(np.asarray(got), np.asarray(want)), (fn, gi)
            else:
                ga, wa = got.as_list(), want.as_list()
                assert len(ga) == len(wa) and all(np.array_equal(a, b) for a, b in zip(ga, wa)), (fn, gi)
