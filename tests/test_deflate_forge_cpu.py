"""DEFLATE conformance of the decode core on the CPU.  The forge (deflate_forge.py) writes streams that zlib's encoder never
writes - distances up to 32768, mixed and empty blocks, single-code and literal-only distance trees, 15-bit codes, length
258 as 284 + 31 - and streams that no decoder may accept.  zlib's decoder is the reference, asked at run time.  The decode
core shared with the GPU kernel (inflate_core.cuh, compiled into tests/host_inflate_cases.cpp under ASan / UBSan) must
give zlib's bytes for every stream zlib accepts and refuse every stream zlib refuses - by itself: the trailer of a refused
stream carries the CRC32 and ISIZE of what a lenient decoder would produce."""
import os
import subprocess
import zlib

import pytest

import deflate_forge as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def corpus():
    return F.corpus()


def _build(tmp_path_factory, src):
    exe = str(tmp_path_factory.mktemp("forge_harness") / os.path.splitext(src)[0])
    subprocess.check_call(["g++", "-O1", "-g", "-fsanitize=address,undefined", "-fno-sanitize-recover=undefined", "-o", exe,
                           os.path.join(ROOT, "tests", src), "-lz"])
    return exe


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    """per stream of a corpus (tests/host_inflate_cases.cpp)"""
    return _build(tmp_path_factory, "host_inflate_cases.cpp")


@pytest.fixture(scope="module")
def file_harness(tmp_path_factory):
    """per BGZF block of a file, checked against its CRC32 and ISIZE (tests/host_inflate_harness.cpp)"""
    return _build(tmp_path_factory, "host_inflate_harness.cpp")


def test_zlib_version_recorded():
    print(f"zlib {zlib.ZLIB_RUNTIME_VERSION} (built against {zlib.ZLIB_VERSION})")
    assert zlib.ZLIB_RUNTIME_VERSION


def test_corpus_names_unique(corpus):
    names = [c.name for c in corpus]
    assert len(names) == len(set(names))
    assert sum(c.valid for c in corpus) >= 40 and sum(not c.valid for c in corpus) >= 20
    assert sum(c.code_check for c in corpus) >= 6


def test_forge_agrees_with_zlib(corpus):
    """Every valid case decodes in zlib to exactly the bytes the forge meant; every refusal case is refused by zlib."""
    for c in corpus:
        ok, out, _ = F.zlib_verdict(c.stream, c.isize, c.crc)
        if c.valid:
            assert ok and out == c.data, c.name
        else:
            assert not ok, c.name


def test_zlib_pins(corpus):
    """What zlib does at the edges the corpus relies on."""
    by = {c.name: c for c in corpus}
    # bytes after the final block: zlib stops at the final block and leaves them unused (so do both library paths)
    ok, out, tail = F.zlib_verdict(*(lambda c: (c.stream, c.isize, c.crc))(by["trailing_bytes_after_final_block"]))
    assert ok and tail == b"\xde\xad\xbe\xef"
    # the single-code exceptions: zlib accepts one literal/length code of one bit, one distance code of one bit, and
    # no distance code at all
    for name in ("eob_only_single_code", "single_distance_code_1bit", "hlit257_hdist1_literal_only"):
        assert F.zlib_verdict(by[name].stream, by[name].isize, by[name].crc)[0], name
    d = zlib.decompressobj(-15)
    with pytest.raises(zlib.error, match="invalid literal/lengths set"):
        d.decompress(by["incomplete_literal_code"].stream)
    with pytest.raises(zlib.error, match="invalid distances set"):
        zlib.decompressobj(-15).decompress(by["incomplete_distance_code"].stream)
    with pytest.raises(zlib.error, match="invalid code lengths set"):
        zlib.decompressobj(-15).decompress(by["incomplete_code_length_code"].stream)


def test_forge_huffman_and_rle():
    for freqs, limit in (([1] * 286, 15), ([2 ** min(i, 20) for i in range(40)], 7), ([5, 0, 0, 7], 15), ([1, 1], 1)):
        lens = F.huffman_lengths(freqs, limit)
        assert max(lens) <= limit
        assert sum(2.0 ** -x for x in lens if x) == 1.0
        assert all((f > 0) == (x > 0) for f, x in zip(freqs, lens))
    lens = [3] * 20 + [0] * 150 + [7, 7, 7, 7] + [0] * 5
    out = []
    for s, e in F.rle_lengths(lens):
        out += [s] if s < 16 else [out[-1]] * (3 + e) if s == 16 else [0] * ((3 if s == 17 else 11) + e)
    assert out == lens


def run_cases(exe, corpus, path):
    F.write_corpus(path, corpus)
    r = subprocess.run([exe, path], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "runtime error" not in r.stderr and "AddressSanitizer" not in r.stderr, r.stderr[-4000:]
    res = {}
    for line in r.stdout.splitlines():
        _, i, _, p, _, rc, _, crc = line.split()
        res[(int(i), int(p))] = (int(rc), int(crc))
    assert len(res) == 8 * len(corpus)
    return res


def test_decode_core_matches_zlib(harness, corpus, tmp_path):
    """The shared decode core at every input byte phase: zlib's bytes (CRC32 of exactly ISIZE bytes) on every stream zlib
    accepts, a refusal (non-zero return code) on every stream zlib refuses."""
    res = run_cases(harness, corpus, str(tmp_path / "corpus.bin"))
    wrong = []
    for i, c in enumerate(corpus):
        for p in range(8):
            rc, crc = res[(i, p)]
            if c.valid and (rc != 0 or crc != zlib.crc32(c.data) & 0xFFFFFFFF):
                wrong.append(f"{c.name} phase {p}: rc {rc}, crc {crc:#x}")
            if not c.valid and rc == 0:
                wrong.append(f"{c.name} phase {p}: accepted")
    assert not wrong, wrong


@pytest.mark.parametrize("name", ["incomplete_literal_code", "incomplete_distance_code", "incomplete_code_length_code",
                                  "oversubscribed_literal_code", "oversubscribed_distance_code",
                                  "oversubscribed_code_length_code", "incomplete_literal_code_two_bits",
                                  "incomplete_distance_code_single_2bit"])
def test_invalid_codes_refused(harness, corpus, tmp_path, name):
    """Huffman codes zlib refuses (inftrees.c: over-subscribed, or incomplete unless a single one-bit code) are refused
    by the decode core too - before it produces a byte, so a matching trailer cannot let them through."""
    c = next(c for c in corpus if c.name == name)
    assert c.code_check and not F.zlib_verdict(c.stream, c.isize, c.crc)[0]
    res = run_cases(harness, [c], str(tmp_path / "one.bin"))
    assert all(res[(0, p)][0] != 0 for p in range(8)), res


def test_foreign_bgzf_blocks(file_harness, tmp_path):
    """The foreign encoder's streams in BGZF blocks (bgzf_wrap), through the harness that checks CRC32 and ISIZE."""
    import random
    rng = random.Random(3)
    blob = bytearray()
    for seed in range(6):
        d = bytes(rng.choice(b"ACGTN") for _ in range(rng.randint(100, 50000)))
        blob += F.bgzf_wrap(F.foreign_deflate(d, seed), len(d), zlib.crc32(d))
    p = tmp_path / "f.bgzf"
    p.write_bytes(bytes(blob))
    r = subprocess.run([file_harness, str(p)], capture_output=True, text=True)
    assert r.returncode == 0 and "blocks 6 bad 0" in r.stdout, r.stdout + r.stderr


def test_reencoded_bams_read_the_same(tmp_path):
    """reencode_bam (the BAMs of other encoders the GPU tests count): recompressed blocks and inserted ISIZE-0 blocks,
    with the index's virtual offsets moved along, give the CPU oracle the same counts as the zlib-written original."""
    import numpy as np
    import bamwriter as W
    import edge_cases as E
    import oracle_api as O
    src = str(tmp_path / "src.bam")
    W.write_bam(src, E.REFS, E.variety_reads(n=800), block_payload=12000)
    gr = E.variety_regions()
    want = O.bamCount(src, gr, ss=True)
    for k, rk in enumerate((dict(deflate=lambda d: F.foreign_deflate(d, len(d))), dict(empty_before={1, 2, 5}),
                            dict(deflate=lambda d: F.foreign_deflate(d, 7), empty_before={3, 4}))):
        p = str(tmp_path / f"r{k}.bam")
        F.reencode_bam(src, p, **rk)
        assert open(p, "rb").read() != open(src, "rb").read()
        assert np.array_equal(O.bamCount(p, gr, ss=True), want), rk
