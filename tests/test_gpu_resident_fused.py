"""Staged pileup calls on the fused path (DESIGN.md §13): with opts.resident_scheme 0 (auto), 1 (decode every resident
record, join against the read table) and 2 (the session's record index, K3f + K4f), host and device output, every
result equals the oracle's element for element (the scaled presets: the streaming call's, which the other suites check
against the oracle), also when the session's records sit in several resident batches, and the resident records'
status bits raise on every staged call what the table path raises."""
import os
import sys
import warnings

import numpy as np
import pytest

import bamsignals_b200 as B
import bamwriter as W
import oracle_api as O
import random_cases as RC

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import workloads as WL  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:some ranges' widths")]
DEV = "cuda:0"


def ext_of(args):
    return abs(args["shift"]) + (args["tlen_filter"][1] if args["pe_mid"] else 0)


def oracle_flat(bam, gr, fn, kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return RC.flat(getattr(O, fn)(bam, gr, **kw), fn)


def staged(st, args):
    """(host result, device result, timings of the host call) of one staged pileup call."""
    h = st.pileup(**args)
    t = B.timings()
    if len(h) == 0:
        return h, h, t
    d = torch.full((len(h),), -7, dtype=torch.int32, device=DEV)
    assert st.pileup(**args, out=d) is d
    return h, d.cpu().numpy(), t


def check_all_schemes(bam, gr, fn, kw, want, batch_bytes=0, min_batches=0):
    args = B.core_args(fn, **kw)
    kept = {}
    for scheme in (0, 1, 2):
        o = B.default_opts(resident_scheme=scheme, batch_bytes=batch_bytes)
        with B.Stage(bam, gr, ext_hint=ext_of(args), opts=o) as st:
            assert B.timings()["n_batches"] >= min_batches
            for _ in range(2):                              # the second call reuses the tiles and the path estimate
                h, d, t = staged(st, args)
                assert np.array_equal(h, want) and np.array_equal(d, want), (scheme, fn, kw, batch_bytes)
            kept[scheme] = t["records_kept"]
    assert kept[1] >= 0 and kept[2] == -1 and kept[0] in (-1, kept[1])
    return kept


def _fetches_records(sc):
    return sc["fn"] != "bamCoverage" and len(sc["reads"]) >= 60 and len(sc["gr"]) >= 3


PILEUP_SEEDS = [s for s in range(200) if _fetches_records(RC.scenario(s))][:24]


@pytest.mark.parametrize("seed", PILEUP_SEEDS)
def test_random_scenarios(tmp_path, seed):
    """All CIGAR operators, long N spans, flag-0x4 reads with a position, unplaced reads, shifts of +-100 k, midpoints
    with tlen filters at their edges, regions below 1 / zero-width / past the contig end / seqlevels in another order."""
    sc = RC.scenario(seed)
    bam = RC.write(sc, str(tmp_path / "r.bam"))
    want = oracle_flat(bam, sc["gr"], sc["fn"], sc["kw"])
    assert np.array_equal(want, RC.spec_counts(sc))
    check_all_schemes(bam, sc["gr"], sc["fn"], sc["kw"], want)


def _multi_batch_reads(rng, n=40000, length=3_000_000):
    """40 k reads of ~140 bytes, 2 % of them spliced over 5-40 kb (the long list), over a 3 Mb contig: stored
    uncompressed, the fetch plan of windows over the whole contig is five ~1 MB segments, and every segment is a batch of
    its own when batch_bytes is smaller than one."""
    reads = []
    for p in np.sort(rng.integers(0, length - 70000, n)):
        u = rng.random()
        cigar = "60M" if u < .96 else (f"30M{int(rng.integers(5000, 40000))}N30M" if u < .98 else "20M2D10I30M")
        reads.append(dict(tid=0, pos=int(p), flag=int(rng.choice([0, 16, 99, 147])), mapq=int(rng.integers(0, 61)),
                          cigar=cigar, tlen=int(rng.choice([150, -150, 300, -301])), l_seq=60))
    return reads


MULTI_BATCH_CALLS = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamProfile", dict(binsize=7, shift=-500)),
                     ("bamProfile", dict(binsize=2, paired_end="midpoint", tlenFilter=(150, 300))),
                     ("bamCount", dict(ss=True, shift=40))]


@pytest.fixture(scope="module")
def multi_batch_bam(tmp_path_factory):
    bam = str(tmp_path_factory.mktemp("mb") / "mb.bam")
    W.write_bam(bam, [("chrM", 3_000_000)], _multi_batch_reads(np.random.default_rng(11)), level=0)
    return bam


@pytest.mark.parametrize("fn,kw", MULTI_BATCH_CALLS, ids=[f"{f}-{i}" for i, (f, _) in enumerate(MULTI_BATCH_CALLS)])
def test_tiles_across_resident_batches(multi_batch_bam, fn, kw):
    """3 kb windows every 1 kb plus the whole contig, staged in five resident batches: tiles' row ranges and long-list
    entries cross every batch boundary."""
    starts = np.arange(1, 2_990_000, 1000)
    gr = B.GRanges(["chrM"] * (len(starts) + 1), np.append(starts, 1), np.append(np.full(len(starts), 3000), 3_000_000),
                   (["+", "-", "*"] * len(starts))[:len(starts) + 1])
    assert B.debug_plan(multi_batch_bam, gr, ext=ext_of(B.core_args(fn, **kw)), cap=1)["segments"] >= 4
    want = oracle_flat(multi_batch_bam, gr, fn, kw)
    assert want.sum() > 0
    check_all_schemes(multi_batch_bam, gr, fn, kw, want, batch_bytes=1 << 16, min_batches=4)


def _wide_reads(rng):
    """Reads larger than a CTA's staging buffer (SEQ/QUAL of 10-20 kb), spliced reads with 5-60 kb N operations,
    both strands, paired flags and tlen values at the filter's edges."""
    reads = []
    for p in np.sort(rng.integers(0, 400000, 3000)):
        u = rng.random()
        cigar = "60M" if u < .7 else (f"30M{int(rng.integers(5000, 60000))}N30M" if u < .85 else "25M3D10I25M")
        flag = int(rng.choice([0, 16, 99, 147, 83, 163]))
        tl = int(rng.choice([149, -149, 150, -150, 300, -300, 301, -301, 0, -2147483648]))
        l_seq = int(rng.integers(10000, 20000)) if rng.random() < .05 else 60
        reads.append(dict(tid=0, pos=int(p), flag=flag, mapq=int(rng.integers(0, 61)), cigar=cigar, tlen=tl, l_seq=l_seq))
    return reads


WIDE_CALLS = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamProfile", dict(binsize=7, shift=-100000)),
              ("bamProfile", dict(binsize=1, shift=100000, ss=True)),
              ("bamProfile", dict(binsize=3, paired_end="midpoint", tlenFilter=(150, 300), ss=True)),
              ("bamCount", dict(ss=True, paired_end="midpoint", tlenFilter=(149, 301))),
              ("bamCount", dict(shift=20)), ("bamProfile", dict(binsize=200, mapqual=30, filteredFlag=1024))]


@pytest.mark.parametrize("fn,kw", WIDE_CALLS, ids=[f"{f}-{i}" for i, (f, _) in enumerate(WIDE_CALLS)])
def test_large_records_and_long_spans(tmp_path, fn, kw):
    rng = np.random.default_rng(3)
    bam = str(tmp_path / "wide.bam")
    W.write_bam(bam, [("chrW", 500000)], _wide_reads(rng))
    start = rng.integers(-50, 499000, 300)
    gr = B.GRanges(["chrW"] * 300, start, rng.integers(0, 3000, 300), rng.choice(["+", "-", "*"], 300).tolist())
    want = oracle_flat(bam, gr, fn, kw)
    assert want.sum() > 0
    for bb in (0, 1 << 16):
        check_all_schemes(bam, gr, fn, kw, want, batch_bytes=bb)


@pytest.fixture(scope="module")
def gen_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("gen"))


@pytest.mark.parametrize("preset,gs,fused", [("c2", 0.002, True), ("c4", 0.002, False), ("c5", 0.002, False)])
def test_scaled_configs_choose_their_path(gen_dir, preset, gs, fused):
    """Auto takes the fused path on C2's sparse windows and the table path on C4's whole contigs and C5's overlapping
    windows; both paths give the streaming call's result."""
    bam, _ = WL.make_bam(preset, gs, gen_dir, unplaced=7)
    gr, kw, fn = WL.regions(preset, gs)
    want = WL.as_flat(getattr(B, fn)(bam, gr, **kw))
    kept = check_all_schemes(bam, gr, fn, kw, want)
    assert (kept[0] == -1) == fused and int(want.sum()) > 0


def test_empty_bam(tmp_path):
    bam = str(tmp_path / "empty.bam")
    W.write_bam(bam, [("chrE", 10000)], [])
    gr = B.GRanges(["chrE", "chrE"], [1, 500], [100, 0])
    for fn, kw in (("bamProfile", dict(binsize=1, ss=True)), ("bamCount", {})):
        check_all_schemes(bam, gr, fn, kw, oracle_flat(bam, gr, fn, kw))


def test_changing_parameters_interleaved_with_a_table_session(fixture_bam):
    """One fused session called with changing parameters, interleaved with a second session forced onto the table path
    (the two share the device's tile buffers)."""
    rng = np.random.default_rng(7)
    gr = B.GRanges(rng.choice(["chr1", "chr2", "chr3"], 200).tolist(), rng.integers(1, 9000, 200), rng.integers(0, 1500, 200),
                   rng.choice(["+", "-", "*"], 200).tolist())
    gr2 = gr[np.arange(0, 200, 3)]
    calls = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamProfile", dict(binsize=5)),
             ("bamCount", dict(ss=True)), ("bamProfile", dict(binsize=2, paired_end="midpoint", tlenFilter=(0, 300))),
             ("bamProfile", dict(binsize=1, shift=-40, mapqual=20)), ("bamCount", dict(paired_end="filter", tlenFilter=(50, 200)))]
    with B.Stage(fixture_bam, gr, ext_hint=1000, opts=B.default_opts(resident_scheme=2)) as fused, \
            B.Stage(fixture_bam, gr2, ext_hint=1000, opts=B.default_opts(resident_scheme=1)) as table:
        for _ in range(2):
            for fn, kw in calls:
                args = B.core_args(fn, **kw)
                for st, g, k in ((fused, gr, -1), (table, gr2, None)):
                    want = oracle_flat(fixture_bam, g, fn, kw)
                    h, d, t = staged(st, args)
                    assert np.array_equal(h, want) and np.array_equal(d, want), (fn, kw, k)
                    assert (t["records_kept"] == -1) == (k == -1)


def _bad_cigar_bam(path):
    """A BAM whose third record claims 0xffff CIGAR operations: they run past the record's end."""
    orig = W.record_bytes

    def patched(tid, pos, flag, mapq, cigar, tlen, name="r", *a, **k):
        b, rl = orig(tid, pos, flag, mapq, cigar, tlen, name, *a, **k)
        if name == "bad":
            b = bytearray(b)
            b[16:18] = (0xFFFF).to_bytes(2, "little")
            b = bytes(b)
        return b, rl
    W.record_bytes = patched
    try:
        reads = [dict(tid=0, pos=x, flag=0, mapq=30, cigar="20M", tlen=0, name="bad" if i == 2 else f"q{i}")
                 for i, x in enumerate(range(100, 4000, 100))]
        W.write_bam(path, [("chrA", 5000)], reads)
    finally:
        W.record_bytes = orig
    return path


def _unsorted_at_batch_boundary(path):
    """chrB's reads stored before chrA's, with 3000 unfetched chrB reads between: the windows chrA:1-5000 and
    chrB:1-5000 are two fetch segments, and the only pair out of order is the last record of the first and the first
    record of the second - the boundary between two resident batches."""
    reads = [dict(tid=1, pos=p, flag=0, mapq=30, cigar="50M", tlen=0) for p in range(100, 3100, 10)]
    reads += [dict(tid=1, pos=p, flag=0, mapq=30, cigar="50M", tlen=0) for p in range(50000, 95000, 15)]
    reads += [dict(tid=0, pos=p, flag=0, mapq=30, cigar="50M", tlen=0) for p in range(100, 3100, 10)]
    W.write_bam(path, [("chrA", 100000), ("chrB", 100000)], reads, block_payload=4000)
    return path


@pytest.mark.parametrize("kind", ["unsorted", "unsorted_at_batch_boundary", "cigar_past_end"])
def test_resident_status_raises_on_every_call(tmp_path, kind):
    p = str(tmp_path / f"{kind}.bam")
    gr = B.GRanges(["chrA", "chrA"], [1, 2000], [1000, 1000])
    batch_bytes, min_batches = 0, 1
    if kind == "unsorted":
        W.write_bam(p, [("chrA", 5000)], [dict(tid=0, pos=x, flag=0, mapq=30, cigar="20M", tlen=0) for x in (100, 500, 300, 900)])
    elif kind == "unsorted_at_batch_boundary":
        _unsorted_at_batch_boundary(p)
        gr = B.GRanges(["chrA", "chrB"], [1, 1], [1000, 1000])
        plan = B.debug_plan(p, gr, cap=1000)
        assert plan["segments"] == 2 and list(plan["tid"][299:301]) == [1, 0]
        batch_bytes, min_batches = 4096, 2
    else:
        _bad_cigar_bam(p)
    codes = {}
    for scheme in (1, 0, 2):
        with B.Stage(p, gr, opts=B.default_opts(resident_scheme=scheme, batch_bytes=batch_bytes)) as st:   # opens: the status is the calls'
            assert B.timings()["n_batches"] >= min_batches
            for args in (B.core_args("bamProfile", binsize=1, ss=True), B.core_args("bamCount"), B.core_args("bamProfile", binsize=1, ss=True)):
                with pytest.raises(B.BamsignalsError) as e:
                    st.pileup(**args)
                codes.setdefault(scheme, set()).add(e.value.code)
                with pytest.raises(B.BamsignalsError) as e:
                    st.pileup(**args, out=torch.zeros(4000, dtype=torch.int32, device=DEV))
                codes[scheme].add(e.value.code)
    assert codes[1] == {-5 if kind.startswith("unsorted") else -4} and codes[0] == codes[1] == codes[2], codes
