"""Strand-specific bamCoverage on the GPU (bsg_coverage_ss*, `ss=True`): the dense result equals the oracle identity
(sense / antisense from coverage with requiredF and requiredF | 16) and the GPU's own unstranded pair, every form (dense
host, dense device, out= buffers, staged sessions, runs to host and to device) gives the same result element for
element, run properties hold, tiles of every size and halved tiles of whole contigs are exact, device output lands only
inside the caller's slice at every 16-byte phase and after the caller's stream, both inflate paths, result packing and
early tile counting agree, and two devices give what one gives."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import bamsignals_b200 as B
import oracle_api as O
from bamsignals_b200 import api

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import workloads as WL  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
LEVELS = ["chr1", "chr2", "chr3"]
DEV = "cuda:0"
EARG = -8

COVERAGE_KW = [dict(paired_end="ignore"), dict(paired_end="extend"), dict(paired_end="extend", tlenFilter=(50, 300)),
               dict(paired_end="ignore", mapqual=20), dict(paired_end="ignore", filteredFlag=1024 + 16),
               dict(paired_end="extend", tlenFilter=(0, 250), mapqual=10, filteredFlag=256)]
KW_IDS = ["-".join(f"{k}{v}" for k, v in kw.items()) for kw in COVERAGE_KW]


def fixture_regions(seed=31, n=120):
    """Shuffled, duplicated and overlapping regions on '+', '-' and '*', some of them zero-width."""
    rng = np.random.default_rng(seed)
    start = rng.integers(1, 9001, n)
    width = rng.integers(1, 1000, n)
    width[::9] = 0
    chrom = rng.choice(LEVELS, n)
    strand = rng.choice(["+", "-", "*"], n)
    idx = np.concatenate([np.arange(n), rng.integers(0, n, n // 4)])
    rng.shuffle(idx)
    return B.GRanges(chrom[idx].tolist(), start[idx], width[idx], strand[idx].tolist())


def host(x):
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def identity(cov, gr, a):
    """The stranded result from two unstranded ones: cov(**args) with requiredF and with requiredF | 16, per region a
    (2, w) [sense; antisense] matrix."""
    tot = cov(**a)
    rev = cov(**dict(a, requiredF=a["requiredF"] | 16))
    out = []
    for t, r, s in zip(tot, rev, gr.strand):
        t, r = host(t).astype(np.int32), host(r).astype(np.int32)
        out.append(np.stack([r, t - r]) if s < 0 else np.stack([t - r, r]))
    return out


def oracle_identity(bam, gr, **kw):
    return identity(lambda **a: O.coverage_core(bam, gr, **a), gr, api.core_args("bamCoverage", **kw))


def same(got, want):
    got = [host(g) for g in got]
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and np.array_equal(g, w), i


def flat_of(mats):
    return np.concatenate([m.reshape(-1, order="F") for m in mats]) if mats else np.zeros(0, np.int32)


def check_runs(runs, want, timed=True):
    """runs (CoverageRuns with ss) against the dense (2, w) matrices: the lists expand to the rows, lengths >= 1 sum to
    the width, adjacent values differ, zero-width regions have no runs."""
    assert runs.ss and len(runs) == len(want) and len(runs.offsets) == 2 * len(want) + 1
    off = runs.offsets
    L, V = host(runs.lengths), host(runs.values)
    assert L.dtype == np.int32 and V.dtype == np.int32
    for i, w in enumerate(want):
        for a in (0, 1):
            k = 2 * i + a
            lg, vg = L[off[k]:off[k + 1]], V[off[k]:off[k + 1]]
            assert (lg >= 1).all() and int(lg.sum()) == w.shape[1], (i, a)
            assert (vg[1:] != vg[:-1]).all(), (i, a)
            assert np.array_equal(np.repeat(vg, lg), w[a]), (i, a)
    same(runs.to_dense().as_list(), want)
    if timed:
        t = B.timings()
        assert t["out_elems"] == 2 * off[-1]
        assert t["bytes_d2h"] <= 4096 + 8 * len(off)


@pytest.mark.parametrize("kw", COVERAGE_KW, ids=KW_IDS)
def test_fixture_identity_and_every_form(fixture_bam, kw):
    gr = fixture_regions()
    want = oracle_identity(fixture_bam, gr, **kw)
    dense = B.bamCoverage(fixture_bam, gr, ss=True, **kw)
    assert dense.ss and isinstance(dense._flat, np.ndarray)
    same(dense.as_list(), want)
    # the GPU's own unstranded pair gives the same identity
    same(dense.as_list(), identity(lambda **a: B.coverage_core(fixture_bam, gr, **a), gr, api.core_args("bamCoverage", **kw)))
    # sense + antisense is today's unstranded coverage
    same([m.sum(0) for m in want], [host(x).astype(np.int64) for x in B.bamCoverage(fixture_bam, gr, **kw).as_list()])
    dd = B.bamCoverage(fixture_bam, gr, ss=True, device=DEV, **kw)
    assert dd._flat.is_cuda and dd.ss
    same(dd.as_list(), want)
    a = api.core_args("bamCoverage", **kw)
    off = api.output_layout(gr.width, 1, True)
    buf = torch.full((int(off[-1]),), -5, dtype=torch.int32, device=DEV)
    assert B.coverage_core(fixture_bam, gr, **a, out=buf, ss=True) is buf
    assert np.array_equal(buf.cpu().numpy(), flat_of(want))
    same(B.coverage_core(fixture_bam, gr, **a, ss=True), want)
    r = B.bamCoverage(fixture_bam, gr, ss=True, runs=True, **kw)
    assert isinstance(r, B.CoverageRuns) and isinstance(r.lengths, np.ndarray)
    check_runs(r, want)
    rd = B.bamCoverage(fixture_bam, gr, ss=True, runs=True, device=DEV, **kw)
    assert rd.lengths.is_cuda and np.array_equal(rd.offsets, r.offsets)
    check_runs(rd, want)
    td = rd.to_dense()
    assert td._flat.is_cuda
    # without ss every entry point is the existing one
    same(B.bamCoverage(fixture_bam, gr, ss=False, **kw).as_list(), [host(x) for x in O.bamCoverage(fixture_bam, gr, **kw).as_list()])


def test_staged_session_interleaves_every_form(fixture_bam):
    gr = fixture_regions(seed=32)
    settings = [dict(tlen_filter=None, requiredF=0, tspan=False),
                dict(tlen_filter=(0, 1000), requiredF=66, tspan=True),
                dict(tlen_filter=(50, 300), requiredF=66, tspan=True, mapqual=10)]
    want = [identity(lambda **a: O.coverage_core(fixture_bam, gr, **a), gr, kw) for kw in settings]
    plain = [O.coverage_core(fixture_bam, gr, **kw) for kw in settings]
    off = api.output_layout(gr.width, 1, True)
    with B.Stage(fixture_bam, gr, ext_hint=1000) as st:
        for _ in range(2):
            for kw, w, p in zip(settings, want, plain):
                assert np.array_equal(st.coverage(**kw, ss=True), flat_of(w))
                assert np.array_equal(st.coverage(**kw), np.concatenate(p))
                buf = torch.empty(int(off[-1]), dtype=torch.int32, device=DEV)
                st.coverage(**kw, out=buf, ss=True)
                assert np.array_equal(buf.cpu().numpy(), flat_of(w))
                check_runs(st.coverage_runs(**kw, ss=True), w)
                check_runs(st.coverage_runs(**kw, ss=True, device=DEV), w)
                rr = st.coverage_runs(**kw)
                assert not rr.ss and len(rr.offsets) == len(gr) + 1
                st.pileup(None, binsize=3, ss=True)
        with pytest.raises(B.BamsignalsError, match="halo"):
            st.coverage((0, 5000), requiredF=66, tspan=True, ss=True)


def test_tile_edges_and_whole_contigs(fixture_bam):
    """Widths around 256, 2048, 4096 and 8192 bases (tiles of 512 to 8192 ints hold half as many bases), on every
    strand, then the whole contigs alone, so that the engine halves its tiles to fill the machine."""
    w = [255, 256, 257, 2047, 2048, 2049, 4095, 4096, 4097, 8191, 8192, 8193, 12289]
    n = len(w)
    strands = (["+"] * n) + (["-"] * n) + (["*"] * n)
    gr = B.GRanges(["chr1"] * 3 * n, [1 + 41 * k for k in range(3 * n)], w * 3, strands)
    for kw in (dict(paired_end="extend"), dict(paired_end="ignore")):
        want = oracle_identity(fixture_bam, gr, **kw)
        same(B.bamCoverage(fixture_bam, gr, ss=True, **kw).as_list(), want)
        check_runs(B.bamCoverage(fixture_bam, gr, ss=True, runs=True, device=DEV, **kw), want)
    names, lens = O.header(fixture_bam)
    gr = B.GRanges(names + names[:1], [1] * (len(names) + 1), lens + lens[:1], ["+", "-", "*", "-"][:len(names) + 1])
    want = oracle_identity(fixture_bam, gr, paired_end="extend")
    got = B.bamCoverage(fixture_bam, gr, ss=True, paired_end="extend")
    assert B.timings()["n_tiles"] > 4
    same(got.as_list(), want)
    check_runs(B.bamCoverage(fixture_bam, gr, ss=True, paired_end="extend", runs=True), want)


def test_device_output_at_every_phase_with_guard_bands(fixture_bam):
    gr = fixture_regions(seed=33)
    want = flat_of(oracle_identity(fixture_bam, gr))
    n = len(want)
    G = 4096
    a = api.core_args("bamCoverage")
    for k in range(4):
        big = torch.full((2 * G + n + 4,), -7, dtype=torch.int32, device=DEV)
        B.coverage_core(fixture_bam, gr, **a, out=big[G + k:G + k + n], ss=True)
        h = big.cpu().numpy()
        assert np.array_equal(h[G + k:G + k + n], want), k
        assert (h[:G + k] == -7).all() and (h[G + k + n:] == -7).all(), k
    with B.Stage(fixture_bam, gr) as st:
        for k in range(4):
            big = torch.full((2 * G + n + 4,), -7, dtype=torch.int32, device=DEV)
            st.coverage(None, out=big[G + k:G + k + n], ss=True)
            h = big.cpu().numpy()
            assert np.array_equal(h[G + k:G + k + n], want), k
            assert (h[:G + k] == -7).all() and (h[G + k + n:] == -7).all(), k


@pytest.mark.parametrize("side_stream", [False, True])
def test_device_output_ordered_after_the_callers_stream(fixture_bam, side_stream):
    gr = fixture_regions(seed=34)
    want = flat_of(oracle_identity(fixture_bam, gr))
    torch.cuda.synchronize()
    s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s):
        buf = torch.empty(len(want), dtype=torch.int32, device=DEV)
        torch.cuda._sleep(int(3e8))                       # ~150 ms of device time
        buf.fill_(-7)
        B.coverage_core(fixture_bam, gr, **api.core_args("bamCoverage"), out=buf, ss=True)
        got = buf.cpu().numpy()
    assert np.array_equal(got, want)


@pytest.fixture(scope="module")
def gen_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("gen"))


@pytest.mark.parametrize("inflate", [-1, 1])
def test_scaled_c3_against_the_unstranded_pair(gen_dir, inflate):
    bam, _ = WL.make_bam("c3", 0.004, gen_dir, unplaced=7)
    gr, kw, _ = WL.regions("c3", 0.004)
    a = api.core_args("bamCoverage", **kw)
    o = B.default_opts(gpu_inflate=inflate)
    want = identity(lambda **x: B.coverage_core(bam, gr, opts=o, **x), gr, a)
    assert sum(int(m[1].sum()) for m in want) > 0 and sum(int(m[0].sum()) for m in want) > 0
    for rp in (0, -1):
        for smi in (0, -1):
            o = B.default_opts(gpu_inflate=inflate, result_pack=rp, stream_min_ints=smi, batch_bytes=1 << 17)
            got = B.bamCoverage(bam, gr, ss=True, opts=o, **kw)
            assert B.timings()["n_tiles"] > len(gr)
            same(got.as_list(), want)
    o = B.default_opts(gpu_inflate=inflate)
    same(B.bamCoverage(bam, gr, ss=True, opts=o, device=DEV, **kw).as_list(), want)
    check_runs(B.bamCoverage(bam, gr, ss=True, opts=o, runs=True, device=DEV, **kw), want)


def test_two_devices(fixture_bam):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    gr = fixture_regions(seed=35)
    wide = B.GRanges(["chr1", "chr2", "chr3"], [1, 1, 1], [30000, 30000, 30000], ["-", "+", "*"])
    for g in (gr, wide):
        one = B.bamCoverage(fixture_bam, g, ss=True, paired_end="extend")
        two = B.bamCoverage(fixture_bam, g, ss=True, paired_end="extend", opts=B.default_opts(devices=[0, 1]))
        assert B.timings()["n_devices"] == 2
        same(two.as_list(), [host(x) for x in one.as_list()])


def _raw_dense(bam, gr, ss, off, opts=None, device_buf=None):
    m = api.marshal_regions(gr)
    args = [bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32), api._p(m.loc, C.c_int32),
            api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8), None, 0, 0, -1, 0, ss, 16385]
    o = None if opts is None else C.byref(opts)
    if device_buf is not None:
        return B.lib().bsg_coverage_ss_device(*args, device_buf.data_ptr(), api._p(off, C.c_int64), None, o)
    out = np.empty(max(int(off[-1]), 1), np.int32)
    return B.lib().bsg_coverage_ss(*args, api._p(out, C.c_int32), api._p(off, C.c_int64), None, o)


def test_refusals(fixture_bam):
    gr = fixture_regions(seed=36)
    plain = api.output_layout(gr.width, 1, False)
    stranded = api.output_layout(gr.width, 1, True)
    buf = torch.empty(int(stranded[-1]), dtype=torch.int32, device=DEV)
    assert _raw_dense(fixture_bam, gr, 1, plain) == EARG
    assert "strand-specific" in B.lib().bsg_last_error().decode()
    assert _raw_dense(fixture_bam, gr, 1, plain, device_buf=buf) == EARG
    assert _raw_dense(fixture_bam, gr, 0, stranded) == EARG                     # ss off wants the plain layout
    assert _raw_dense(fixture_bam, gr, 1, stranded, opts=B.default_opts(devices=[0, 1]), device_buf=buf) == EARG
    assert _raw_dense(fixture_bam, gr, 1, stranded) == 0
    neg = B.GRanges(["chr1"], [0], [10])
    with pytest.raises(B.BamsignalsError, match="position 1"):
        B.bamCoverage(fixture_bam, neg, ss=True)
    with B.Stage(fixture_bam, gr) as st:
        with pytest.raises(B.BamsignalsError, match="out_offsets"):
            api._check(B.lib().bsg_coverage_ss_staged(st._h, None, 0, 0, -1, 0, 1, None, api._p(plain, C.c_int64)))
        h = C.c_void_p()
        assert B.lib().bsg_coverage_runs_ss_staged(st._h, None, 0, 0, -1, 0, 1, None, C.byref(h)) == EARG
        assert B.lib().bsg_coverage_runs_ss_staged(st._h, None, 0, 0, -1, 0, 1, api._p(stranded, C.c_int64), None) == EARG
