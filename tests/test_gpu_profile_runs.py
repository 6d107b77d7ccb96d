"""bamProfile as runs on the GPU (bsg_profile_runs, `runs=True`): expanded runs equal dense bamProfile element for
element (and the oracle on the reference fixture) with and without ss, the run properties hold, reads land only inside
the caller's slice whatever its 16-byte phase and are ordered after the caller's stream, results can be read many
times, staged sessions interleave dense, device, coverage-runs and profile-runs calls, bsg_shutdown frees a live
result, and the refusals come before any work."""
import ctypes as C
import itertools
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
pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:some ranges' widths")]
LEVELS = ["chr1", "chr2", "chr3"]
DEV = "cuda:0"
EARG = -8


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
    return x.cpu().numpy() if isinstance(x, torch.Tensor) else x


def check_runs(runs, dense, timed=True):
    """runs (ProfileRuns) against a dense bamProfile result (CountSignals): every row of every region equal after
    expansion, and the run properties: lengths >= 1 summing to the bin count, adjacent values different, zero-width
    regions without runs.  timed: the last library call made `runs`, so its timings count 2 x runs output elements."""
    sig = [host(s) for s in dense.as_list()]
    assert len(runs) == len(sig) and runs.ss == dense.ss
    mult = 2 if runs.ss else 1
    off = runs.offsets
    assert off.dtype == np.int64 and len(off) == mult * len(sig) + 1 and off[0] == 0 and (np.diff(off) >= 0).all()
    L, V = host(runs.lengths), host(runs.values)
    assert L.dtype == np.int32 and V.dtype == np.int32 and len(L) == len(V) == off[-1]
    for i, s in enumerate(sig):
        rows = s if runs.ss else [s]
        for a, row in enumerate(rows):
            k = mult * i + a
            lg, vg = L[off[k]:off[k + 1]], V[off[k]:off[k + 1]]
            assert (lg >= 1).all() and int(lg.sum()) == len(row), (i, a)
            assert (vg[1:] != vg[:-1]).all(), (i, a)
            assert np.array_equal(np.repeat(vg, lg), row), (i, a)
    if timed:
        assert B.timings()["out_elems"] == 2 * off[-1]


def assert_only_offsets_over_pcie(runs):
    assert B.timings()["bytes_d2h"] <= 4096 + 8 * len(runs.offsets)


PE = [dict(paired_end="ignore"), dict(paired_end="filter"), dict(paired_end="midpoint", tlenFilter=(50, 300))]
FILTERS = [dict(), dict(mapqual=20, filteredFlag=1024 + 16)]
GRID = [dict(binsize=b, ss=ss, shift=sh, **pe, **fl)
        for b, ss, sh, pe, fl in itertools.product((1, 3, 4, 50), (False, True), (0, 75), PE, FILTERS)]


@pytest.mark.parametrize("kw", GRID, ids=["-".join(f"{k}{v}" for k, v in kw.items()) for kw in GRID])
def test_fixture_against_dense_and_oracle(fixture_bam, kw):
    gr = fixture_regions()
    dense = B.bamProfile(fixture_bam, gr, **kw)
    want = O.bamProfile(fixture_bam, gr, **kw)
    assert all(np.array_equal(a, b) for a, b in zip(dense.as_list(), want.as_list()))
    r = B.bamProfile(fixture_bam, gr, runs=True, **kw)
    assert isinstance(r, B.ProfileRuns) and isinstance(r.lengths, np.ndarray)
    check_runs(r, want)
    assert_only_offsets_over_pcie(r)
    rd = B.bamProfile(fixture_bam, gr, runs=True, device=DEV, **kw)
    assert rd.lengths.is_cuda and rd.values.is_cuda
    check_runs(rd, want)
    assert_only_offsets_over_pcie(rd)
    assert np.array_equal(rd.offsets, r.offsets)
    td = rd.to_dense()
    assert td._flat.is_cuda and td.ss == dense.ss
    assert all(np.array_equal(host(a), b) for a, b in zip(td.as_list(), want.as_list()))
    assert np.array_equal(host(td._flat), dense._flat)
    assert all(np.array_equal(a, b) for a, b in zip(r.to_dense().as_list(), want.as_list()))


@pytest.fixture(scope="module")
def gen_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("gen"))


@pytest.mark.parametrize("inflate", [-1, 1])
@pytest.mark.parametrize("preset", ["c2", "c4"])
def test_scaled_c2_c4(gen_dir, preset, inflate):
    bam, _ = WL.make_bam(preset, 0.004, gen_dir, unplaced=7)
    gr, kw, _ = WL.regions(preset, 0.004)
    o = B.default_opts(gpu_inflate=inflate)
    dense = B.bamProfile(bam, gr, opts=o, **kw)
    r = B.bamProfile(bam, gr, opts=o, runs=True, **kw)
    check_runs(r, dense)
    assert_only_offsets_over_pcie(r)
    if preset == "c4":
        assert B.timings()["n_tiles"] > len(gr)                   # whole contigs: many tiles per region
    o = B.default_opts(gpu_inflate=inflate, batch_bytes=1 << 17, stream_min_ints=1)
    rd = B.bamProfile(bam, gr, opts=o, runs=True, device=DEV, **kw)
    check_runs(rd, dense)
    assert_only_offsets_over_pcie(rd)
    assert np.array_equal(host(rd.to_dense()._flat), dense._flat)


def test_whole_contigs_read_ends(gen_dir):
    """Every contig as one '*' region at binsize 1 with ss: the genome-wide read-end profile, many tiles per list."""
    bam, _ = WL.make_bam("c2", 0.004, gen_dir)
    lens = WL.contig_lens("c2", 0.004)
    gr = B.GRanges.from_codes(WL.NAMES[:len(lens)], np.arange(len(lens)), np.ones(len(lens)), np.asarray(lens),
                              np.zeros(len(lens), np.int8))
    dense = B.bamProfile(bam, gr, ss=True)
    for dev in (None, DEV):
        r = B.bamProfile(bam, gr, ss=True, runs=True, device=dev)
        assert B.timings()["n_tiles"] > 4 * len(gr)
        check_runs(r, dense)
        assert_only_offsets_over_pcie(r)
        assert int(r.offsets[-1]) < len(dense._flat) // 4            # sparse: far fewer runs than bins


def test_region_tiles_of_every_size(fixture_bam):
    """Widths around the tile sizes the engine picks (512..8192 ints) and multiples of them, on both strands, with and
    without ss (a strand-specific tile holds half the bins)."""
    w = [511, 512, 513, 1024, 4096, 8191, 8192, 8193, 16384, 24577]
    gr = B.GRanges(["chr1"] * len(w) * 2, [1 + 37 * k for k in range(len(w) * 2)], w * 2, ["+"] * len(w) + ["-"] * len(w))
    for ss in (False, True):
        dense = B.bamProfile(fixture_bam, gr, ss=ss)
        check_runs(B.bamProfile(fixture_bam, gr, ss=ss, runs=True, device=DEV), dense)


def _raw_runs(bam, gr, binsize=1, ss=True, opts=None):
    m = api.marshal_regions(gr)
    off = np.zeros((2 if ss else 1) * m.R + 1, dtype=np.int64)
    h = C.c_void_p()
    rc = B.lib().bsg_profile_runs(bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32),
                                  api._p(m.loc, C.c_int32), api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8),
                                  None, 0, binsize, 75, int(ss), 0, -1, 0, 16385, api._p(off, C.c_int64), C.byref(h),
                                  None if opts is None else C.byref(opts))
    return rc, h, off


def test_reads_at_every_phase_with_guard_bands(fixture_bam):
    gr = fixture_regions(seed=32)
    rc, h, off = _raw_runs(fixture_bam, gr)
    assert rc == 0
    try:
        n = int(off[-1])
        L, V = np.empty(n, np.int32), np.empty(n, np.int32)
        assert B.lib().bsg_runs_read(h, L.ctypes.data, V.ctypes.data, None) == 0
        G = 4096
        for k in range(4):
            bl = torch.full((2 * G + n + 4,), -7, dtype=torch.int32, device=DEV)
            bv = torch.full((2 * G + n + 4,), -9, dtype=torch.int32, device=DEV)
            for rep in range(2):                                                  # repeated reads of one result
                assert B.lib().bsg_runs_read(h, bl[G + k:].data_ptr(), bv[G + k:].data_ptr(), None) == 0
                hl, hv = bl.cpu().numpy(), bv.cpu().numpy()
                assert np.array_equal(hl[G + k:G + k + n], L) and np.array_equal(hv[G + k:G + k + n], V), (k, rep)
                assert (hl[:G + k] == -7).all() and (hl[G + k + n:] == -7).all()
                assert (hv[:G + k] == -9).all() and (hv[G + k + n:] == -9).all()
            assert B.lib().bsg_runs_read(h, bl[G + k:].data_ptr() + 2, bv[G + k:].data_ptr(), None) == EARG
            assert "aligned" in B.lib().bsg_last_error().decode()
        L2, V2 = np.empty(n, np.int32), np.empty(n, np.int32)
        assert B.lib().bsg_runs_read(h, L2.ctypes.data, V2.ctypes.data, None) == 0
        assert np.array_equal(L, L2) and np.array_equal(V, V2)
        check_runs(B.ProfileRuns(L, V, off, ss=True), B.bamProfile(fixture_bam, gr, ss=True, shift=75), timed=False)
    finally:
        B.lib().bsg_runs_free(h)


@pytest.mark.parametrize("side_stream", [False, True])
def test_read_ordered_after_the_callers_stream(fixture_bam, side_stream):
    gr = fixture_regions(seed=33)
    want = B.bamProfile(fixture_bam, gr, ss=True, shift=75, runs=True)
    torch.cuda.synchronize()
    s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s):
        rc, h, off = _raw_runs(fixture_bam, gr)
        assert rc == 0 and np.array_equal(off, want.offsets)
        n = int(off[-1])
        bl = torch.empty(n, dtype=torch.int32, device=DEV)
        bv = torch.empty(n, dtype=torch.int32, device=DEV)
        torch.cuda._sleep(int(3e8))                       # ~150 ms of device time
        bl.fill_(-7)
        bv.fill_(-7)
        assert B.lib().bsg_runs_read(h, bl.data_ptr(), bv.data_ptr(), s.cuda_stream) == 0
        B.lib().bsg_runs_free(h)
        hl, hv = bl.cpu().numpy(), bv.cpu().numpy()
    assert np.array_equal(hl, want.lengths) and np.array_equal(hv, want.values)


def test_staged_session_interleaves_dense_device_and_runs(fixture_bam):
    gr = fixture_regions(seed=34)
    settings = [dict(tlen_filter=None, binsize=1, ss=True, shift=75),
                dict(tlen_filter=(0, 1000), binsize=4, ss=False, requiredF=66, pe_mid=True),
                dict(tlen_filter=(50, 300), binsize=3, ss=True, requiredF=66, mapqual=10)]
    want = [B.pileup_core(fixture_bam, gr, **kw) for kw in settings]
    cov_want = B.bamCoverage(fixture_bam, gr)
    with B.Stage(fixture_bam, gr, ext_hint=1000) as st:
        for _ in range(2):
            for kw, w in zip(settings, want):
                dense = B.CountSignals(w, kw["ss"])
                flat = np.concatenate([x.ravel(order="F") for x in w])
                check_runs(st.profile_runs(**kw), dense)
                assert np.array_equal(st.pileup(**kw), flat)
                off = api.output_layout(gr.width, kw["binsize"], kw["ss"])
                buf = torch.empty(int(off[-1]), dtype=torch.int32, device=DEV)
                st.pileup(**kw, out=buf)
                assert np.array_equal(buf.cpu().numpy(), flat)
                rd = st.profile_runs(**kw, device=DEV)
                check_runs(rd, dense)
                cr = st.coverage_runs(None)
                assert all(np.array_equal(host(a), b) for a, b in zip(cr.to_dense().as_list(), cov_want.as_list()))
        with pytest.raises(B.BamsignalsError, match="halo"):
            st.profile_runs(None, shift=5000)
        with pytest.raises(B.BamsignalsError, match="binsize"):
            st.profile_runs(None, binsize=0)


def test_shutdown_frees_a_live_result(fixture_bam):
    gr = fixture_regions(seed=35)
    rc, h, off = _raw_runs(fixture_bam, gr)
    assert rc == 0 and off[-1] > 0
    st = B.Stage(fixture_bam, gr, ext_hint=75)
    hs = C.c_void_p()
    off2 = np.zeros(2 * len(gr) + 1, np.int64)
    assert B.lib().bsg_profile_runs_staged(st._h, None, 0, 1, 75, 1, 0, -1, 0, api._p(off2, C.c_int64), C.byref(hs)) == 0
    assert np.array_equal(off, off2)
    B.lib().bsg_shutdown()
    L = np.empty(int(off[-1]), np.int32)
    for x in (h, hs):
        assert B.lib().bsg_runs_read(x, L.ctypes.data, L.ctypes.data, None) == EARG
        assert "bsg_shutdown" in B.lib().bsg_last_error().decode()
        B.lib().bsg_runs_free(x)
    st.close()
    dense = B.bamProfile(fixture_bam, gr, ss=True, shift=75)
    check_runs(B.bamProfile(fixture_bam, gr, ss=True, shift=75, runs=True), dense)            # the library works on


def test_refusals(fixture_bam):
    gr = fixture_regions(seed=36)
    rc, h, _ = _raw_runs(fixture_bam, gr, opts=B.default_opts(devices=[0, 1]))
    assert rc == EARG and h.value is None
    rc, h, _ = _raw_runs(fixture_bam, gr, binsize=0)
    assert rc == EARG and h.value is None and "binsize" in B.lib().bsg_last_error().decode()
    m = api.marshal_regions(gr)
    off = np.zeros(2 * m.R + 1, dtype=np.int64)
    args = (fixture_bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32), api._p(m.loc, C.c_int32),
            api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8))
    hh = C.c_void_p()
    assert B.lib().bsg_profile_runs(*args, None, 0, 1, 0, 1, 0, -1, 0, 16385, api._p(off, C.c_int64), None, None) == EARG
    assert B.lib().bsg_profile_runs(*args, None, 0, 1, 0, 1, 0, -1, 0, 16385, None, C.byref(hh), None) == EARG
    assert B.lib().bsg_profile_runs(*args, None, 0, 1, 0, 1, 0, -1, 1, 16385, api._p(off, C.c_int64), C.byref(hh), None) == EARG
    assert hh.value is None
    rc, h, off = _raw_runs(fixture_bam, gr)
    assert rc == 0
    try:
        n = int(off[-1])
        ok = torch.empty(n, dtype=torch.int32, device=DEV)
        assert B.lib().bsg_runs_read(h, None, ok.data_ptr(), None) == EARG
        if torch.cuda.device_count() > 1:
            other = torch.empty(n, dtype=torch.int32, device="cuda:1")
            assert B.lib().bsg_runs_read(h, other.data_ptr(), ok.data_ptr(), None) == EARG
    finally:
        B.lib().bsg_runs_free(h)
