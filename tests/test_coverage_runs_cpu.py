"""CPU-only checks of bamCoverage as runs (bsg_coverage_runs, `runs=True`): the entry points exist and refuse bad
arguments and a missing GPU, the Python side validates before the library sees anything, CoverageRuns indexes and
expands hand-built runs, and a numpy restatement of the three kernels (count pass, tile/region scans, write pass with
atomically added lengths) gives exactly the run-length encoding of the dense coverage."""
import ctypes as C

import numpy as np
import pytest

import bamsignals_b200 as B
from bamsignals_b200 import api

EARG, ECUDA = -8, -6
TILE_SIZES = (512, 1024, 2048, 4096, 8192)          # what the engine can choose (prepare_tiles: 8192 halved down to 512)


def no_gpu():
    return B.lib().bsg_device_count() == 0


# ---- the C ABI and the Python surface --------------------------------------------------------------------------------
def test_runs_symbols_exported():
    L = B.lib()
    for s in ("bsg_coverage_runs", "bsg_coverage_runs_staged", "bsg_runs_read", "bsg_runs_free"):
        assert hasattr(L, s)
    assert B.CoverageRuns is api.CoverageRuns and B.coverage_runs_core is api.coverage_runs_core
    assert hasattr(B.Stage, "coverage_runs")


def _call_runs(bam, gr, runs_ptr, opts=None):
    m = api.marshal_regions(gr)
    off = np.zeros(m.R + 1, dtype=np.int64)
    rc = B.lib().bsg_coverage_runs(bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32),
                                   api._p(m.loc, C.c_int32), api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8),
                                   None, 0, 0, -1, 0, 16385, api._p(off, C.c_int64), runs_ptr,
                                   None if opts is None else C.byref(opts))
    return rc


def test_refusals_come_before_the_device(fixture_bam):
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    assert _call_runs(fixture_bam, gr, None) == EARG                                       # runs == NULL
    h = C.c_void_p()
    assert _call_runs(fixture_bam, gr, C.byref(h), B.default_opts(devices=[0, 1])) == EARG  # n_devices > 1
    assert "one device" in B.lib().bsg_last_error().decode()
    assert h.value is None
    off = np.zeros(3, dtype=np.int64)
    assert B.lib().bsg_coverage_runs_staged(None, None, 0, 0, -1, 0, api._p(off, C.c_int64), C.byref(h)) == EARG
    assert B.lib().bsg_coverage_runs_staged(None, None, 0, 0, -1, 0, api._p(off, C.c_int64), None) == EARG
    buf = np.zeros(4, dtype=np.int32)
    assert B.lib().bsg_runs_read(None, buf.ctypes.data, buf.ctypes.data, None) == EARG
    B.lib().bsg_runs_free(None)                                                            # a no-op


def test_runs_need_a_gpu(fixture_bam):
    if not no_gpu():
        pytest.skip("a GPU is present")
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    h = C.c_void_p()
    assert _call_runs(fixture_bam, gr, C.byref(h)) == ECUDA
    assert h.value is None
    for call in (lambda: B.coverage_runs_core(fixture_bam, gr, None),
                 lambda: B.bamCoverage(fixture_bam, gr, runs=True),
                 lambda: B.bamCoverage(fixture_bam, gr, paired_end="extend", runs=True)):
        with pytest.raises(B.BamsignalsError, match="no CUDA device") as e:
            call()
        assert e.value.code == ECUDA


def test_python_validation(fixture_bam):
    gr = B.GRanges(["chr1"], [1], [10])
    with pytest.raises(TypeError):
        B.bamCoverage(fixture_bam, "not a GRanges", runs=True)
    with pytest.raises(ValueError):
        B.bamCoverage(fixture_bam, gr, paired_end="midpoint", runs=True)
    pytest.importorskip("torch")
    with pytest.raises(TypeError, match="CUDA device"):
        B.bamCoverage(fixture_bam, gr, runs=True, device="cpu")
    with pytest.raises(TypeError, match="CUDA device"):
        B.coverage_runs_core(fixture_bam, gr, None, device="cpu")


# ---- CoverageRuns over hand-built arrays -----------------------------------------------------------------------------
def test_coverage_runs_container():
    lengths = np.array([3, 2, 1, 4, 5], np.int32)
    values = np.array([0, 7, 0, 2, 1], np.int32)
    offsets = np.array([0, 2, 2, 4, 5], np.int64)                  # region 1 is zero-width
    r = B.CoverageRuns(lengths, values, offsets)
    assert len(r) == 4
    lr, vr = r[0]
    assert lr.tolist() == [3, 2] and vr.tolist() == [0, 7]
    assert np.shares_memory(lr, lengths) and np.shares_memory(vr, values)       # views, not copies
    assert [len(x) for x in r[1]] == [0, 0]
    assert r[3][0].tolist() == [5] and r[3][1].tolist() == [1]
    with pytest.raises(IndexError):
        r[4]
    with pytest.raises(IndexError):
        r[-1]
    d = r.to_dense()
    assert isinstance(d, B.CountSignals) and len(d) == 4
    want = [[0, 0, 0, 7, 7], [], [0, 2, 2, 2, 2], [1] * 5]
    assert [x.tolist() for x in d.as_list()] == want
    assert d.width().tolist() == [5, 0, 5, 5]
    assert repr(r) == "CoverageRuns object with 4 regions and 5 runs"
    empty = B.CoverageRuns(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(1, np.int64))
    assert len(empty) == 0 and len(empty.to_dense()) == 0
    for bad in (np.array([0, 2, 1, 4, 5]), np.array([1, 2, 2, 4, 5]), np.array([0, 2, 2, 4, 6])):
        with pytest.raises(ValueError):
            B.CoverageRuns(lengths, values, bad)


def test_coverage_runs_container_torch():
    torch = pytest.importorskip("torch")
    r = B.CoverageRuns(torch.tensor([2, 1], dtype=torch.int32), torch.tensor([4, 0], dtype=torch.int32),
                       np.array([0, 0, 2], np.int64))
    d = r.to_dense()
    assert isinstance(d._flat, torch.Tensor)
    assert [x.tolist() for x in d.as_list()] == [[], [4, 4, 0]]


# ---- numpy restatement of the kernels ---------------------------------------------------------------------------------
def tiles_of(widths, strands, tile_ints, order):
    """make_tiles for bamCoverage: regions in `order` (the engine's (chromosome, start) order), each cut into tiles of
    tile_ints bases from its output start; (region, rel, len) per tile.  Zero-width regions have no tiles."""
    out = []
    for i in order:
        for rel in range(0, int(widths[i]), tile_ints):
            out.append((int(i), rel, min(int(widths[i]), rel + tile_ints) - rel))
    return out


def tile_diff(s, e, loc, width, neg, rel, ln):
    """scatter_coverage: the tile's difference array from the reads' inclusive [s, e] (genome coordinates)."""
    tloc = loc + width - rel - ln if neg else loc + rel
    rend = tloc + ln
    keep = (s < rend) & (e >= tloc)
    s, e = s[keep], e[keep]
    up, down = (rend - 1 - e, rend - s) if neg else (s - tloc, e + 1 - tloc)
    d = np.zeros(ln, np.int64)
    np.add.at(d, np.maximum(up, 0), 1)
    inside = down < ln
    np.add.at(d, down[inside], -1)
    return d


def runs_like_the_kernels(reads, locs, widths, strands, tile_ints, order):
    tiles = tiles_of(widths, strands, tile_ints, order)
    T, R = len(tiles), len(widths)
    ds = [tile_diff(*reads[i], locs[i], widths[i], strands[i] < 0, rel, ln) for i, rel, ln in tiles]
    # count pass
    nnz = np.array([np.count_nonzero(d[1:]) for d in ds], np.int64)
    first = np.array([d[0] for d in ds], np.int64)
    last = np.array([d.sum() for d in ds], np.int64)
    reg = np.array([t[0] for t in tiles], np.int64)
    head = np.ones(T, bool)
    head[1:] = reg[1:] != reg[:-1]
    start0 = head.copy()
    start0[1:] |= first[1:] != last[:-1]
    # scans: tiles in tile order, then regions in caller order
    runs = nnz + start0
    toff = np.concatenate([[0], np.cumsum(runs)])
    rfirst, rlast = np.zeros(R, np.int64), np.zeros(R, np.int64)
    for t in range(T):
        if head[t]:
            rfirst[reg[t]] = toff[t]
        if t + 1 == T or reg[t + 1] != reg[t]:
            rlast[reg[t]] = toff[t + 1]
    run_off = np.concatenate([[0], np.cumsum(rlast - rfirst)])
    # write pass: starts write the value, lengths are end - start added up from both ends
    n = int(run_off[-1])
    lengths, values = np.zeros(n, np.int64), np.full(n, -1, np.int64)
    for t, ((i, rel, ln), d) in enumerate(zip(tiles, ds)):
        kbeg, kend = run_off[i], run_off[i + 1]
        k = kbeg + toff[t] - rfirst[i]
        flag = d != 0
        flag[0] = start0[t]
        v = np.cumsum(d)
        for j in np.flatnonzero(flag):
            p = rel + j
            values[k] = v[j]
            lengths[k] -= p
            if k > kbeg:
                lengths[k - 1] += p
            k += 1
        assert k == kbeg + toff[t + 1] - rfirst[i]
        if t + 1 == T or tiles[t + 1][0] != i:
            lengths[kend - 1] += rel + ln
    return lengths, values, run_off


def dense_coverage(s, e, loc, width, neg):
    x = np.arange(loc, loc + width)
    cov = ((s[None, :] <= x[:, None]) & (e[None, :] >= x[:, None])).sum(1) if len(s) else np.zeros(width, np.int64)
    return cov[::-1] if neg else cov


def rle(v):
    if len(v) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    starts = np.concatenate([[0], np.flatnonzero(np.diff(v)) + 1])
    return np.diff(np.concatenate([starts, [len(v)]])), v[starts]


def check(reads, locs, widths, strands, tile_ints, order):
    lengths, values, off = runs_like_the_kernels(reads, locs, widths, strands, tile_ints, order)
    assert off[0] == 0 and (np.diff(off) >= 0).all()
    for i in range(len(widths)):
        lw, vw = rle(dense_coverage(*reads[i], locs[i], widths[i], strands[i] < 0))
        lg, vg = lengths[off[i]:off[i + 1]], values[off[i]:off[i + 1]]
        assert np.array_equal(lg, lw) and np.array_equal(vg, vw), (i, tile_ints)
        assert (lg >= 1).all() and lg.sum() == widths[i]
        assert (vg[1:] != vg[:-1]).all()
    return lengths, values, off


def random_reads(rng, loc, width, n, maxlen):
    s = rng.integers(loc - maxlen, loc + width + maxlen, n)
    return s, s + rng.integers(0, maxlen, n)


@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_random(tile_ints):
    rng = np.random.default_rng(tile_ints)
    widths = np.array([1, 7, tile_ints - 1, tile_ints, tile_ints + 1, 2 * tile_ints, 3 * tile_ints + 1, 0, 5, 0], np.int64)
    strands = np.array([1, -1, 0, -1, 1, 0, -1, 1, 0, -1])
    locs = rng.integers(1000, 50000, len(widths))
    reads = [random_reads(rng, l, w, int(rng.integers(0, 3 * max(w, 1) // 50 + 3)), 300) for l, w in zip(locs, widths)]
    check(reads, locs, widths, strands, tile_ints, rng.permutation(len(widths)))


@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_edges(tile_ints):
    T = tile_ints
    locs = np.array([0, 100, 5000, 5000 + 3 * T, 0], np.int64)
    widths = np.array([5 * T, 3 * T, 3 * T, 2 * T + 1, 0], np.int64)
    strands = np.array([0, 1, -1, 1, -1])
    e0 = np.zeros(0, np.int64)
    reads = [(e0, e0)]                                             # a desert over five tiles: one run of zeros
    p = np.arange(100, 100 + 3 * T)                                 # changes at every base: width runs
    reps = 1 + (np.arange(3 * T) % 3)
    reads.append((np.repeat(p, reps), np.repeat(p, reps)))
    # runs that end exactly at tile boundaries (and start there), '-' orientation
    ends = 5000 + np.array([T - 1, 2 * T - 1, 2 * T])
    reads.append((np.full(3, 5000), ends))
    reads.append((np.array([5000 + 3 * T - 10]), np.array([5000 + 4 * T - 1])))   # touches region 2's end, region 3 starts right there
    reads.append((e0, e0))
    lengths, values, off = check(reads, locs, widths, strands, T, np.array([4, 0, 1, 2, 3]))
    assert off[1] - off[0] == 1 and values[off[0]] == 0 and lengths[off[0]] == 5 * T
    assert off[2] - off[1] == 3 * T
    assert off[4] == off[5]


def test_kernel_restatement_touching_regions_do_not_merge():
    e0 = np.zeros(0, np.int64)
    locs, widths, strands = np.array([0, 600, 1200]), np.array([600, 600, 600]), np.array([1, 1, -1])
    reads = [(e0, e0)] * 3
    lengths, values, off = check(reads, locs, widths, strands, 512, np.arange(3))
    assert off.tolist() == [0, 1, 2, 3] and lengths.tolist() == [600] * 3
