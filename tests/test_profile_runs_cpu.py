"""CPU-only checks of bamProfile as runs (bsg_profile_runs, `runs=True`): the entry points exist and refuse bad arguments
and a missing GPU, the Python side validates before the library sees anything, ProfileRuns indexes and expands
hand-built runs (with and without ss, over numpy and CPU torch), and a numpy restatement of the kernels (per-tile
histogram, virtual-tile order, count pass, tile/list scans, write pass with atomically added lengths) gives exactly the
run-length encoding of the dense profile."""
import ctypes as C

import numpy as np
import pytest

import bamsignals_b200 as B
from bamsignals_b200 import api

EARG, ECUDA = -8, -6
TILE_SIZES = (512, 1024, 2048, 4096, 8192)          # what the engine can choose (prepare_tiles: 8192 halved down to 512)
BINSIZES = (1, 3, 4, 7, 200)


def no_gpu():
    return B.lib().bsg_device_count() == 0


# ---- the C ABI and the Python surface --------------------------------------------------------------------------------
def test_profile_runs_symbols_exported():
    L = B.lib()
    for s in ("bsg_profile_runs", "bsg_profile_runs_staged", "bsg_runs_read", "bsg_runs_free"):
        assert hasattr(L, s)
    assert B.ProfileRuns is api.ProfileRuns and B.profile_runs_core is api.profile_runs_core
    assert hasattr(B.Stage, "profile_runs")


def _call(bam, gr, runs_ptr, opts=None, binsize=1, ss=0, tlen=None, pe_mid=0, offsets=True):
    m = api.marshal_regions(gr)
    off = np.zeros((2 if ss else 1) * m.R + 1, dtype=np.int64)
    tl = None if tlen is None else np.asarray(tlen, np.int32)
    return B.lib().bsg_profile_runs(bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32),
                                    api._p(m.loc, C.c_int32), api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8),
                                    None if tl is None else api._p(tl, C.c_int32), 0, binsize, 0, ss, 0, -1, pe_mid, 16385,
                                    api._p(off, C.c_int64) if offsets else None, runs_ptr,
                                    None if opts is None else C.byref(opts))


def test_refusals_come_before_the_device(fixture_bam):
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    assert _call(fixture_bam, gr, None) == EARG                                            # runs == NULL
    h = C.c_void_p()
    assert _call(fixture_bam, gr, C.byref(h), B.default_opts(devices=[0, 1])) == EARG     # n_devices > 1
    assert "one device" in B.lib().bsg_last_error().decode()
    assert _call(fixture_bam, gr, C.byref(h), offsets=False) == EARG                       # run_offsets == NULL
    assert "run_offsets" in B.lib().bsg_last_error().decode()
    for bs in (0, -1):                                                                      # bamCount has no runs form
        assert _call(fixture_bam, gr, C.byref(h), binsize=bs) == EARG
        assert "binsize" in B.lib().bsg_last_error().decode()
    assert _call(fixture_bam, gr, C.byref(h), pe_mid=1) == EARG                            # midpoint without tlen_filter
    assert "tlen_filter" in B.lib().bsg_last_error().decode()
    assert h.value is None
    off = np.zeros(5, dtype=np.int64)
    staged = B.lib().bsg_profile_runs_staged
    assert staged(None, None, 0, 1, 0, 1, 0, -1, 0, api._p(off, C.c_int64), C.byref(h)) == EARG
    assert staged(None, None, 0, 1, 0, 1, 0, -1, 0, api._p(off, C.c_int64), None) == EARG
    assert h.value is None


def test_profile_runs_need_a_gpu(fixture_bam):
    if not no_gpu():
        pytest.skip("a GPU is present")
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    h = C.c_void_p()
    for ss in (0, 1):
        assert _call(fixture_bam, gr, C.byref(h), binsize=3, ss=ss) == ECUDA
        assert h.value is None
    for call in (lambda: B.profile_runs_core(fixture_bam, gr, None),
                 lambda: B.bamProfile(fixture_bam, gr, runs=True),
                 lambda: B.bamProfile(fixture_bam, gr, binsize=5, ss=True, shift=75, paired_end="midpoint", runs=True)):
        with pytest.raises(B.BamsignalsError, match="no CUDA device") as e:
            call()
        assert e.value.code == ECUDA


def test_python_validation(fixture_bam):
    gr = B.GRanges(["chr1"], [1], [10])
    with pytest.raises(TypeError):
        B.bamProfile(fixture_bam, "not a GRanges", runs=True)
    with pytest.raises(ValueError, match="binsize"):
        B.bamProfile(fixture_bam, gr, binsize=0, runs=True)
    with pytest.raises(ValueError):
        B.bamProfile(fixture_bam, gr, paired_end="extend", runs=True)
    with pytest.raises(ValueError, match="tlenFilter"):
        B.bamProfile(fixture_bam, gr, paired_end="midpoint", tlenFilter=(300, 50), runs=True)
    with pytest.warns(UserWarning, match="multiple of the selected binsize"):               # width 10, binsize 3
        try:
            B.bamProfile(fixture_bam, gr, binsize=3, runs=True)
        except B.BamsignalsError:
            assert no_gpu()
    pytest.importorskip("torch")
    with pytest.raises(TypeError, match="CUDA device"):
        B.bamProfile(fixture_bam, gr, runs=True, device="cpu")
    with pytest.raises(TypeError, match="CUDA device"):
        B.profile_runs_core(fixture_bam, gr, None, device="cpu")


# ---- ProfileRuns over hand-built arrays ------------------------------------------------------------------------------
def test_profile_runs_container():
    lengths = np.array([3, 2, 1, 4, 5], np.int32)
    values = np.array([0, 7, 0, 2, 1], np.int32)
    offsets = np.array([0, 2, 2, 4, 5], np.int64)                  # region 1 is zero-width
    r = B.ProfileRuns(lengths, values, offsets, ss=False)
    assert len(r) == 4
    lr, vr = r[0]
    assert lr.tolist() == [3, 2] and vr.tolist() == [0, 7]
    assert np.shares_memory(lr, lengths) and np.shares_memory(vr, values)       # views, not copies
    assert [len(x) for x in r[1]] == [0, 0]
    with pytest.raises(IndexError):
        r[4]
    with pytest.raises(IndexError):
        r[-1]
    with pytest.raises(TypeError):
        r[0:2]
    d = r.to_dense()
    assert isinstance(d, B.CountSignals) and not d.ss
    assert [x.tolist() for x in d.as_list()] == [[0, 0, 0, 7, 7], [], [0, 2, 2, 2, 2], [1] * 5]
    assert repr(r) == "ProfileRuns object with 4 strand-unspecific regions and 5 runs"
    for bad in (np.array([0, 2, 1, 4, 5]), np.array([1, 2, 2, 4, 5]), np.array([0, 2, 2, 4, 6])):
        with pytest.raises(ValueError):
            B.ProfileRuns(lengths, values, bad, ss=False)


def ss_example():
    # region 0: sense [1, 1, 0], antisense [0, 2, 2]; region 1: zero-width; region 2: sense [5, 5], antisense [0, 0]
    lengths = np.array([2, 1, 1, 2, 2, 2], np.int32)
    values = np.array([1, 0, 0, 2, 5, 0], np.int32)
    offsets = np.array([0, 2, 4, 4, 4, 5, 6], np.int64)
    dense = [[[1, 1, 0], [0, 2, 2]], np.zeros((2, 0), np.int32).tolist(), [[5, 5], [0, 0]]]
    return lengths, values, offsets, dense


def test_profile_runs_container_ss():
    lengths, values, offsets, dense = ss_example()
    r = B.ProfileRuns(lengths, values, offsets, ss=True)
    assert len(r) == 3 and r.ss
    (ls, vs), (la, va) = r[0]
    assert ls.tolist() == [2, 1] and vs.tolist() == [1, 0] and la.tolist() == [1, 2] and va.tolist() == [0, 2]
    assert all(len(x) == 0 for row in r[1] for x in row)
    d = r.to_dense()
    assert d.ss and len(d) == 3 and d.width().tolist() == [3, 0, 2]
    assert [x.tolist() for x in d.as_list()] == dense
    assert d._flat.tolist() == [1, 0, 1, 2, 0, 2, 5, 0, 5, 0]                 # interleaved like bsg_pileup's layout
    assert repr(r) == "ProfileRuns object with 3 strand-specific regions and 6 runs"
    with pytest.raises(ValueError, match="2R"):
        B.ProfileRuns(lengths[:5], values[:5], offsets[:6], ss=True)
    with pytest.raises(ValueError, match="same number of bins"):             # region 0's rows differ in width
        B.ProfileRuns(np.array([2, 1, 1, 3], np.int32), np.array([1, 0, 0, 2], np.int32),
                      np.array([0, 2, 4], np.int64), ss=True).to_dense()
    empty = B.ProfileRuns(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(1, np.int64), ss=True)
    assert len(empty) == 0 and len(empty.to_dense()) == 0


def test_profile_runs_container_torch():
    torch = pytest.importorskip("torch")
    lengths, values, offsets, dense = ss_example()
    r = B.ProfileRuns(torch.from_numpy(lengths), torch.from_numpy(values), offsets, ss=True)
    d = r.to_dense()
    assert isinstance(d._flat, torch.Tensor)
    assert [x.tolist() for x in d.as_list()] == dense
    r1 = B.ProfileRuns(torch.tensor([2, 1], dtype=torch.int32), torch.tensor([4, 0], dtype=torch.int32),
                       np.array([0, 0, 2], np.int64), ss=False)
    assert [x.tolist() for x in r1.to_dense().as_list()] == [[], [4, 4, 0]]
    same = B.ProfileRuns(torch.tensor([2, 1, 3], dtype=torch.int32), torch.tensor([1, 0, 6], dtype=torch.int32),
                         np.array([0, 2, 3], np.int64), ss=True).to_dense()
    assert same.alignSignals().tolist() == [[[1], [1], [0]], [[6], [6], [6]]]


# ---- numpy restatement of the kernels ---------------------------------------------------------------------------------
def tiles_of(widths, strands, binsize, mult, tile_ints, order):
    """make_tiles for bamProfile: regions in `order` (the engine's (chromosome, start) order), each cut into tiles of
    tile_ints // mult bins from its 5' end; (region, rel_bin, rel_bp, len_bp) per tile.  Zero-width regions have none."""
    tb = max(1, tile_ints // mult)
    out = []
    for i in order:
        w = int(widths[i])
        nb = -(-w // binsize)
        for k in range(0, nb, tb):
            lo, hi = k * binsize, min(w, (k + tb) * binsize)
            out.append((int(i), k, lo, hi - lo))
    return out


def tile_hist(p5, ng, loc, width, strand, rel_bp, ln, binsize, ss):
    """scatter_profile / scatter_profile_agg: the tile's histogram from the reads' 5' ends and strand bits."""
    flip = 1 if strand < 0 else 0
    tloc = loc + width - rel_bp - ln if flip else loc + rel_bp
    rel = p5 - tloc
    keep = (ng >= 0) & (rel >= 0) & (rel < ln)
    rel, a = rel[keep], (ng[keep] ^ flip) & 1
    if flip:
        rel = ln - 1 - rel
    nb = -(-ln // binsize)
    h = np.zeros((nb, 2 if ss else 1), np.int64)
    np.add.at(h, (rel // binsize, a if ss else 0), 1)
    return h                                                        # h[j, a] = hist[mult * j + a]


def runs_like_the_kernels(reads, locs, widths, strands, binsize, ss, tile_ints, order):
    mult = 2 if ss else 1
    tiles = tiles_of(widths, strands, binsize, mult, tile_ints, order)
    T, R = len(tiles), len(widths)
    L, NV = mult * R, mult * T
    hs = [tile_hist(*reads[i], locs[i], widths[i], strands[i], rel_bp, ln, binsize, ss) for i, _, rel_bp, ln in tiles]
    # virtual tiles: row a of the j-th of region i's n_i tiles, T_i its first, is v = mult T_i + a n_i + j, list mult i + a
    vlist, vrel, vhist = np.zeros(NV, np.int64), np.zeros(NV, np.int64), [None] * NV
    t = 0
    while t < T:
        i = tiles[t][0]
        n_i = next((k for k in range(t, T) if tiles[k][0] != i), T) - t
        for j in range(n_i):
            for a in range(mult):
                v = mult * t + a * n_i + j
                vlist[v], vrel[v], vhist[v] = mult * i + a, tiles[t + j][1], hs[t + j][:, a]
        t += n_i
    assert all(h is not None for h in vhist)
    # count pass
    nnz = np.array([np.count_nonzero(h[1:] != h[:-1]) for h in vhist], np.int64)
    first = np.array([h[0] for h in vhist], np.int64)
    last = np.array([h[-1] for h in vhist], np.int64)
    head = np.ones(NV, bool)
    head[1:] = vlist[1:] != vlist[:-1]
    start0 = head.copy()
    start0[1:] |= first[1:] != last[:-1]
    # k_runs_scan over the virtual tiles, then over the lists in caller order
    runs = nnz + start0
    toff = np.concatenate([[0], np.cumsum(runs)])
    rfirst, rlast = np.zeros(L, np.int64), np.zeros(L, np.int64)
    for v in range(NV):
        if head[v]:
            rfirst[vlist[v]] = toff[v]
        if v + 1 == NV or vlist[v + 1] != vlist[v]:
            rlast[vlist[v]] = toff[v + 1]
    run_off = np.concatenate([[0], np.cumsum(rlast - rfirst)])
    # write pass: every run start writes its bin's value; lengths are end - start added up from both ends
    n = int(run_off[-1])
    lengths, values = np.zeros(n, np.int64), np.full(n, -1, np.int64)
    for v in range(NV):
        lst, h = vlist[v], vhist[v]
        kbeg, kend = run_off[lst], run_off[lst + 1]
        flag = np.concatenate([[start0[v]], h[1:] != h[:-1]])
        j = np.flatnonzero(flag)
        k = kbeg + toff[v] - rfirst[lst] + np.arange(len(j))
        assert len(j) == runs[v]
        p = vrel[v] + j
        values[k] = h[j]
        np.add.at(lengths, k, -p)
        np.add.at(lengths, k[k > kbeg] - 1, p[k > kbeg])
        if v + 1 == NV or vlist[v + 1] != lst:
            lengths[kend - 1] += vrel[v] + len(h)
    return lengths, values, run_off


def dense_profile(p5, ng, loc, width, strand, binsize, ss):
    """bsg_pileup's slice of one region, straight from the reads (src/bamsignals.cpp:349-363)."""
    flip = 1 if strand < 0 else 0
    rel = p5 - loc
    keep = (ng >= 0) & (rel >= 0) & (rel < width)
    rel, a = rel[keep], (ng[keep] ^ flip) & 1
    if flip:
        rel = width - 1 - rel
    mult = 2 if ss else 1
    out = np.zeros(mult * (-(-int(width) // binsize)), np.int64)
    np.add.at(out, mult * (rel // binsize) + (a if ss else 0), 1)
    return out


def rle(v):
    if len(v) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    starts = np.concatenate([[0], np.flatnonzero(np.diff(v)) + 1])
    return np.diff(np.concatenate([starts, [len(v)]])), v[starts]


def check(reads, locs, widths, strands, binsize, ss, tile_ints, order):
    lengths, values, off = runs_like_the_kernels(reads, locs, widths, strands, binsize, ss, tile_ints, order)
    mult = 2 if ss else 1
    assert len(off) == mult * len(widths) + 1 and off[0] == 0 and (np.diff(off) >= 0).all()
    for i in range(len(widths)):
        dense = dense_profile(*reads[i], locs[i], widths[i], strands[i], binsize, ss)
        for a in range(mult):
            lst = mult * i + a
            lw, vw = rle(dense[a::mult])
            lg, vg = lengths[off[lst]:off[lst + 1]], values[off[lst]:off[lst + 1]]
            assert np.array_equal(lg, lw) and np.array_equal(vg, vw), (i, a, binsize, ss, tile_ints)
            assert (lg >= 1).all() and lg.sum() == -(-int(widths[i]) // binsize)
            assert (vg[1:] != vg[:-1]).all()
    return lengths, values, off


def random_reads(rng, loc, width, n, halo=300):
    p5 = rng.integers(loc - halo, loc + width + halo, n)
    ng = rng.integers(-1, 2, n)                                      # -1: a dropped read (k_decode's ng < 0)
    return p5, ng


@pytest.mark.parametrize("ss", [False, True], ids=["ss0", "ss1"])
@pytest.mark.parametrize("binsize", BINSIZES)
@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_random(tile_ints, binsize, ss):
    rng = np.random.default_rng(tile_ints * 1000 + binsize * 2 + ss)
    tb = max(1, tile_ints // (2 if ss else 1)) * binsize               # bases per tile
    widths = np.array([1, 7, tb - 1, tb, tb + 1, 2 * tb, 3 * tb + binsize // 2 + 1, 0, 5, 0], np.int64)
    strands = np.array([1, -1, 0, -1, 1, 0, -1, 1, 0, -1])
    locs = rng.integers(1000, 50000, len(widths))
    # a few reads per bin in some regions, sparse in others
    dens = rng.choice([0.02, 0.3, 2.0], len(widths))
    reads = [random_reads(rng, l, w, int(dens[k] * (w // binsize + 1)) + 1) for k, (l, w) in enumerate(zip(locs, widths))]
    check(reads, locs, widths, strands, binsize, ss, tile_ints, rng.permutation(len(widths)))


@pytest.mark.parametrize("ss", [False, True], ids=["ss0", "ss1"])
@pytest.mark.parametrize("binsize", BINSIZES)
@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_edges(tile_ints, binsize, ss):
    mult = 2 if ss else 1
    tb = max(1, tile_ints // mult)                                  # bins per tile
    B_ = tb * binsize                                               # bases per tile
    locs = np.array([0, 100, 5000, 5000 + 3 * B_, 0, 100, 9 * B_], np.int64)
    widths = np.array([5 * B_, 3 * B_, 3 * B_, 2 * B_ + 1, 0, 3 * B_, 2 * B_ - 1], np.int64)
    strands = np.array([0, 1, -1, 1, -1, 1, -1])
    e0 = np.zeros(0, np.int64)
    reads = [(e0, e0)]                                              # a desert over five tiles: one run of zeros per row
    # a change at every bin (0, 1 or 2 reads per bin, both strands)
    bins = np.arange(3 * tb)
    reps = bins % 3
    p5 = 100 + np.repeat(bins * binsize, reps)
    reads.append((p5, np.repeat(bins % 2, reps)))
    # one read in the first and the last bin of every tile ('-' orientation: counted from the region's end), so that the
    # runs change exactly on tile boundaries
    edge = np.concatenate([[k * tb, k * tb + tb - 1] for k in range(3)])
    reads.append((5000 + 3 * B_ - 1 - edge * binsize, np.zeros(len(edge), np.int64)))
    reads.append((np.array([5000 + 3 * B_]), np.array([1])))          # region 3 starts right where region 2 ends
    reads.append((e0, e0))
    reads.append(reads[1])                                          # region 5 duplicates region 1
    reads.append(random_reads(np.random.default_rng(7), 9 * B_, 2 * B_ - 1, 40))
    lengths, values, off = check(reads, locs, widths, strands, binsize, ss, tile_ints, np.array([4, 0, 1, 5, 2, 3, 6]))
    nb = lambda i: -(-int(widths[i]) // binsize)                   # noqa: E731
    for a in range(mult):
        assert off[a + 1] - off[a] == 1 and values[off[a]] == 0 and lengths[off[a]] == nb(0)
        assert off[mult * 4 + a] == off[mult * 4 + a + 1]                                  # zero width: no runs
    assert np.array_equal(values[off[mult]:off[2 * mult]], values[off[5 * mult]:off[6 * mult]])   # duplicates agree
    if not ss:
        assert off[2] - off[1] == 3 * tb - 1 + 1 and (values[off[1]:off[2]] == np.arange(3 * tb) % 3).all()


@pytest.mark.parametrize("ss", [False, True], ids=["ss0", "ss1"])
def test_kernel_restatement_touching_regions_do_not_merge(ss):
    e0 = np.zeros(0, np.int64)
    locs, widths, strands = np.array([0, 600, 1200, 1200]), np.array([600, 600, 600, 600]), np.array([1, 1, -1, -1])
    lengths, values, off = check([(e0, e0)] * 4, locs, widths, strands, 4, ss, 512, np.arange(4))
    mult = 2 if ss else 1
    assert off.tolist() == list(range(4 * mult + 1)) and lengths.tolist() == [150] * (4 * mult)
