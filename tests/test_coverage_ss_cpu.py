"""CPU-only checks of strand-specific bamCoverage (bsg_coverage_ss*, `ss=True`): the six entry points exist, refuse bad
arguments before any device work and need a GPU, the Python side validates, CoverageRuns with ss indexes and expands
hand-built runs, a numpy restatement of stranded coverage from the fixture's reads satisfies the identity with the CPU
oracle's unstranded coverage (requiredF and requiredF | 16), and a numpy restatement of the interleaved tile scatter and
scan (k_coverage_ss) and of the count, scan and write passes of stranded runs (k_runs_count_ss, k_runs_scan,
k_runs_write_ss) gives exactly the dense result and its np.diff run-length encoding."""
import ctypes as C

import numpy as np
import pytest

import bamsignals_b200 as B
import oracle_api as O
from bamsignals_b200 import api

EARG, ECUDA = -8, -6
TILE_SIZES = (512, 1024, 2048, 4096, 8192)          # ints per tile the engine can choose: half as many bases with ss
ENTRY_POINTS = ("bsg_coverage_ss", "bsg_coverage_ss_device", "bsg_coverage_ss_staged", "bsg_coverage_ss_staged_device",
                "bsg_coverage_runs_ss", "bsg_coverage_runs_ss_staged")
COVERAGE_KW = [dict(paired_end="ignore"), dict(paired_end="extend"), dict(paired_end="extend", tlenFilter=(50, 300)),
               dict(paired_end="ignore", mapqual=20), dict(paired_end="ignore", filteredFlag=1024 + 16),
               dict(paired_end="extend", tlenFilter=(0, 250), mapqual=10, filteredFlag=256)]


def no_gpu():
    return B.lib().bsg_device_count() == 0


def test_entry_points_exported():
    L = B.lib()
    for s in ENTRY_POINTS:
        assert hasattr(L, s), s


def _region_args(bam, gr):
    m = api.marshal_regions(gr)
    return m, [bam.encode(), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32), api._p(m.loc, C.c_int32),
               api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8), None, 0, 0, -1, 0]


def _dense(bam, gr, ss, off, opts=None):
    _, args = _region_args(bam, gr)
    out = np.empty(max(int(off[-1]), 1), np.int32)
    return B.lib().bsg_coverage_ss(*args, ss, 16385, api._p(out, C.c_int32), api._p(off, C.c_int64), None,
                                   None if opts is None else C.byref(opts))


def _device(bam, gr, ss, off, ptr, opts=None):
    _, args = _region_args(bam, gr)
    return B.lib().bsg_coverage_ss_device(*args, ss, 16385, ptr, api._p(off, C.c_int64), None,
                                          None if opts is None else C.byref(opts))


def _runs(bam, gr, ss, off, runs_ptr, opts=None):
    _, args = _region_args(bam, gr)
    return B.lib().bsg_coverage_runs_ss(*args, ss, 16385, None if off is None else api._p(off, C.c_int64), runs_ptr,
                                        None if opts is None else C.byref(opts))


def test_refusals_come_before_the_device(fixture_bam):
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    plain = api.output_layout(gr.width, 1, False)
    assert _dense(fixture_bam, gr, 1, plain) == EARG                                       # the unstranded layout
    assert "strand-specific" in B.lib().bsg_last_error().decode()
    assert _device(fixture_bam, gr, 1, plain, 64) == EARG
    h = C.c_void_p()
    off = np.zeros(2 * len(gr) + 1, np.int64)
    assert _runs(fixture_bam, gr, 1, off, C.byref(h), B.default_opts(devices=[0, 1])) == EARG   # n_devices > 1
    assert "one device" in B.lib().bsg_last_error().decode()
    assert _runs(fixture_bam, gr, 1, off, None) == EARG                                    # runs == NULL
    assert _runs(fixture_bam, gr, 1, None, C.byref(h)) == EARG                              # run_offsets == NULL
    assert h.value is None
    po = api._p(off, C.c_int64)
    assert B.lib().bsg_coverage_ss_staged(None, None, 0, 0, -1, 0, 1, None, po) == EARG
    assert B.lib().bsg_coverage_ss_staged_device(None, None, 0, 0, -1, 0, 1, None, po, None) == EARG
    assert B.lib().bsg_coverage_runs_ss_staged(None, None, 0, 0, -1, 0, 1, po, C.byref(h)) == EARG
    assert B.lib().bsg_coverage_runs_ss_staged(None, None, 0, 0, -1, 0, 1, po, None) == EARG


def test_calls_need_a_gpu(fixture_bam):
    if not no_gpu():
        pytest.skip("a GPU is present")
    gr = B.GRanges(["chr1", "chr2"], [1, 100], [10, 20], ["+", "-"])
    off = api.output_layout(gr.width, 1, True)
    assert _dense(fixture_bam, gr, 1, off) == ECUDA
    assert _device(fixture_bam, gr, 1, off, 64) == ECUDA
    h = C.c_void_p()
    assert _runs(fixture_bam, gr, 1, np.zeros(5, np.int64), C.byref(h)) == ECUDA and h.value is None
    for call in (lambda: B.bamCoverage(fixture_bam, gr, ss=True), lambda: B.bamCoverage(fixture_bam, gr, ss=True, runs=True),
                 lambda: B.coverage_core(fixture_bam, gr, None, ss=True),
                 lambda: B.coverage_runs_core(fixture_bam, gr, (0, 500), requiredF=66, tspan=True, ss=True)):
        with pytest.raises(B.BamsignalsError, match="no CUDA device") as e:
            call()
        assert e.value.code == ECUDA


def test_python_validation(fixture_bam):
    gr = B.GRanges(["chr1"], [1], [10])
    with pytest.raises(TypeError):
        B.bamCoverage(fixture_bam, "not a GRanges", ss=True)
    with pytest.raises(ValueError):
        B.bamCoverage(fixture_bam, gr, paired_end="midpoint", ss=True)
    assert api.output_layout(np.array([3, 0, 5]), 1, True).tolist() == [0, 6, 6, 16]
    pytest.importorskip("torch")
    with pytest.raises(TypeError, match="CUDA device"):
        B.bamCoverage(fixture_bam, gr, ss=True, device="cpu")
    with pytest.raises(TypeError, match="CUDA device"):
        B.bamCoverage(fixture_bam, gr, ss=True, runs=True, device="cpu")


# ---- CoverageRuns with ss over hand-built arrays ---------------------------------------------------------------------
def _hand_built():
    # region 0: width 4, sense [1 1 0 0], antisense [0 2 2 2]; region 1: zero-width; region 2: width 2, [5 5], [0 3]
    lengths = np.array([2, 2, 1, 3, 2, 1, 1], np.int32)
    values = np.array([1, 0, 0, 2, 5, 0, 3], np.int32)
    offsets = np.array([0, 2, 4, 4, 4, 5, 7], np.int64)
    return lengths, values, offsets


def test_coverage_runs_container_ss():
    lengths, values, offsets = _hand_built()
    r = B.CoverageRuns(lengths, values, offsets, ss=True)
    assert r.ss and len(r) == 3
    (ls, vs), (la, va) = r[0]
    assert ls.tolist() == [2, 2] and vs.tolist() == [1, 0] and la.tolist() == [1, 3] and va.tolist() == [0, 2]
    assert [len(x) for pair in r[1] for x in pair] == [0, 0, 0, 0]
    with pytest.raises(IndexError):
        r[3]
    d = r.to_dense()
    assert isinstance(d, B.CountSignals) and d.ss and len(d) == 3
    assert [x.tolist() for x in d.as_list()] == [[[1, 1, 0, 0], [0, 2, 2, 2]], [[], []], [[5, 5], [0, 3]]]
    assert d._flat.tolist() == [1, 0, 1, 2, 0, 2, 0, 2, 5, 0, 5, 3]
    assert d.width().tolist() == [4, 0, 2]
    assert repr(r) == "CoverageRuns object with 3 strand-specific regions and 7 runs"
    with pytest.raises(ValueError, match="two lists per region"):
        B.CoverageRuns(lengths[:4], values[:4], offsets[:4], ss=True)
    plain = B.CoverageRuns(lengths, values, offsets)                       # the same arrays as six unstranded regions
    assert not plain.ss and len(plain) == 6 and plain[0][0].tolist() == [2, 2]
    assert repr(plain) == "CoverageRuns object with 6 regions and 7 runs"


def test_coverage_runs_container_ss_torch():
    torch = pytest.importorskip("torch")
    lengths, values, offsets = _hand_built()
    r = B.CoverageRuns(torch.from_numpy(lengths), torch.from_numpy(values), offsets, ss=True)
    d = r.to_dense()
    assert isinstance(d._flat, torch.Tensor)
    assert [x.tolist() for x in d.as_list()] == [[[1, 1, 0, 0], [0, 2, 2, 2]], [[], []], [[5, 5], [0, 3]]]


# ---- stranded coverage from the reads, against the oracle identity ----------------------------------------------------
def kept_intervals(reads, a):
    """setRead for coverage (src/bamsignals.cpp:392-415) in numpy: the kept reads' tid, inclusive [s, e] and strand."""
    flag = reads["flag"].astype(np.uint32) & 0xffff
    tlen = reads["tlen"].astype(np.int64)
    keep = reads["mapq"] >= a["mapqual"]
    keep &= (np.uint32(a["requiredF"] & 0xffffffff) & ~flag) == 0
    keep &= (np.uint32(a["filteredF"] & 0xffffffff) & ~flag) != 0
    if a["tlen_filter"] is not None:
        keep &= (np.abs(tlen) >= a["tlen_filter"][0]) & (np.abs(tlen) <= a["tlen_filter"][1])
    s, e = reads["pos"].astype(np.int64), reads["endpos"].astype(np.int64) - 1
    neg = (flag & 16) != 0
    if a["tspan"]:
        s = np.where(neg & (tlen < 0), e + tlen + 1, s)
        e = np.where(~neg & (tlen > 0), s + tlen - 1, e)
    return reads["tid"][keep], s[keep], e[keep], neg[keep]


def stranded_coverage(iv, names, gr):
    tid, s, e, neg = iv
    out = []
    for i in range(len(gr)):
        loc, w, st = int(gr.start[i]) - 1, int(gr.width[i]), int(gr.strand[i])
        m = np.zeros((2, w), np.int64)
        sel = (tid == names.index(gr.seqlevels[gr.seq_idx[i]])) & (s < loc + w) & (e >= loc)
        for ss_, ee, nn in zip(s[sel], e[sel], neg[sel]):
            lo, hi = max(ss_, loc) - loc, min(ee, loc + w - 1) - loc + 1
            m[int(nn) ^ int(st < 0), lo:hi] += 1
        out.append(m[:, ::-1] if st < 0 else m)
    return out


def fixture_regions(rng, n=60):
    starts = rng.integers(1, 9500, n)
    widths = rng.integers(0, 700, n)
    return B.GRanges(rng.choice(["chr1", "chr2", "chr3"], n).tolist(), starts, widths,
                     rng.choice(["+", "-", "*"], n).tolist())


@pytest.mark.parametrize("k", range(len(COVERAGE_KW)))
def test_restatement_against_the_oracle_identity(fixture_bam, k):
    kw = COVERAGE_KW[k]
    gr = fixture_regions(np.random.default_rng(100 + k))
    names, _ = O.header(fixture_bam)
    a = api.core_args("bamCoverage", **kw)
    got = stranded_coverage(kept_intervals(O.dump_reads(fixture_bam), a), names, gr)
    tot = O.coverage_core(fixture_bam, gr, **a)
    rev = O.coverage_core(fixture_bam, gr, **dict(a, requiredF=a["requiredF"] | 16))
    assert sum(int(m.sum()) for m in got) > 0
    for i, (m, t, r) in enumerate(zip(got, tot, rev)):
        sense, anti = (r, t - r) if gr.strand[i] < 0 else (t - r, r)
        assert np.array_equal(m[0], sense) and np.array_equal(m[1], anti), i
        assert np.array_equal(m.sum(0), t), i


# ---- numpy restatement of the kernels ---------------------------------------------------------------------------------
def tiles_of(widths, tile_ints, order):
    """make_tiles for strand-specific coverage: tile_ints // 2 bases per tile, (region, rel, len) in `order`."""
    tb = tile_ints // 2
    return [(int(i), rel, min(int(widths[i]), rel + tb) - rel) for i in order for rel in range(0, int(widths[i]), tb)]


def tile_diff_ss(s, e, neg_read, loc, width, neg, rel, ln):
    """scatter_coverage<true>: the interleaved difference array d[2j + a], a = read strand XOR region strand."""
    tloc = loc + width - rel - ln if neg else loc + rel
    rend = tloc + ln
    keep = (s < rend) & (e >= tloc)
    s, e, a = s[keep], e[keep], (neg_read[keep].astype(np.int64) ^ int(neg))
    up, down = (rend - 1 - e, rend - s) if neg else (s - tloc, e + 1 - tloc)
    d = np.zeros(2 * ln, np.int64)
    np.add.at(d, 2 * np.maximum(up, 0) + a, 1)
    inside = down < ln
    np.add.at(d, 2 * down[inside] + a[inside], -1)
    return d


def scan_like_k_coverage_ss(d, ph):
    """k_coverage_ss's scan: d placed ph ints into quads, per quad x -> z and y -> w, two carries over the quads."""
    total = ph + len(d)
    sm = np.zeros(4 * ((total + 3) // 4), np.int64)
    sm[ph:total] = d
    q = sm.reshape(-1, 4)
    q[:, 2] += q[:, 0]
    q[:, 3] += q[:, 1]
    incl = np.cumsum(q[:, 2:], axis=0)
    prefix = incl - q[:, 2:]
    q[:, 0] += prefix[:, 0]
    q[:, 2] += prefix[:, 0]
    q[:, 1] += prefix[:, 1]
    q[:, 3] += prefix[:, 1]
    return sm[ph:total]


def runs_like_the_kernels(reads, locs, widths, strands, tile_ints, order):
    tiles = tiles_of(widths, tile_ints, order)
    T, R = len(tiles), len(widths)
    ds = [tile_diff_ss(*reads[i], locs[i], widths[i], strands[i] < 0, rel, ln) for i, rel, ln in tiles]
    # virtual tiles: row a of the j-th of region i's n_i tiles (T_i its first) is v = 2 T_i + a n_i + j, list 2i + a
    V = 2 * T
    vt = np.zeros((2, T), np.int64)
    vlist, vrel = np.zeros(V, np.int64), np.zeros(V, np.int64)
    t0 = 0
    while t0 < T:
        t1 = t0 + 1
        while t1 < T and tiles[t1][0] == tiles[t0][0]:
            t1 += 1
        for t in range(t0, t1):
            for a in (0, 1):
                v = 2 * t0 + a * (t1 - t0) + (t - t0)
                vt[a, t], vlist[v], vrel[v] = v, 2 * tiles[t][0] + a, tiles[t][1]
        t0 = t1
    # count pass (k_runs_count_ss)
    nnz, first, last = np.zeros(V, np.int64), np.zeros(V, np.int64), np.zeros(V, np.int64)
    for t, d in enumerate(ds):
        for a in (0, 1):
            row = d[a::2]
            v = vt[a, t]
            nnz[v], first[v], last[v] = np.count_nonzero(row[1:]), row[0], row.sum()
    # k_runs_scan over the virtual tiles and 2R lists
    head = np.ones(V, bool)
    head[1:] = vlist[1:] != vlist[:-1]
    start0 = head.copy()
    start0[1:] |= first[1:] != last[:-1]
    runs = nnz + start0
    toff = np.concatenate([[0], np.cumsum(runs)])
    rfirst, rlast = np.zeros(2 * R, np.int64), np.zeros(2 * R, np.int64)
    for v in range(V):
        if head[v]:
            rfirst[vlist[v]] = toff[v]
        if v + 1 == V or vlist[v + 1] != vlist[v]:
            rlast[vlist[v]] = toff[v + 1]
    run_off = np.concatenate([[0], np.cumsum(rlast - rfirst)])
    # write pass (k_runs_write_ss): per row the value scan and the run starts, lengths by the two atomics
    n = int(run_off[-1])
    lengths, values = np.zeros(n, np.int64), np.full(n, -1, np.int64)
    for t, ((i, rel, ln), d) in enumerate(zip(tiles, ds)):
        for a in (0, 1):
            v, lst = vt[a, t], 2 * i + a
            kbeg, kend = run_off[lst], run_off[lst + 1]
            k = kbeg + toff[v] - rfirst[lst]
            row = d[a::2]
            flag = row != 0
            flag[0] = start0[v]
            x = np.cumsum(row)
            for j in np.flatnonzero(flag):
                p = rel + j
                values[k] = x[j]
                lengths[k] -= p
                if k > kbeg:
                    lengths[k - 1] += p
                k += 1
            assert k == kbeg + toff[v + 1] - rfirst[lst]
            if v + 1 == V or vlist[v + 1] != lst:
                lengths[kend - 1] += rel + ln
    return tiles, ds, lengths, values, run_off


def dense_ss(s, e, neg_read, loc, width, neg):
    x = np.arange(loc, loc + width)
    cover = (s[None, :] <= x[:, None]) & (e[None, :] >= x[:, None])
    a = neg_read.astype(bool) ^ bool(neg)
    m = np.stack([(cover & ~a[None, :]).sum(1), (cover & a[None, :]).sum(1)]) if len(s) else np.zeros((2, width), np.int64)
    return m[:, ::-1] if neg else m


def rle(v):
    if len(v) == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    starts = np.concatenate([[0], np.flatnonzero(np.diff(v)) + 1])
    return np.diff(np.concatenate([starts, [len(v)]])), v[starts]


def check(reads, locs, widths, strands, tile_ints, order):
    tiles, ds, lengths, values, off = runs_like_the_kernels(reads, locs, widths, strands, tile_ints, order)
    want = [dense_ss(*reads[i], locs[i], widths[i], strands[i] < 0) for i in range(len(widths))]
    # the dense kernel: every tile's scan at every 16-byte phase is its slice of the interleaved region
    for (i, rel, ln), d in zip(tiles, ds):
        for ph in range(4):
            got = scan_like_k_coverage_ss(d, ph)
            assert np.array_equal(got, want[i][:, rel:rel + ln].reshape(-1, order="F")), (i, rel, ph)
    assert off[0] == 0 and (np.diff(off) >= 0).all() and len(off) == 2 * len(widths) + 1
    for i in range(len(widths)):
        for a in (0, 1):
            k = 2 * i + a
            lw, vw = rle(want[i][a])
            lg, vg = lengths[off[k]:off[k + 1]], values[off[k]:off[k + 1]]
            assert np.array_equal(lg, lw) and np.array_equal(vg, vw), (i, a, tile_ints)
            assert (lg >= 1).all() and lg.sum() == widths[i]
    return lengths, values, off


def random_reads(rng, loc, width, n, maxlen):
    s = rng.integers(loc - maxlen, loc + width + maxlen, n)
    return s, s + rng.integers(0, maxlen, n), rng.integers(0, 2, n)


@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_random(tile_ints):
    rng = np.random.default_rng(tile_ints + 7)
    tb = tile_ints // 2
    widths = np.array([1, 7, tb - 1, tb, tb + 1, 2 * tb, 3 * tb + 1, 0, 5, 0, tb + 3, 2 * tb - 1], np.int64)
    strands = np.array([1, -1, 0, -1, 1, 0, -1, 1, 0, -1, 0, 1])
    locs = rng.integers(1000, 50000, len(widths))
    reads = [random_reads(rng, l, w, int(rng.integers(0, 3 * max(w, 1) // 50 + 3)), 300) for l, w in zip(locs, widths)]
    check(reads, locs, widths, strands, tile_ints, rng.permutation(len(widths)))


@pytest.mark.parametrize("tile_ints", TILE_SIZES)
def test_kernel_restatement_one_strand_and_edges(tile_ints):
    """Only forward or only reverse reads (the other row is one run of zeros), runs that change at every base on one
    row, and reads ending exactly on tile boundaries, on '+', '-' and '*'."""
    tb = tile_ints // 2
    locs = np.array([100, 100, 5000, 0], np.int64)
    widths = np.array([3 * tb, 3 * tb, 2 * tb + 1, 0], np.int64)
    strands = np.array([1, -1, 0, -1])
    p = np.arange(100, 100 + 3 * tb)
    reps = 1 + (np.arange(3 * tb) % 3)
    fw = (np.repeat(p, reps), np.repeat(p, reps), np.zeros(int(reps.sum()), np.int64))
    ends = 5000 + np.array([tb - 1, 2 * tb - 1, 2 * tb])
    reads = [fw, fw, (np.full(3, 5000), ends, np.ones(3, np.int64)), (np.zeros(0, np.int64),) * 3]
    lengths, values, off = check(reads, locs, widths, strands, tile_ints, np.array([3, 1, 0, 2]))
    assert off[2] - off[1] == 1 and values[off[1]] == 0                  # region 0 '+': no antisense reads
    assert off[3] - off[2] == 1 and values[off[2]] == 0                  # region 1 '-': forward reads are antisense
    assert off[7] == off[8]
