"""Results on the GPU (bsg_*_device; `device=` / `out=` in the Python API): the device result equals the host path's
element for element (and the oracle's on the reference fixture), lands only inside the caller's range however the
buffer is aligned, is ordered after the caller's stream, shares the staged tile cache with host calls correctly, and
does not cross PCIe."""
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
pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:some ranges' widths")]
LEVELS = ["chr1", "chr2", "chr3"]
DEV = "cuda:0"
EARG = -8


def fixture_regions(seed=11, n=120):
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


def host_flat(res):
    return WL.as_flat(res)


def dev_flat(res):
    """A device result (bamCount tensor / CountSignals over a CUDA buffer) -> host vector in bsg_output_layout() order."""
    if isinstance(res, torch.Tensor):
        assert res.is_cuda
        return res.cpu().numpy().ravel(order="F")
    sig = res.as_list()
    assert all(isinstance(s, torch.Tensor) and s.is_cuda for s in sig)
    return np.concatenate([s.cpu().numpy().ravel(order="F") for s in sig]) if sig else np.zeros(0, np.int32)


def assert_no_result_over_pcie(total):
    t = B.timings()
    assert t["out_elems"] == total
    assert t["bytes_d2h"] <= 4096


def same_shapes(dev, host):
    if isinstance(host, np.ndarray):
        assert tuple(dev.shape) == host.shape
    else:
        assert [tuple(x.shape) for x in dev.as_list()] == [x.shape for x in host.as_list()]


MODES = [("bamCount", dict(ss=False)), ("bamCount", dict(ss=True, shift=13))] + \
        [("bamProfile", dict(binsize=b, ss=s)) for b in (1, 2, 3, 4, 200) for s in (False, True)] + \
        [("bamCoverage", dict(paired_end="ignore")), ("bamCoverage", dict(paired_end="extend"))]


@pytest.mark.parametrize("fn,kw", MODES, ids=[f"{f}-{'-'.join(f'{k}{v}' for k, v in kw.items())}" for f, kw in MODES])
def test_every_mode_on_the_fixture(fixture_bam, fn, kw):
    gr = fixture_regions()
    host = getattr(B, fn)(fixture_bam, gr, **kw)
    want = host_flat(host)
    assert np.array_equal(want, host_flat(getattr(O, fn)(fixture_bam, gr, **kw)))
    got = getattr(B, fn)(fixture_bam, gr, device=DEV, **kw)
    assert_no_result_over_pcie(len(want))
    same_shapes(got, host)
    assert np.array_equal(dev_flat(got), want)


@pytest.fixture(scope="module")
def gen_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("gen"))


@pytest.mark.parametrize("inflate", [-1, 1])
@pytest.mark.parametrize("preset,gs", [("c2", 0.002), ("c3", 0.004), ("c4", 0.002), ("c5", 0.002)])
def test_scaled_configs(gen_dir, preset, gs, inflate):
    """C4's whole contigs and C3's 100 kb windows are cut into many tiles each."""
    bam, _ = WL.make_bam(preset, gs, gen_dir, unplaced=7)
    gr, kw, fn = WL.regions(preset, gs)
    o = B.default_opts(gpu_inflate=inflate)
    want = host_flat(getattr(B, fn)(bam, gr, opts=o, **kw))
    got = getattr(B, fn)(bam, gr, opts=o, device=DEV, **kw)
    assert_no_result_over_pcie(len(want))
    assert B.timings()["n_tiles"] > len(gr) or fn == "bamCount" or preset == "c2"
    assert np.array_equal(dev_flat(got), want) and int(want.sum()) > 0


@pytest.mark.parametrize("preset,gs", [("c2", 0.002), ("c3", 0.004)])
def test_tiles_counted_early_into_the_callers_buffer(gen_dir, preset, gs):
    """Small batches and stream_min_ints = 1: finished tiles are counted while later batches still inflate."""
    bam, _ = WL.make_bam(preset, gs, gen_dir, unplaced=7)
    gr, kw, fn = WL.regions(preset, gs)
    perm = np.random.default_rng(5).permutation(len(gr))
    gr = gr[np.concatenate([perm, perm[:7]])]
    want = host_flat(getattr(B, fn)(bam, gr, **kw))
    o = B.default_opts(batch_bytes=1 << 17, stream_min_ints=1, gpu_inflate=1)
    got = getattr(B, fn)(bam, gr, opts=o, device=DEV, **kw)
    t = B.timings()
    assert t["n_batches"] >= 2
    assert_no_result_over_pcie(len(want))
    assert np.array_equal(dev_flat(got), want)


CORES = {"count": dict(binsize=-1, ss=True), "profile_b1": dict(binsize=1, ss=True), "profile_b3": dict(binsize=3),
         "profile_agg": dict(binsize=5, ss=True), "coverage": None}


@pytest.mark.parametrize("what", list(CORES))
def test_misaligned_destinations(fixture_bam, what):
    """buf[k:k + total] for k = 0..3 at the start of an allocation, and big[G + k:G + k + total] inside 16 KiB guard bands
    of one allocation: only 4-byte aligned destinations; everything outside the slice must stay untouched."""
    gr = fixture_regions(seed=12)
    kw = CORES[what]

    def call(**extra):
        if kw is None:
            return B.coverage_core(fixture_bam, gr, (0, 1000), requiredF=66, tspan=True, **extra)
        return B.pileup_core(fixture_bam, gr, None, **kw, **extra)

    want = np.concatenate([x.ravel(order="F") for x in call()]) if kw is None or kw["binsize"] > 0 else \
        call()[0].ravel(order="F")
    total = len(want)
    G = 4096
    for lead in (0, G):
        big = torch.empty(lead + total + G, dtype=torch.int32, device=DEV)
        for k in range(4):
            big.fill_(-7)
            view = big[lead + k:lead + k + total]
            assert call(out=view) is view
            h = big.cpu().numpy()
            assert np.array_equal(h[lead + k:lead + k + total], want), (lead, k)
            assert (h[:lead + k] == -7).all() and (h[lead + k + total:] == -7).all(), (lead, k)


@pytest.mark.parametrize("side_stream", [False, True])
def test_ordered_after_the_callers_stream(fixture_bam, side_stream):
    """Work the caller queued on its stream before the call (here: a long sleep, then a fill) runs before the
    library writes: the result is the counts, not the fill value."""
    gr = fixture_regions(seed=13)
    want = np.concatenate(B.coverage_core(fixture_bam, gr, None))
    buf = torch.empty(len(want), dtype=torch.int32, device=DEV)
    torch.cuda.synchronize()
    s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(3e8))                       # ~150 ms of device time
        buf.fill_(-7)
        B.coverage_core(fixture_bam, gr, None, out=buf)
        h = buf.cpu().numpy()
    assert np.array_equal(h, want)


def test_host_device_host_calls(fixture_bam):
    gr = fixture_regions(seed=14)
    for fn, kw in (("bamProfile", dict(binsize=3, ss=True)), ("bamCoverage", {}), ("bamCount", dict(ss=True))):
        a = host_flat(getattr(B, fn)(fixture_bam, gr, **kw))
        b = dev_flat(getattr(B, fn)(fixture_bam, gr, device=DEV, **kw))
        c = host_flat(getattr(B, fn)(fixture_bam, gr, **kw))
        assert np.array_equal(a, b) and np.array_equal(a, c), fn


def test_staged_device_calls_interleaved_with_host_calls(fixture_bam):
    """A staged session caches its tile table; device calls (caller layout) and host calls (tile order) alternate."""
    gr = fixture_regions(seed=15)
    settings = [("bamProfile", dict(binsize=1)), ("bamProfile", dict(binsize=1, ss=True)),
                ("bamProfile", dict(binsize=4, ss=True, shift=20)), ("bamCount", dict(ss=True)),
                ("bamCoverage", dict(paired_end="extend")), ("bamCoverage", {})]
    with B.Stage(fixture_bam, gr, ext_hint=1000) as st:
        for _ in range(2):
            for fn, kw in settings:
                args = B.core_args(fn, **kw)
                if fn == "bamCoverage":
                    want = np.concatenate(B.coverage_core(fixture_bam, gr, **args))
                    run = st.coverage
                else:
                    res = B.pileup_core(fixture_bam, gr, **args)
                    want = np.concatenate([x.ravel(order="F") for x in res])
                    run = st.pileup
                h1 = run(**args)
                d = torch.full((len(want),), -7, dtype=torch.int32, device=DEV)
                assert run(**args, out=d) is d
                assert_no_result_over_pcie(len(want))
                h2 = run(**args)
                d2 = run(**args, out=torch.full((len(want),), -7, dtype=torch.int32, device=DEV))
                for r in (h1, d.cpu().numpy(), h2, d2.cpu().numpy()):
                    assert np.array_equal(r, want), (fn, kw)


def _raw_pileup(bam, gr, ptr, off, opts=None, stream=None):
    m = api.marshal_regions(gr)
    return B.lib().bsg_pileup_device(os.fsencode(bam), m.R, m.levels, m.n_levels, api._p(m.seq_idx, C.c_int32),
                                     api._p(m.loc, C.c_int32), api._p(m.width, C.c_int32), api._p(m.strand, C.c_int8),
                                     None, 0, 1, 0, 1, 0, -1, 0, 16385, ptr, api._p(off, C.c_int64), stream,
                                     None if opts is None else C.byref(opts))


def test_refusals_leave_the_buffer_unchanged(fixture_bam):
    gr = fixture_regions(seed=16)
    off = api.output_layout(gr.width, 1, True)
    total = int(off[-1])
    buf = torch.full((total + 1,), -7, dtype=torch.int32, device=DEV)
    host = np.full(total, -7, dtype=np.int32)
    pinned = torch.full((total,), -7, dtype=torch.int32).pin_memory()
    bad_off = off.copy()
    bad_off[1] += 1
    cases = [("host memory", host.ctypes.data, off, None),
             ("page-locked host memory", pinned.data_ptr(), off, None),
             ("two devices", buf.data_ptr(), off, B.default_opts(devices=[0, 1])),
             ("wrong layout", buf.data_ptr(), bad_off, None),
             ("misaligned", buf.data_ptr() + 2, off, None),
             ("NULL with elements", None, off, None)]
    if torch.cuda.device_count() >= 2:
        cases.append(("another device than opts", buf.data_ptr(), off, B.default_opts(devices=[1])))
    for name, ptr, o, opts in cases:
        rc = _raw_pileup(fixture_bam, gr, ptr, o, opts)
        assert rc == EARG, (name, rc, B.lib().bsg_last_error())
        torch.cuda.synchronize()
        assert (buf.cpu().numpy() == -7).all() and (host == -7).all() and (pinned.numpy() == -7).all(), name
    # the empty layout needs no buffer
    empty = B.GRanges([], [], [], [])
    assert _raw_pileup(fixture_bam, empty, None, np.zeros(1, np.int64)) == 0


def test_staged_refusals(fixture_bam):
    gr = fixture_regions(seed=17)
    off = api.output_layout(gr.width, 1, False)
    total = int(off[-1])
    host = np.full(total, -7, dtype=np.int32)
    with B.Stage(fixture_bam, gr) as st:
        rc = B.lib().bsg_pileup_staged_device(st._h, None, 0, 1, 0, 0, 0, -1, 0, host.ctypes.data, api._p(off, C.c_int64), None)
        assert rc == EARG and (host == -7).all()
        if torch.cuda.device_count() >= 2:
            other = torch.full((total,), -7, dtype=torch.int32, device="cuda:1")
            rc = B.lib().bsg_coverage_staged_device(st._h, None, 0, 0, -1, 0, other.data_ptr(), api._p(off, C.c_int64), None)
            assert rc == EARG and "staged session" in B.lib().bsg_last_error().decode()
            assert (other.cpu().numpy() == -7).all()
        good = torch.full((total,), -7, dtype=torch.int32, device=DEV)
        st.coverage(None, out=good)
        assert np.array_equal(good.cpu().numpy(), st.coverage(None))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_result_on_the_second_device(fixture_bam):
    gr = fixture_regions(seed=18)
    want = host_flat(B.bamProfile(fixture_bam, gr, binsize=2, ss=True))
    got = B.bamProfile(fixture_bam, gr, binsize=2, ss=True, device=1)
    assert all(x.device == torch.device("cuda", 1) for x in got.as_list())
    assert np.array_equal(dev_flat(got), want)
