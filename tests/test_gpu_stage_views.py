"""Region views of staged sessions on the GPU (bsg_stage_view, Stage.view): every counting form of a view equals a
fresh library call on the same regions and arguments (and the oracle where the other suites use it), on host and
device output and as runs; views of whole-contig sessions, of widened random scenarios and of sessions in several
resident batches; resident_scheme 0 / 1 / 2 agree; the coverage rule accepts exactly what the session's index queries
cover; views need no file; and handles may be closed in any order, nest, interleave, and end with bsg_shutdown()."""
import os
import shutil
import sys
import warnings

import numpy as np
import pytest

import bamsignals_b200 as B
import bamwriter as W
import oracle_api as O
import random_cases as RC
import spec_r

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import workloads as WL  # noqa: E402

torch = pytest.importorskip("torch")
pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore:some ranges' widths")]
DEV = "cuda:0"
EARG, ENOCHROM = -8, -3


def whole_contigs(bam):
    names, lens = O.header(bam)
    return B.GRanges(names, np.ones(len(names), np.int64), lens)


def annot_regions(seed=5):
    """The fixture's annotation, shuffled and duplicated, plus overlapping copies on '-' and zero-width regions."""
    a = spec_r.load_annot()
    rng = np.random.default_rng(seed)
    n = len(a["start"])
    idx = np.concatenate([np.arange(n), rng.integers(0, n, n // 2)])
    rng.shuffle(idx)
    names = [a["seqnames"][i] for i in idx]
    start = [int(a["start"][i]) for i in idx]
    width = [int(a["width"][i]) for i in idx]
    strand = [a["strand"][i] for i in idx]
    for i in range(0, n, 2):                       # overlapping the original by half, on '-'
        names.append(a["seqnames"][i]); start.append(int(a["start"][i]) + int(a["width"][i]) // 2)
        width.append(int(a["width"][i])); strand.append("-")
    for i in range(3):                             # zero-width
        names.append(a["seqnames"][i]); start.append(int(a["start"][i]) + 7); width.append(0); strand.append("*")
    return B.GRanges(names, start, width, strand)


def ext_of(fn, args):
    if fn == "bamCoverage":
        return args["tlen_filter"][1] if args["tspan"] else 0
    return abs(args["shift"]) + (args["tlen_filter"][1] if args["pe_mid"] else 0)


def fresh_flat(bam, gr, fn, kw):
    return WL.as_flat(getattr(B, fn)(bam, gr, **kw))


def oracle_flat(bam, gr, fn, kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return RC.flat(getattr(O, fn)(bam, gr, **kw), fn)


def staged_call(st, fn, kw, out=None):
    """The staged form of the R-level call fn(**kw) on session or view `st` (host result, or `out` filled on the GPU)."""
    if fn == "bamCoverage":
        k = dict(kw)
        ss = k.pop("ss", False)
        return st.coverage(**B.core_args(fn, **k), ss=ss, out=out)
    return st.pileup(**B.core_args(fn, **kw), out=out)


def check_view(st, bam, gr, fn, kw, want):
    """Host and device output of a staged call equal `want`; returns the host call's timings."""
    h = staged_call(st, fn, kw)
    t = B.timings()
    assert np.array_equal(h, want), (fn, kw)
    if len(want):
        d = torch.full((len(want),), -7, dtype=torch.int32, device=DEV)
        assert staged_call(st, fn, kw, out=d) is d
        assert np.array_equal(d.cpu().numpy(), want), (fn, kw, "device")
    return t


FORMS = [("bamCount", {}), ("bamCount", dict(ss=True, shift=40)),
         ("bamProfile", dict(binsize=1)), ("bamProfile", dict(binsize=1, ss=True, shift=75)),
         ("bamProfile", dict(binsize=5, ss=True)), ("bamProfile", dict(binsize=5, shift=-30)),
         ("bamProfile", dict(binsize=200)), ("bamProfile", dict(binsize=200, ss=True, mapqual=20)),
         ("bamProfile", dict(binsize=1, paired_end="midpoint", tlenFilter=(50, 300))),
         ("bamProfile", dict(binsize=5, ss=True, paired_end="filter", tlenFilter=(0, 400))),
         ("bamCoverage", {}), ("bamCoverage", dict(paired_end="extend")),
         ("bamCoverage", dict(ss=True)), ("bamCoverage", dict(paired_end="extend", ss=True))]


@pytest.fixture(scope="module")
def fixture_view(fixture_bam):
    gr = annot_regions()
    with B.Stage(fixture_bam, whole_contigs(fixture_bam), ext_hint=2000) as st:
        v = st.view(gr)
        yield v, gr
        v.close()


@pytest.mark.parametrize("fn,kw", FORMS, ids=[f"{f}-{i}" for i, (f, _) in enumerate(FORMS)])
def test_fixture_forms(fixture_bam, fixture_view, fn, kw):
    v, gr = fixture_view
    want = fresh_flat(fixture_bam, gr, fn, kw)
    if not (fn == "bamCoverage" and kw.get("ss")):               # the oracle has no strand-specific coverage
        assert np.array_equal(want, oracle_flat(fixture_bam, gr, fn, kw))
    assert want.sum() > 0
    for _ in range(2):                                          # the second call reuses the view's tiles
        t = check_view(v, fixture_bam, gr, fn, kw, want)
    assert t["bytes_inflated"] > 0 and t["n_batches"] >= 1      # carried over from the open


RUNS = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamProfile", dict(binsize=5)),
        ("bamCoverage", {}), ("bamCoverage", dict(paired_end="extend", ss=True))]


@pytest.mark.parametrize("fn,kw", RUNS, ids=[f"{f}-{i}" for i, (f, _) in enumerate(RUNS)])
@pytest.mark.parametrize("device", [None, DEV])
def test_fixture_runs(fixture_bam, fixture_view, fn, kw, device):
    v, gr = fixture_view
    k = dict(kw)
    ss = k.pop("ss", False)
    args = B.core_args(fn, **k)
    got = v.coverage_runs(**args, ss=ss, device=device) if fn == "bamCoverage" else \
        v.profile_runs(**B.core_args(fn, **kw), device=device)
    want = getattr(B, fn)(fixture_bam, gr, runs=True, **kw)
    host = lambda x: x.cpu().numpy() if isinstance(x, torch.Tensor) else x       # noqa: E731
    assert np.array_equal(got.offsets, want.offsets)
    assert np.array_equal(host(got.lengths), want.lengths) and np.array_equal(host(got.values), want.values)


def _scenario_seeds(n_pileup=12, n_coverage=6):
    """The first seeds whose scenario fetches records for several regions (test_gpu_resident_fused's choice), of
    bamCount / bamProfile and of bamCoverage."""
    pileup, cover = [], []
    for s in range(200):
        sc = RC.scenario(s)
        if len(sc["reads"]) < 60 or len(sc["gr"]) < 3:
            continue
        (cover if sc["fn"] == "bamCoverage" else pileup).append(s)
        if len(pileup) >= n_pileup and len(cover) >= n_coverage:
            break
    return pileup[:n_pileup] + cover[:n_coverage]


@pytest.mark.parametrize("seed", _scenario_seeds())
def test_random_scenarios(tmp_path, seed):
    """A session over the scenario's regions widened by more than the call's halo; the view is the scenario's own
    region set (regions below 1, zero-width, past the contig end, seqlevels in another order)."""
    sc = RC.scenario(seed)
    bam = RC.write(sc, str(tmp_path / "r.bam"))
    gr, fn, kw = sc["gr"], sc["fn"], sc["kw"]
    want = oracle_flat(bam, gr, fn, kw)
    assert np.array_equal(want, RC.spec_counts(sc))
    assert np.array_equal(want, fresh_flat(bam, gr, fn, kw))
    margin = ext_of(fn, B.core_args(fn, **kw)) + 1
    wide = B.GRanges.from_codes(gr.seqlevels, gr.seq_idx, gr.start.astype(np.int64) - margin,
                                gr.width.astype(np.int64) + 2 * margin, gr.strand)
    with B.Stage(bam, wide, ext_hint=0) as st, st.view(gr) as v:
        check_view(v, bam, gr, fn, kw, want)


@pytest.mark.parametrize("fn,kw", [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamCount", dict(ss=True)),
                                   ("bamProfile", dict(binsize=200, paired_end="midpoint", tlenFilter=(50, 300)))])
def test_schemes_agree_and_small_views_take_the_fused_path(fixture_bam, fn, kw):
    gr = annot_regions()
    small = gr[np.arange(5)]
    want, want_small = fresh_flat(fixture_bam, gr, fn, kw), fresh_flat(fixture_bam, small, fn, kw)
    for scheme in (0, 1, 2):
        with B.Stage(fixture_bam, whole_contigs(fixture_bam), ext_hint=1000, opts=B.default_opts(resident_scheme=scheme)) as st:
            with st.view(gr) as v, st.view(small) as vs:
                t = check_view(v, fixture_bam, gr, fn, kw, want)
                ts = check_view(vs, fixture_bam, small, fn, kw, want_small)
                if scheme == 1:
                    assert t["records_kept"] >= 0 and ts["records_kept"] >= 0
                else:
                    assert ts["records_kept"] == -1, scheme
                    assert scheme == 0 or t["records_kept"] == -1


def _multi_batch_reads(rng, n=40000, length=3_000_000):
    reads = []
    for p in np.sort(rng.integers(0, length - 70000, n)):
        u = rng.random()
        cigar = "60M" if u < .96 else (f"30M{int(rng.integers(5000, 40000))}N30M" if u < .98 else "20M2D10I30M")
        reads.append(dict(tid=0, pos=int(p), flag=int(rng.choice([0, 16, 99, 147])), mapq=int(rng.integers(0, 61)),
                          cigar=cigar, tlen=int(rng.choice([150, -150, 300, -301])), l_seq=60))
    return reads


@pytest.fixture(scope="module")
def multi_batch_bam(tmp_path_factory):
    bam = str(tmp_path_factory.mktemp("views_mb") / "mb.bam")
    W.write_bam(bam, [("chrM", 3_000_000)], _multi_batch_reads(np.random.default_rng(12)), level=0)
    return bam


@pytest.mark.parametrize("scheme", [1, 2])
def test_view_regions_cross_resident_batches(multi_batch_bam, scheme):
    """The whole contig staged in several resident batches; 3 kb view windows every 1 kb cross every batch boundary."""
    starts = np.arange(1, 2_990_000, 1000)
    gr = B.GRanges(["chrM"] * len(starts), starts, np.full(len(starts), 3000), (["+", "-", "*"] * len(starts))[:len(starts)])
    calls = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamCount", dict(shift=-40)),
             ("bamCoverage", dict(paired_end="extend"))]
    o = B.default_opts(resident_scheme=scheme, batch_bytes=1 << 16)
    with B.Stage(multi_batch_bam, whole_contigs(multi_batch_bam), ext_hint=1000, opts=o) as st:
        assert B.timings()["n_batches"] >= 4
        with st.view(gr) as v:
            for fn, kw in calls:
                want = fresh_flat(multi_batch_bam, gr, fn, kw)
                assert want.sum() > 0
                if fn == "bamCount":
                    assert np.array_equal(want, oracle_flat(multi_batch_bam, gr, fn, kw))
                check_view(v, multi_batch_bam, gr, fn, kw, want)


# ---- the coverage rule ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rule_bam(tmp_path_factory):
    rng = np.random.default_rng(4)
    reads = []
    for tid in (0, 1):
        for p in np.sort(rng.integers(0, 399_000, 16000)):
            reads.append(dict(tid=tid, pos=int(p), flag=int(rng.choice([0, 16, 99, 147])), mapq=30, cigar="50M",
                              tlen=int(rng.choice([150, -150])), l_seq=50))
    bam = str(tmp_path_factory.mktemp("rule") / "rule.bam")
    W.write_bam(bam, [("chrR", 400_000), ("chrS", 400_000)], reads)
    return bam


def gr0(chrom, loc, width, strand=None):
    """Regions from 0-based starts, as in the C ABI ('+' unless `strand` says otherwise)."""
    return B.GRanges(chrom, np.asarray(loc, np.int64) + 1, width, strand or ["+"] * len(loc))


def test_rule_halo_of_a_narrower_view(rule_bam):
    with B.Stage(rule_bam, gr0(["chrR"], [100_000], [10_000]), ext_hint=0) as st, \
            st.view(gr0(["chrR", "chrR"], [100_075, 100_075], [9850, 9850], ["+", "-"])) as v:
        g = gr0(["chrR", "chrR"], [100_075, 100_075], [9850, 9850], ["+", "-"])
        for shift in (75, -75):
            kw = dict(binsize=1, ss=True, shift=shift)
            want = fresh_flat(rule_bam, g, "bamProfile", kw)
            assert want.sum() > 0
            check_view(v, rule_bam, g, "bamProfile", kw, want)
        with pytest.raises(B.BamsignalsError, match="reach 75 bp") as e:
            v.pileup(**B.core_args("bamProfile", binsize=1, shift=76))
        assert e.value.code == EARG
        with pytest.raises(B.BamsignalsError) as e:
            v.coverage(**B.core_args("bamCoverage", paired_end="extend", tlenFilter=(0, 76)))
        assert e.value.code == EARG
        want = fresh_flat(rule_bam, g, "bamCoverage", dict(paired_end="extend", tlenFilter=(0, 75)))
        check_view(v, rule_bam, g, "bamCoverage", dict(paired_end="extend", tlenFilter=(0, 75)), want)


def test_rule_refuses_at_creation(rule_bam):
    with B.Stage(rule_bam, gr0(["chrR"], [100_000], [10_000]), ext_hint=0) as st:
        with pytest.raises(B.BamsignalsError, match="region 2 ") as e:
            st.view(gr0(["chrR", "chrR"], [100_075, 99_999], [100, 100]))
        assert e.value.code == EARG
        with pytest.raises(B.BamsignalsError, match="region 1 ") as e:
            st.view(gr0(["chrS"], [100_100], [100]))                  # a contig the session did not stage
        assert e.value.code == EARG
        with pytest.raises(B.BamsignalsError, match="chromosome chrZ not present in the bam file") as e:
            st.view(B.GRanges(["chrZ"], [1], [10]))
        assert e.value.code == ENOCHROM
        with st.view(gr0(["chrR", "chrS"], [100_000, 5], [10_000, 0])) as v:     # zero-width regions need nothing
            v.pileup(**B.core_args("bamCount"))


def test_rule_merge_gap(rule_bam):
    gap = gr0(["chrR"], [112_000], [6000])
    with B.Stage(rule_bam, gr0(["chrR", "chrR"], [100_000, 120_000], [10_000, 10_000]), ext_hint=0) as st, st.view(gap) as v:
        for fn, kw in (("bamCoverage", {}), ("bamProfile", dict(binsize=10, shift=500))):
            want = fresh_flat(rule_bam, gap, fn, kw)
            assert want.sum() > 0
            check_view(v, rule_bam, gap, fn, kw, want)
    with B.Stage(rule_bam, gr0(["chrR", "chrR"], [100_000, 160_000], [10_000, 10_000]), ext_hint=0) as st:
        with pytest.raises(B.BamsignalsError, match="region 1 ") as e:
            st.view(gr0(["chrR"], [130_000], [1000]))
        assert e.value.code == EARG


# ---- no file access, lifetime ------------------------------------------------------------------------------------
def test_views_need_no_file(fixture_bam, tmp_path):
    bam = str(tmp_path / "gone.bam")
    shutil.copyfile(fixture_bam, bam)
    shutil.copyfile(fixture_bam + ".bai", bam + ".bai")
    gr = annot_regions(seed=9)
    with B.Stage(bam, whole_contigs(fixture_bam), ext_hint=500) as st:
        os.remove(bam)
        os.remove(bam + ".bai")
        for fn, kw in (("bamProfile", dict(binsize=5, ss=True, shift=75)), ("bamCoverage", dict(paired_end="extend",
                                                                                               tlenFilter=(0, 400)))):
            with st.view(gr) as v:
                check_view(v, fixture_bam, gr, fn, kw, fresh_flat(fixture_bam, gr, fn, kw))


def test_close_order_nesting_and_interleaving(fixture_bam):
    gr1, gr2 = annot_regions(seed=1), annot_regions(seed=2)[np.arange(0, 30, 2)]
    whole = whole_contigs(fixture_bam)
    calls = [("bamProfile", dict(binsize=1, ss=True, shift=75)), ("bamCount", dict(ss=True)), ("bamCoverage", {}),
             ("bamProfile", dict(binsize=5, paired_end="midpoint", tlenFilter=(0, 300))),
             ("bamProfile", dict(binsize=1, shift=-40, mapqual=20)), ("bamCoverage", dict(ss=True))]
    want = {(id(g), i): fresh_flat(fixture_bam, g, fn, kw) for g in (whole, gr1, gr2) for i, (fn, kw) in enumerate(calls)}
    st = B.Stage(fixture_bam, whole, ext_hint=1000)
    v1 = st.view(gr1)
    v2 = v1.view(gr2)                                  # a view of a view counts against the session's records
    for _ in range(2):
        for i, (fn, kw) in enumerate(calls):
            for h, g in ((st, whole), (v1, gr1), (v2, gr2)):
                check_view(h, fixture_bam, g, fn, kw, want[(id(g), i)])
    st.close()                                         # the session first: its views keep the resident records
    v1.close()
    for i, (fn, kw) in enumerate(calls):
        check_view(v2, fixture_bam, gr2, fn, kw, want[(id(gr2), i)])
    v3 = v2.view(gr1)
    v2.close()
    check_view(v3, fixture_bam, gr1, *calls[0], want[(id(gr1), 0)])
    v3.close()


def test_shutdown_ends_session_and_views(fixture_bam):
    st = B.Stage(fixture_bam, whole_contigs(fixture_bam), ext_hint=100)
    v1, v2 = st.view(annot_regions(seed=3)), st.view(annot_regions(seed=4))
    B.lib().bsg_shutdown()
    for h in (st, v1, v2):
        with pytest.raises(B.BamsignalsError, match="ended by bsg_shutdown") as e:
            h.pileup(**B.core_args("bamProfile", binsize=1))
        assert e.value.code == EARG
    with pytest.raises(B.BamsignalsError) as e:
        st.view(annot_regions())
    assert e.value.code == EARG
    for h in (v1, st, v2):
        h.close()
    gr = annot_regions()
    assert np.array_equal(fresh_flat(fixture_bam, gr, "bamCount", {}), oracle_flat(fixture_bam, gr, "bamCount", {}))


def test_scaled_c2_view_of_a_whole_genome_session(tmp_path_factory):
    gs = 0.002
    bam, _ = WL.make_bam("c2", gs, str(tmp_path_factory.mktemp("c2v")), unplaced=7)
    gr, kw, fn = WL.regions("c2", gs)
    lens = WL.contig_lens("c2", gs)
    whole = B.GRanges(WL.NAMES[:len(lens)], np.ones(len(lens), np.int64), lens)
    want = fresh_flat(bam, gr, fn, kw)
    assert want.sum() > 0
    with B.Stage(bam, whole, ext_hint=75) as st, st.view(gr) as v:
        t = check_view(v, bam, gr, fn, kw, want)
        assert t["records_kept"] == -1                     # a small view of a whole-genome session: the fused path
