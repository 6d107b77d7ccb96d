#!/usr/bin/env python
"""Every kernel of the path once on the reference's toy BAM, for runs under compute-sanitizer:
    compute-sanitizer --tool memcheck  python tools/sanitize_smoke.py
    compute-sanitizer --tool racecheck python tools/sanitize_smoke.py
Covers K0a inflate, K0b CRC32, K0c walk (speculate / link / scan / write), K1 decode (pileup and coverage
instantiations), K3 join, K4 count, K4 profile (binsize 1 and the aggregated binsize >= 4 kernel, ss and not), K5
coverage, the result-narrowing kernels and the one-thread publishers, K5r coverage runs and K4r profile runs (every
instantiation: binsize 1, 2..3 and >= 4, ss and not), and (where torch is installed) the tile kernels writing
into a caller's device buffer at every 16-byte phase (bsg_*_device); results are checked against the oracle so that a
sanitizer-clean run is also a correct one.  (The device-inflate path is forced: a job this small would otherwise be
inflated by the host pool.)"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import bamsignals_b200 as B  # noqa: E402
import oracle_api as O  # noqa: E402
import spec_r  # noqa: E402

bam = os.path.join(ROOT, "tests", "golden", "randomBam.bam")
g = spec_r.test_regions(seed=3, n=40)
# 40 short regions + two whole chromosomes (several tiles each, one on the - strand)
gr = B.GRanges([["chr1", "chr2", "chr3"][i] for i in g["rname"]] + ["chr2", "chr1"], g["start"] + [1, 1],
               g["width"] + [10279, 10237], g["strand"] + ["-", "*"])
opts = B.default_opts(gpu_inflate=1, stream_min_ints=1 << 14)
launches = 0
for kw in (dict(ss=True, shift=75), dict(mapqual=20, filteredFlag=1024)):
    assert np.array_equal(B.bamCount(bam, gr, opts=opts, **kw), O.bamCount(bam, gr, **kw))
    launches += B.timings()["n_launches"]
for kw in (dict(binsize=1, ss=True, shift=75), dict(binsize=1), dict(binsize=5, ss=True, paired_end="midpoint"), dict(binsize=50)):
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a, b = B.bamProfile(bam, gr, opts=opts, **kw).as_list(), O.bamProfile(bam, gr, **kw).as_list()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    launches += B.timings()["n_launches"]
for kw in (dict(), dict(paired_end="extend")):
    a, b = B.bamCoverage(bam, gr, opts=opts, **kw).as_list(), O.bamCoverage(bam, gr, **kw).as_list()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    launches += B.timings()["n_launches"]
# a result large enough (>= 64 Ki elements per portion) for the byte-packed transfer, with and without a roomy pair list
big = B.GRanges(["chr1", "chr2", "chr3"] * 8, [1] * 24, [10000] * 24, ["+", "-", "*"] * 8)
for rp in (0, 2):
    o2 = B.default_opts(gpu_inflate=1, result_pack=rp)
    a, b = B.bamCoverage(bam, big, paired_end="extend", opts=o2).as_list(), O.bamCoverage(bam, big, paired_end="extend").as_list()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    launches += B.timings()["n_launches"]
# run-length results (bsg_coverage_runs, bsg_profile_runs), expanded and compared with the oracle
for kw in (dict(), dict(paired_end="extend")):
    a, b = B.bamCoverage(bam, gr, opts=opts, runs=True, **kw).to_dense().as_list(), O.bamCoverage(bam, gr, **kw).as_list()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    launches += B.timings()["n_launches"]
for kw in (dict(binsize=1, ss=True, shift=75), dict(binsize=1), dict(binsize=3, ss=True), dict(binsize=2),
           dict(binsize=5, ss=True, paired_end="midpoint"), dict(binsize=50)):
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        a, b = B.bamProfile(bam, gr, opts=opts, runs=True, **kw).to_dense().as_list(), O.bamProfile(bam, gr, **kw).as_list()
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    launches += B.timings()["n_launches"]
# device output (bsg_*_device) into slices of every 16-byte phase of one allocation: the tile kernels place their shared
# buffers and 128-bit stores by the destination ADDRESS, which a caller's buffer only guarantees to 4 bytes
try:
    import torch
except ImportError:
    torch = None
if torch is not None:
    import warnings
    for fn, kw in (("bamProfile", dict(binsize=1, ss=True)), ("bamProfile", dict(binsize=5, ss=True)),
                   ("bamProfile", dict(binsize=3)), ("bamCount", dict(ss=True)), ("bamCoverage", dict(paired_end="extend"))):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = getattr(O, fn)(bam, gr, **kw)
        want = ref.ravel(order="F") if fn == "bamCount" else np.concatenate([x.ravel(order="F") for x in ref.as_list()])
        args = B.core_args(fn, **kw)
        buf = torch.full((len(want) + 8,), -7, dtype=torch.int32, device="cuda:0")
        for k in range(4):
            view = buf[k:k + len(want)]
            if fn == "bamCoverage":
                B.coverage_core(bam, gr, opts=opts, out=view, **args)
            else:
                B.pileup_core(bam, gr, opts=opts, out=view, **args)
            assert np.array_equal(view.cpu().numpy(), want), (fn, kw, k)
            launches += B.timings()["n_launches"]
B.lib().bsg_shutdown()
print(f"sanitize_smoke ok: {launches} kernel launches, results equal to the oracle")
