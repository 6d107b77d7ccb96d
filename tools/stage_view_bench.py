"""Stage once, count many annotations: python tools/stage_view_bench.py [--gscale 1] [--sets 3] [--reps 5]

One staged session holds C2's BAM (tools/workloads.py) over all 24 whole contigs.  For --sets seeded annotation sets of
each kind below, every result is obtained two ways, each timed --reps times after one untimed call:
  fresh   the streaming call (bamProfile / bamCoverage): plan, fetch, inflate, decode and count the BAM again;
  view    Stage.view(gr) + the staged call on the session's resident records, with host output ('view_host') and
          with out= a torch tensor on the device ('view_device'; the tensor is allocated once, outside the timing).
Kinds:  c2_windows   C2's 100 k x 2 kb promoter windows, bamProfile binsize=1 ss=TRUE shift=75;
        gene_bodies  20 k x 10 kb windows, bamCoverage;
        ss_windows   50 k x 4 kb windows, strand-specific bamCoverage (ss=True).
(counts scale with --gscale, as the contigs do.)  Every view result is compared element by element with the fresh one.
One JSON line per (kind, set) with the median wall times, the path the view's staged call took under
resident_scheme auto (records_kept == -1: fused) and the number of annotation sets after which staging pays off
(open + n x view <= n x fresh); a first line reports the open's cost; every line carries the card's name and power limit,
read in the same run."""
import argparse
import json
import math
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
import workloads as WL  # noqa: E402
from device_output_bench import data_dir, flat_of, gpu_info  # noqa: E402

KINDS = {"c2_windows": (100000, 2000, "bamProfile", dict(binsize=1, ss=True, shift=75)),
         "gene_bodies": (20000, 10000, "bamCoverage", {}),
         "ss_windows": (50000, 4000, "bamCoverage", dict(ss=True))}
EXT_HINT = 75                      # the largest halo of the calls above (C2's shift)


def annotation(kind, gscale, seed):
    """Seeded windows of the kind's width over the genome, placed in proportion to contig length."""
    if kind == "c2_windows":
        return WL.regions("c2", gscale, seed=seed)[0]
    n0, width, _, _ = KINDS[kind]
    lens = np.asarray(WL.contig_lens("c2", gscale), dtype=np.int64)
    rng = np.random.default_rng(seed)
    n = max(8, int(round(n0 * gscale)))
    ci = rng.choice(len(lens), n, p=lens / lens.sum())
    start = (rng.random(n) * (lens[ci] - width)).astype(np.int64) + 1
    return WL.GRanges.from_codes(WL.NAMES[:len(lens)], ci, start, np.full(n, width), rng.choice(np.array([1, -1], np.int8), n))


def staged(B, st, fn, kw, out=None):
    if fn == "bamCoverage":
        k = dict(kw)
        ss = k.pop("ss", False)
        return st.coverage(**B.core_args(fn, **k), ss=ss, out=out)
    return st.pileup(**B.core_args(fn, **kw), out=out)


def timed(f, reps):
    """f() once untimed, then reps times: (median ms, all ms, last result, timings of the last call)."""
    import bamsignals_b200 as B
    f()
    ms, res, t = [], None, None
    for _ in range(reps):
        res = None
        t0 = time.perf_counter()
        res = f()
        ms.append((time.perf_counter() - t0) * 1e3)
        t = B.timings()
    return statistics.median(ms), [round(x, 2) for x in ms], res, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gscale", type=float, default=1.0, help="1.0 = the full C2 configuration")
    ap.add_argument("--sets", type=int, default=3, help="annotation sets (seeds) per kind")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--kinds", default=",".join(KINDS))
    args = ap.parse_args()
    if args.sets < 1 or args.reps < 1:
        ap.error("--sets and --reps must be at least 1")
    import torch
    import bamsignals_b200 as B
    if B.lib().bsg_device_count() < 1:
        raise SystemExit("stage_view_bench needs a CUDA device")
    card = gpu_info()
    bam, info = WL.make_bam("c2", args.gscale, data_dir())
    lens = WL.contig_lens("c2", args.gscale)
    whole = WL.GRanges.from_codes(WL.NAMES[:len(lens)], np.arange(len(lens)), np.ones(len(lens)), np.asarray(lens),
                                  np.zeros(len(lens), np.int8))
    torch.empty(1, device="cuda:0")                       # CUDA context + allocator set-up outside the timings
    t0 = time.perf_counter()
    st = B.Stage(bam, whole, ext_hint=EXT_HINT)
    open_ms = (time.perf_counter() - t0) * 1e3
    to = B.timings()
    head = dict(what="open", gscale=args.gscale, reads_in_bam=info["records"], contigs=len(lens), ext_hint=EXT_HINT,
                open_wall_ms=round(open_ms, 2), ms_total=round(to["ms_total"], 2), ms_fetch=round(to["ms_fetch"], 2),
                ms_decode=round(to["ms_decode"], 2), bytes_compressed=to["bytes_compressed"],
                bytes_inflated=to["bytes_inflated"], records=to["records"], n_batches=to["n_batches"], **card)
    print(json.dumps(head), flush=True)
    bad = []
    for kind in args.kinds.split(","):
        _, width, fn, kw = KINDS[kind]
        for s in range(args.sets):
            gr = annotation(kind, args.gscale, seed=100 + s)
            fresh_ms, fresh_all, res, _ = timed(lambda: getattr(B, fn)(bam, gr, **kw), args.reps)
            want = np.array(flat_of(res), copy=True)
            res = None

            def view_host():
                with st.view(gr) as v:
                    return staged(B, v, fn, kw)
            host_ms, host_all, got, th = timed(view_host, args.reps)
            same_host = bool(np.array_equal(got, want))
            got = None
            out = torch.empty(len(want), dtype=torch.int32, device="cuda:0")

            def view_device():
                with st.view(gr) as v:
                    return staged(B, v, fn, kw, out=out)
            dev_ms, dev_all, _, td = timed(view_device, args.reps)
            same_dev = bool(np.array_equal(out.cpu().numpy(), want))
            t0 = time.perf_counter()
            st.view(gr).close()
            view_only_ms = (time.perf_counter() - t0) * 1e3

            def pays_off(view_ms):              # open + n * view <= n * fresh
                return math.ceil(open_ms / (fresh_ms - view_ms)) if fresh_ms > view_ms else None
            line = dict(what="annotation", kind=kind, set=s, call=f"{fn} {kw}", regions=len(gr), width=width,
                        out_elems=int(len(want)), median_ms=dict(fresh=round(fresh_ms, 2), view_host=round(host_ms, 2),
                                                                 view_device=round(dev_ms, 2)),
                        all_ms=dict(fresh=fresh_all, view_host=host_all, view_device=dev_all),
                        view_create_ms=round(view_only_ms, 3), staged_ms_total_host=round(th["ms_total"], 2),
                        staged_ms_total_device=round(td["ms_total"], 2),
                        path="fused" if th["records_kept"] == -1 else "table", records_kept=th["records_kept"],
                        open_wall_ms=round(open_ms, 2), sets_to_pay_off=dict(host=pays_off(host_ms), device=pays_off(dev_ms)),
                        identical=dict(host=same_host, device=same_dev), gscale=args.gscale, **card)
            print(json.dumps(line), flush=True)
            if not (same_host and same_dev):
                bad.append((kind, s))
            out = None
            torch.cuda.empty_cache()
    st.close()
    if bad:
        raise SystemExit(f"view results differ from fresh calls: {bad}")


if __name__ == "__main__":
    main()
