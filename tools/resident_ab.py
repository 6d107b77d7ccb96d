#!/usr/bin/env python
"""A/B of the staged pileup step: the table path (opts.resident_scheme 1: K1 decodes every resident record, K3 + K4)
against the fused path (2: K3f + K4f over the session's record index), on the same staged BAM and regions.

  python tools/resident_ab.py [--preset c2] [--gscale 1.0] [--steps 20] [--warmup 5] [--widths 1,4,10] [--out FILE]

For every width factor w the preset's regions are widened w times (same starts), which raises the share of the resident
rows the fused join examines; per factor, two sessions (one per scheme) are opened on the same BAM and the steps
alternate between them.  Per step: CUDA-event times of the library's kernels (ms_decode, ms_join, ms_count) and
ms_device.  The full results of both schemes are compared element for element on the device.  One JSON line per
factor; `share` = rows examined by the fused join / resident rows (the quantity the auto choice compares with
kFusedShare).  `estimate_ms`: what the auto choice's host-side row estimate adds to a call whose halos the session has
not seen yet (a scheme-0 session, first call with a new shift minus the median of repeated ones).  Card name and power
limit are read in the same run.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import bamsignals_b200 as B  # noqa: E402
import workloads as WL  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", default="c2")
    ap.add_argument("--gscale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--widths", default="1,4,10")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    d = os.environ.get("BSG_BENCH_DIR") or os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"bsg_bench_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    bam, info = WL.make_bam(a.preset, a.gscale, d)
    gr0, kw, fn = WL.regions(a.preset, a.gscale)
    args = B.core_args(fn, **kw)
    ext = abs(args["shift"]) + (args["tlen_filter"][1] if args["pe_mid"] else 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    lines = []
    for w in [int(x) for x in a.widths.split(",")]:
        gr = gr0 if w == 1 else B.GRanges.from_codes(gr0.seqlevels, gr0.seq_idx, gr0.start, gr0.width.astype(np.int64) * w, gr0.strand)
        st = {s: B.Stage(bam, gr, ext_hint=ext, opts=B.default_opts(resident_scheme=s)) for s in (1, 2)}
        index_ms = B.timings()["ms_decode"]          # the second open (scheme 2) is the last: its index pass
        per = {1: [], 2: []}
        for i in range(a.warmup + a.steps):
            for s in (1, 2):
                st[s].pileup(**args, want_output=False)
                t = B.timings()
                if i >= a.warmup:
                    per[s].append({k: t[k] for k in ("ms_decode", "ms_join", "ms_count", "ms_device", "candidates", "records", "records_kept")})
        outs = {}
        for s in (1, 2):
            total = int(B.api.output_layout(gr.width, int(args["binsize"]), bool(args["ss"]))[-1])
            outs[s] = torch.full((total,), -7, dtype=torch.int32, device="cuda:0")
            st[s].pileup(**args, out=outs[s])
            st[s].close()
        torch.cuda.synchronize()
        equal = bool(torch.equal(outs[1], outs[2]))
        del outs
        est = []
        with B.Stage(bam, gr, ext_hint=ext + 8, opts=B.default_opts(resident_scheme=0)) as s0:
            for k in range(4):
                a2 = dict(args, shift=args["shift"] + k)           # new halos: the first call of each estimates
                s0.pileup(**a2, want_output=False)
                first = B.timings()["ms_total"]
                again = []
                for _ in range(3):
                    s0.pileup(**a2, want_output=False)
                    again.append(B.timings()["ms_total"])
                est.append(first - float(np.median(again)))
        med = {s: {k: float(np.median([x[k] for x in per[s]])) for k in ("ms_decode", "ms_join", "ms_count", "ms_device")} for s in (1, 2)}
        spread = {s: [round(min(x["ms_device"] for x in per[s]), 4), round(max(x["ms_device"] for x in per[s]), 4)] for s in (1, 2)}
        rec = per[2][-1]
        line = {"preset": a.preset, "gscale": a.gscale, "width_factor": w, "regions": len(gr), "steps": a.steps,
                "resident_records": rec["records"], "fused_rows_examined": rec["candidates"],
                "share": rec["candidates"] / max(1, rec["records"]), "table": med[1], "fused": med[2],
                "ms_device_min_max": {"table": spread[1], "fused": spread[2]},
                "speedup": med[1]["ms_device"] / max(1e-9, med[2]["ms_device"]), "index_pass_ms": index_ms,
                "estimate_ms": round(float(np.median(est)), 3), "results_equal": equal, "gpu": gpu}
        print(json.dumps(line), flush=True)
        lines.append(line)
        if not equal:
            sys.exit(1)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
