"""Strand-specific coverage in one pass vs the two-call workaround:
python tools/coverage_ss_bench.py --preset c3|genome [--gscale 1] [--calls 7] [--out profiles/coverage_ss_<preset>.jsonl]

Presets as in tools/coverage_runs_bench.py: 'c3' is BASELINE's C3 (bamCoverage paired_end="extend" over 10k 100 kb
windows on chr1), 'genome' is bamCoverage over C2's BAM with every contig as one '*' region.  Four arms, each in a fresh
process of its own:
  ss_dense_host    bamCoverage(ss=True) -> numpy (bsg_coverage_ss)
  ss_dense_device  bamCoverage(ss=True, device="cuda:0") (bsg_coverage_ss_device)
  ss_runs_device   bamCoverage(ss=True, runs=True, device="cuda:0") -> torch tensors (bsg_coverage_runs_ss)
  pair_device      the workaround without ss: bamCoverage(device=) with requiredF and with requiredF | 16, then the
                   sense / antisense rows by a subtraction on the device (torch), interleaved into the stranded layout
After --warmup untimed calls, --calls timed calls.  Medians of the wall time of the whole Python call, of the library's
ms_total and of ms_count (the coverage kernels: K5 with SS in the ss arms, two unstranded K5 in the pair arm; summed over
the pair's two library calls, as are ms_total and ms_fetch), and the peak rise of the device's used memory
(cudaMemGetInfo polled every millisecond).  Every arm digests its last result in the dense stranded layout; the parent
checks that all digests agree (the same sense and antisense everywhere).  Each line carries the card name and power
limit read in the same run."""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
from coverage_runs_bench import MemPoll, digest, run_arms, workload  # noqa: E402
from device_output_bench import gpu_info  # noqa: E402

ARMS = ("ss_dense_host", "ss_dense_device", "ss_runs_device", "pair_device")


class _Flat:
    """A dense stranded result held as one flat tensor (what digest() reads from a CountSignals)."""

    def __init__(self, flat):
        self._flat = flat


def pair_call(B, torch, bam, gr, opts, kw):
    """The two-call workaround on the device: cov(requiredF) and cov(requiredF | 16), subtracted and interleaved."""
    a = B.core_args("bamCoverage", **kw)
    tot, off = B.coverage_core(bam, gr, **a, opts=opts, _lazy=True, out=B.api._empty_on("cuda:0", gr, 1, False))
    t1 = B.timings()
    rev, _ = B.coverage_core(bam, gr, **dict(a, requiredF=a["requiredF"] | 16), opts=opts, _lazy=True,
                             out=B.api._empty_on("cuda:0", gr, 1, False))
    t2 = B.timings()
    fwd = tot - rev
    # per base: reverse reads are sense on '-' regions, antisense elsewhere
    minus = torch.from_numpy(gr.strand < 0).to(tot.device)
    widths = torch.from_numpy(gr.width.astype("int64")).to(tot.device)
    neg = torch.repeat_interleave(minus, widths)
    out = torch.empty(2 * tot.numel(), dtype=torch.int32, device=tot.device)
    out[0::2] = torch.where(neg, rev, fwd)
    out[1::2] = torch.where(neg, fwd, rev)
    both = {k: t1[k] + t2[k] for k in ("ms_total", "ms_count", "ms_fetch", "ms_kernels", "bytes_d2h")}
    return _Flat(out), both


def run_arm(args):
    import torch
    import bamsignals_b200 as B
    if B.lib().bsg_device_count() < 1:
        raise SystemExit("coverage_ss_bench needs a CUDA device")
    bam, info, gr, kw = workload(args.preset, args.gscale, 1.0)
    opts = B.default_opts(gpu_inflate=args.gpu_inflate)
    bases = int(sum(int(w) for w in gr.width))
    torch.empty(1, device="cuda:0")                          # CUDA context + allocator set-up outside the timed calls
    arm = args.arm

    def call():
        if arm == "pair_device":
            return pair_call(B, torch, bam, gr, opts, kw)
        device = None if arm == "ss_dense_host" else "cuda:0"
        res = B.bamCoverage(bam, gr, opts=opts, device=device, runs=arm == "ss_runs_device", ss=True, **kw)
        t = B.timings()
        return res, {k: t[k] for k in ("ms_total", "ms_count", "ms_fetch", "ms_kernels", "bytes_d2h")}
    poll, th, rows, res = MemPoll(torch), None, [], None
    for i in range(args.warmup + args.calls):
        if i == args.warmup:
            th = threading.Thread(target=poll.run, daemon=True)
            th.start()
        res = None
        t0 = time.perf_counter()
        res, t = call()
        torch.cuda.synchronize()
        t["wall_ms"] = (time.perf_counter() - t0) * 1e3
        if i >= args.warmup:
            rows.append(t)
    poll.stop = True
    th.join()
    dig, total = digest(res)
    keys = ("wall_ms", "ms_total", "ms_count", "ms_fetch", "ms_kernels", "bytes_d2h")
    line = dict(preset=args.preset, gscale=args.gscale, arm=arm, call=f"bamCoverage {kw} ss", regions=len(gr), bases=bases,
                reads_in_bam=info["records"], warmup=args.warmup, calls=args.calls, gpu_inflate=args.gpu_inflate,
                median={k: statistics.median(r[k] for r in rows) for k in keys},
                ms_total_all=[round(r["ms_total"], 2) for r in rows], ms_count_all=[round(r["ms_count"], 3) for r in rows],
                runs=int(res.offsets[-1]) if hasattr(res, "offsets") and hasattr(res, "lengths") else None,
                device_mb_peak=round(poll.peak / 2 ** 20, 1), result_sum=total, result_blake2b=dig)
    line.update(gpu_info())
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", default="c3", choices=["c3", "genome"])
    ap.add_argument("--gscale", type=float, default=1.0, help="1.0 = the full configuration")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=7)
    ap.add_argument("--gpu-inflate", type=int, default=1)
    ap.add_argument("--arms", default=",".join(ARMS))
    ap.add_argument("--out", help="append the JSON lines to this file")
    ap.add_argument("--arm", choices=ARMS, help="(internal) run one arm in this process")
    args = ap.parse_args()
    if args.calls < 1:
        ap.error("--calls must be at least 1")
    if args.arm:
        return run_arm(args)
    workload(args.preset, args.gscale, 1.0)                 # generate once, outside the arms
    run_arms(args, __file__, ["--preset", args.preset, "--gscale", repr(args.gscale), "--warmup", str(args.warmup),
                              "--calls", str(args.calls), "--gpu-inflate", str(args.gpu_inflate)])


if __name__ == "__main__":
    main()
