"""Dense vs run-length profiles: python tools/profile_runs_bench.py --preset c2|genome_ends|c4 [--gscale 1] [--calls 7]

Presets: 'c2' is BASELINE's C2 (bamProfile binsize=1 ss=TRUE shift=75 over 100k 2 kb windows); 'genome_ends' is
bamProfile binsize=1 ss=TRUE over C2's BAM with every contig as one '*' region (the genome-wide read-end profile of
ATAC insertion sites, ChIP-exo, CAGE or MNase dyads); 'c4' is BASELINE's C4 (binsize=200 midpoint tlenFilter=c(70,200)
over the 24 whole contigs), the dense regime: it shows what runs cost where they do not pay.  Four arms, each in a
fresh process of its own:
  dense_host    bamProfile -> numpy (bsg_pileup: result streamer, PCIe, host scatter)
  dense_device  bamProfile(device="cuda:0") (bsg_pileup_device)
  runs_host     bamProfile(runs=True) -> numpy lengths / values (bsg_profile_runs + bsg_runs_read into host memory)
  runs_device   bamProfile(runs=True, device="cuda:0") -> torch tensors
The timed calls, the medians, the peak device memory and the digests are those of tools/coverage_runs_bench.py, whose
driver this uses; a strand-specific result is digested in the dense interleaved order.  The dense_host arm of
genome_ends holds a 24.7 GB result at gscale 1: it is skipped, with the reason in its line, when the host has less
than twice the result's size available."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
import workloads as WL  # noqa: E402
from coverage_runs_bench import ARMS, measure_arm, run_arms  # noqa: E402
from device_output_bench import data_dir  # noqa: E402


def workload(preset, gscale):
    import numpy as np
    import bamsignals_b200 as B
    if preset in ("c2", "c4"):
        bam, info = WL.make_bam(preset, gscale, data_dir())
        gr, kw, _ = WL.regions(preset, gscale)
        return bam, info, gr, kw
    bam, info = WL.make_bam("c2", gscale, data_dir())
    lens = WL.contig_lens("c2", gscale)
    gr = B.GRanges.from_codes(WL.NAMES[:len(lens)], np.arange(len(lens)), np.ones(len(lens)), np.asarray(lens),
                              np.zeros(len(lens), np.int8))
    return bam, info, gr, dict(binsize=1, ss=True)


def bins_of(gr, kw):
    b = int(kw.get("binsize", 1))
    return (2 if kw.get("ss") else 1) * sum((int(w) + b - 1) // b for w in gr.width)


def host_bytes_available():
    with open("/proc/meminfo") as f:
        for ln in f:
            if ln.startswith("MemAvailable:"):
                return int(ln.split()[1]) * 1024
    return 0


def run_arm(args):
    import bamsignals_b200 as B
    if B.lib().bsg_device_count() < 1:
        raise SystemExit("profile_runs_bench needs a CUDA device")
    bam, info, gr, kw = workload(args.preset, args.gscale)
    opts = B.default_opts(gpu_inflate=args.gpu_inflate)
    head = dict(preset=args.preset, gscale=args.gscale, arm=args.arm, call=f"bamProfile {kw}", regions=len(gr),
                reads_in_bam=info["records"])
    measure_arm(args, lambda device, runs: B.bamProfile(bam, gr, opts=opts, device=device, runs=runs, **kw),
                bins_of(gr, kw), "bin", head)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", default="c2", choices=["c2", "genome_ends", "c4"])
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
    _, _, gr, kw = workload(args.preset, args.gscale)       # generate once, outside the arms
    need = 2 * 4 * bins_of(gr, kw)

    def skip(arm):
        if arm == "dense_host" and args.preset == "genome_ends" and host_bytes_available() < need:
            return (f"the dense host result needs {need / 2 ** 30 / 2:.1f} GiB; the host has "
                    f"{host_bytes_available() / 2 ** 30:.1f} GiB available, less than twice that")
        return None
    run_arms(args, __file__, ["--preset", args.preset, "--gscale", repr(args.gscale), "--warmup", str(args.warmup),
                              "--calls", str(args.calls), "--gpu-inflate", str(args.gpu_inflate)], skip)


if __name__ == "__main__":
    main()
