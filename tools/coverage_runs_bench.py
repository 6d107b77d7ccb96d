"""Dense vs run-length coverage: python tools/coverage_runs_bench.py --preset c3|genome|genome_low [--gscale 1] [--calls 7]

Presets: 'c3' is BASELINE's C3 (bamCoverage paired_end="extend" over 10k 100 kb windows on chr1); 'genome' is
bamCoverage over C2's BAM (100 M single-end 100 bp reads at gscale 1) with every contig as one '*' region; 'genome_low'
the same over a BAM with a quarter of the reads (--density).  Four arms, each in a fresh process of its own:
  dense_host    bamCoverage -> numpy (bsg_coverage: result streamer, PCIe, host scatter)
  dense_device  bamCoverage(device="cuda:0") (bsg_coverage_device)
  runs_host     bamCoverage(runs=True) -> numpy lengths / values (bsg_coverage_runs + bsg_runs_read into host memory)
  runs_device   bamCoverage(runs=True, device="cuda:0") -> torch tensors
After --warmup untimed calls, --calls timed calls; medians of the library's ms_total / ms_d2h / bytes_d2h and of the
wall time of the whole Python call (for runs_host this includes reading the runs over PCIe; bytes_pcie adds those
bytes to bytes_d2h).  device_mb_peak: the largest rise of the device's used memory (cudaMemGetInfo, polled every
millisecond from a second thread during the timed calls) over what the process held before its first call - on a
shared GPU, other processes' allocations would show up in it too.  Every arm digests its last result in dense
bsg_output_layout() order (runs are expanded in chunks); the parent checks that all digests agree.
tools/profile_runs_bench.py drives its arms with the same code (measure_arm, run_arms)."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
import workloads as WL  # noqa: E402
from device_output_bench import data_dir, gpu_info  # noqa: E402

ARMS = ("dense_host", "dense_device", "runs_host", "runs_device")
CHUNK = 1 << 24


def workload(preset, gscale, density):
    import numpy as np
    import bamsignals_b200 as B
    if preset == "c3":
        bam, info = WL.make_bam("c3", gscale, data_dir())
        gr, kw, _ = WL.regions("c3", gscale)
        return bam, info, gr, kw
    d = density if preset == "genome_low" else 1.0
    bam, info = WL.make_bam("c2", gscale, data_dir(), density=d)
    lens = WL.contig_lens("c2", gscale)
    gr = B.GRanges.from_codes(WL.NAMES[:len(lens)], np.arange(len(lens)), np.ones(len(lens)), np.asarray(lens),
                              np.zeros(len(lens), np.int8))
    return bam, info, gr, {}


def digest(res):
    """blake2b of the result in bsg_output_layout() order, and its sum; runs are expanded CHUNK runs at a time.  A
    strand-specific ProfileRuns is walked region by region, CHUNK bins at a time, its two rows interleaved
    [s_0, a_0, s_1, ...] as in the dense layout."""
    import numpy as np
    h, total = hashlib.blake2b(), 0

    def host(x):
        return x if isinstance(x, np.ndarray) else x.cpu().numpy()
    if getattr(res, "ss", False) and hasattr(res, "lengths"):
        lengths, values, off = host(res.lengths).astype(np.int64), host(res.values), res.offsets
        ends = np.cumsum(lengths)
        for i in range(len(res)):
            rows = [(int(off[k]), int(off[k + 1])) for k in (2 * i, 2 * i + 1)]
            base = [int(ends[a] - lengths[a]) if b > a else 0 for a, b in rows]    # the list's first bin, flat
            nb = int(lengths[rows[0][0]:rows[0][1]].sum())
            for b0 in range(0, nb, CHUNK):
                b1 = min(nb, b0 + CHUNK)
                part = np.empty(2 * (b1 - b0), np.int32)
                for a, ((k0, k1), z) in enumerate(zip(rows, base)):
                    e = ends[k0:k1] - z                                             # run ends, relative to the list
                    lo, hi = np.searchsorted(e, b0, "right"), np.searchsorted(e, b1 - 1, "right") + 1
                    seg = np.minimum(e[lo:hi], b1) - np.maximum(e[lo:hi] - lengths[k0 + lo:k0 + hi], b0)
                    part[a::2] = np.repeat(values[k0 + lo:k0 + hi], seg)
                h.update(memoryview(part))
                total += int(part.sum(dtype=np.int64))
    elif hasattr(res, "lengths"):
        n = int(res.offsets[-1])
        for a in range(0, n, CHUNK):
            dense = np.repeat(host(res.values[a:a + CHUNK]), host(res.lengths[a:a + CHUNK])).astype(np.int32)
            h.update(memoryview(dense))
            total += int(dense.sum(dtype=np.int64))
    else:
        flat = res._flat
        for a in range(0, len(flat), CHUNK):
            part = np.ascontiguousarray(host(flat[a:a + CHUNK]))
            h.update(memoryview(part))
            total += int(part.sum(dtype=np.int64))
    return h.hexdigest(), total


class MemPoll:
    def __init__(self, torch):
        self.torch, self.base, self.peak, self.stop = torch, None, 0, False
        free, tot = torch.cuda.mem_get_info(0)
        self.base = tot - free

    def run(self):
        while not self.stop:
            free, tot = self.torch.cuda.mem_get_info(0)
            self.peak = max(self.peak, tot - free - self.base)
            time.sleep(0.001)


def measure_arm(args, call, n_elems, elem, head):
    """Run `call(device, runs)` --warmup + --calls times for args.arm and print its JSON line: `head` first, then the
    medians, the runs per output element (`elem`: "base", "bin") over n_elems, the peak device memory, the digest."""
    import torch
    import bamsignals_b200 as B
    device = "cuda:0" if args.arm.endswith("device") else None
    is_runs = args.arm.startswith("runs")
    torch.empty(1, device="cuda:0")                          # CUDA context + allocator set-up outside the timed calls
    poll = MemPoll(torch)
    th = None
    rows, res = [], None
    for i in range(args.warmup + args.calls):
        if i == args.warmup:
            th = threading.Thread(target=poll.run, daemon=True)
            th.start()
        res = None                                           # a fresh result per call, as a user's call has
        t0 = time.perf_counter()
        res = call(device, is_runs)
        if device:
            torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        t = B.timings()
        if i >= args.warmup:
            runs = int(res.offsets[-1]) if is_runs else None
            read = 8 * runs if args.arm == "runs_host" else 0
            rows.append(dict(wall_ms=wall, ms_total=t["ms_total"], ms_d2h=t["ms_d2h"], bytes_d2h=t["bytes_d2h"],
                             bytes_pcie=t["bytes_d2h"] + read, ms_fetch=t["ms_fetch"], ms_kernels=t["ms_kernels"],
                             out_elems=t["out_elems"]))
    poll.stop = True
    th.join()
    runs = int(res.offsets[-1]) if is_runs else None
    dig, total = digest(res)
    med = {k: statistics.median(r[k] for r in rows) for k in ("wall_ms", "ms_total", "ms_d2h", "bytes_d2h", "bytes_pcie",
                                                                "ms_fetch", "ms_kernels")}
    line = dict(head)
    line.update({"arm": args.arm, elem + "s": n_elems, "warmup": args.warmup, "calls": args.calls,
                 "gpu_inflate": args.gpu_inflate, "median": med,
                 "ms_total_all": [round(r["ms_total"], 2) for r in rows], "wall_ms_all": [round(r["wall_ms"], 2) for r in rows],
                 "out_elems": int(rows[-1]["out_elems"]), "runs": runs,
                 f"runs_per_{elem}": None if runs is None else runs / n_elems,
                 "device_mb_peak": round(poll.peak / 2 ** 20, 1), "result_sum": total, "result_blake2b": dig})
    line.update(gpu_info())
    print(json.dumps(line), flush=True)


def run_arm(args):
    import bamsignals_b200 as B
    if B.lib().bsg_device_count() < 1:
        raise SystemExit("coverage_runs_bench needs a CUDA device")
    bam, info, gr, kw = workload(args.preset, args.gscale, args.density)
    opts = B.default_opts(gpu_inflate=args.gpu_inflate)
    head = dict(preset=args.preset, gscale=args.gscale, density=args.density if args.preset == "genome_low" else 1.0,
                arm=args.arm, call=f"bamCoverage {kw}", regions=len(gr))
    bases = int(sum(int(w) for w in gr.width))
    head.update(bases=bases, reads_in_bam=info["records"])
    measure_arm(args, lambda device, runs: B.bamCoverage(bam, gr, opts=opts, device=device, runs=runs, **kw), bases, "base", head)


def run_arms(args, script, child_args, skip=None):
    """Every arm of args.arms in a fresh process (`script --arm <arm> child_args`); skip(arm) may return a reason to
    leave an arm out, which becomes that arm's line.  Prints the lines (appended to args.out) with digests_equal over
    the arms that ran; exits non-zero if they differ."""
    lines = []
    for arm in args.arms.split(","):
        why = skip(arm) if skip else None
        if why:
            lines.append(dict(preset=args.preset, gscale=args.gscale, arm=arm, skipped=why, **gpu_info()))
            continue
        cmd = [sys.executable, os.path.abspath(script), "--arm", arm] + child_args
        out = subprocess.run(cmd, check=True, stdout=subprocess.PIPE, text=True, cwd=ROOT).stdout
        lines.append(json.loads(out.strip().splitlines()[-1]))
    same = len({(ln["result_blake2b"], ln["result_sum"]) for ln in lines if "skipped" not in ln}) == 1
    for ln in lines:
        ln["digests_equal"] = same
        print(json.dumps(ln), flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(json.dumps(ln) + "\n")
    if not same:
        raise SystemExit("the arms' results differ")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", default="c3", choices=["c3", "genome", "genome_low"])
    ap.add_argument("--gscale", type=float, default=1.0, help="1.0 = the full configuration")
    ap.add_argument("--density", type=float, default=0.25, help="genome_low: fraction of C2's reads")
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
    workload(args.preset, args.gscale, args.density)       # generate once, outside the arms
    run_arms(args, __file__, ["--preset", args.preset, "--gscale", repr(args.gscale), "--density", repr(args.density),
                              "--warmup", str(args.warmup), "--calls", str(args.calls), "--gpu-inflate", str(args.gpu_inflate)])


if __name__ == "__main__":
    main()
