"""Host output vs device output on one preset: python tools/device_output_bench.py --preset c3 [--gscale 1] [--calls 7]

Each arm runs in a fresh process of its own (one BAM, same region set, same options): 'host' is the R-level call that
returns numpy arrays (bsg_pileup / bsg_coverage: result streamer, PCIe, host scatter), 'device' the same call with
device="cuda:0" (bsg_*_device: the counting kernels write the torch tensor directly).  After --warmup untimed calls,
--calls timed calls; the medians of the library's own ms_total / ms_d2h / bytes_d2h (and the wall time of the Python
call) are reported.  Both arms hash their last result in bsg_output_layout() order; the parent checks that the two
digests agree and prints one JSON line per arm.  The BAM is generated (or reused) through tools/workloads.py in the
per-user cache directory bench.py uses."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, ROOT)
import workloads as WL  # noqa: E402


def data_dir():
    d = os.environ.get("BSG_BENCH_DIR") or os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp",
                                                        f"bsg_bench_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


def flat_of(res):
    """The result's flat buffer in bsg_output_layout() order, as a host numpy array (no copy for host results)."""
    import numpy as np
    if isinstance(res, np.ndarray):                          # bamCount: (R,) or the (2, R) Fortran view of the flat buffer
        return res.ravel(order="F")
    if hasattr(res, "_flat"):                                # CountSignals over the flat buffer
        res = res._flat
    else:                                                    # bamCount on the device: (R,) or flat.view(R, 2).t()
        res = res.t().reshape(-1) if res.dim() == 2 else res
    return res.cpu().numpy() if not isinstance(res, np.ndarray) else res


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in q.split(",")]
        return dict(gpu=name, power_limit=limit)
    except Exception as e:                                  # noqa: BLE001 - informational only
        return dict(gpu=f"unknown ({e})")


def run_arm(args):
    import bamsignals_b200 as B
    if B.lib().bsg_device_count() < 1:
        raise SystemExit("device_output_bench needs a CUDA device")
    bam, info = WL.make_bam(args.preset, args.gscale, data_dir())
    gr, kw, fn = WL.regions(args.preset, args.gscale)
    call = getattr(B, fn)
    opts = B.default_opts(gpu_inflate=args.gpu_inflate)
    device = None
    if args.arm == "device":
        import torch
        device = "cuda:0"
        torch.empty(1, device=device)                         # CUDA context + allocator set-up outside the timed calls
    rows, res = [], None
    for i in range(args.warmup + args.calls):
        res = None                                           # a fresh result buffer per call, as a user's call has
        t0 = time.perf_counter()
        res = call(bam, gr, opts=opts, device=device, **kw) if device else call(bam, gr, opts=opts, **kw)
        wall = (time.perf_counter() - t0) * 1e3
        t = B.timings()
        if i >= args.warmup:
            rows.append(dict(wall_ms=wall, ms_total=t["ms_total"], ms_d2h=t["ms_d2h"], bytes_d2h=t["bytes_d2h"],
                             ms_fetch=t["ms_fetch"], ms_kernels=t["ms_kernels"], out_elems=t["out_elems"]))
    flat = flat_of(res)
    med = {k: statistics.median(r[k] for r in rows) for k in ("wall_ms", "ms_total", "ms_d2h", "bytes_d2h", "ms_fetch", "ms_kernels")}
    line = dict(preset=args.preset, gscale=args.gscale, arm=args.arm, call=f"{fn} {kw}", regions=len(gr),
                reads_in_bam=info["records"], warmup=args.warmup, calls=args.calls, gpu_inflate=args.gpu_inflate,
                median=med, ms_total_all=[round(r["ms_total"], 2) for r in rows], out_elems=int(rows[-1]["out_elems"]),
                result_sum=int(flat.sum(dtype="int64")), result_blake2b=hashlib.blake2b(memoryview(flat)).hexdigest())
    line.update(gpu_info())
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--preset", default="c3", choices=["c2", "c3", "c4", "c5"])
    ap.add_argument("--gscale", type=float, default=1.0, help="1.0 = the full configuration")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--calls", type=int, default=7)
    ap.add_argument("--gpu-inflate", type=int, default=1)
    ap.add_argument("--arm", choices=["host", "device"], help="(internal) run one arm in this process")
    args = ap.parse_args()
    if args.calls < 1:
        ap.error("--calls must be at least 1")
    if args.arm:
        return run_arm(args)
    WL.make_bam(args.preset, args.gscale, data_dir())         # generate once, outside both arms
    lines = []
    for arm in ("host", "device"):
        cmd = [sys.executable, os.path.abspath(__file__), "--arm", arm, "--preset", args.preset, "--gscale", repr(args.gscale),
               "--warmup", str(args.warmup), "--calls", str(args.calls), "--gpu-inflate", str(args.gpu_inflate)]
        out = subprocess.run(cmd, check=True, stdout=subprocess.PIPE, text=True, cwd=ROOT).stdout
        lines.append(json.loads(out.strip().splitlines()[-1]))
    same = lines[0]["result_blake2b"] == lines[1]["result_blake2b"] and lines[0]["out_elems"] == lines[1]["out_elems"]
    for ln in lines:
        ln["results_identical"] = same
        print(json.dumps(ln), flush=True)
    if not same:
        raise SystemExit("host and device results differ")


if __name__ == "__main__":
    main()
