"""Per-launch cost of the headline blur (blur_rows_kernel<9>, csrc/blur.cu) against its per-image cost.

Times plan.blur(src, dst) on n x 1360x765 images for n in SIZES, the way bench.py times it (warm-up, then CUDA events
around a loop of calls, here at least 0.3 s per size), and fits t(n) = F + n * c: F is what every launch costs on top
of moving its bytes, c the time per image, 2 * 3 * 1360 * 765 / c the steady-state rate.  A separate torch.profiler
pass splits each call into the kernel and the rest of its period (memset / launch gaps), and its fit gives the
kernel's own fixed part.  dst.copy_(src) at n = 256 is the copy ceiling of the same card.  Inputs at every n but 32
are larger than the 126 MB L2 (n = 32: 200 MB in + out).

Each --lib NAME=PATH is run in its own process (one library per process), alternating the libraries for --rounds rounds.
Usage: python tools/time_blur_launch.py [--lib parent=build/parent/librod_b200.so --lib new=...] [--rounds 3] --out F.json
       (no --lib: the in-tree library)"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W = 765, 1360
IMG_BYTES = 3 * H * W
SIZES = [32, 64, 128, 256, 384]
MIN_SECONDS = 0.3
PROFILED_CALLS = 60


def fit(ns, ts):
    import numpy as np
    c, f = np.polyfit(np.asarray(ns, float), np.asarray(ts, float), 1)
    return float(f), float(c)


def worker(lib_path):
    """One library: the event sweep, the profiler pass and the copy ceiling; prints one JSON line."""
    sys.path.insert(0, ROOT)
    import torch
    from robust_object_detection_b200 import _native as N
    if lib_path:
        N.LIB_PATH = os.path.abspath(lib_path)
    from robust_object_detection_b200.batch import CorruptionPlan

    gen = torch.Generator(device="cuda")
    gen.manual_seed(2000)
    src = torch.randint(0, 256, (max(SIZES), H, W, 3), dtype=torch.uint8, device="cuda", generator=gen)
    dst = torch.empty_like(src)
    plans = {n: CorruptionPlan.uniform(n, H, W) for n in SIZES}

    def events_us(fn, calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return 1e3 * e0.elapsed_time(e1) / calls

    def timed(fn):
        for _ in range(5):
            fn()
        est = events_us(fn, 20)
        calls = max(50, int(MIN_SECONDS * 1e6 / est) + 1)
        return events_us(fn, calls), calls

    sweep = {}
    for n in SIZES:
        s, d, p = src[:n], dst[:n], plans[n]
        us, calls = timed(lambda: p.blur(s, d))
        sweep[n] = {"us_per_call": us, "calls": calls}
    f, c = fit(SIZES, [sweep[n]["us_per_call"] for n in SIZES])

    # profiler pass: kernel time of each call and the rest of its period (start of one blur kernel to the next)
    from torch.profiler import ProfilerActivity, profile
    prof_rows = {}
    for n in SIZES:
        s, d, p = src[:n], dst[:n], plans[n]
        for _ in range(5):
            p.blur(s, d)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(PROFILED_CALLS):
                p.blur(s, d)
            torch.cuda.synchronize()
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            with open(path) as fh:
                trace = json.load(fh)["traceEvents"]
        ks = sorted((e["ts"], e["dur"]) for e in trace
                    if e.get("cat") == "kernel" and "blur_rows_kernel" in e.get("name", ""))
        memsets = [e["dur"] for e in trace if e.get("cat") == "gpu_memset"]
        assert len(ks) == PROFILED_CALLS, f"{len(ks)} blur kernels traced for {PROFILED_CALLS} calls"
        kern = [dur for _, dur in ks]
        period = [(ks[i + 1][0] - ks[i][0]) for i in range(len(ks) - 1)]
        kern.sort()
        period.sort()
        prof_rows[n] = {"kernel_us_median": kern[len(kern) // 2], "period_us_median": period[len(period) // 2],
                        "gap_us_median": period[len(period) // 2] - kern[len(kern) // 2],
                        "memsets_per_call": len(memsets) / PROFILED_CALLS,
                        "memset_us_mean": (sum(memsets) / len(memsets)) if memsets else 0.0}
    fk, ck = fit(SIZES, [prof_rows[n]["kernel_us_median"] for n in SIZES])
    gaps = [prof_rows[n]["gap_us_median"] for n in SIZES]

    m = 256
    copy_us, _ = timed(lambda: dst[:m].copy_(src[:m]))
    out = {
        "lib": lib_path or N.LIB_PATH,
        "sweep": {str(n): v for n, v in sweep.items()},
        "fit": {"F_us": f, "c_us_per_image": c, "steady_GBs": 2 * IMG_BYTES / c / 1e3},
        "profiler": {str(n): v for n, v in prof_rows.items()},
        "profiler_fit": {"kernel_F_us": fk, "kernel_c_us_per_image": ck, "gap_us_median_over_sizes": sorted(gaps)[len(gaps) // 2]},
        "copy_256": {"us_per_call": copy_us, "GBs": 2 * IMG_BYTES * m / copy_us / 1e3},
    }
    print(json.dumps(out), flush=True)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", help="write the JSON result here (default: stdout only)")
    ap.add_argument("--worker", metavar="PATH", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker is not None:
        worker(args.worker)
        return
    libs = [tuple(s.split("=", 1)) for s in args.lib] or [("in-tree", "")]
    res = {"gpu": gpu_info(), "image": f"{W}x{H}x3 uint8", "sizes": SIZES, "min_seconds_per_size": MIN_SECONDS,
           "rounds": []}
    for r in range(args.rounds):
        for name, path in libs:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", path], capture_output=True, text=True)
            if p.returncode != 0:
                sys.stderr.write(p.stderr)
                raise SystemExit(f"worker for {name} failed (exit {p.returncode})")
            rec = json.loads(p.stdout.strip().splitlines()[-1])
            rec.update(name=name, round=r)
            res["rounds"].append(rec)
            print(f"[round {r} {name}] F {rec['fit']['F_us']:.2f} us  c {rec['fit']['c_us_per_image']:.4f} us/img  "
                  f"{rec['fit']['steady_GBs']:.0f} GB/s  kernel F {rec['profiler_fit']['kernel_F_us']:.2f} us  "
                  f"gap {rec['profiler_fit']['gap_us_median_over_sizes']:.2f} us  "
                  f"t(256) {rec['sweep']['256']['us_per_call']:.1f} us  copy {rec['copy_256']['GBs']:.0f} GB/s",
                  file=sys.stderr, flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
