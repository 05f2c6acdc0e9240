"""Device JPEG decoder on progressive files: device time per call for 128 progressive 1360x765 q95 files written by
OpenCV (smooth and noise content), the time of each scan level's kernel (torch.profiler, a separate pass), and
cv2.imdecode of the same files on all host threads; the card's name and power limit are read in the same run.
`--baseline` times the decoder on 128 baseline files of the same size instead, through the entry points every build has
(rod_jpegdec_create / _decode / _status), so that `--lib PATH` can time another build of librod_b200.so for comparison.
Prints one JSON line; with --out also appends it there.

    python tools/time_jpegdec_progressive.py [--baseline] [--lib PATH] [--out profiles/x.json]"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2
import numpy as np
import torch

ap = argparse.ArgumentParser()
ap.add_argument("--baseline", action="store_true")
ap.add_argument("--lib", default=None)
ap.add_argument("--out", default=None)
ap.add_argument("-n", type=int, default=128)
args = ap.parse_args()

import ctypes  # noqa: E402

from robust_object_detection_b200 import _native  # noqa: E402
from robust_object_detection_b200.batch import CorruptionPlan  # noqa: E402
from robust_object_detection_b200.jpeg import JpegDecoder  # noqa: E402



class BaselineDecoder:
    """rod_jpegdec_create / _decode / _status / _destroy through ctypes: present in every build of the library."""

    def __init__(self, files, offsets):
        lib = self.lib = ctypes.CDLL(os.path.abspath(args.lib) if args.lib else _native.LIB_PATH)
        vp = ctypes.c_void_p
        lib.rod_jpegdec_create.argtypes = [vp, vp, ctypes.c_int, vp, vp, ctypes.c_int, ctypes.POINTER(vp)]
        lib.rod_jpegdec_decode.argtypes = [vp, vp, vp]
        lib.rod_jpegdec_status.argtypes = [vp, vp, vp]
        lib.rod_jpegdec_destroy.argtypes = [vp]
        self.bufs = [np.frombuffer(f, np.uint8) for f in files]
        n = self.n = len(files)
        ptrs = (vp * n)(*[b.ctypes.data for b in self.bufs])
        lens = (ctypes.c_uint64 * n)(*[b.size for b in self.bufs])
        offs = (ctypes.c_uint64 * n)(*[int(o) for o in offsets])
        self.h = vp()
        assert lib.rod_jpegdec_create(ptrs, lens, n, offs, None, 16, ctypes.byref(self.h)) == 0

    def decode(self, pix):
        assert self.lib.rod_jpegdec_decode(self.h, pix.data_ptr(), torch.cuda.current_stream().cuda_stream) == 0

    def status(self):
        st = np.zeros(self.n, np.int32)
        assert self.lib.rod_jpegdec_status(self.h, st.ctypes.data, torch.cuda.current_stream().cuda_stream) == 0
        return st

assert torch.cuda.is_available(), "this measurement needs the GPU"
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
H, W, n = 765, 1360, args.n
rng = np.random.default_rng(4)
params = [] if args.baseline else [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]
out = {"gpu": gpu[0] if gpu else None, "lib": args.lib or "in-tree", "files": "baseline" if args.baseline else "progressive"}


def device_ms(dec, pix, reps=10):
    e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e[0].record()
        dec.decode(pix)
        e[1].record()
        torch.cuda.synchronize()
        ts.append(e[0].elapsed_time(e[1]))
    return ts


for kind in ("smooth", "noise"):
    files = []
    for _ in range(n):
        im = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        files.append(cv2.imencode(".jpg", cv2.GaussianBlur(im, (0, 0), 3.0) if kind == "smooth" else im, params)[1].tobytes())
    plan = CorruptionPlan.uniform(n, H, W)
    pix = torch.empty(plan.src_bytes, dtype=torch.uint8, device="cuda")
    dec = BaselineDecoder(files, plan.src_offsets) if args.baseline else JpegDecoder(files, plan.src_offsets, host_threads=16, progressive=True)
    dec.decode(pix)   # warm-up, and the check that the timed work is the right work
    assert (dec.status() == 0).all()
    got = pix.cpu().numpy()
    for i in range(0, n, 16):
        assert np.array_equal(got[plan.src_offsets[i]:plan.src_offsets[i] + 3 * H * W].reshape(H, W, 3),
                              cv2.imdecode(np.frombuffer(files[i], np.uint8), cv2.IMREAD_COLOR)), i
    ts = device_ms(dec, pix)
    r = {"images": n, "compressed_MB": round(sum(len(f) for f in files) / 1e6, 1),
         "device_call_ms_min": round(min(ts), 2), "device_call_ms_median": round(float(np.median(ts)), 2)}
    if not args.baseline:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            dec.decode(pix)
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and "jpegdec" in ev.name:
                name = ev.name.split("(")[0].split("::")[-1]
                kern.setdefault(name, []).append(round(ev.time_range.elapsed_us() / 1e3, 3))
        r["kernel_ms"] = kern   # jpegdec_prog_kernel: one entry per scan level, in launch order
        threads = os.cpu_count()
        with ThreadPoolExecutor(threads) as pool:
            best = None
            for _ in range(3):
                t0 = time.perf_counter()
                list(pool.map(lambda f: cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR), files))
                t = time.perf_counter() - t0
                best = t if best is None else min(best, t)
        r["cv2_host_threads"] = threads
        r["cv2_all_threads_ms"] = round(best * 1e3, 1)
    out[kind] = r
line = json.dumps(out)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(line + "\n")
