"""Timing of the Faster R-CNN loader path (train_frcnn_augmented.py:61-67: RandomCorruption(0.5) + ToImage +
ToDtype(float32, scale=True), then .to(device)) on the GPU, in one process.

  convert_only   rod_corrupt_chw_f32 on 256 clean 1360x765 frames (device-resident, 0.8 GB source + 3.2 GB output: larger
                 than L2).  CUDA events over the whole call (it also launches the noise / blur / LowRes kernels, which find
                 no image of theirs), and the conversion kernel's own time from torch.profiler in a separate pass.
                 Algorithmic bytes: 3 read + 12 written per pixel.
  mixed          the same call on a p = 0.5 Philox mix: a clean image costs 15 B/px, a corrupted one 21 B/px (3 + 3 through
                 the scratch, then 3 + 12).
  files          DetectionCorruptionBatcher.run from q95 JPEG files (1360x765) on tmpfs, batch 2 (the reference's) and 16,
                 compat and philox noise, in images/s; against the reference's per-item pipeline on the host (PIL open,
                 RandomCorruption over oracle/cv2_port.py, ToImage, ToDtype, .to(device)) timed in the same run.

Usage: python tools/time_detection_batcher.py > profiles/<tag>_detection_batcher.json   (imports oracle/: bench infra)"""
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cv2  # noqa: E402
import torch  # noqa: E402

from oracle import cv2_port  # noqa: E402
from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions  # noqa: E402
from robust_object_detection_b200.training import DetectionCorruptionBatcher  # noqa: E402

H, W, N = 765, 1360, 256
MEASURED_COPY_GBS = 6459.0  # the project's measured device copy bandwidth on a B200 (README)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_call(fn, warmup=3, iters=20):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters * 1e-3  # seconds per call


def kernel_time(fn, name, iters=20):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    ts = [e.device_time for e in prof.events() if name in e.name and e.device_time > 0]
    return (sum(ts) / len(ts) * 1e-6) if ts else None  # seconds per launch


def device_paths():
    plan = CorruptionPlan.uniform(N, H, W)
    g = torch.Generator(device="cuda").manual_seed(0)
    src = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, device="cuda", generator=g)
    out = torch.empty(plan.chw_offsets()[-1], dtype=torch.float32, device="cuda")
    px = N * H * W
    res = {}
    clean = torch.zeros(N, dtype=torch.uint8, device="cuda")
    t = time_call(lambda: plan.corrupt_chw_f32(src, clean, out, seed=1))
    tk = kernel_time(lambda: plan.corrupt_chw_f32(src, clean, out, seed=1), "chw_f32_kernel")
    res["convert_only"] = {
        "frames": N, "shape": [H, W], "algorithmic_bytes": 15 * px,
        "call_ms": t * 1e3, "call_GBps": 15 * px / t / 1e9,
        "kernel_ms": tk * 1e3 if tk else None, "kernel_GBps": 15 * px / tk / 1e9 if tk else None,
        "kernel_share_of_measured_copy_bw": 15 * px / tk / 1e9 / MEASURED_COPY_GBS if tk else None,
        "bound_ms_at_measured_copy_bw": 15 * px / (MEASURED_COPY_GBS * 1e9) * 1e3}
    random.seed(3)
    ops = draw_decisions(N, gate="pil", p=0.5)
    nc = int((ops != 0).sum())
    nbytes = (15 * (N - nc) + 21 * nc) * H * W
    ops_d = torch.from_numpy(ops).cuda()
    t = time_call(lambda: plan.corrupt_chw_f32(src, ops_d, out, seed=1))
    res["mixed_p05_philox"] = {"frames": N, "corrupted": nc, "algorithmic_bytes": nbytes, "call_ms": t * 1e3,
                               "call_GBps": nbytes / t / 1e9,
                               "share_of_measured_copy_bw": nbytes / t / 1e9 / MEASURED_COPY_GBS}
    del src, out
    torch.cuda.empty_cache()
    return res


class RefRandomCorruption:
    """augmentations.py:60-74 over the live OpenCV / NumPy calls."""

    def __call__(self, img):
        from PIL import Image
        if random.random() > 0.5:
            return img
        img_bgr = cv2.cvtColor(np.array(img), cv2.COLOR_RGB2BGR)
        out = cv2_port.OPS[random.choice(["noise", "blur", "lowres"])](img_bgr)
        return Image.fromarray(cv2.cvtColor(out, cv2.COLOR_BGR2RGB))


def file_paths(n_files=64, n_ref=24):
    from PIL import Image
    import torchvision.transforms.v2 as T
    d = tempfile.mkdtemp(prefix="rod_frcnn_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    res = {}
    try:
        rng = np.random.default_rng(5)
        yy, xx = np.mgrid[0:H, 0:W]
        base = np.stack([xx * 255 // (W - 1), yy * 255 // (H - 1), (xx + yy) % 256], -1)
        paths = []
        for i in range(n_files):
            img = np.clip(base + rng.integers(-30, 31, (H, W, 3)), 0, 255).astype(np.uint8)
            p = os.path.join(d, f"{i:04d}.jpg")
            cv2.imwrite(p, img, [cv2.IMWRITE_JPEG_QUALITY, 95])
            paths.append(p)
        for noise in ("compat", "philox"):
            for bs in (2, 16):
                b = DetectionCorruptionBatcher(p=0.5, noise=noise, seed=1)
                batches = [paths[i:i + bs] for i in range(0, n_files, bs)]
                for _ in b.run(batches[:2]):  # warm-up: plans, pinned buffers, decoder caches
                    pass
                random.seed(0)
                np.random.seed(0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in b.run(batches):
                    pass
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                res[f"ours_{noise}_batch{bs}_img_per_s"] = n_files / dt
        tf = T.Compose([RefRandomCorruption(), T.ToImage(), T.ToDtype(torch.float32, scale=True)])
        random.seed(0)
        np.random.seed(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for p in paths[:n_ref]:
            x = tf(Image.open(p).convert("RGB")).to("cuda")
        torch.cuda.synchronize()
        res["reference_per_item_img_per_s"] = n_ref / (time.perf_counter() - t0)
        res["files"] = n_files
        res["reference_items_timed"] = n_ref
        del x
    finally:
        shutil.rmtree(d, ignore_errors=True)
    return res


def main():
    torch.cuda.init()
    out = {"gpu": gpu_info(), "device_resident": device_paths(), "from_files": file_paths(),
           "host_cpus": len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()}
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
