"""Times the Philox-mode noise kernels on 256 x 1360x765 (device-resident): the table generator, its Philox4x32-7
variant, Box-Muller.  Usage: python tools/sweep_noise.py [n_images]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from robust_object_detection_b200.batch import CorruptionPlan

n, h, w = int(sys.argv[1]) if len(sys.argv) > 1 else 256, 765, 1360
torch.cuda.set_device(0)
src = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device="cuda")
dst = torch.empty_like(src)
plan = CorruptionPlan.uniform(n, h, w)
bytes_per = 2 * 3 * h * w * n


def rate(fn, steps=10, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return round(bytes_per / ms / 1e6, 1)


out = {}
for gen, name in ((0, "table"), (2, "table_philox7"), (1, "boxmuller")):
    plan.set_gaussian_generator(gen)
    out[name] = rate(lambda: plan.noise(src, dst, None, 15.0, seed=1))
plan.set_gaussian_generator(0)
out["copy_GBs"] = rate(lambda: dst.copy_(src))
print(json.dumps(out))
