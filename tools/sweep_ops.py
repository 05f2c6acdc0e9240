"""Quick per-op timing for knob sweeps: prints GB/s of noise (Philox), lowres and blur on 256 x 1360x765."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from robust_object_detection_b200.batch import CorruptionPlan
n, h, w = 256, 765, 1360
src = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device="cuda"); dst = torch.empty_like(src)
plan = CorruptionPlan.uniform(n, h, w)
def t(fn, steps=10):
    for _ in range(3): fn()
    torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps): fn()
    e1.record(); torch.cuda.synchronize()
    return 2 * 3 * h * w * n / (e0.elapsed_time(e1) / steps) / 1e6
which = sys.argv[1:] or ["noise", "lowres", "blur"]
out = []
if "noise" in which: out.append(("noise", t(lambda: plan.noise(src, dst, None, 15.0, seed=1))))
if "lowres" in which: out.append(("lowres", t(lambda: plan.lowres(src, dst))))
if "blur" in which: out.append(("blur", t(lambda: plan.blur(src, dst))))
print(" ".join(f"{k}={v:.0f}" for k, v in out))
