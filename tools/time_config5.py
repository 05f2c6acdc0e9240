"""Config 5 timing: corrupt + letterbox 640 + normalise for batch 16 (and 64) of 1360x765 frames."""
import os, random, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
for n in (16, 64):
    h, w = 765, 1360
    src = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device="cuda")
    plan = CorruptionPlan.uniform(n, h, w)
    random.seed(42)
    ops = torch.from_numpy(draw_decisions(n)).cuda()
    out = torch.empty((n, 3, 640, 640), dtype=torch.float16, device="cuda")
    fn = lambda: plan.corrupt_letterbox(src, ops, out, 640, 640, 114, seed=1)
    for _ in range(5): fn()
    torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50): fn()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 50 * 1e3
    print(f"config5 n={n}: {us:.1f} us  {n / us * 1e6:.0f} img/s")
