"""Config 5 by op class: corrupt + letterbox 640 + normalise for batch 16 / 64 of 1360x765 frames with every image on the
same op (0 clean, 1 noise, 2 blur, 3 LowRes) and with the seed-42 mix."""
import os, random, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
for n in (16, 64):
    h, w = 765, 1360
    src = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device="cuda")
    plan = CorruptionPlan.uniform(n, h, w)
    out = torch.empty((n, 3, 640, 640), dtype=torch.float16, device="cuda")
    random.seed(42)
    mixes = {"mix": draw_decisions(n)}
    for op in range(4):
        mixes[f"op{op}"] = np.full(n, op, np.uint8)
    res = {}
    for name, dec in mixes.items():
        ops = torch.from_numpy(dec).cuda()
        fn = lambda: plan.corrupt_letterbox(src, ops, out, 640, 640, 114, seed=1)
        for _ in range(5): fn()
        torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(40): fn()
        e1.record(); torch.cuda.synchronize()
        res[name] = round(e0.elapsed_time(e1) / 40 * 1e3, 1)
    print(f"config5 n={n} us:", res)
