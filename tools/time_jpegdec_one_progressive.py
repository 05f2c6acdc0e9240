"""FileCorruptionBatcher on 16 1360x765 q95 files of which one is progressive (smooth or noise content): time per call,
against the same call on 16 baseline files.  argv[1]: the repository tree whose package is timed (to compare two
commits).  Prints one JSON line.

    python tools/time_jpegdec_one_progressive.py <tree>"""
import json
import os
import sys
import time

sys.path.insert(0, sys.argv[1])
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
from robust_object_detection_b200.training import FileCorruptionBatcher
rng = np.random.default_rng(3)
out = {"tree": os.path.basename(sys.argv[1].rstrip("/"))}
for kind in ("smooth", "noise"):
    imgs = [rng.integers(0, 256, (765, 1360, 3), dtype=np.uint8) for _ in range(16)]
    if kind == "smooth":
        imgs = [cv2.GaussianBlur(im, (0, 0), 3.0) for im in imgs]
    base = [cv2.imencode(".jpg", im)[1].tobytes() for im in imgs]
    mixed = list(base)
    mixed[5] = cv2.imencode(".jpg", imgs[5], [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    fb = FileCorruptionBatcher(out_hw=(640, 640), seed=1, io_threads=16)
    for name, files in (("all_baseline", base), ("one_progressive", mixed)):
        for _ in range(3):
            fb(files)
            torch.cuda.synchronize()
        ts = []
        for _ in range(15):
            t0 = time.perf_counter()
            fb(files)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        out[f"{kind}_{name}_ms_median"] = round(1e3 * float(np.median(ts)), 2)
print(json.dumps(out))
