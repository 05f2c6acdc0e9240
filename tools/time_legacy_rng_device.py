"""Times the device draw of compat noise (rod_numpy_legacy_normal_f32_device, csrc/legacy_rng.cu) against the host
generator (rod_numpy_legacy_normal_f32, csrc/np_legacy_rng.cpp, all host threads) and np.random.normal, per call, and
checks every device field against NumPy bit for bit.  The device and host generators alternate within each repeat.
Cases: one 1360x765x3 field; 16 such fields as 16 segments; one restoration batch (16 samples of 256x256x3, the noise
samples -- every other one -- as segments); and the first call of the process (jump-table set-up included), timed once.
Usage: python tools/time_legacy_rng_device.py [repeats] > profiles/<run>_legacy_rng_device.json"""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from robust_object_detection_b200 import augmentations as aug  # noqa: E402

F = 1360 * 765 * 3
P = 256 * 256 * 3
CASES = {
    "field_1360x765": [(0, F)],
    "fields_16x1360x765": [(i * F, F) for i in range(16)],
    "restoration_16x256": [(i * P, P) for i in range(0, 16, 2)],
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def device_call(out, spans):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fix = aug.legacy_normal_f32_device(15.0, out, spans)
    torch.cuda.synchronize()  # the patch kernel queued after the state came back
    return (time.perf_counter() - t0) * 1e3, fix


def host_call(buf, n):
    t0 = time.perf_counter()
    aug.legacy_normal_f32(15.0, (n,), out=buf[:n])
    return (time.perf_counter() - t0) * 1e3


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7
    out = torch.empty(16 * F, dtype=torch.float32, device="cuda")
    buf = np.empty(16 * F, dtype=np.float32)
    res = {"gpu": gpu_info(), "host_cores": os.cpu_count(), "repeats": reps, "sigma": 15.0}
    np.random.seed(1)
    t, fix = device_call(out, CASES["field_1360x765"])
    res["first_call_field_1360x765"] = {"device_ms": round(t, 3), "host_fixups": fix}
    for name, spans in CASES.items():
        n = sum(c for _, c in spans)
        dev, host, npy, fixes = [], [], [], []
        for r in range(reps):
            np.random.seed(100 + r)
            t, fix = device_call(out, spans)
            dev.append(t)
            fixes.append(fix)
            st_dev = np.random.get_state(legacy=True)
            np.random.seed(100 + r)
            host.append(host_call(buf, n))
            st_host = np.random.get_state(legacy=True)
            assert np.array_equal(st_dev[1], st_host[1]) and st_dev[2:] == st_host[2:], name
            got = out.cpu().numpy()
            k = 0
            for o, c in spans:
                assert np.array_equal(got[o:o + c], buf[k:k + c]), name
                k += c
            if r < 2:  # NumPy itself: slow, a couple of samples
                np.random.seed(100 + r)
                t0 = time.perf_counter()
                np.random.normal(0, 15.0, n).astype(np.float32)
                npy.append((time.perf_counter() - t0) * 1e3)
        res[name] = {"values": n, "device_ms": [round(x, 3) for x in dev], "host_ms": [round(x, 3) for x in host],
                     "numpy_ms": [round(x, 1) for x in npy], "host_fixups": fixes,
                     "device_ms_median": round(float(np.median(dev)), 3), "host_ms_median": round(float(np.median(host)), 3)}
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
