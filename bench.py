#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 corruption path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): horizontal motion blur k=9 / angle 0 on 256 synthetic
1360x765 uint8 BGR images PER GPU (device-resident [256,765,1360,3], 799 MB in + 799 MB out,
far larger than the 126 MB L2).  A step is one pass of the blur kernel over the batch.  Metric:
corrupted images/s, whole job.  Images shard by index over ranks with no collective (weak
scaling: per-GPU work fixed); only per-rank timings are gathered.

One JSON line on stdout (rank 0); see the keys in main().  `--impl reference` times the
reference's own CPU implementation of the same workload (OpenCV filter2D via oracle/cv2_port.py)
on the host cores.  `--dump-outputs DIR` writes what the last timed step computed (see
dump_outputs()); the inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, N_PER_GPU = 765, 1360, 256
IMG_BYTES = 3 * H * W              # 3 121 200
ALGO_BYTES_PER_IMAGE = 2 * IMG_BYTES  # read + write, SURVEY 8d
METRIC = "corrupted images/sec (1360x765 RGB), motion blur k=9"
UNIT = "images/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profile(name):
    """dram bytes per launch from the committed ncu summary of this kernel, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return float(json.load(f)[name]["dram_bytes"])
    except Exception:
        return None


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out = self.proc.communicate(timeout=5)[0]
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own library calls (oracle/cv2_port.py) on the box's host cores.
# A "pass" is the bench workload's batch -- 256 images of 1360x765 -- spread over a persistent pool of one process
# per core with cv2.setNumThreads(1) each (the best case for the reference: np.random.normal is single-threaded and
# OpenCV's own thread pool scales worse than processes).  Passes are timed INSIDE the loop, for at least min_seconds.
# ---------------------------------------------------------------------------------------------------------
def _host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


class CpuPool:
    def __init__(self):
        import multiprocessing as mp
        from oracle import cv2_port
        self.cv2_port = cv2_port
        self.workers = _host_cores()
        self.pool = mp.get_context("spawn").Pool(self.workers, initializer=cv2_port._pool_init)

    def one_pass(self, op, n_images=N_PER_GPU):
        """n_images images of `op` through the pool; returns wall seconds of the pass."""
        per, extra = divmod(n_images, self.workers)
        tasks = [(op, s, H, W, per + (1 if s < extra else 0)) for s in range(self.workers)]
        tasks = [t for t in tasks if t[4] > 0]
        t0 = time.perf_counter()
        self.pool.map(self.cv2_port._pool_task, tasks)
        return time.perf_counter() - t0

    def rate(self, op, warmup=1, passes=1, min_seconds=2.0, n_images=N_PER_GPU, max_seconds=30.0):
        for _ in range(warmup):
            self.one_pass(op, min(n_images, 2 * self.workers))
        times = []
        while len(times) < passes or (sum(times) < min_seconds and sum(times) < max_seconds):
            times.append(self.one_pass(op, n_images))
        return {"value": n_images * len(times) / sum(times), "passes": len(times), "seconds": sum(times),
                "ms_per_pass": 1e3 * sum(times) / len(times), "images_per_pass": n_images}

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_baseline():
    """The reference's CPU path on a bounded sample of the same workload, per corruption (BASELINE.md section 3): the
    process-pool figure (headline) and the single-process figure with OpenCV's own thread pool."""
    from oracle import cv2_port
    if not cv2_port.available():  # numpy restatement (opencv not importable): a scalar port
        from oracle import corruption_oracle as orc
        import numpy as np
        img = np.random.default_rng(0).integers(0, 256, (H, W, 3), dtype=np.uint8)
        t0 = time.perf_counter()
        n = 4
        for _ in range(n):
            orc.apply_motion_blur(img, 9, 0)
        return {"value": n / (time.perf_counter() - t0), "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"{n} images 1360x765, numpy restatement (opencv not importable)", "cpu_model": cpu_model()}
    pool = CpuPool()
    per_op = {}
    try:
        for op, n_img in (("blur", N_PER_GPU), ("lowres", N_PER_GPU), ("noise", 64)):
            r = pool.rate(op, warmup=1, passes=1, min_seconds=2.0, n_images=n_img)
            thr, nthr = cv2_port.time_op(op, H, W, 48 if op != "noise" else 8, "threads")
            per_op[op] = {"pool_images_per_s": r["value"], "pool_workers": pool.workers, "pool_passes": r["passes"],
                          "pool_seconds": r["seconds"], "images_per_pass": r["images_per_pass"],
                          "single_process_images_per_s": thr, "opencv_threads": nthr}
    finally:
        pool.close()
    b = per_op["blur"]
    return {"value": b["pool_images_per_s"], "unit": UNIT, "cores": pool.workers, "kind": "port",
            "sample": f"{b['pool_passes']} passes x {N_PER_GPU} images 1360x765 (motion blur k=9), {pool.workers} processes x "
                      f"cv2.setNumThreads(1), timed {b['pool_seconds']:.1f} s; single process with OpenCV's own "
                      f"{b['opencv_threads']}-thread pool: {b['single_process_images_per_s']:.0f} images/s",
            "per_op": per_op, "cpu_model": cpu_model()}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the SAME workload (configs[1]: motion blur k=9 on 256
    images of 1360x765 per step; OpenCV filter2D through oracle/cv2_port.py, the calls augmentations.py:36-38 makes) on
    all host cores.  W warm-up + K timed steps, each step one pass over 256 images, timed inside the loop."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cv2_port
    if not cv2_port.available():
        base = cpu_baseline()
        v, cores, desc, ms, passes = base["value"], base["cores"], base["sample"], 1e3 * N_PER_GPU / max(base["value"], 1e-9), 0
    else:
        pool = CpuPool()
        try:
            r = pool.rate("blur", warmup=max(1, args.warmup), passes=args.steps, min_seconds=0.0)
        finally:
            pool.close()
        v, cores, ms, passes = r["value"], pool.workers, r["ms_per_pass"], r["passes"]
        desc = (f"{N_PER_GPU} images 1360x765 per step over {cores} processes x cv2.setNumThreads(1); {passes} timed passes, "
                f"{r['seconds']:.2f} s")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "configs[1]: motion blur k=9 angle=0 on 256 x 1360x765x3 uint8 per step, host memory",
                       "images_per_step": N_PER_GPU, "timed_passes": passes, "sample": desc},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc,
                             "cpu_model": cpu_model()},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bind_to_gpu_cpus(gpu_index):
    """Pin this process to the CPUs NVML reports as local to its GPU (same NUMA node / PCIe root), so that the pinned
    staging buffers of the e2e leg are allocated next to the GPU.  Best effort: returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        allowed = os.sched_getaffinity(0)
        pick = cpus & allowed
        if pick and pick != allowed:
            os.sched_setaffinity(0, pick)
            return f"{len(pick)} of {len(allowed)} allowed CPUs (GPU-local)"
        return f"unchanged ({len(allowed)} allowed CPUs, {len(cpus)} GPU-local)"
    except Exception as e:  # NVML missing, cpuset restrictions, ...
        return f"unavailable ({type(e).__name__})"


DUMP_SAMPLE = 1 << 22   # elements of the seeded sample of the batch: 16 MiB as float32


def dump_outputs(out_dir, dst, torch, np):
    """--dump-outputs: the blurred batch dst [n, 765, 1360, 3] uint8 (799 MB), reduced to 29 MB of .npy files:
      blur_dst_image0.npy      image 0 in full, float32 [765, 1360, 3]
      blur_dst_sample.npy      float32 [4 Mi]: dst.reshape(-1) at the sorted flat indices
                               np.random.default_rng(0).integers(0, dst.numel(), 4 Mi) (the same on every run)
      blur_dst_image_sums.npy  float64 [n]: the sum of every image's bytes (exact: at most 3 121 200 * 255)"""
    os.makedirs(out_dir, exist_ok=True)
    flat = dst.reshape(-1)
    idx = np.sort(np.random.default_rng(0).integers(0, flat.numel(), DUMP_SAMPLE))
    arrays = {"blur_dst_image0": dst[0].float(),
              "blur_dst_sample": flat[torch.from_numpy(idx).to(dst.device)].float(),
              "blur_dst_image_sums": dst.reshape(dst.shape[0], -1).sum(1).double()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def time_device(fn, steps, warmup, torch, dist=None):
    """W untimed + K timed calls of fn() bracketed by barrier + synchronize; CUDA events on the
    current stream; returns this rank's elapsed ms."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the per-op side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the output of the last one as DIR/<name>.npy (rank 0's shard)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the device output of --impl ours")
    if args.impl == "reference":
        run_reference(args)
        return

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # CPU baseline first (rank 0, N=1 only), before CUDA is initialised in this process
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_baseline()

    import numpy as np
    import torch
    from robust_object_detection_b200 import _native as N
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.sharding import gather_records, shard_range

    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_cpus(local_rank) if world > 1 else "not applied (single GPU)"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # this rank's shard of the global batch (weak scaling: N_PER_GPU images per rank)
    g_lo, g_hi = shard_range(N_PER_GPU * world, rank, world)
    n = g_hi - g_lo
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2000 + rank)
    src = torch.randint(0, 256, (n, H, W, 3), dtype=torch.uint8, device="cuda", generator=gen)
    dst = torch.empty_like(src)
    plan = CorruptionPlan.uniform(n, H, W)

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms = time_device(lambda: plan.blur(src, dst), args.steps, args.warmup, torch, dist)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:   # before the side measurements below reuse dst
        dump_outputs(args.dump_outputs, dst, torch, np)
    rec = gather_records({"rank": rank, "ms": ms, "images": n})
    max_ms = max(r["ms"] for r in rec)
    total_images = sum(r["images"] for r in rec)
    value = total_images * args.steps / (max_ms / 1e3)

    # end-to-end through the host-buffer C-ABI call (pinned host memory, H2D + kernel + D2H per step)
    h_src = torch.empty((n, H, W, 3), dtype=torch.uint8).pin_memory()
    h_src.copy_(src.cpu())
    h_dst = torch.empty_like(h_src).pin_memory()
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_step():
        plan.apply_host(N.OP_BLUR, h_src.data_ptr(), h_dst.data_ptr())

    for _ in range(2):
        e2e_step()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    e2e_s = time.perf_counter() - t0
    rec2 = gather_records({"rank": rank, "s": e2e_s})
    e2e_value = total_images * e2e_steps / max(r["s"] for r in rec2)

    # configs 4 and 5 are defined across GPUs (BASELINE.json): measured at every N, all ranks take part
    peak, peak_src = peaks()
    multi = {} if args.no_extras else multi_gpu_configs(torch, np, rank, world, dist, peak)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    launch_ms = ms / args.steps  # rank 0's kernel: one launch per step
    achieved = ALGO_BYTES_PER_IMAGE * n / (launch_ms / 1e3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": max_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": "configs[1]: motion blur k=9 angle=0 on 256 x 1360x765x3 uint8 per GPU, device-resident",
                   "images_per_gpu": n, "l2": "inputs (799 MB in + 799 MB out per step) larger than the 126 MB L2",
                   "sharding": "image index, no collective"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic_from_profile("bench:blur_rows_kernel<9>"), "peak_source": peak_src,
                     "kernel": "rod::blur_rows_kernel<9>", "algorithmic_bytes_per_launch": ALGO_BYTES_PER_IMAGE * n,
                     "frac_of_nominal_8TBs": achieved / 8000.0,
                     "traffic_source": "dram read+write of this launch from the committed ncu --set full capture (profiles/ncu_traffic.json)"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": IMG_BYTES * n, "d2h_bytes_per_step": IMG_BYTES * n,
                "steps": e2e_steps, "api": "rod_apply_host (pinned host buffers, chunked H2D/kernel/D2H pipeline)"},
        "gpu_launches": args.steps * plan.launches(N.OP_BLUR),
        "clocks": clocks,
        "per_rank_ms": [r["ms"] for r in rec],
        "cpu_binding": numa,
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if multi:
        line["configs"] = multi
    if world == 1 and not args.no_extras:
        line["ops"] = extras(torch, np, plan, src, dst, peak)
        if cpu is not None:
            line["ops"]["drop_in_per_call_ms"] = per_call_latency(np)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


VISDRONE_SHAPES = [(765, 1360), (1050, 1400), (788, 1400), (1078, 1916), (1080, 1920), (1500, 2000), (540, 960), (360, 480)]
ODD_SHAPES = [(765, 1361), (1079, 1917), (1499, 1999)]


def multi_gpu_configs(torch, np, rank, world, dist, peak):
    """BASELINE.json configs[3] and configs[4], at whatever N this run has (every rank takes part; rank 0 reports).

    config 4 -- build_corrupted_testsets equivalent: 1610 VisDrone-test-dev-shaped images x {Noise (Philox), Blur, LowRes},
    the image list cut into `world` contiguous blocks balanced by byte count (sharding.shard_by_bytes): STRONG scaling,
    total work fixed.  Counted in corrupted OUTPUTS per second (3 per image).
    config 5 -- training path: random one-of-three (decisions drawn with random.seed(42)) fused with letterbox 640 +
    normalise -> fp16 NCHW, batch 16 PER GPU: weak scaling."""
    import random
    from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
    from robust_object_detection_b200.sharding import gather_records, shard_by_bytes
    out = {}
    rng = np.random.default_rng(4000)
    shapes = [VISDRONE_SHAPES[i] for i in rng.integers(0, 8, 1610)]
    sizes = [3 * h * w for h, w in shapes]
    lo, hi = shard_by_bytes(sizes, world)[rank]
    tp = CorruptionPlan.ragged(shapes[lo:hi])
    gen = torch.Generator(device="cuda")
    gen.manual_seed(4000 + rank)
    tsrc = torch.randint(0, 256, (tp.src_bytes,), dtype=torch.uint8, device="cuda", generator=gen)
    tdst = torch.empty_like(tsrc)

    def testset():
        tp.noise(tsrc, tdst, None, 15.0, seed=42, first_image_index=lo)
        tp.blur(tsrc, tdst)
        tp.lowres(tsrc, tdst)

    steps, warm = 5, 3
    ms = time_device(testset, steps, warm, torch, dist) / steps
    per_op = {}
    for name, fn in (("noise_philox", lambda: tp.noise(tsrc, tdst, None, 15.0, seed=42, first_image_index=lo)),
                     ("blur", lambda: tp.blur(tsrc, tdst)), ("lowres", lambda: tp.lowres(tsrc, tdst))):
        t = time_device(fn, 3, 2, torch, dist) / 3
        per_op[name] = 2 * tp.payload_bytes / (t / 1e3) / 1e9
    rec = gather_records({"rank": rank, "ms": ms, "images": hi - lo, "bytes": tp.payload_bytes, "per_op": per_op})
    t_max = max(r["ms"] for r in rec)
    tot_bytes = sum(r["bytes"] for r in rec)
    out["config4_testset_1610x3"] = {
        "workload": "configs[3]: Noise(Philox)/Blur/LowRes over 1610 VisDrone-shaped images, sharded by byte count",
        "scaling": "strong", "outputs_per_s": 3 * 1610 / (t_max / 1e3), "images": 1610, "ms_per_step": t_max,
        "GB/s": 3 * 2 * tot_bytes / (t_max / 1e3) / 1e9,
        "frac_of_measured_peak_per_gpu": [3 * 2 * r["bytes"] / (r["ms"] / 1e3) / 1e9 / peak for r in rec],
        "per_rank_ms": [r["ms"] for r in rec], "per_rank_images": [r["images"] for r in rec],
        "per_op_GB/s_rank0": rec[0]["per_op"], "unit": "corrupted outputs/s (3 per image)"}
    del tsrc, tdst, tp
    torch.cuda.empty_cache()

    random.seed(42)
    ops_host = draw_decisions(16 * world)[16 * rank:16 * rank + 16]
    p16 = CorruptionPlan.uniform(16, H, W)
    gen.manual_seed(5000 + rank)
    src16 = torch.randint(0, 256, (16, H, W, 3), dtype=torch.uint8, device="cuda", generator=gen)
    ops = torch.from_numpy(np.ascontiguousarray(ops_host)).cuda()
    f16 = torch.empty((16, 3, 640, 640), dtype=torch.float16, device="cuda")
    ms = time_device(lambda: p16.corrupt_letterbox(src16, ops, f16, 640, 640, 114, seed=1, first_image_index=16 * rank),
                     30, 5, torch, dist) / 30
    # the same call replayed from a CUDA graph: at ~40 us per batch the eager loop above is close to the host's launch rate
    # (Python + ctypes + one kernel launch per call), the replay is the device time of the batch
    ms_graph = None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                p16.corrupt_letterbox(src16, ops, f16, 640, 640, 114, seed=1, first_image_index=16 * rank)
        torch.cuda.current_stream().wait_stream(side)
        ms_graph = time_device(g.replay, 30, 5, torch, dist) / 30
    except Exception as e:  # capture is optional evidence; the eager number stands on its own
        print(f"[bench] CUDA-graph replay of config 5 skipped: {e}", file=sys.stderr)
    rec = gather_records({"rank": rank, "ms": ms, "ms_graph": ms_graph})
    t_max = max(r["ms"] for r in rec)
    b16 = 16 * (IMG_BYTES + 640 * 640 * 3 * 2)
    out["config5_train_letterbox_b16"] = {
        "workload": "configs[4]: random one-of-three + letterbox 640 + normalise -> fp16 NCHW, batch 16 per GPU (1360x765 sources)",
        "scaling": "weak", "images_per_s": 16 * world / (t_max / 1e3), "ms_per_batch": t_max, "per_rank_ms": [r["ms"] for r in rec],
        "GB/s": b16 * world / (t_max / 1e3) / 1e9, "frac_of_measured_peak_per_gpu": [b16 / (r["ms"] / 1e3) / 1e9 / peak for r in rec],
        "ms_per_batch_graph_replay": (max(r["ms_graph"] for r in rec) if all(r.get("ms_graph") for r in rec) else None),
        "note": "latency-bound at batch 16 (one ~40 us launch; the eager loop is near the host's launch rate, the CUDA-graph replay "
                "is the device time); inputs fit L2"}
    return out


def per_call_latency(np):
    """One 1360x765 frame through the drop-in functions (host array in, fresh host array out: the call the training
    scripts make), next to the reference's own library calls for the same frame (oracle/cv2_port.py: part of the CPU
    baseline leg).  compat noise is bit-exact, i.e. it includes drawing NumPy's legacy normal stream."""
    from oracle import cv2_port
    from robust_object_detection_b200 import augmentations as aug
    img = np.random.default_rng(7).integers(0, 256, (H, W, 3), dtype=np.uint8)

    def ms(fn, reps):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return 1e3 * (time.perf_counter() - t0) / reps

    out = {"apply_noise_compat": {"ours": ms(lambda: aug.apply_noise(img, 15), 10)},
           "apply_motion_blur": {"ours": ms(lambda: aug.apply_motion_blur(img, 9, 0), 20)},
           "apply_lowres": {"ours": ms(lambda: aug.apply_lowres(img, 0.5), 20)}}
    if cv2_port.available():
        out["apply_noise_compat"]["reference"] = ms(lambda: cv2_port.noise(img, 15), 3)
        out["apply_motion_blur"]["reference"] = ms(lambda: cv2_port.blur(img, 9, 0), 10)
        out["apply_lowres"]["reference"] = ms(lambda: cv2_port.lowres(img, 0.5), 10)
    return out


def extras(torch, np, plan, src, dst, peak):
    """Side measurements of the other kernels on one GPU (not the headline): images/s and HBM fraction.  Configs 4 and 5
    are in multi_gpu_configs (measured at every N)."""
    from robust_object_detection_b200.batch import CorruptionPlan
    out = {}
    n = src.shape[0]

    def rate(fn, bytes_per_call, images, steps=10, warmup=3):
        ms = time_device(fn, steps, warmup, torch) / steps
        gbs = bytes_per_call / (ms / 1e3) / 1e9
        return {"images_per_s": images / (ms / 1e3), "ms": ms, "GB/s": gbs, "frac_of_measured_peak": gbs / peak}

    out["noise_philox"] = rate(lambda: plan.noise(src, dst, None, 15.0, seed=1), ALGO_BYTES_PER_IMAGE * n, n)
    out["lowres_1360x765"] = rate(lambda: plan.lowres(src, dst), ALGO_BYTES_PER_IMAGE * n, n)
    # compat noise needs a 4-byte field per element: 64 images (config 1)
    m = min(64, n)
    plan64 = CorruptionPlan.uniform(m, H, W)
    field = torch.randn((m, H, W, 3), dtype=torch.float32, device="cuda") * 15.0
    out["noise_compat_64"] = rate(lambda: plan64.noise(src[:m], dst[:m], field, 15.0), (2 + 4) * IMG_BYTES * m, m)
    del field
    # config 3: 256 mixed-resolution images, fused lowres
    rng = np.random.default_rng(3000)
    pool = VISDRONE_SHAPES + ODD_SHAPES
    shapes = [pool[i] for i in rng.integers(0, len(pool), 256)]
    rp = CorruptionPlan.ragged(shapes)
    rsrc = torch.randint(0, 256, (rp.src_bytes,), dtype=torch.uint8, device="cuda")
    rdst = torch.empty_like(rsrc)
    out["lowres_mixed_256"] = rate(lambda: rp.lowres(rsrc, rdst), 2 * rp.payload_bytes, 256)
    out["lowres_mixed_256"]["shapes"] = "VisDrone set + odd-dimension variants (1361x765, 1917x1079, 1999x1499)"
    out["blur_mixed_256"] = rate(lambda: rp.blur(rsrc, rdst), 2 * rp.payload_bytes, 256)
    out["noise_philox_mixed_256"] = rate(lambda: rp.noise(rsrc, rdst, None, 15.0, seed=3), 2 * rp.payload_bytes, 256)
    del rsrc, rdst, rp
    # LowRes on the 1610-image VisDrone mix alone (config 4's resolution histogram)
    rng = np.random.default_rng(4000)
    shapes = [VISDRONE_SHAPES[i] for i in rng.integers(0, 8, 1610)]
    tp = CorruptionPlan.ragged(shapes)
    tsrc = torch.randint(0, 256, (tp.src_bytes,), dtype=torch.uint8, device="cuda")
    tdst = torch.empty_like(tsrc)
    out["lowres_visdrone_1610"] = rate(lambda: tp.lowres(tsrc, tdst), 2 * tp.payload_bytes, 1610, steps=4, warmup=2)
    del tsrc, tdst, tp
    torch.cuda.empty_cache()
    # even x even frame (the packed-integer kernel) and batch 64 of the training path
    p1080 = CorruptionPlan.uniform(128, 1080, 1920)
    s1080 = torch.randint(0, 256, (128, 1080, 1920, 3), dtype=torch.uint8, device="cuda")
    d1080 = torch.empty_like(s1080)
    out["lowres_1920x1080_128"] = rate(lambda: p1080.lowres(s1080, d1080), 2 * s1080.numel(), 128)
    del s1080, d1080, p1080
    # odd width and height (the odd-width kernel: general INTER_AREA taps in both axes, rows at every byte phase)
    podd = CorruptionPlan.uniform(64, 1079, 1917)
    sodd = torch.randint(0, 256, (64, 1079, 1917, 3), dtype=torch.uint8, device="cuda")
    dodd = torch.empty_like(sodd)
    out["lowres_1917x1079_64"] = rate(lambda: podd.lowres(sodd, dodd), 2 * sodd.numel(), 64)
    del sodd, dodd, podd
    # SURVEY 8f rank 1: device JPEG encoder (files byte-identical to cv2.imwrite's) on 64 frames of the batch; bytes = pixels
    # read + stream written.  Content: uniform noise (the worst case for a JPEG encoder: every coefficient is coded).
    try:
        from robust_object_detection_b200 import _native as N
        from robust_object_detection_b200.batch import _ptr
        from robust_object_detection_b200.jpeg import JpegEncoder
        nj = min(64, n)
        enc = JpegEncoder([(H, W)] * nj, [i * IMG_BYTES for i in range(nj)])
        files = enc.encode(src[:nj])
        stream_bytes = sum(len(f) for f in files if f is not None)
        r = rate(lambda: N.check(N.lib().rod_jpeg_encode(enc._h, _ptr(src), None), "rod_jpeg_encode"), IMG_BYTES * nj + stream_bytes, nj)
        r["compressed_bytes_per_image"] = stream_bytes // nj
        r["content"] = "uniform noise"
        r["bound"] = "entropy coding (instruction / latency), not HBM: the fraction of the copy bandwidth is for scale only"
        out["jpeg_encode_64"] = r
        # ... and the device JPEG decoder (pixels identical to cv2.imread's) on those 64 files: bytes = stream read + pixels
        # written; the call includes the upload of the streams and the host round trips of the synchronisation rounds
        from robust_object_detection_b200.jpeg import JpegDecoder
        dec = JpegDecoder([bytes(f) for f in files], [i * IMG_BYTES for i in range(nj)], host_threads=16)
        back = torch.empty(nj * IMG_BYTES, dtype=torch.uint8, device="cuda")
        r = rate(lambda: dec.decode(back), IMG_BYTES * nj + stream_bytes, nj, steps=5, warmup=2)
        assert (dec.status() == 0).all()
        r["content"] = "the 64 files of jpeg_encode_64 (uniform noise, 1.2 MB each: the slowest content to decode)"
        r["bound"] = "Huffman decoding (dependent bit-buffer chain per symbol, synchronisation rounds), not HBM"
        out["jpeg_decode_64"] = r
        # the same on smooth content (9 x 9 box average of the noise frames: ~0.2 MB per file, what camera frames compress to)
        smooth = torch.nn.functional.avg_pool2d(src[:nj].permute(0, 3, 1, 2).float(), 9, 1, 4).round_().clamp_(0, 255) \
            .to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        files_s = enc.encode(smooth.reshape(-1))
        sbytes = sum(len(f) for f in files_s if f is not None)
        dec_s = JpegDecoder([bytes(f) for f in files_s], [i * IMG_BYTES for i in range(nj)], host_threads=16)
        r = rate(lambda: dec_s.decode(back), IMG_BYTES * nj + sbytes, nj, steps=5, warmup=2)
        assert (dec_s.status() == 0).all()
        r["compressed_bytes_per_image"] = sbytes // nj
        r["content"] = "box-averaged noise (smooth)"
        r["bound"] = "Huffman decoding, not HBM"
        out["jpeg_decode_64_smooth"] = r
        del enc, dec, dec_s, back, smooth
    except Exception as e:  # cv2 (for the header template) is the only extra dependency
        print(f"[bench] JPEG encoder line skipped: {e}", file=sys.stderr)
    import random
    from robust_object_detection_b200.batch import draw_decisions
    random.seed(42)
    p64 = CorruptionPlan.uniform(64, H, W)
    ops = torch.from_numpy(draw_decisions(64)).cuda()
    f16 = torch.empty((64, 3, 640, 640), dtype=torch.float16, device="cuda")
    out["train_letterbox_b64"] = rate(lambda: p64.corrupt_letterbox(src[:64], ops, f16, 640, 640, 114, seed=1),
                                      64 * (IMG_BYTES + 640 * 640 * 3 * 2), 64, steps=20, warmup=3)
    return out


if __name__ == "__main__":
    main()
