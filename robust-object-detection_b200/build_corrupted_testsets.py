"""Drop-in for scripts/build_corrupted_testsets.py of ysbbin/Robust-Object-Detection (SURVEY 8a row a9, 8f rank 1).

Same module surface (constants, set_seed, build_yolo_testsets, build_coco_testsets, main), same on-disk result:
for Test_Clean / Test_Noise / Test_Blur / Test_LowRes the images of `images/val` are read with cv2.imread, corrupted and
written with cv2.imwrite under the same file name; labels / annotations are copied; data.yaml is written
(build_corrupted_testsets.py:62-166).  The corruption itself runs on the GPU, one ragged batch at a time
and so does the JPEG codec on both sides of it.  JPEG DECODING (`DECODER = "gpu"`: rod_jpegdec_decode, libjpeg-turbo's
Huffman decoding / islow IDCT / fancy upsampling / colour conversion restated in CUDA, pixels identical to cv2.imread's): the
I/O threads only read the files; a file of a layout the device decoder does not take (progressive, other chroma sampling,
EXIF rotation, CMYK, PNG ...) is read with cv2.imread like the reference does.  A tree's decoded batches stay on
the device for its four variants.  `DECODER = "host"` decodes with cv2.imread on the I/O threads (the next batch decodes
while a batch is on the GPU; a tree's decoded frames are reused by its four variants).  JPEG ENCODING runs on the GPU too
(`ENCODER = "gpu"`: rod_jpeg_encode, libjpeg-turbo's integer algorithms restated in CUDA, the header bytes taken from
OpenCV itself): the corrupted frames never leave the device, only the compressed streams do, and the files are
byte-identical to cv2.imwrite's (tested).  `ENCODER = "host"` keeps cv2.imwrite on the I/O threads (rod_apply_host:
pinned staging, chunked H2D / kernel / D2H); other file types than .jpg / .jpeg always take that route.

RNG: Test_Noise draws each image's field from NumPy's global legacy generator in glob order after np.random.seed(SEED)
-- the same stream as the reference's np.random.normal calls, regenerated bit for bit: on the GPU, one draw per batch
(csrc/legacy_rng.cu) with the device encoder; on the host (csrc/np_legacy_rng.cpp, per-sample math on all host threads)
with `ENCODER = "host"` -- so the noisy files are byte-identical too.
`NOISE_MODE = "philox"` generates the field on the GPU instead (statistically equivalent, not byte-identical).

Several GPUs (BASELINE configs[3], SURVEY 8e): started under `torchrun --nproc-per-node N` (RANK / WORLD_SIZE / LOCAL_RANK
in the environment) every rank builds the same directory trees, owns one contiguous block of each image directory's glob
list -- blocks balanced by file size (sharding.shard_by_bytes), no pixel ever crosses ranks, no collective -- and uses
GPU LOCAL_RANK; rank 0 alone copies labels / annotations and writes data.yaml.  The files are the ones a single process
writes: Philox noise is keyed by an image's position in the glob list, and compat noise -- one serial NumPy stream -- is
left to rank 0 for the whole directory while the other ranks go on with Test_Blur / Test_LowRes.
"""
from __future__ import annotations

import os
import shutil
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

from . import _native as N
from .augmentations import apply_lowres, apply_motion_blur, apply_noise  # noqa: F401  (same names as the reference)
from .augmentations import legacy_normal_f32, legacy_normal_f32_device
from .augmentations import _motion_blur_kernel as motion_blur_kernel  # noqa: F401
from .batch import CorruptionPlan
from .sharding import shard_by_bytes

# ====== paths (same defaults as the reference, build_corrupted_testsets.py:8-10) ======
YOLO_SRC = Path("data/processed/visdrone_yolo6")
COCO_SRC = Path("data/processed/visdrone_coco6")
OUT_ROOT = Path("data/testsets")

# ====== corruption parameters (build_corrupted_testsets.py:13-23) ======
SEED = 42
NOISE_SIGMA = 15
BLUR_KERNEL = 9
BLUR_ANGLE_DEG = 0
DOWNSCALE_FACTOR = 0.5

# ====== B200 path knobs ======
NOISE_MODE = "compat"      # "compat": host np.random stream (byte-identical) | "philox": in-kernel RNG
PHILOX_SEED = SEED
BATCH_BYTES = 512 << 20    # decoded source bytes per GPU batch
NOISE_BATCH_BYTES = 128 << 20   # ... of a compat-noise batch on the host-encoder path (its float32 field is 4x that, page-locked)
IO_THREADS = 16
DECODER = "gpu"            # "gpu": device JPEG decoder for .jpg / .jpeg sources (same pixels as cv2.imread; needs ENCODER = "gpu") | "host": cv2.imread
ENCODER = "gpu"            # "gpu": device JPEG encoder for .jpg / .jpeg outputs (same bytes as cv2.imwrite) | "host": cv2.imwrite
DECODE_CACHE_BYTES = 8 << 30  # decoded frames of one tree kept for its later variants (548 VisDrone val frames ~ 2.3 GB)
DEVICE_CACHE_BYTES = 8 << 30   # ... and their uploaded batches kept on the GPU with their JPEG encoders (ENCODER = "gpu"; ~5 bytes of device memory per cached byte)

SHARD = "env"              # "env": RANK / WORLD_SIZE of torchrun decide | (rank, world) | None: this process does everything

VARIANTS = ["Test_Clean", "Test_Noise", "Test_Blur", "Test_LowRes"]
_OPS = {"Test_Noise": N.OP_NOISE, "Test_Blur": N.OP_BLUR, "Test_LowRes": N.OP_LOWRES}


def _rank_world():
    """(rank, world) of this process: torchrun's environment, or the SHARD knob."""
    if SHARD is None:
        return 0, 1
    if SHARD == "env":
        rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    else:
        rank, world = (int(v) for v in SHARD)
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad shard {rank} of {world}")
    return rank, world


def _shard_of(paths, variant: str):
    """[lo, hi) of the glob list this rank owns for one variant (see the module docstring)."""
    rank, world = _rank_world()
    if world == 1:
        return 0, len(paths)
    if variant == "Test_Noise" and NOISE_MODE == "compat":   # np.random's stream is serial: one rank draws all of it
        return (0, len(paths)) if rank == 0 else (0, 0)
    return shard_by_bytes([p.stat().st_size for p in paths], world)[rank]


def set_seed(seed: int):
    np.random.seed(seed)


def ensure_dir(p: Path):
    p.mkdir(parents=True, exist_ok=True)


def write_yolo_valonly_yaml(dst_root: Path):
    """data.yaml that evaluates on this test set's val folder (build_corrupted_testsets.py:66-82)."""
    lines = [f"path: {dst_root.as_posix()}", "train: images/val", "val: images/val", "", "names:",
             "  0: pedestrian", "  1: car", "  2: van", "  3: truck", "  4: bus", "  5: motor"]
    (dst_root / "data.yaml").write_text("\n".join(lines), encoding="utf-8")


def _corrupt_batch(variant: str, images, philox_index: int, run: "_TreeRun" = None):
    """One ragged batch through the GPU; returns the corrupted arrays (views into one host buffer).  With a _TreeRun the
    batch is packed into / returned in page-locked buffers (packing spread over the I/O threads): pageable buffers cost
    more in the two PCIe copies than the corruption itself."""
    shapes = [(im.shape[0], im.shape[1]) for im in images]
    plan = CorruptionPlan.ragged(shapes)
    if run is not None:
        src = run.pinned("src", plan.src_bytes)
        dst = run.pinned_out(plan.dst_bytes)

        def put(args):
            im, off = args
            src[off:off + im.size].reshape(im.shape)[...] = im

        list(run.pool.map(put, zip(images, plan.src_offsets)))
    else:
        src = plan.pack(images)
        dst = np.empty(plan.dst_bytes, dtype=np.uint8)
    op = _OPS[variant]
    noise = None
    if variant == "Test_Noise" and NOISE_MODE == "compat":
        # the draws of augmentations.py:31, one per image, in order
        total = sum(im.size for im in images)
        # drawn straight into a page-locked buffer kept for the run (a fresh pageable 4-bytes-per-pixel array costs
        # more in page faults and in the upload than the GPU work)
        noise = run.pinned("noise", 4 * total).view(np.float32) if run is not None else np.empty(total, dtype=np.float32)
        o = 0
        for im in images:  # np.random.normal(0, NOISE_SIGMA, im.shape).astype(np.float32), bit for bit, multi-threaded
            legacy_normal_f32(NOISE_SIGMA, im.shape, out=noise[o:o + im.size])
            o += im.size
    if variant == "Test_Blur" and float(BLUR_ANGLE_DEG) != 0.0:
        plan.set_blur_kernel(motion_blur_kernel(BLUR_KERNEL, BLUR_ANGLE_DEG))
    plan.apply_host(op, src, dst, noise_host=noise, sigma=float(NOISE_SIGMA), k=int(BLUR_KERNEL),
                    factor=float(DOWNSCALE_FACTOR), seed=PHILOX_SEED, first_image_index=philox_index)
    return plan.unpack(dst)


def _write_bytes(path: str, data) -> bool:
    """data: (header bytes, view of the downloaded stream): written by the I/O threads straight from the page-locked buffer"""
    with open(path, "wb") as f:
        f.write(data[0])
        f.write(data[1])
    return True


class _Encoded:
    """A source file the device decoder takes: its bytes and the size cv2.imread would return."""
    __slots__ = ("data", "shape")

    def __init__(self, data, shape):
        self.data, self.shape = data, shape


def _load_source(path: Path, run: "_TreeRun"):
    """What an I/O thread does for one source file: with the device decoder the file bytes (+ the frame size from the
    header); else -- host decoder, other file types, layouts the device decoder does not take -- cv2.imread's array.  None:
    unreadable (the reference skips such files, build_corrupted_testsets.py:110-111)."""
    if DECODER == "gpu" and ENCODER == "gpu" and path.suffix.lower() in (".jpg", ".jpeg"):
        from .jpeg import probe
        try:
            data = path.read_bytes()
        except OSError:
            return None
        shape = probe(data)
        if shape is not None:
            return _Encoded(data, shape)
    return run.decode(path)


class _DeviceRun:
    """Consecutive readable files of one directory on the device: the plan of their sizes, the decoded frames, the JPEG
    encoder for that layout; `skip`: images whose entropy-coded data turned out to be broken and that OpenCV cannot read either."""
    __slots__ = ("pos", "paths", "plan", "src_dev", "enc", "skip")


def _upload_run(pos: int, items, run: "_TreeRun") -> "_DeviceRun":
    """items: [(path, _Encoded | ndarray)].  Decodes / uploads them into one device batch."""
    import cv2
    import torch
    from .jpeg import JpegDecoder, JpegEncoder
    r = _DeviceRun()
    r.pos, r.paths, r.skip = pos, [p for p, _ in items], set()
    shapes = [(it.shape[0], it.shape[1]) for _, it in items]
    r.plan = CorruptionPlan.ragged(shapes)
    r.src_dev = torch.empty(r.plan.src_bytes, dtype=torch.uint8, device="cuda")
    enc_idx = [i for i, (_, it) in enumerate(items) if isinstance(it, _Encoded)]
    dec = None
    if enc_idx:
        dec = JpegDecoder([items[i][1].data for i in enc_idx], [r.plan.src_offsets[i] for i in enc_idx], host_threads=IO_THREADS)
        dec.decode(r.src_dev)

    def put(i, arr):   # (late, rare: pageable copy)
        off = r.plan.src_offsets[i]
        r.src_dev[off:off + arr.size].copy_(torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)))

    host_idx = [i for i, (_, it) in enumerate(items) if not isinstance(it, _Encoded)]
    if host_idx:   # frames decoded by the host codec: packed into page-locked memory by the I/O threads, then uploaded
        src = run.pinned("src", r.plan.src_bytes)

        def pack(i):
            im, off = items[i][1], r.plan.src_offsets[i]
            src[off:off + im.size].reshape(im.shape)[...] = im

        list(run.pool.map(pack, host_idx))
        pinned = run.pinned_tensor("src", r.plan.src_bytes)
        if len(host_idx) == len(items):
            r.src_dev = pinned.cuda(non_blocking=True)
        else:
            for i in host_idx:
                off, n = r.plan.src_offsets[i], items[i][1].size
                r.src_dev[off:off + n].copy_(pinned[off:off + n], non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the page-locked buffer is repacked for the next run
    if dec is not None:
        for i, st in zip(enc_idx, dec.status()):
            if st != 0:   # broken entropy-coded data: whatever OpenCV makes of the file is the reference's answer
                arr = cv2.imread(str(items[i][0]))
                if arr is not None and arr.shape[:2] == shapes[i] and arr.ndim == 3:
                    put(i, arr)
                else:
                    r.skip.add(i)
    r.enc = JpegEncoder(shapes, r.plan.dst_offsets)
    return r


def _corrupt_encode(variant: str, r: "_DeviceRun", run: "_TreeRun"):
    """One device batch: corrupt (Test_Clean: nothing), JPEG-encode; returns the write jobs [(function, path, payload)]
    -- encoded files as bytes, everything that is not a .jpg / .jpeg (or did not fit the encoder's buffers) as a decoded
    array for cv2.imwrite."""
    import cv2
    import torch
    plan, src_dev = r.plan, r.src_dev
    if variant == "Test_Clean":
        pix = src_dev
    else:
        pix = torch.empty(plan.dst_bytes, dtype=torch.uint8, device="cuda")
        if variant == "Test_Noise":
            field = None
            if NOISE_MODE == "compat":   # the draws of augmentations.py:31, one per image, in order: one device draw
                # (indexed by the plan's packed element index -- images back to back -- as rod_noise_u8 expects)
                total = sum(3 * h * w for h, w in plan.shapes)
                field = torch.empty(total, dtype=torch.float32, device="cuda")
                legacy_normal_f32_device(NOISE_SIGMA, field, [(0, total)])
            plan.noise(src_dev, pix, field, float(NOISE_SIGMA), seed=PHILOX_SEED, first_image_index=r.pos)
        elif variant == "Test_Blur":
            if float(BLUR_ANGLE_DEG) != 0.0:
                plan.set_blur_kernel(motion_blur_kernel(BLUR_KERNEL, BLUR_ANGLE_DEG))
            plan.blur(src_dev, pix, int(BLUR_KERNEL), float(BLUR_ANGLE_DEG))
        else:
            plan.lowres(src_dev, pix, float(DOWNSCALE_FACTOR))
    files = r.enc.encode(pix, copy=False)   # views into a ring of three download buffers; at most two batches of writes are pending
    jobs = []
    for i, (p, data, off, (h, w)) in enumerate(zip(r.paths, files, plan.dst_offsets, plan.shapes)):
        if i in r.skip:
            continue
        if data is not None and p.suffix.lower() in (".jpg", ".jpeg"):
            jobs.append((_write_bytes, p, data))
        else:
            jobs.append((cv2.imwrite, p, pix[off:off + 3 * h * w].cpu().numpy().reshape(h, w, 3)))
    return jobs


class _TreeRun:
    """Host-side pipeline state of one source tree (its four variants): the I/O thread pool, the decoded frames of the
    tree (the reference re-reads every file for every variant, build_corrupted_testsets.py:109/:149; here variants 2-4
    reuse the arrays of variant 1 while they fit DECODE_CACHE_BYTES) and the imwrite futures still in flight (encoding
    of one batch overlaps decoding / corrupting the next; at most two batches of output buffers are alive)."""

    def __init__(self):
        # compat noise draws np.random.normal on the calling thread (the serial bottleneck of that mode): leave it a core
        import os
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self.pool = ThreadPoolExecutor(max(1, min(IO_THREADS, cores - 2)) if NOISE_MODE == "compat" else IO_THREADS)
        self.cache = {}
        self.cache_bytes = 0
        self.dev_cache = {}    # batch (tuple of paths) -> [_DeviceRun]: decoded frames, plan and JPEG encoder of its readable runs
        self.dev_cache_bytes = 0
        self.pending = []  # one list of futures per batch in flight
        self._pinned = {}  # name -> page-locked torch uint8 tensor (grow-only)
        self._out_turn = 0

    def pinned(self, name: str, nbytes: int) -> np.ndarray:
        """A page-locked host buffer of at least nbytes, kept for the run (pinning is slow: ~0.3 s per GB)."""
        import torch
        t = self._pinned.get(name)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(int(nbytes), 1), dtype=torch.uint8).pin_memory()
            self._pinned[name] = t
        return t.numpy()[:nbytes]

    def pinned_tensor(self, name: str, nbytes: int):
        """The page-locked torch tensor behind pinned(name, ...) (for asynchronous uploads)."""
        return self._pinned[name][:nbytes]

    def pinned_out(self, nbytes: int) -> np.ndarray:
        """Output buffers rotate over three slots: the imwrite futures of at most two batches still read theirs."""
        self._out_turn = (self._out_turn + 1) % 3
        return self.pinned(f"dst{self._out_turn}", nbytes)

    def decode(self, path: Path):
        import cv2
        im = self.cache.get(path)
        return im if im is not None else cv2.imread(str(path))

    def remember(self, path: Path, im):
        if path not in self.cache and self.cache_bytes + im.nbytes <= DECODE_CACHE_BYTES:
            self.cache[path] = im
            self.cache_bytes += im.nbytes

    def drain(self, keep: int = 0):
        while len(self.pending) > keep:
            for f in self.pending.pop(0):
                if not f.result():
                    raise IOError("cv2.imwrite failed")

    def submit_writes(self, jobs):
        """[(function, path, payload)] spread over the I/O threads, a slice of the files per task (a future per file costs
        more than writing a VisDrone-sized JPEG to a page-cached file system)"""
        n = max(1, min(len(jobs), self.pool._max_workers))

        def write_slice(part):
            return all(fn(path, payload) for fn, path, payload in part)

        return [self.pool.submit(write_slice, jobs[k::n]) for k in range(n)]

    def close(self):
        self.drain()
        self.pool.shutdown()


def _process_images(src_img_dir: Path, dst_img_dir: Path, variant: str, run: "_TreeRun" = None):
    """The image loop of build_corrupted_testsets.py:108-124 / :148-164 for one variant, batched."""
    import cv2
    own = run is None
    if own:
        run = _TreeRun()
    paths = list(src_img_dir.glob("*.*"))  # filesystem order, like the reference (it fixes the noise stream order)
    lo, hi = _shard_of(paths, variant)
    paths = paths[lo:hi]

    device = ENCODER == "gpu"
    # the host-encoder path stages compat noise as a float32 field of 4 bytes per pixel byte in page-locked memory:
    # smaller batches there.  The device path draws the field on the GPU, so its batches are those of the other variants
    # (and so hit the device cache of the tree's decoded batches).
    host_field = variant == "Test_Noise" and NOISE_MODE == "compat" and not device
    cap = min(BATCH_BYTES, NOISE_BATCH_BYTES) if host_field else BATCH_BYTES

    def submit_loads(i):
        """read / decode ahead until the batch is full (cv2 and file reads release the GIL); a batch that is still on the
        device from an earlier variant of this tree is not read again"""
        batch_paths, nbytes = [], 0
        while i < len(paths) and (nbytes < cap or not batch_paths):
            batch_paths.append((lo + i, paths[i]))
            i += 1
            nbytes += 6 << 20  # ~ a decoded VisDrone frame; the real size is known after decoding
        key = tuple(p for _, p in batch_paths)
        if device and key in run.dev_cache:
            return i, batch_paths, None
        load = (lambda p: _load_source(p, run)) if device else run.decode
        return i, batch_paths, [run.pool.submit(load, p) for _, p in batch_paths]

    def readable_runs(batch_paths, futs):
        """The batch without its unreadable files (skipped like the reference does, :110-111), cut where one was skipped:
        a GPU batch numbers its images consecutively from its first one's position in the glob list (the Philox key)."""
        runs, prev = [], None
        for (pos, p), f in zip(batch_paths, futs):
            im = f.result()
            if im is None:
                continue
            if prev is None or pos != prev + 1:
                runs.append((pos, []))
            runs[-1][1].append((p, im))
            prev = pos
        return runs

    dst_dir_s = str(dst_img_dir)
    i, batch_paths, futs = submit_loads(0)
    while batch_paths:
        cur_paths, cur_futs = batch_paths, futs
        if device:
            key = tuple(p for _, p in cur_paths)
            dev_runs = run.dev_cache.get(key)
            if dev_runs is None:
                work = readable_runs(cur_paths, cur_futs)
                i, batch_paths, futs = submit_loads(i)  # the next batch is read while this one is decoded, corrupted and encoded
                dev_runs = [_upload_run(pos, items, run) for pos, items in work]
                nbytes = sum(r.plan.src_bytes for r in dev_runs)
                if run.dev_cache_bytes + nbytes <= DEVICE_CACHE_BYTES:
                    run.dev_cache[key] = dev_runs
                    run.dev_cache_bytes += nbytes
            else:
                i, batch_paths, futs = submit_loads(i)
            for r in dev_runs:
                run.drain(keep=1)  # the encoder's download ring has three buffers: at most two batches of writes are pending
                jobs = _corrupt_encode(variant, r, run)
                run.pending.append(run.submit_writes([(fn, os.path.join(dst_dir_s, p.name), payload) for fn, p, payload in jobs]))
            continue
        work = readable_runs(cur_paths, cur_futs)
        i, batch_paths, futs = submit_loads(i)  # the next batch decodes while this one is corrupted and encoded
        for philox_index, decoded in work:
            for p, im in decoded:
                run.remember(p, im)
            images = [im for _, im in decoded]
            if variant == "Test_Clean":
                outs = images
            else:
                run.drain(keep=1)  # before the third output slot back is reused
                outs = _corrupt_batch(variant, images, philox_index, run)
            run.drain(keep=1)
            run.pending.append([run.pool.submit(cv2.imwrite, str(dst_img_dir / p.name), o) for (p, _), o in zip(decoded, outs)])
    if own:
        run.close()


def build_yolo_testsets():
    src_img_dir = YOLO_SRC / "images" / "val"
    src_lbl_dir = YOLO_SRC / "labels" / "val"
    if not src_img_dir.exists() or not src_lbl_dir.exists():
        raise FileNotFoundError("YOLO val images/labels not found. Check YOLO_SRC path.")
    run = _TreeRun()
    for v in VARIANTS:
        dst_root = OUT_ROOT / "yolo6" / v
        dst_img_dir = dst_root / "images" / "val"
        dst_lbl_dir = dst_root / "labels" / "val"
        ensure_dir(dst_img_dir)
        ensure_dir(dst_lbl_dir)
        if _rank_world()[0] == 0:
            for lbl in src_lbl_dir.glob("*.txt"):
                shutil.copy2(lbl, dst_lbl_dir / lbl.name)
            write_yolo_valonly_yaml(dst_root)
        _process_images(src_img_dir, dst_img_dir, v, run)
    run.close()
    if _rank_world()[0] == 0:
        print("YOLO test sets created:", (OUT_ROOT / "yolo6").resolve())


def build_coco_testsets():
    src_img_dir = COCO_SRC / "images" / "val"
    src_ann = COCO_SRC / "annotations" / "instances_val.json"
    if not src_img_dir.exists() or not src_ann.exists():
        raise FileNotFoundError("COCO val images or instances_val.json not found. Check COCO_SRC path.")
    run = _TreeRun()
    for v in VARIANTS:
        dst_root = OUT_ROOT / "coco6" / v
        dst_img_dir = dst_root / "images" / "val"
        dst_ann_dir = dst_root / "annotations"
        ensure_dir(dst_img_dir)
        ensure_dir(dst_ann_dir)
        if _rank_world()[0] == 0:
            shutil.copy2(src_ann, dst_ann_dir / "instances_val.json")
        _process_images(src_img_dir, dst_img_dir, v, run)
    run.close()
    if _rank_world()[0] == 0:
        print("COCO test sets created:", (OUT_ROOT / "coco6").resolve())


def main():
    set_seed(SEED)
    rank, world = _rank_world()
    if world > 1 and "LOCAL_RANK" in os.environ:   # one process per GPU
        import torch
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]) % max(1, torch.cuda.device_count()))
    build_yolo_testsets()
    build_coco_testsets()
    if rank == 0:
        print("\nAll corrupted test sets are ready under:", OUT_ROOT.resolve(),
              "" if world == 1 else f"(this is rank 0 of {world}: the other ranks finish on their own)")


if __name__ == "__main__":
    main()
