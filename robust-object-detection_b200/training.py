"""Main-process training hook (SURVEY 8f rank 2): corruption + detector-input formatting on the GPU, fed from
pinned host memory, for the Ultralytics launchers of the reference.

The reference runs the corruption inside 8 DataLoader workers (scripts/augmentations.py:91-95,
scripts/train_yolo_augmented.py:33).  The unmodified launchers keep working through the per-image drop-in functions in
spawned workers (augmentations.patch_ultralytics_augmentations selects the start method); per-image host calls are
PCIe-latency bound, though, so for custom training loops this module offers the batch form in the main process: raw HWC BGR uint8 frames of one batch go through ONE pinned staging buffer and ONE H2D copy, the
decisions are drawn from Python's `random` in the reference's order (random() < 0.5, then random.choice), and
`rod_corrupt_letterbox_f16` produces the fp16 NCHW tensor the detector consumes.  Two staging slots and a copy
stream let batch i+1 upload while batch i is being corrupted.
"""
from __future__ import annotations

from typing import Iterable, Iterator, List, Optional, Sequence, Tuple

import numpy as np

from .batch import CorruptionPlan, draw_decisions


class CorruptionBatcher:
    """Double-buffered host->device pipeline around CorruptionPlan.corrupt_letterbox.

        batcher = CorruptionBatcher(out_hw=(640, 640), seed=42)
        for x in batcher.run(batches):      # batches: iterable of lists of HWC BGR uint8 arrays
            loss = model(x)                 # x: torch.float16 [B,3,640,640] RGB in [0,1], on the GPU

    Per batch: `draw_decisions(B, gate)` consumes the global `random` stream exactly as B consecutive calls of the
    reference hook would; Philox noise is keyed by (seed, running global image index), so a run is reproducible
    and independent of how images are grouped into batches.
    """

    def __init__(self, out_hw: Tuple[int, int] = (640, 640), pad_value: int = 114, gate: str = "ultralytics",
                 seed: int = 0, max_cached_plans: int = 16):
        import torch
        self._torch = torch
        self.out_h, self.out_w = int(out_hw[0]), int(out_hw[1])
        self.pad_value, self.gate, self.seed = int(pad_value), gate, int(seed)
        self._plans: dict = {}
        self._max_plans = max_cached_plans
        self._copy_stream = torch.cuda.Stream()
        from concurrent.futures import ThreadPoolExecutor
        import os
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        self._pack_pool = ThreadPoolExecutor(max(1, min(int(os.environ.get("ROD_PACK_THREADS", "8")), cores)))
        self._slots: List[dict] = [{}, {}]
        self.images_seen = 0

    # ------------------------------------------------------------------ internals
    def _plan(self, shapes: Sequence[Tuple[int, int]]) -> CorruptionPlan:
        key = tuple(shapes)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) >= self._max_plans:
                self._plans.pop(next(iter(self._plans)))
            plan = CorruptionPlan.ragged(shapes)
            self._plans[key] = plan
        return plan

    def _stage(self, slot: dict, images: Sequence[np.ndarray], ops: Optional[np.ndarray]):
        """Pack one batch into the slot's pinned buffer and start its H2D copy on the copy stream."""
        torch = self._torch
        shapes = [(int(im.shape[0]), int(im.shape[1])) for im in images]
        plan = self._plan(shapes)
        nbytes = plan.src_bytes
        if slot.get("cap", 0) < nbytes:
            cap = max(nbytes, 2 * slot.get("cap", 0))
            slot["host"] = torch.empty(cap, dtype=torch.uint8).pin_memory()
            slot["dev"] = torch.empty(cap, dtype=torch.uint8, device="cuda")
            slot["cap"] = cap
            # the caching allocator may hand out a block whose last use (a previous step's output, activations) is still
            # pending on the compute stream; the copy stream must not write it before that work has finished
            self._copy_stream.wait_stream(torch.cuda.current_stream())
        ev = slot.get("free")
        if ev is not None:
            ev.synchronize()  # the compute that last read this slot's device buffer has finished
        hbuf = slot["host"].numpy()
        for im in images:
            if im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3:
                raise ValueError("expected HWC uint8 BGR frames")

        def pack(args):  # one frame into the pinned buffer (NumPy releases the GIL for the copy)
            im, off, (h, w) = args
            hbuf[off:off + 3 * h * w].reshape(h, w, 3)[...] = im

        # the packing copy is the host-side cost of a batch (50 MB for 16 VisDrone frames): spread it over threads
        list(self._pack_pool.map(pack, zip(images, plan.src_offsets, shapes)))
        if ops is None:
            ops = draw_decisions(len(images), gate=self.gate)
        n = len(images)
        if slot.get("ops_cap", 0) < n:
            slot["ops_host"] = torch.empty(max(n, 64), dtype=torch.uint8).pin_memory()
            slot["ops_dev"] = torch.empty(max(n, 64), dtype=torch.uint8, device="cuda")
            slot["ops_cap"] = max(n, 64)
            self._copy_stream.wait_stream(torch.cuda.current_stream())
        slot["ops_host"][:n] = torch.from_numpy(np.asarray(ops, dtype=np.uint8))
        with torch.cuda.stream(self._copy_stream):
            slot["dev"][:nbytes].copy_(slot["host"][:nbytes], non_blocking=True)
            slot["ops_dev"][:n].copy_(slot["ops_host"][:n], non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._copy_stream)
        slot.update(plan=plan, n=n, ready=ready, ops=np.asarray(ops, dtype=np.uint8), first_index=self.images_seen)
        self.images_seen += n

    def _compute(self, slot: dict):
        torch = self._torch
        cur = torch.cuda.current_stream()
        cur.wait_event(slot["ready"])
        n = slot["n"]
        out = torch.empty((n, 3, self.out_h, self.out_w), dtype=torch.float16, device="cuda")
        slot["plan"].corrupt_letterbox(slot["dev"], slot["ops_dev"], out, self.out_h, self.out_w, self.pad_value,
                                       seed=self.seed, first_image_index=slot["first_index"])
        free = torch.cuda.Event()
        free.record(cur)
        slot["free"] = free
        return out

    # ------------------------------------------------------------------ public
    def __call__(self, images: Sequence[np.ndarray], ops: Optional[np.ndarray] = None):
        """One batch, no overlap: returns the fp16 [B,3,H,W] tensor (and leaves the drawn op-codes in .last_ops)."""
        slot = self._slots[0]
        self._stage(slot, images, ops)
        self.last_ops = slot["ops"]
        return self._compute(slot)

    def run(self, batches: Iterable[Sequence[np.ndarray]]) -> Iterator:
        """Pipelined: while batch i is corrupted on the current stream, batch i+1 is packed and uploaded."""
        it = iter(batches)
        try:
            first = next(it)
        except StopIteration:
            return
        k = 0
        self._stage(self._slots[0], first, None)
        while True:
            cur = self._slots[k & 1]
            try:
                nxt = next(it)
            except StopIteration:
                nxt = None
            if nxt is not None:
                self._stage(self._slots[(k + 1) & 1], nxt, None)
            self.last_ops = cur["ops"]
            yield self._compute(cur)
            if nxt is None:
                return
            k += 1


class FileCorruptionBatcher:
    """The augmented dataloader path from image FILES (BASELINE config 5 as the trainers meet it: Ultralytics' workers
    start from `cv2.imread`): a batch of JPEG files is read by I/O threads, decoded on the GPU (jpeg.JpegDecoder: the pixels
    of cv2.imread), corrupted and letterboxed by the fused kernel -- decoded frames never exist in host memory.  Files the
    device decoder does not take (progressive, PNG, ...) are decoded by the host codec and uploaded into their slot.

        batcher = FileCorruptionBatcher(out_hw=(640, 640), seed=42)
        for x in batcher.run(batches):      # batches: iterable of lists of paths (or of bytes objects)
            loss = model(x)                 # x: torch.float16 [B,3,640,640] RGB in [0,1], on the GPU

    Decisions and Philox keying as in CorruptionBatcher: the result equals CorruptionBatcher's on the cv2.imread frames.
    """

    def __init__(self, out_hw: Tuple[int, int] = (640, 640), pad_value: int = 114, gate: str = "ultralytics",
                 seed: int = 0, io_threads: int = 16, max_cached_plans: int = 16):
        import torch
        from concurrent.futures import ThreadPoolExecutor
        self._torch = torch
        self.out_h, self.out_w = int(out_hw[0]), int(out_hw[1])
        self.pad_value, self.gate, self.seed = int(pad_value), gate, int(seed)
        self._plans: dict = {}
        self._max_plans = max_cached_plans
        self._pool = ThreadPoolExecutor(max(1, int(io_threads)))
        self._io_threads = max(1, int(io_threads))
        self.images_seen = 0

    def _plan(self, shapes) -> CorruptionPlan:
        key = tuple(shapes)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) >= self._max_plans:
                self._plans.pop(next(iter(self._plans)))
            plan = self._plans[key] = CorruptionPlan.ragged(shapes)
        return plan

    @staticmethod
    def _load(item):
        """I/O thread: (file bytes, (h, w)) for a file the device decoder takes, else (decoded array, (h, w))."""
        from .jpeg import probe
        data = item if isinstance(item, (bytes, bytearray, memoryview)) else open(item, "rb").read()
        shape = probe(data)
        if shape is not None:
            return data, shape
        import cv2
        arr = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        if arr is None:
            raise IOError(f"unreadable image: {item if not isinstance(item, (bytes, bytearray, memoryview)) else '<bytes>'}")
        return arr, (int(arr.shape[0]), int(arr.shape[1]))

    def _submit(self, items):
        return [self._pool.submit(self._load, it) for it in items]

    def _finish(self, items, futs, ops):
        torch = self._torch
        from .jpeg import JpegDecoder
        loaded = [f.result() for f in futs]
        shapes = [sh for _, sh in loaded]
        plan = self._plan(shapes)
        dev = torch.empty(plan.src_bytes, dtype=torch.uint8, device="cuda")
        enc = [i for i, (d, _) in enumerate(loaded) if not isinstance(d, np.ndarray)]
        if enc:
            dec = JpegDecoder([loaded[i][0] for i in enc], [plan.src_offsets[i] for i in enc], host_threads=self._io_threads)
            dec.decode(dev)
        for i, (d, (h, w)) in enumerate(loaded):
            if isinstance(d, np.ndarray):
                off = plan.src_offsets[i]
                dev[off:off + 3 * h * w].copy_(torch.from_numpy(np.ascontiguousarray(d).reshape(-1)))
        if enc:
            import cv2
            for i, st in zip(enc, dec.status()):
                if st != 0:   # broken entropy-coded data: OpenCV's reading of the file is the reference's answer
                    arr = cv2.imdecode(np.frombuffer(loaded[i][0], np.uint8), cv2.IMREAD_COLOR)
                    if arr is None or (int(arr.shape[0]), int(arr.shape[1])) != shapes[i]:
                        raise IOError("unreadable image in batch")
                    off = plan.src_offsets[i]
                    dev[off:off + arr.size].copy_(torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)))
        n = len(items)
        if ops is None:
            ops = draw_decisions(n, gate=self.gate)
        self.last_ops = np.asarray(ops, dtype=np.uint8)
        ops_dev = torch.from_numpy(self.last_ops).cuda()
        out = torch.empty((n, 3, self.out_h, self.out_w), dtype=torch.float16, device="cuda")
        plan.corrupt_letterbox(dev, ops_dev, out, self.out_h, self.out_w, self.pad_value, seed=self.seed,
                               first_image_index=self.images_seen)
        self.images_seen += n
        return out

    def __call__(self, items: Sequence, ops: Optional[np.ndarray] = None):
        """One batch of paths / bytes objects -> the fp16 [B,3,H,W] tensor (the drawn op-codes are left in .last_ops)."""
        return self._finish(items, self._submit(items), ops)

    def run(self, batches: Iterable[Sequence]) -> Iterator:
        """Pipelined: the files of batch i+1 are read while batch i is decoded, corrupted and letterboxed."""
        it = iter(batches)
        try:
            cur = next(it)
        except StopIteration:
            return
        futs = self._submit(cur)
        while True:
            try:
                nxt = next(it)
            except StopIteration:
                nxt = None
            nfuts = self._submit(nxt) if nxt is not None else None
            yield self._finish(cur, futs, None)
            if nxt is None:
                return
            cur, futs = nxt, nfuts


class RestorationPairBatcher:
    """Host-level drop-in for the pair generation of RestorationDataset.__getitem__ (train_restoration.py:104-129), one
    batch at a time: for every decoded frame (HWC BGR uint8; smaller than patch_size: enlarged first like the reference) the decisions are
    drawn in the reference's order (random crop position, flip, random.choice of the corruption; centre crop and no
    flip for validation), only the CROP is uploaded (the frame itself never leaves the host), and
    rod_restoration_pairs_f32 produces both tensors on the device:

        pairs = RestorationPairBatcher(patch_size=256, is_train=True)
        corrupted, clean = pairs(frames)        # float32 [B,3,P,P] RGB in [0,1], on the GPU

    noise="compat" draws each noise patch's field from NumPy's global legacy stream (bit-identical to the reference under
    the same seeds: augmentations.legacy_normal_f32_device, one draw per batch on the GPU); noise="philox" generates it in the kernel, keyed by (seed, running
    sample index)."""

    def __init__(self, patch_size: int = 256, is_train: bool = True, noise: str = "compat", seed: int = 0):
        import torch
        if noise not in ("compat", "philox"):
            raise ValueError("noise must be 'compat' or 'philox'")
        self._torch = torch
        self.size, self.is_train, self.noise, self.seed = int(patch_size), bool(is_train), noise, int(seed)
        self._plans: dict = {}
        self.samples_seen = 0
        self.last_decisions: List[tuple] = []

    def __call__(self, frames: Sequence[np.ndarray]):
        from .batch import draw_restoration_decisions, resize_linear_u8
        torch, P, n = self._torch, self.size, len(frames)
        if n not in self._plans:  # crops are staged back to back: one plan per batch size
            offs = [i * 3 * P * P for i in range(n)]
            self._plans[n] = (CorruptionPlan([(P, P)] * n, offs, [0] * n),
                              torch.empty(n * 3 * P * P, dtype=torch.uint8).pin_memory())
        plan, hbuf = self._plans[n]
        crops = hbuf.numpy().reshape(n, P, P, 3)
        dec = []
        for i, im in enumerate(frames):
            if im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3:
                raise ValueError("expected HWC uint8 BGR frames")
            if im.shape[0] < P or im.shape[1] < P:  # the reference enlarges such a frame first (train_restoration.py:79-81)
                im = resize_linear_u8(im, max(int(im.shape[0]), P), max(int(im.shape[1]), P))
            y, x, flip, op = draw_restoration_decisions(int(im.shape[0]), int(im.shape[1]), P, self.is_train)
            crops[i] = im[y:y + P, x:x + P]
            dec.append((y, x, flip, op))
        self.last_decisions = dec
        src = hbuf.cuda()  # (synchronous for the host: the pinned crop buffer is rewritten by the next call)
        return self._pairs(plan, src, dec)

    def _pairs(self, plan, src, dec):
        """src: the n crops back to back on the device; dec: (y, x, flip, op) per sample.  Compat mode draws the noise
        samples' fields here, in sample order, in one device draw (the decisions consume only `random`, so drawing them
        after all decisions is the reference's np.random stream)."""
        from .augmentations import NOISE_SIGMA, legacy_normal_f32_device
        torch, P, n = self._torch, self.size, len(dec)
        flips = torch.tensor([int(d[2]) for d in dec], dtype=torch.uint8).cuda()
        ops = torch.tensor([d[3] for d in dec], dtype=torch.uint8).cuda()
        nz = None
        noisy = [i for i, d in enumerate(dec) if d[3] == 1]
        if self.noise == "compat" and noisy:
            nz = torch.empty(n * 3 * P * P, dtype=torch.float32, device="cuda")
            legacy_normal_f32_device(NOISE_SIGMA, nz, [(i * 3 * P * P, 3 * P * P) for i in noisy])
        corrupted = torch.empty((n, 3, P, P), dtype=torch.float32, device="cuda")
        clean = torch.empty_like(corrupted)
        plan.restoration_pairs(src, flips, ops, corrupted, clean, noise=nz, sigma=float(NOISE_SIGMA), seed=self.seed,
                               first_image_index=self.samples_seen)
        self.samples_seen += n
        return corrupted, clean

    def from_files(self, items: Sequence, io_threads: int = 8):
        """The same pairs starting from image files (`cv2.imread(str(path))`, train_restoration.py:105): paths or bytes
        objects are read on I/O threads, decoded on the GPU (jpeg.JpegDecoder: the pixels of cv2.imread; other layouts
        through the host codec), cropped on the device.  Equals __call__([cv2.imread(p) for p in items]) under the same
        `random` / `np.random` state."""
        from concurrent.futures import ThreadPoolExecutor
        from . import _native as N
        from .batch import _ptr, _stream_handle, draw_restoration_decisions
        from .jpeg import JpegDecoder
        torch, P, n = self._torch, self.size, len(items)
        with ThreadPoolExecutor(max(1, min(int(io_threads), n))) as pool:
            loaded = list(pool.map(FileCorruptionBatcher._load, items))
        shapes = [sh for _, sh in loaded]
        fplan = CorruptionPlan.ragged(shapes)
        dev = torch.empty(fplan.src_bytes, dtype=torch.uint8, device="cuda")
        enc = [i for i, (d, _) in enumerate(loaded) if not isinstance(d, np.ndarray)]
        if enc:
            dec_ = JpegDecoder([loaded[i][0] for i in enc], [fplan.src_offsets[i] for i in enc], host_threads=io_threads)
            dec_.decode(dev)
        for i, (d, (h, w)) in enumerate(loaded):
            if isinstance(d, np.ndarray):
                dev[fplan.src_offsets[i]:fplan.src_offsets[i] + 3 * h * w].copy_(torch.from_numpy(np.ascontiguousarray(d).reshape(-1)))
        if enc:
            import cv2
            for i, st in zip(enc, dec_.status()):
                if st != 0:
                    arr = cv2.imdecode(np.frombuffer(loaded[i][0], np.uint8), cv2.IMREAD_COLOR)
                    if arr is None or (int(arr.shape[0]), int(arr.shape[1])) != shapes[i]:
                        raise IOError("unreadable image in batch")
                    dev[fplan.src_offsets[i]:fplan.src_offsets[i] + arr.size].copy_(torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)))
        if n not in self._plans:
            offs = [i * 3 * P * P for i in range(n)]
            self._plans[n] = (CorruptionPlan([(P, P)] * n, offs, [0] * n), torch.empty(n * 3 * P * P, dtype=torch.uint8).pin_memory())
        plan = self._plans[n][0]
        crops = torch.empty((n, P, P, 3), dtype=torch.uint8, device="cuda")
        dec = []
        for i, (h, w) in enumerate(shapes):
            frame = dev[fplan.src_offsets[i]:fplan.src_offsets[i] + 3 * h * w].view(h, w, 3)
            if h < P or w < P:  # the reference enlarges such a frame first (train_restoration.py:79-81)
                nh, nw = max(h, P), max(w, P)
                big = torch.empty((nh, nw, 3), dtype=torch.uint8, device="cuda")
                N.check(N.lib().rod_resize_linear_u8(_ptr(frame), h, w, 3 * w, _ptr(big), nh, nw, 3 * nw, _stream_handle()), "rod_resize_linear_u8")
                frame, h, w = big, nh, nw
            y, x, flip, op = draw_restoration_decisions(h, w, P, self.is_train)
            crops[i].copy_(frame[y:y + P, x:x + P])
            dec.append((y, x, flip, op))
        self.last_decisions = dec
        return self._pairs(plan, crops.reshape(-1), dec)


class DetectionCorruptionBatcher:
    """Batched device path of the torchvision Faster R-CNN loader (train_frcnn_augmented.py:61-67,131-134): per item
    `PIL.Image.open(p).convert("RGB")` -> RandomCorruption(p) (augmentations.py:60-74) -> ToImage() ->
    ToDtype(torch.float32, scale=True), then `.to(device)` in the loop.  Here one call takes a whole batch and returns
    CUDA float32 [3,H,W] RGB tensors (views into one flat buffer, rod_corrupt_chw_f32):

        batcher = DetectionCorruptionBatcher(p=0.5)               # noise="compat": the reference's tensors, bit for bit
        images = batcher(paths)                                  # or bytes objects, PIL images, HWC RGB uint8 arrays
        loader = DataLoader(dataset_without_transforms, batch_size=2, shuffle=True, num_workers=0,
                            collate_fn=batcher.collate)          # (images, targets) with the images already on the GPU

    Decisions: `random` is consumed as the per-item gate would (skip iff random() > p, then random.choice), for the whole
    batch first; in compat mode the fields of the noise images are then drawn from NumPy's global legacy stream in image
    order (np.random.normal(0, 15, (H, W, 3)).astype(float32) for the BGR array), in one device draw per batch
    (augmentations.legacy_normal_f32_device).  The two
    streams are independent, so this equals the reference's per-item interleaving.  noise="philox" generates the field in
    the kernel instead (the plan's generator, keyed by (seed, running image index)).  The drawn op-codes are left in
    .last_ops.

    Files: JPEGs the device decoder takes are decoded on the GPU (PIL and cv2.imdecode give the same pixels for them);
    every other file -- EXIF-rotated (PIL does not apply the orientation; OpenCV would), progressive, CMYK, PNG, corrupt
    entropy data -- is read with `Image.open(...).convert("RGB")` like the reference's dataset, so PIL's own errors and
    settings (ImageFile.LOAD_TRUNCATED_IMAGES) apply.  The batcher uses CUDA in the calling process: with a DataLoader, keep
    num_workers=0 (the reference's setting) so that collate runs in the main process.
    """

    def __init__(self, p: float = 0.5, noise: str = "compat", seed: int = 0, io_threads: int = 16,
                 max_cached_plans: int = 16):
        import torch
        from concurrent.futures import ThreadPoolExecutor
        if noise not in ("compat", "philox"):
            raise ValueError("noise must be 'compat' or 'philox'")
        self._torch = torch
        self.p, self.noise, self.seed = float(p), noise, int(seed)
        self._plans: dict = {}
        self._max_plans = max_cached_plans
        self._io_threads = max(1, int(io_threads))
        self._pool = ThreadPoolExecutor(self._io_threads)
        self._copy_stream = torch.cuda.Stream()
        self._slots: List[dict] = [{}, {}]
        self.images_seen = 0
        self.last_ops: Optional[np.ndarray] = None

    # ------------------------------------------------------------------ internals
    def _plan(self, shapes) -> CorruptionPlan:
        key = tuple(shapes)
        plan = self._plans.get(key)
        if plan is None:
            if len(self._plans) >= self._max_plans:
                self._plans.pop(next(iter(self._plans)))
            plan = self._plans[key] = CorruptionPlan.ragged(shapes)
        return plan

    @staticmethod
    def _read_pil(data) -> np.ndarray:
        import io
        from PIL import Image
        with Image.open(io.BytesIO(data)) as im:
            return np.asarray(im.convert("RGB"))

    @classmethod
    def _load(cls, item):
        """I/O thread: (file bytes, (h, w)) for a JPEG the device decoder takes, else (HWC RGB uint8 array, (h, w))."""
        if isinstance(item, np.ndarray):
            if item.dtype != np.uint8 or item.ndim != 3 or item.shape[2] != 3:
                raise ValueError("expected HWC RGB uint8 arrays")
            return item, (int(item.shape[0]), int(item.shape[1]))
        if not isinstance(item, (bytes, bytearray, memoryview)) and hasattr(item, "convert"):  # a PIL image
            arr = np.asarray(item if item.mode == "RGB" else item.convert("RGB"))
            return arr, (int(arr.shape[0]), int(arr.shape[1]))
        from .jpeg import probe
        data = item if isinstance(item, (bytes, bytearray, memoryview)) else open(item, "rb").read()
        shape = probe(data)
        if shape is not None:
            return data, shape
        arr = cls._read_pil(data)
        return arr, (int(arr.shape[0]), int(arr.shape[1]))

    def _stage(self, slot: dict, items: Sequence, futs) -> None:
        """Read / decode / pack one batch into the slot's buffers on the copy stream and draw its decisions."""
        torch = self._torch
        from .augmentations import NOISE_SIGMA, legacy_normal_f32_device
        from .jpeg import JpegDecoder
        loaded = [f.result() for f in futs]
        shapes = [sh for _, sh in loaded]
        plan = self._plan(shapes)
        n = len(items)
        elems = [3 * h * w for h, w in shapes]
        elem_base = np.concatenate([[0], np.cumsum(elems)]).astype(np.int64)
        grow = False
        for name, dtype, size in (("src", torch.uint8, plan.src_bytes), ("noise", torch.float32, int(elem_base[-1])),
                                  ("ops", torch.uint8, max(n, 64))):
            if slot.get(name + "_cap", 0) < size:
                cap = max(size, 2 * slot.get(name + "_cap", 0))
                if name != "noise":  # (the compat field is drawn on the device)
                    slot[name + "_host"] = torch.empty(cap, dtype=dtype).pin_memory()
                slot[name + "_dev"] = torch.empty(cap, dtype=dtype, device="cuda")
                slot[name + "_cap"] = cap
                grow = True
        if grow:  # a fresh block's previous use may still be pending on the compute stream
            self._copy_stream.wait_stream(torch.cuda.current_stream())
        ev = slot.get("free")
        if ev is not None:
            ev.synchronize()  # the compute that last read this slot's buffers has finished
        dev, hbuf = slot["src_dev"], slot["src_host"].numpy()
        offs = plan.src_offsets
        host_idx = [i for i, (d, _) in enumerate(loaded) if isinstance(d, np.ndarray)]
        enc = [i for i, (d, _) in enumerate(loaded) if not isinstance(d, np.ndarray)]
        with torch.cuda.stream(self._copy_stream):
            if enc:
                dec = JpegDecoder([loaded[i][0] for i in enc], [offs[i] for i in enc], host_threads=self._io_threads)
                dec.decode(dev, stream=self._copy_stream)
                for i, st in zip(enc, dec.status(stream=self._copy_stream)):
                    if st != 0:  # not decodable here after all, or corrupt entropy data: PIL's reading is the reference's
                        arr = self._read_pil(loaded[i][0])
                        if (int(arr.shape[0]), int(arr.shape[1])) != shapes[i]:
                            raise IOError("image size differs between the file header and its decoded pixels")
                        loaded[i] = (arr, shapes[i])
                        host_idx.append(i)
                host_idx.sort()

            def pack(i):  # RGB -> BGR into the pinned buffer (NumPy releases the GIL for the copy)
                (h, w), off = shapes[i], offs[i]
                hbuf[off:off + 3 * h * w].reshape(h, w, 3)[...] = loaded[i][0][:, :, ::-1]

            packing = [self._pool.submit(pack, i) for i in host_idx]
            ops = draw_decisions(n, gate="pil", p=self.p)
            noise = None
            if self.noise == "compat" and (ops == 1).any():  # the noise images' fields in image order: one device draw
                noise = slot["noise_dev"]
                legacy_normal_f32_device(NOISE_SIGMA, noise, [(int(elem_base[i]), elems[i]) for i in np.flatnonzero(ops == 1)])
            for f in packing:
                f.result()
            # one copy per run of consecutive host-sourced images
            k = 0
            while k < len(host_idx):
                j = k
                while j + 1 < len(host_idx) and host_idx[j + 1] == host_idx[j] + 1:
                    j += 1
                lo = offs[host_idx[k]]
                hi = offs[host_idx[j]] + elems[host_idx[j]]
                dev[lo:hi].copy_(slot["src_host"][lo:hi], non_blocking=True)
                k = j + 1
            slot["ops_host"][:n] = torch.from_numpy(ops)
            slot["ops_dev"][:n].copy_(slot["ops_host"][:n], non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._copy_stream)
        slot.update(plan=plan, n=n, ready=ready, ops=ops, noise=noise, first_index=self.images_seen)
        self.images_seen += n

    def _compute(self, slot: dict) -> List:
        torch = self._torch
        from .augmentations import NOISE_SIGMA
        cur = torch.cuda.current_stream()
        cur.wait_event(slot["ready"])
        plan = slot["plan"]
        out = torch.empty(plan.chw_offsets()[-1], dtype=torch.float32, device="cuda")
        plan.corrupt_chw_f32(slot["src_dev"], slot["ops_dev"], out, noise=slot["noise"], sigma=float(NOISE_SIGMA),
                             seed=self.seed, first_image_index=slot["first_index"])
        free = torch.cuda.Event()
        free.record(cur)
        slot["free"] = free
        self.last_ops = slot["ops"]
        return plan.chw_views(out)

    def _submit(self, items):
        return [self._pool.submit(self._load, it) for it in items]

    # ------------------------------------------------------------------ public
    def __call__(self, items: Sequence) -> List:
        """One batch -> list of CUDA float32 [3,H,W] RGB tensors in [0, 1] (the drawn op-codes in .last_ops)."""
        items = list(items)
        slot = self._slots[0]
        self._stage(slot, items, self._submit(items))
        return self._compute(slot)

    def run(self, batches: Iterable[Sequence]) -> Iterator[List]:
        """Pipelined: while batch i is corrupted and converted on the current stream, batch i+1 is read, packed and
        uploaded on a copy stream."""
        it = iter(batches)
        try:
            cur = list(next(it))
        except StopIteration:
            return
        k = 0
        self._stage(self._slots[0], cur, self._submit(cur))
        while True:
            out = self._compute(self._slots[k & 1])  # enqueued first: the GPU works while the next batch is staged
            try:
                nxt = list(next(it))
            except StopIteration:
                nxt = None
            if nxt is not None:
                self._stage(self._slots[(k + 1) & 1], nxt, self._submit(nxt))
            yield out
            if nxt is None:
                return
            k += 1

    def collate(self, batch: Sequence[Tuple[object, object]]):
        """collate_fn for DataLoader(num_workers=0) over a dataset of (PIL image, target) built without transforms:
        returns (tuple of CUDA float32 [3,H,W] tensors, tuple of targets) like the reference's tuple(zip(*batch))."""
        images, targets = zip(*batch)
        return tuple(self(list(images))), tuple(targets)
