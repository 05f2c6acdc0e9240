"""Device-resident batches for the corruption path (the batch driver of
scripts/build_corrupted_testsets.py:108-124 and the training-time hook of
scripts/augmentations.py:91-95, moved onto the GPU).

A `CorruptionPlan` wraps one `rod_plan` (include/rod_b200.h): a descriptor table for a
uniform [N,H,W,3] tensor or for a ragged flat buffer of mixed-resolution images.  PyTorch is
used only for device memory and the current stream; all pixel work happens in librod_b200.so.
"""
from __future__ import annotations

import ctypes
import random
from typing import Iterable, Optional, Sequence, Tuple

import numpy as np

from . import _native as N

NOISE_SIGMA = 15
BLUR_KERNEL = 9
BLUR_ANGLE_DEG = 0
DOWNSCALE_FACTOR = 0.5
IMAGE_ALIGN = 256  # byte alignment of each image inside a ragged flat buffer


def _ptr(t) -> Optional[int]:
    """Device (or host) address of a torch tensor / numpy array / int / None."""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    if isinstance(t, np.ndarray):
        return t.ctypes.data
    return t.data_ptr()


def _stream_handle(stream=None) -> Optional[int]:
    import torch
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream or None


def draw_decisions(n: int, gate: str = "ultralytics", p: float = 0.5) -> np.ndarray:
    """Op-codes for n consecutive images, consuming Python's global `random` exactly as n
    consecutive reference hook calls would: gate 'ultralytics' = apply iff random() < 0.5
    (augmentations.py:93), gate 'pil' = skip iff random() > p (augmentations.py:70); then
    random.choice(["noise","blur","lowres"]) (augmentations.py:50)."""
    ops = np.zeros(n, dtype=np.uint8)
    for i in range(n):
        r = random.random()
        applied = (r < 0.5) if gate == "ultralytics" else not (r > p)
        if applied:
            ops[i] = 1 + ("noise", "blur", "lowres").index(random.choice(["noise", "blur", "lowres"]))
    return ops


def resize_linear_u8(img: np.ndarray, nh: int, nw: int) -> np.ndarray:
    """cv2.resize(img, (nw, nh)) with the default INTER_LINEAR for an HWC uint8 frame that is enlarged (or kept) in both
    axes, computed on the GPU (rod_resize_linear_u8; bit-exact against OpenCV's 8-bit fixed-point path).  The
    resize-first branch of RestorationDataset._random_crop / _center_crop (train_restoration.py:79-81,88-90)."""
    import torch
    N.require_device()
    if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
        raise ValueError("expected an HWC uint8 image")
    h, w = int(img.shape[0]), int(img.shape[1])
    src = torch.from_numpy(np.ascontiguousarray(img)).cuda()
    dst = torch.empty((int(nh), int(nw), 3), dtype=torch.uint8, device="cuda")
    N.check(N.lib().rod_resize_linear_u8(_ptr(src), h, w, 3 * w, _ptr(dst), int(nh), int(nw), 3 * int(nw), _stream_handle()),
            "rod_resize_linear_u8")
    return dst.cpu().numpy()


def draw_restoration_decisions(h: int, w: int, size: int, is_train: bool = True):
    """(y, x, flip, op) of one RestorationDataset.__getitem__ call (train_restoration.py:77-102,108-121), consuming
    Python's global `random` in the reference's order: randint(0, h - size), randint(0, w - size), random() > 0.5,
    random.choice([...]); validation items take the centre crop and no flip.  A frame smaller than the patch is first
    enlarged to (max(h, size), max(w, size)) in the reference (:79-81, 88-90); the positions are drawn for that size."""
    h, w = max(h, size), max(w, size)
    if is_train:
        y = random.randint(0, h - size)
        x = random.randint(0, w - size)
        flip = random.random() > 0.5
    else:
        y, x, flip = (h - size) // 2, (w - size) // 2, False
    op = 1 + ("noise", "blur", "lowres").index(random.choice(["noise", "blur", "lowres"]))
    return y, x, flip, op


class CorruptionPlan:
    """Descriptor table + tile lists + resize tables for one batch layout."""

    def __init__(self, shapes: Sequence[Tuple[int, int]], src_offsets: Sequence[int], dst_offsets: Sequence[int],
                 src_pitches: Optional[Sequence[int]] = None, dst_pitches: Optional[Sequence[int]] = None):
        N.require_device()
        n = len(shapes)
        if n < 1:
            raise ValueError("a plan needs at least one image")
        descs = (N.ImageDesc * n)()
        for i, (h, w) in enumerate(shapes):
            descs[i].src_offset = int(src_offsets[i])
            descs[i].dst_offset = int(dst_offsets[i])
            descs[i].height, descs[i].width = int(h), int(w)
            descs[i].src_pitch = int(src_pitches[i]) if src_pitches is not None else 3 * int(w)
            descs[i].dst_pitch = int(dst_pitches[i]) if dst_pitches is not None else 3 * int(w)
        handle = ctypes.c_void_p()
        N.check(N.lib().rod_plan_create(descs, n, ctypes.byref(handle)), "rod_plan_create")
        self._h = handle
        self.shapes = [(int(h), int(w)) for h, w in shapes]
        self.n_images = n
        self.src_offsets = [int(o) for o in src_offsets]
        self.dst_offsets = [int(o) for o in dst_offsets]
        self.payload_bytes = int(N.lib().rod_plan_payload_bytes(handle))
        last = n - 1
        self.src_bytes = max(o + (h - 1) * (src_pitches[i] if src_pitches is not None else 3 * w) + 3 * w
                             for i, (o, (h, w)) in enumerate(zip(self.src_offsets, self.shapes)))
        self.dst_bytes = max(o + (h - 1) * (dst_pitches[i] if dst_pitches is not None else 3 * w) + 3 * w
                             for i, (o, (h, w)) in enumerate(zip(self.dst_offsets, self.shapes)))
        del last

    # -- constructors ------------------------------------------------------------------
    @classmethod
    def uniform(cls, n: int, h: int, w: int) -> "CorruptionPlan":
        """Contiguous [n, h, w, 3] uint8 tensors for both src and dst."""
        size = 3 * h * w
        offs = [i * size for i in range(n)]
        return cls([(h, w)] * n, offs, offs)

    @classmethod
    def ragged(cls, shapes: Iterable[Tuple[int, int]], align: int = IMAGE_ALIGN) -> "CorruptionPlan":
        """Mixed-resolution images packed into one flat buffer, each image contiguous and
        starting at a multiple of `align` bytes (same layout for src and dst)."""
        shapes = list(shapes)
        offs, cur = [], 0
        for h, w in shapes:
            offs.append(cur)
            cur += (3 * h * w + align - 1) // align * align
        return cls(shapes, offs, offs)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                N.lib().rod_plan_destroy(h)
            except Exception:
                pass
            self._h = None

    # -- helpers -----------------------------------------------------------------------
    def launches(self, op: int) -> int:
        return int(N.lib().rod_plan_launches(self._h, int(op)))

    def pack(self, images: Sequence[np.ndarray]) -> np.ndarray:
        """Host flat uint8 buffer holding `images` at this plan's source offsets."""
        buf = np.zeros(self.src_bytes, dtype=np.uint8)
        for img, off, (h, w) in zip(images, self.src_offsets, self.shapes):
            assert img.shape == (h, w, 3) and img.dtype == np.uint8
            buf[off:off + 3 * h * w] = np.ascontiguousarray(img).reshape(-1)
        return buf

    def unpack(self, flat: np.ndarray):
        """Views of the images inside a host flat buffer laid out by the dst offsets."""
        return [flat[off:off + 3 * h * w].reshape(h, w, 3) for off, (h, w) in zip(self.dst_offsets, self.shapes)]

    # -- device ops (torch CUDA uint8 tensors or raw device addresses) -------------------
    def noise(self, src, dst, noise=None, sigma: float = NOISE_SIGMA, seed: int = 0, first_image_index: int = 0,
              offset: int = 0, opcodes=None, stream=None) -> None:
        N.check(N.lib().rod_noise_u8(self._h, _ptr(src), _ptr(dst), _ptr(noise), float(sigma), int(seed),
                                     int(first_image_index), int(offset), _ptr(opcodes), _stream_handle(stream)),
                "rod_noise_u8")

    def noise_field(self, out, sigma: float = NOISE_SIGMA, seed: int = 0, first_image_index: int = 0, offset: int = 0,
                    stream=None) -> None:
        N.check(N.lib().rod_noise_field_f32(self._h, _ptr(out), float(sigma), int(seed), int(first_image_index),
                                            int(offset), _stream_handle(stream)), "rod_noise_field_f32")

    @staticmethod
    def prewarm_noise(sigma: float = NOISE_SIGMA, device: Optional[int] = None) -> None:
        """Upload the table-generator table of `sigma` now, so that the first Philox-mode launch with this sigma does
        no allocation / blocking copy (required before capturing it in a CUDA graph).  rod_noise_prewarm."""
        if device is None:
            import torch
            device = torch.cuda.current_device()
        N.check(N.lib().rod_noise_prewarm(int(device), float(sigma)), "rod_noise_prewarm")

    def set_gaussian_generator(self, generator: int) -> None:
        """Philox-mode Gaussian generator of this plan: 0 = auto (256-entry table + Hadamard mix when 3 <= sigma <= 20,
        else Box-Muller), 1 = Box-Muller, 2 = auto with the table generator on Philox4x32-7.  include/rod_b200.h
        rod_plan_set_gaussian_generator."""
        N.check(N.lib().rod_plan_set_gaussian_generator(self._h, int(generator)), "rod_plan_set_gaussian_generator")

    def blur(self, src, dst, k: int = BLUR_KERNEL, angle_deg: float = BLUR_ANGLE_DEG, opcodes=None, stream=None) -> None:
        N.check(N.lib().rod_blur_h_u8(self._h, _ptr(src), _ptr(dst), int(k), float(angle_deg), _ptr(opcodes),
                                      _stream_handle(stream)), "rod_blur_h_u8")

    def set_blur_kernel(self, kernel: Optional[np.ndarray]) -> None:
        """Install the k x k float32 kernel of _motion_blur_kernel(k, angle != 0) for this plan's blur op
        (cv2.filter2D semantics, k*k < 130), or None to return to the horizontal angle-0 box."""
        if kernel is None:
            N.check(N.lib().rod_set_blur_kernel(self._h, None, 0), "rod_set_blur_kernel")
            return
        kern = np.ascontiguousarray(kernel, dtype=np.float32)
        if kern.ndim != 2 or kern.shape[0] != kern.shape[1]:
            raise ValueError("kernel must be k x k")
        N.check(N.lib().rod_set_blur_kernel(self._h, kern.ctypes.data, int(kern.shape[0])), "rod_set_blur_kernel")

    def lowres(self, src, dst, factor: float = DOWNSCALE_FACTOR, opcodes=None, stream=None) -> None:
        N.check(N.lib().rod_lowres_u8(self._h, _ptr(src), _ptr(dst), float(factor), _ptr(opcodes),
                                      _stream_handle(stream)), "rod_lowres_u8")

    def corrupt(self, src, dst, opcodes, noise=None, sigma: float = NOISE_SIGMA, k: int = BLUR_KERNEL,
                factor: float = DOWNSCALE_FACTOR, seed: int = 0, first_image_index: int = 0, offset: int = 0,
                stream=None) -> None:
        """opcodes: device uint8[n_images] (0 none / 1 noise / 2 blur / 3 lowres)."""
        N.check(N.lib().rod_corrupt_batch_u8(self._h, _ptr(src), _ptr(dst), _ptr(opcodes), _ptr(noise), float(sigma),
                                             int(k), float(factor), int(seed), int(first_image_index), int(offset),
                                             _stream_handle(stream)), "rod_corrupt_batch_u8")

    def corrupt_letterbox(self, src, opcodes, out_f16, out_h: int = 640, out_w: int = 640, pad_value: int = 114,
                          noise=None, sigma: float = NOISE_SIGMA, k: int = BLUR_KERNEL,
                          factor: float = DOWNSCALE_FACTOR, seed: int = 0, first_image_index: int = 0,
                          offset: int = 0, stream=None) -> None:
        """Training path: corruption + letterbox + BGR->RGB + CHW + /255 -> fp16 [n,3,out_h,out_w]."""
        N.check(N.lib().rod_corrupt_letterbox_f16(self._h, _ptr(src), _ptr(opcodes), _ptr(out_f16), int(out_h),
                                                  int(out_w), int(pad_value), _ptr(noise), float(sigma), int(k),
                                                  float(factor), int(seed), int(first_image_index), int(offset),
                                                  _stream_handle(stream)), "rod_corrupt_letterbox_f16")

    def chw_offsets(self) -> list:
        """Float offsets of the images' [3,H,W] blocks in the output of corrupt_chw_f32, plus the total size in floats as
        the last entry (rod_plan_chw_offset: blocks in plan order, each starting at a multiple of 256 bytes)."""
        if getattr(self, "_chw_offsets", None) is None:
            self._chw_offsets = [int(N.lib().rod_plan_chw_offset(self._h, i)) for i in range(self.n_images + 1)]
        return self._chw_offsets

    def chw_views(self, out) -> list:
        """The [3,H,W] tensors of the images inside a flat output buffer of corrupt_chw_f32."""
        offs = self.chw_offsets()
        return [out[o:o + 3 * h * w].view(3, h, w) for o, (h, w) in zip(offs, self.shapes)]

    def corrupt_chw_f32(self, src, opcodes, out, noise=None, sigma: float = NOISE_SIGMA, k: int = BLUR_KERNEL,
                        factor: float = DOWNSCALE_FACTOR, seed: int = 0, first_image_index: int = 0, offset: int = 0,
                        stream=None) -> None:
        """Faster R-CNN loader path (RandomCorruption + ToImage + ToDtype(float32, scale=True)): the corruption of
        corrupt() for opcodes, then BGR->RGB, HWC->CHW and float(v) * float32(1/255) into `out`, a flat CUDA float32
        buffer of chw_offsets()[-1] elements (256-byte aligned) laid out by chw_offsets()."""
        N.check(N.lib().rod_corrupt_chw_f32(self._h, _ptr(src), _ptr(opcodes), _ptr(out), _ptr(noise), float(sigma),
                                            int(k), float(factor), int(seed), int(first_image_index), int(offset),
                                            _stream_handle(stream)), "rod_corrupt_chw_f32")

    def restoration_pairs(self, src, flips, opcodes, corrupted_out, clean_out, noise=None, sigma: float = NOISE_SIGMA,
                          k: int = BLUR_KERNEL, factor: float = DOWNSCALE_FACTOR, seed: int = 0,
                          first_image_index: int = 0, offset: int = 0, stream=None) -> None:
        """RestorationDataset.__getitem__ (train_restoration.py:104-129) for a batch: this plan's source descriptors
        are the crops; outputs are float32 [n,3,P,P] RGB in [0,1] (corrupted input, clean target)."""
        N.check(N.lib().rod_restoration_pairs_f32(self._h, _ptr(src), _ptr(flips), _ptr(opcodes), _ptr(corrupted_out),
                                                  _ptr(clean_out), _ptr(noise), float(sigma), int(k), float(factor),
                                                  int(seed), int(first_image_index), int(offset), _stream_handle(stream)),
                "rod_restoration_pairs_f32")

    # -- host-buffer path (H2D + kernel + D2H inside the call) ---------------------------
    def apply_host(self, op: int, src_host, dst_host, noise_host=None, sigma: float = NOISE_SIGMA,
                   k: int = BLUR_KERNEL, factor: float = DOWNSCALE_FACTOR, seed: int = 0, first_image_index: int = 0,
                   offset: int = 0) -> None:
        N.check(N.lib().rod_apply_host(self._h, int(op), _ptr(src_host), _ptr(dst_host), _ptr(noise_host),
                                       float(sigma), int(k), float(factor), int(seed), int(first_image_index),
                                       int(offset)), "rod_apply_host")
