"""torch.library custom ops over the C ABI (SURVEY 8b: "the same entry points are registered as torch.library custom
ops taking CUDA uint8 tensors"; north_star: "a thin PyTorch custom-op / C-ABI layer").

    import robust_object_detection_b200.torch_ops            # registers the ops
    y = torch.ops.rod.blur(x, 9, 0.0)                         # x: CUDA uint8 [N,H,W,3] (or [H,W,3]) BGR

    op                          entry point (include/rod_b200.h)   reference (scripts/augmentations.py)
    rod::noise                  rod_noise_u8                       apply_noise                    :30-33
    rod::blur                   rod_blur_h_u8                      apply_motion_blur              :36-38
    rod::lowres                 rod_lowres_u8                      apply_lowres                   :41-45
    rod::corrupt_batch          rod_corrupt_batch_u8               _apply_random_corruption + gate :48-56, :93
    rod::corrupt_letterbox      rod_corrupt_letterbox_f16          hook + Ultralytics LetterBox / Format / /255
    rod::corrupt_chw            rod_corrupt_chw_f32                RandomCorruption + ToImage + ToDtype(float32, scale=True)

All ops are functional (fresh output tensor, input untouched -- the reference's ownership convention), run on the
CURRENT CUDA stream of the input's device, have fake (meta) implementations so they trace under torch.compile /
torch.export, and have no CPU implementation: a CPU tensor raises.  The tensors are contiguous uniform batches; ragged
mixed-resolution batches use batch.CorruptionPlan directly.  Pixel work happens in librod_b200.so only.
"""
from __future__ import annotations

import threading
from typing import Optional

import torch

from .batch import CorruptionPlan

_plans: dict = {}
_plans_lock = threading.Lock()
_PLAN_CACHE_MAX = 32


def _plan(n: int, h: int, w: int, device: torch.device) -> CorruptionPlan:
    """One cached plan per (batch, shape, device, thread): a plan carries per-call state (resize tables, installed
    blur kernel), so threads do not share one."""
    key = (n, h, w, device.index, threading.get_ident())
    with _plans_lock:
        plan = _plans.get(key)
        if plan is None:
            if len(_plans) >= _PLAN_CACHE_MAX:
                _plans.pop(next(iter(_plans)))
            with torch.cuda.device(device):
                plan = CorruptionPlan.uniform(n, h, w)
            _plans[key] = plan
    return plan


def _check(img: torch.Tensor):
    if not img.is_cuda:
        raise RuntimeError("rod ops run on CUDA tensors only (there is no CPU fallback)")
    if img.dtype != torch.uint8 or img.dim() not in (3, 4) or img.shape[-1] != 3:
        raise ValueError("expected a uint8 [N,H,W,3] or [H,W,3] tensor (HWC, BGR)")
    x = img.contiguous()
    n = 1 if x.dim() == 3 else int(x.shape[0])
    return x, n, int(x.shape[-3]), int(x.shape[-2])


@torch.library.custom_op("rod::noise", mutates_args=(), device_types="cuda")
def noise(img: torch.Tensor, sigma: float, seed: int, first_image_index: int, field: Optional[torch.Tensor] = None) -> torch.Tensor:
    """apply_noise for a batch.  field = None: Philox mode (seed, first_image_index key the stream); field = float32 tensor
    of img's shape: compat mode, out = uint8(trunc(clip(float32(img) + field, 0, 255))) bit-exactly."""
    x, n, h, w = _check(img)
    if field is not None:
        if not field.is_cuda or field.dtype != torch.float32 or field.numel() != x.numel():
            raise ValueError("field must be a CUDA float32 tensor with img's element count")
        field = field.contiguous()
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _plan(n, h, w, x.device).noise(x, out, field, float(sigma), seed=int(seed), first_image_index=int(first_image_index))
    return out


@torch.library.custom_op("rod::blur", mutates_args=(), device_types="cuda")
def blur(img: torch.Tensor, k: int, angle_deg: float) -> torch.Tensor:
    """apply_motion_blur for a batch (angle 0: the k-tap horizontal box; other angles: the rotated k x k kernel, k <= 11)."""
    x, n, h, w = _check(img)
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        plan = _plan(n, h, w, x.device)
        if float(angle_deg) != 0.0:
            from .augmentations import _motion_blur_kernel
            plan.set_blur_kernel(_motion_blur_kernel(int(k), float(angle_deg)))
        else:
            plan.set_blur_kernel(None)
        plan.blur(x, out, int(k), 0.0)
    return out


@torch.library.custom_op("rod::lowres", mutates_args=(), device_types="cuda")
def lowres(img: torch.Tensor, factor: float) -> torch.Tensor:
    """apply_lowres for a batch: INTER_AREA down + INTER_LINEAR up, fused (the low-res image never touches HBM)."""
    x, n, h, w = _check(img)
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _plan(n, h, w, x.device).lowres(x, out, float(factor))
    return out


@torch.library.custom_op("rod::corrupt_batch", mutates_args=(), device_types="cuda")
def corrupt_batch(img: torch.Tensor, opcodes: torch.Tensor, sigma: float, k: int, factor: float, seed: int,
                  first_image_index: int) -> torch.Tensor:
    """The random one-of-three apply for a batch: opcodes uint8[N] (0 none / 1 noise / 2 blur / 3 lowres), drawn on the
    host in the reference's order by batch.draw_decisions."""
    x, n, h, w = _check(img)
    if not opcodes.is_cuda or opcodes.dtype != torch.uint8 or opcodes.numel() != n:
        raise ValueError("opcodes must be a CUDA uint8 tensor with one entry per image")
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        plan = _plan(n, h, w, x.device)
        plan.set_blur_kernel(None)
        plan.corrupt(x, out, opcodes.contiguous(), None, float(sigma), int(k), float(factor), int(seed), int(first_image_index))
    return out


@torch.library.custom_op("rod::corrupt_letterbox", mutates_args=(), device_types="cuda")
def corrupt_letterbox(img: torch.Tensor, opcodes: torch.Tensor, out_h: int, out_w: int, pad_value: int, sigma: float, k: int,
                      factor: float, seed: int, first_image_index: int) -> torch.Tensor:
    """Training path: corruption + letterbox + BGR->RGB + CHW + /255 -> float16 [N,3,out_h,out_w], one pass over the source."""
    x, n, h, w = _check(img)
    if not opcodes.is_cuda or opcodes.dtype != torch.uint8 or opcodes.numel() != n:
        raise ValueError("opcodes must be a CUDA uint8 tensor with one entry per image")
    out = torch.empty((n, 3, int(out_h), int(out_w)), dtype=torch.float16, device=x.device)
    with torch.cuda.device(x.device):
        plan = _plan(n, h, w, x.device)
        plan.set_blur_kernel(None)
        plan.corrupt_letterbox(x, opcodes.contiguous(), out, int(out_h), int(out_w), int(pad_value), None, float(sigma), int(k),
                               float(factor), int(seed), int(first_image_index))
    return out


def _chw_strides(h: int, w: int):
    """Strides of the [N,3,H,W] float32 result of rod::corrupt_chw: image blocks start at multiples of 64 floats
    (include/rod_b200.h rod_plan_chw_offset), so the batch stride is 3*H*W rounded up to 64."""
    return ((3 * h * w + 63) // 64 * 64, h * w, w, 1)


@torch.library.custom_op("rod::corrupt_chw", mutates_args=(), device_types="cuda")
def corrupt_chw(img: torch.Tensor, opcodes: torch.Tensor, sigma: float, k: int, factor: float, seed: int,
                first_image_index: int) -> torch.Tensor:
    """Faster R-CNN loader path: the corruption of rod::corrupt_batch, then BGR->RGB, HWC->CHW and float32 scaling as
    torchvision's ToDtype(float32, scale=True) -> float32 [N,3,H,W] (batch stride rounded up to 64 floats)."""
    x, n, h, w = _check(img)
    if not opcodes.is_cuda or opcodes.dtype != torch.uint8 or opcodes.numel() != n:
        raise ValueError("opcodes must be a CUDA uint8 tensor with one entry per image")
    strides = _chw_strides(h, w)
    out = torch.empty_strided((n, 3, h, w), strides, dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        plan = _plan(n, h, w, x.device)
        plan.set_blur_kernel(None)
        plan.corrupt_chw_f32(x, opcodes.contiguous(), out, None, float(sigma), int(k), float(factor), int(seed),
                             int(first_image_index))
    return out


@noise.register_fake
def _(img, sigma, seed, first_image_index, field=None):
    return torch.empty_like(img.contiguous())


@blur.register_fake
def _(img, k, angle_deg):
    return torch.empty_like(img.contiguous())


@lowres.register_fake
def _(img, factor):
    return torch.empty_like(img.contiguous())


@corrupt_batch.register_fake
def _(img, opcodes, sigma, k, factor, seed, first_image_index):
    return torch.empty_like(img.contiguous())


@corrupt_letterbox.register_fake
def _(img, opcodes, out_h, out_w, pad_value, sigma, k, factor, seed, first_image_index):
    n = 1 if img.dim() == 3 else img.shape[0]
    return img.new_empty((n, 3, out_h, out_w), dtype=torch.float16)


@corrupt_chw.register_fake
def _(img, opcodes, sigma, k, factor, seed, first_image_index):
    n = 1 if img.dim() == 3 else img.shape[0]
    h, w = img.shape[-3], img.shape[-2]
    return img.new_empty_strided((n, 3, h, w), _chw_strides(h, w), dtype=torch.float32)
