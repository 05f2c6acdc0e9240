"""Drop-in for scripts/augmentations.py of ysbbin/Robust-Object-Detection.

Same module surface, same signatures, same observable RNG behaviour -- but every pixel is
computed on a B200 by librod_b200.so (hand-written sm_100a CUDA, include/rod_b200.h).
There is no CPU fallback: without the built library or without a GPU the calls raise.

    reference (scripts/augmentations.py)            here
    ---------------------------------------------   --------------------------------------------
    NOISE_SIGMA .. DOWNSCALE_FACTOR      :14-17     same names and values
    _motion_blur_kernel(k, angle_deg)    :21-27     same (host-side, float32 k x k; angle 0 only)
    apply_noise(img_bgr, sigma)          :30-33     rod_apply_host(ROD_OP_NOISE)
    apply_motion_blur(img_bgr, k, angle) :36-38     rod_apply_host(ROD_OP_BLUR)
    apply_lowres(img_bgr, factor)        :41-45     rod_apply_host(ROD_OP_LOWRES)
    _apply_random_corruption(img_bgr)    :48-56     same dispatch, same `random.choice`
    RandomCorruption(p)                  :60-74     same gate (skip iff random() > p)
    patch_ultralytics_augmentations()    :78-98     same gate (apply iff random() < 0.5)

Noise modes.  'compat' (default) draws the field on the host with
np.random.normal(0, sigma, shape).astype(float32) -- consuming NumPy's global legacy stream
exactly like the reference -- and the GPU does the add/clip/truncate, so outputs are
bit-identical to the reference under the same np.random.seed.  'philox' generates the field
inside the kernel (Philox4x32-10 keyed by seed and a running image counter; for 3 <= sigma <= 20 four 8-bit draws per
Philox word from a 256-entry table, mixed by a 4 x 4 Hadamard transform in integer arithmetic; Box-Muller otherwise):
no host RNG work, statistically equivalent, not bit-identical.

Process and thread model (SURVEY 8b).  The functions are re-entrant: a module lock serialises the short critical section
(plan cache, the shared page-locked noise buffer, the launch) so concurrent threads corrupting same-shaped images get
the right bytes; the GPU runs one call at a time anyway.  In DataLoader WORKER PROCESSES each process needs its own
CUDA context, which only the 'spawn' (or 'forkserver') start method gives: patch_ultralytics_augmentations() therefore
switches multiprocessing to 'spawn' (the reference's launchers already call the patch at import time precisely so that
spawned workers re-apply it, train_yolo_augmented.py:16-19).  A fork()ed child of a process that has used CUDA cannot
use it: calling into this module from such a child raises a RuntimeError that names the fix instead of a raw CUDA error.
"""
from __future__ import annotations

import os
import random
import threading

import numpy as np

from . import _native as N
from .batch import CorruptionPlan

# ---- Parameters (same as build_corrupted_testsets.py:13-23) ----
NOISE_SIGMA = 15
BLUR_KERNEL = 9
BLUR_ANGLE_DEG = 0
DOWNSCALE_FACTOR = 0.5

_noise_mode = "compat"
_philox_seed = 0
_philox_counter = 0
_plans: dict = {}
_PLAN_CACHE_MAX = 64
_lock = threading.RLock()     # plan cache, pinned noise buffers, Philox counter, launch: one call at a time
_owner_pid = None             # the process that first ran a corruption through this module (owns the CUDA context)


def _check_process() -> None:
    """Fail clearly in a fork()ed child of a process that already uses CUDA (the reference's hook runs inside DataLoader
    workers, train_yolo_augmented.py:33 workers=8): CUDA cannot be re-initialised there and there is no CPU fallback."""
    global _owner_pid
    pid = os.getpid()
    if _owner_pid == pid:
        return
    bad = _owner_pid is not None          # this module already ran in the parent, and we are a fork of it
    if not bad:
        try:  # the parent initialised CUDA through torch before forking (the usual Ultralytics situation)
            import sys
            torch = sys.modules.get("torch")
            bad = bool(torch is not None and torch.cuda._is_in_bad_fork())
        except Exception:
            bad = False
    if bad:
        raise RuntimeError(
            "robust_object_detection_b200: this process was fork()ed from a parent that already uses CUDA, and CUDA cannot "
            "be initialised in such a child (there is no CPU fallback).  Start DataLoader workers with the 'spawn' start "
            "method -- patch_ultralytics_augmentations() selects it; or torch.multiprocessing.set_start_method('spawn') / "
            "DataLoader(multiprocessing_context='spawn') -- or use workers=0, or the main-process batch driver "
            "robust_object_detection_b200.training.CorruptionBatcher.")
    _owner_pid = pid


def set_noise_mode(mode: str, seed: int = 0) -> None:
    """'compat' (bit-exact, host RNG) or 'philox' (in-kernel RNG; `seed` keys the stream)."""
    global _noise_mode, _philox_seed, _philox_counter
    if mode not in ("compat", "philox"):
        raise ValueError("mode must be 'compat' or 'philox'")
    _noise_mode, _philox_seed, _philox_counter = mode, int(seed), 0


def _as_rows(img: np.ndarray):
    """Validate an HWC uint8 image; return (array whose rows are contiguous, row pitch in bytes)."""
    if not isinstance(img, np.ndarray) or img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] != 3:
        raise ValueError("expected a uint8 HxWx3 numpy image")
    h, w, _ = img.shape
    if h < 1 or w < 1:
        raise ValueError("empty image")  # cv2 raises cv2.error on empty input as well
    if img.strides[2] != 1 or img.strides[1] != 3 or img.strides[0] < 3 * w:
        img = np.ascontiguousarray(img)  # exotic views (flipped, channel-sliced): compact first
    return img, img.strides[0]


def _plan_for(h: int, w: int, pitch: int) -> CorruptionPlan:
    key = (h, w, pitch)
    plan = _plans.get(key)
    if plan is None:
        if len(_plans) >= _PLAN_CACHE_MAX:
            _plans.pop(next(iter(_plans)))
        plan = CorruptionPlan([(h, w)], [0], [0], src_pitches=[pitch], dst_pitches=[3 * w])
        _plans[key] = plan
    return plan


def _run(op: int, img_bgr: np.ndarray, *, noise=None, sigma=0.0, k=BLUR_KERNEL, factor=DOWNSCALE_FACTOR,
         seed=0, index=0, kernel=None) -> np.ndarray:
    img, pitch = _as_rows(img_bgr)
    h, w, _ = img.shape
    out = np.empty((h, w, 3), dtype=np.uint8)  # fresh, C-contiguous, caller-owned (SURVEY 8b)
    with _lock:  # the cached plan (its staging buffers, its installed blur kernel) is shared by all threads
        _check_process()
        plan = _plan_for(h, w, pitch)
        if op == N.OP_BLUR:
            plan.set_blur_kernel(kernel)  # None: the angle-0 box
        plan.apply_host(op, img, out, noise_host=noise, sigma=sigma, k=k, factor=factor, seed=seed, first_image_index=index)
    return out


# ---- Low-level corruption functions ----
def _motion_blur_kernel(k: int, angle_deg: float):
    """The k x k float32 kernel of augmentations.py:21-27.  At angle 0 the warpAffine there is the identity, so the
    kernel is row k//2 filled with float32(1)/float32(k).  Other angles need the same host-side OpenCV calls as the
    reference (cv2.getRotationMatrix2D + cv2.warpAffine on a k x k array, ~30 us): coefficient construction only --
    every pixel is still filtered on the GPU."""
    kernel = np.zeros((k, k), dtype=np.float32)
    kernel[k // 2, :] = 1.0
    if float(angle_deg) != 0.0:
        try:
            import cv2
        except ImportError as e:  # pragma: no cover
            raise NotImplementedError("angle_deg != 0 needs OpenCV on the host to rotate the k x k kernel") from e
        center = (k / 2 - 0.5, k / 2 - 0.5)
        kernel = cv2.warpAffine(kernel, cv2.getRotationMatrix2D(center, angle_deg, 1.0), (k, k))
    return kernel / (kernel.sum() + 1e-8)


_pinned_fields: dict = {}   # element count -> page-locked float32 buffer for the compat field of apply_noise


def _pinned_field(n: int) -> np.ndarray:
    """A reusable page-locked float32 buffer of n elements (the 12.5 MB field of a VisDrone frame uploads in 0.2 ms from
    pinned memory, 1.2 ms from pageable memory); a handful of sizes are kept."""
    buf = _pinned_fields.get(n)
    if buf is None:
        try:
            import torch
            buf = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
        except Exception:  # no torch / pinning refused: a pageable buffer works too, just slower to upload
            buf = np.empty(n, dtype=np.float32)
        if len(_pinned_fields) >= 8:
            _pinned_fields.pop(next(iter(_pinned_fields)))
        _pinned_fields[n] = buf
    return buf


def _legacy_state(sigma: float):
    """NumPy's global legacy state as (key, pos, has_gauss, cached) for the native generators, or None when the draw must
    be NumPy's own: a state that is not MT19937, or a sigma that is negative (NumPy raises) or NaN."""
    import ctypes
    state = np.random.get_state(legacy=True)
    if state[0] != "MT19937" or not (float(sigma) >= 0.0):
        return None
    return (np.array(state[1], dtype=np.uint32, copy=True), ctypes.c_int32(int(state[2])), ctypes.c_int32(int(state[3])),
            ctypes.c_double(float(state[4])))


def _set_legacy_state(st) -> None:
    key, pos, has, cached = st
    np.random.set_state(("MT19937", key, pos.value, has.value, cached.value))


def legacy_normal_f32(sigma: float, shape, out: np.ndarray = None) -> np.ndarray:
    """np.random.normal(0, sigma, shape).astype(np.float32) -- the draw of augmentations.py:31 -- bit for bit, consuming
    and advancing NumPy's GLOBAL legacy generator exactly like that call, but with the per-sample log / sqrt / divide of
    the polar method spread over all host threads (csrc/np_legacy_rng.cpp; the MT19937 word stream itself stays
    sequential).  The reference spends 104 of its 137 ms per 1360x765 frame in this draw."""
    import ctypes
    n = int(np.prod(shape))
    st = _legacy_state(sigma)
    if st is None:
        return np.random.normal(0, sigma, shape).astype(np.float32)  # (raises ValueError for sigma < 0, like the reference)
    if out is None:
        out = np.empty(n, dtype=np.float32)
    elif out.dtype != np.float32 or out.size != n or not out.flags.c_contiguous:
        raise ValueError("out must be a C-contiguous float32 array of prod(shape) elements")
    key, pos, has, cached = st
    N.check(N.lib().rod_numpy_legacy_normal_f32(key.ctypes.data, ctypes.byref(pos), ctypes.byref(has), ctypes.byref(cached),
                                                float(sigma), n, out.ctypes.data, 0), "rod_numpy_legacy_normal_f32")
    _set_legacy_state(st)
    return out.reshape(shape)


def legacy_normal_f32_device(sigma: float, out, spans) -> int:
    """The same stream as legacy_normal_f32, drawn on the GPU (csrc/legacy_rng.cu) straight into device memory: `out` is
    a CUDA float32 tensor, `spans` a list of (offset, count) element ranges of it, sorted and disjoint.  The values of
    np.random.normal(0, sigma, total).astype(np.float32) fill the spans in order -- one draw per image, back to back, is
    the same stream as one draw per span -- and NumPy's global state ends where that call would leave it.  The draw is
    queued on the current stream; the call returns once the state is known.  Returns the number of values that were
    recomputed on the host (those whose float32 could depend on the last ulps of the device log())."""
    import ctypes

    import torch
    if not (isinstance(out, torch.Tensor) and out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()):
        raise ValueError("out must be a contiguous CUDA float32 tensor")
    offs = np.array([int(o) for o, _ in spans], dtype=np.uint64)
    counts = np.array([int(c) for _, c in spans], dtype=np.uint64)
    if any(int(o) < 0 or int(c) < 0 or int(o) + int(c) > out.numel() for o, c in spans):
        raise ValueError("a span lies outside `out`")
    st = _legacy_state(sigma) if float(sigma) != float("inf") else None
    if st is None:  # NumPy's own draw (raises for sigma < 0 before any state changes)
        vals = torch.from_numpy(np.random.normal(0, sigma, int(counts.sum())).astype(np.float32))
        k = 0
        for o, c in zip(offs.tolist(), counts.tolist()):
            out[o:o + c].copy_(vals[k:k + c])
            k += c
        return 0
    key, pos, has, cached = st
    fix = ctypes.c_int(0)
    with torch.cuda.device(out.device):
        N.check(N.lib().rod_numpy_legacy_normal_f32_device(
            key.ctypes.data, ctypes.byref(pos), ctypes.byref(has), ctypes.byref(cached), float(sigma), offs.ctypes.data,
            counts.ctypes.data, len(spans), out.data_ptr(), ctypes.byref(fix), torch.cuda.current_stream().cuda_stream or None),
            "rod_numpy_legacy_normal_f32_device")
    _set_legacy_state(st)
    return fix.value


def apply_noise(img_bgr: np.ndarray, sigma: float) -> np.ndarray:
    global _philox_counter
    if _noise_mode == "compat":
        # the exact draw of augmentations.py:31 (global legacy NumPy RNG, float64 -> float32).  The draw goes into a
        # page-locked buffer shared by all calls of this size, so draw + upload are one critical section (like the
        # reference, whose np.random.normal holds NumPy's own lock for the draw).
        with _lock:
            _check_process()
            if float(sigma) >= 0.0:
                noise = legacy_normal_f32(sigma, img_bgr.shape, out=_pinned_field(int(np.prod(img_bgr.shape))))
            else:
                noise = legacy_normal_f32(sigma, img_bgr.shape)  # raises like the reference
            return _run(N.OP_NOISE, img_bgr, noise=noise, sigma=float(sigma))
    with _lock:
        idx = _philox_counter
        _philox_counter += 1
    return _run(N.OP_NOISE, img_bgr, sigma=float(sigma), seed=_philox_seed, index=idx)


def apply_motion_blur(img_bgr: np.ndarray, k: int, angle_deg: float) -> np.ndarray:
    if int(k) != k or k < 1 or k % 2 == 0:
        raise NotImplementedError("apply_motion_blur: k must be odd on the B200 path")
    if float(angle_deg) == 0.0:
        if k > 31:
            raise NotImplementedError("apply_motion_blur: k <= 31 at angle 0 on the B200 path")
        return _run(N.OP_BLUR, img_bgr, k=int(k))
    if k * k >= 130:
        raise NotImplementedError("apply_motion_blur: at angle != 0 OpenCV filters kernels of 130+ elements (k >= 13) by "
                                  "DFT, which cannot be reproduced bit-exactly; k <= 11 is implemented")
    return _run(N.OP_BLUR, img_bgr, k=int(k), kernel=_motion_blur_kernel(int(k), angle_deg))


def apply_lowres(img_bgr: np.ndarray, factor: float) -> np.ndarray:
    return _run(N.OP_LOWRES, img_bgr, factor=float(factor))


# name -> call with the module constants looked up at call time (augmentations.py:51-56)
_DISPATCH = {
    "noise": lambda im: apply_noise(im, NOISE_SIGMA),
    "blur": lambda im: apply_motion_blur(im, BLUR_KERNEL, BLUR_ANGLE_DEG),
    "lowres": lambda im: apply_lowres(im, DOWNSCALE_FACTOR),
}


def _apply_random_corruption(img_bgr: np.ndarray) -> np.ndarray:
    """One of the three corruptions, picked with the same `random.choice` draw as the reference."""
    return _DISPATCH[random.choice(["noise", "blur", "lowres"])](img_bgr)


# ---- FRCNN: PIL Image transform ----
class RandomCorruption:
    """PIL Image transform that randomly applies one corruption (torchvision pipelines).

    The reference converts RGB -> BGR, corrupts, converts back (augmentations.py:72-74).  The angle-0 blur and LowRes act
    on each channel separately and identically, so they are applied to the RGB array as it is (same bytes, no swaps).
    The image IS swapped for noise (the channel order decides which plane of the field meets which channel) and for a
    blur at BLUR_ANGLE_DEG != 0 (the general 2-D filter mirrors OpenCV's FMA body / non-FMA row tail split, which is a
    function of the byte position, so the channel order can move a rounding tie): cv2.cvtColor when OpenCV is importable,
    a NumPy reversal otherwise.  The `random` draws are the reference's: random() for the gate, then random.choice
    inside _apply_random_corruption's dispatch."""

    def __init__(self, p: float = 0.5):
        self.p = p

    @staticmethod
    def _swap(arr: np.ndarray) -> np.ndarray:
        try:
            import cv2
            return cv2.cvtColor(arr, cv2.COLOR_RGB2BGR)
        except ImportError:  # pragma: no cover
            return np.ascontiguousarray(arr[:, :, ::-1])

    def __call__(self, img):
        from PIL import Image
        if random.random() > self.p:
            return img
        rgb = np.array(img)
        name = random.choice(["noise", "blur", "lowres"])  # the draw of _apply_random_corruption (augmentations.py:50)
        if name == "noise" or (name == "blur" and float(BLUR_ANGLE_DEG) != 0.0):
            out = self._swap(_DISPATCH[name](self._swap(rgb)))
        else:
            out = _DISPATCH[name](rgb)
        return Image.fromarray(out)


# ---- Ultralytics: monkey-patch Albumentations ----
def patch_ultralytics_augmentations():
    """Inject the corruption into Ultralytics' Albumentations transform (call ONCE before model.train()), like
    augmentations.py:78-98.

    With DataLoader workers > 0 (the reference launchers use workers=8, train_yolo_augmented.py:33) the hook runs inside
    worker processes, and each needs its own CUDA context: the multiprocessing start method is switched to 'spawn'
    here, before Ultralytics builds its DataLoader (the launchers call this function at import time, so spawned workers
    re-import the launcher and re-apply the patch -- the Windows behaviour the reference was written for).  Set
    ROD_KEEP_START_METHOD=1 to leave the start method alone; a fork()ed worker then raises the RuntimeError of
    _check_process() on its first image."""
    from ultralytics.data import augment as _augment

    if os.environ.get("ROD_KEEP_START_METHOD", "0") != "1":
        import multiprocessing
        if multiprocessing.get_start_method(allow_none=True) != "spawn":
            multiprocessing.set_start_method("spawn", force=True)

    _OrigCall = _augment.Albumentations.__call__

    def _patched_call(self, labels):
        if random.random() < 0.5:
            labels["img"] = _apply_random_corruption(labels["img"])
        return _OrigCall(self, labels)

    _augment.Albumentations.__call__ = _patched_call
    print("[augmentations] Ultralytics Albumentations patched with corruption augmentations (B200 path)")
