"""Which kernel writes the trainers' inputs, for the output stages: letterbox (training path), CHW float32 (Faster R-CNN
loader) and restoration pairs.

Like test_kernel_paths.py, every case runs its call under torch.profiler, asserts the exact kernels it launched (with
their counts), compares every output element with an exact reference, and checks that the elements around the output
keep a sentinel bit pattern: the bytes in front of the output base and behind its end, the gaps between CHW blocks and
the floats around the restoration tensors.  Philox noise is compared with the device's own corrupt() on the same seed,
first index and offset followed by the oracle's formatting: 0 differing bytes.

OUTPUT_KERNELS is the list of entry points of letterbox.cu, chw.cu and restoration.cu; a CPU test holds it against the
built library and test_every_output_kernel_is_reached runs the whole matrix and asserts that it reaches each of them.

Path selection of rod_corrupt_letterbox_f16 (api.cu), restated by expected_letterbox():
  fused path, ONE launch of fused_letterbox2_kernel<4>, when all of
    out_w is even and the fp16 output base is 4-byte aligned (the kernel stores pairs of halves);
    every source shape is a plain INTER_LINEAR letterbox (neither an identity nor an exact 2x2 decimation);
    no general-angle blur kernel is installed, 3 <= k <= 31 (odd), and Philox sigma <= 2048 or a supplied field;
    the shared memory of its per-warp row buffers fits 227 KB: 544 + 12 * (192 + round_up_16(3 * max_w)) bytes, i.e.
      every source row is at most 6373 pixels wide.
  LowRes on the fused path runs inside the kernel when every shape that LowRes does not map onto itself is eligible
    for the exact-2x kernels (w % 4 == 0, families P / H / F and wide exact-2x shapes), every source row offset and
    pitch is 4-byte aligned, and so is the `src` base; otherwise the LowRes kernels (expected_lowres) write the LowRes
    images to the plan's scratch first, once per call.
  unfused path otherwise: the noise kernel (noise_kernel<0> for a supplied field, noise_kernel<1>: the training path
    always uses Box-Muller), the blur (blur_rows_kernel<9> / <0>, the copy kernel for k = 1, filter2d_kernel for an
    installed kernel), the LowRes kernels, then letterbox_kernel; 3 + the LowRes count = plan.launches(101).
"""
import collections
import types

import numpy as np
import pytest

from oracle import corruption_oracle as orc
from oracle import cv2_port
from tests.test_kernel_paths import (COPY, FAMILY, FIRST, OFFSET, SEED, SIGMA, TAIL, Layout, angle_kernel,
                                     expected_lowres, image_of, launched, library_kernels, reference, trace)
from tests.test_kernel_paths import torch_  # noqa: F401  (the module-scoped fixture of the tests below)

gpu = pytest.mark.gpu

OUTPUT_KERNELS = {
    "letterbox.cu": ["fused_letterbox2_kernel<4>", "letterbox_kernel"],
    "chw.cu": ["chw_f32_kernel"],
    "restoration.cu": ["format_pairs_kernel", "gather_patches_kernel", "resize_linear_kernel"],
}
ALL_OUTPUT_KERNELS = sorted(k for ks in OUTPUT_KERNELS.values() for k in ks)
FUSED, UNFUSED = "fused_letterbox2_kernel<4>", "letterbox_kernel"


def test_output_kernel_list_matches_library():
    """OUTPUT_KERNELS holds every entry point of letterbox.cu, chw.cu and restoration.cu in the built library, and
    nothing else."""
    for ident, got in library_kernels(OUTPUT_KERNELS).items():
        assert got == sorted(OUTPUT_KERNELS[ident]), (ident, sorted(set(got) ^ set(OUTPUT_KERNELS[ident])))
    assert len(ALL_OUTPUT_KERNELS) == 6


# ------------------------------------------------------------------ shapes: LowRes family at factor 0.5, exact-2x flag
# (classes of the table in test_kernel_paths.py; the trace assertions below check every classification)
X2W = {(96, 160), (97, 160), (66, 100), (67, 100), (64, 136), (765, 1360), (5, 100), (2, 512), (64, 64), (128, 128)}
OUT_FAMILY = {**FAMILY, **{
    (96, 160): "P", (97, 160): "H", (66, 100): "P", (67, 100): "H", (64, 136): "P", (765, 1360): "H", (5, 100): "H",
    (65, 101): "I+", (66, 101): "I-", (33, 47): "I+", (3, 5): "I+", (5, 9): "I+", (7, 9): "I+", (20, 30): "R",
    (1, 40): "R", (1, 1): "GEN", (40, 1): "GEN", (8, 6373): "GEN", (8, 6374): "R",
    # CHW widths around the staging segment
    (4, 1): "GEN", (3, 2): "R", (2, 3): "GEN", (4, 5): "I-", (3, 6): "R", (2, 7): "I-", (3, 8): "R", (4, 9): "I-",
    (5, 509): "I+", (3, 510): "R", (5, 511): "I+", (2, 512): "P", (5, 513): "I+", (2, 1021): "I-", (3, 1022): "R",
    (4, 1023): "I-", (3, 1024): "R", (2, 1025): "I-", (3, 2048): "R",
    # restoration patches
    (2, 2): "R", (3, 3): "GEN", (7, 7): "I+", (63, 63): "I+", (64, 64): "P", (65, 65): "I+", (128, 128): "P",
    (255, 255): "I+",
}}
LOWRES_IDENTITY = {(1, 1)}   # max(1, int(0.5 * 1)) == 1: LowRes maps (1, 1) onto itself


def lowres_expected(ns):
    """(Counter, strip) of one LowRes call over the images of ns (shapes, so / sp / do / dp, src / dst)."""
    if all(s in LOWRES_IDENTITY for s in ns.shapes):
        return collections.Counter({COPY: 1}), False
    return expected_lowres(ns, 0.5, family=OUT_FAMILY)


class _Ptr:
    def __init__(self, p):
        self.p = p

    def data_ptr(self):
        return self.p


SCRATCH = _Ptr(0)   # the plan's scratch (cudaMalloc): 256-byte aligned


# ------------------------------------------------------------------ sources
class Source:
    """Images image_of(h, w) at offsets aligned to `align` with row pitch 3 w + pad (pad: int or per-image list) in a
    buffer of random bytes, the plan's base at buf[lead:]; destination (scratch) descriptors dense and 256-aligned."""

    def __init__(self, torch, shapes, align=256, pad=0, lead=0):
        from robust_object_detection_b200.batch import CorruptionPlan
        self.shapes, self.align, self.pad, self.lead = list(shapes), align, pad, lead
        self.so, self.sp, cur = [], [], 0
        for i, (h, w) in enumerate(shapes):
            p = 3 * w + Layout._get(pad, i)
            o = (cur + align - 1) // align * align
            self.so.append(o)
            self.sp.append(p)
            cur = o + (h - 1) * p + 3 * w
        self.do, self.dp, d = [], [], 0
        for h, w in shapes:
            self.do.append(d)
            self.dp.append(3 * w)
            d += (3 * h * w + 255) // 256 * 256
        self.plan = CorruptionPlan(shapes, self.so, self.do, self.sp, self.dp)
        self.imgs = [image_of(h, w) for h, w in shapes]
        hsrc = np.random.default_rng(len(shapes) + cur).integers(0, 256, lead + cur + TAIL, dtype=np.uint8)
        for img, o, p in zip(self.imgs, self.so, self.sp):
            h, w, _ = img.shape
            hsrc[lead + o + np.arange(h)[:, None] * p + np.arange(3 * w)[None, :]] = img.reshape(h, 3 * w)
        self.buf = torch.from_numpy(hsrc).cuda()
        self.src = self.buf[lead:]
        self.dst = SCRATCH

    def __repr__(self):
        return f"align{self.align}_pad{self.pad}_lead{self.lead}"

    def corrupt_on_device(self, torch, ops, field, k):
        """The plan's own corrupt() into a fresh buffer (dst descriptors): the reference of Philox noise."""
        dbuf = torch.zeros(self.plan.dst_bytes + 64, dtype=torch.uint8, device="cuda")
        self.plan.corrupt(self.src, dbuf, ops, noise=field, sigma=SIGMA, k=k, factor=0.5, seed=SEED,
                          first_image_index=FIRST, offset=OFFSET)
        host = dbuf.cpu().numpy()
        return [host[o:o + 3 * h * w].reshape(h, w, 3) for o, (h, w) in zip(self.do, self.shapes)]

    def fields(self, torch, compat):
        if not compat:
            return None, None
        fs = [np.random.default_rng(300 + i).normal(0, SIGMA, img.shape).astype(np.float32)
              for i, img in enumerate(self.imgs)]
        return fs, torch.from_numpy(np.concatenate([f.reshape(-1) for f in fs])).cuda()


def corrupted_want(s, ops, fields, k, angle, dev):
    """The corrupted uint8 images: the oracle for every op but Philox noise, the device's corrupt() for that."""
    want = []
    for i, ((h, w), img, op) in enumerate(zip(s.shapes, s.imgs, ops)):
        if op == 0:
            cor = img
        elif op == 1:
            cor = orc.add_noise_field(img, fields[i]) if fields is not None else dev[i]
        elif op == 2:
            cor = reference("filter2d", h, w, k, angle) if angle else (img if k == 1 else reference("blur", h, w, k))
        else:
            cor = reference("lowres", h, w, 0.5)
        if dev is not None and not (op == 1 and fields is None):
            assert np.array_equal(dev[i], cor), ("device corrupt() != oracle", i, (h, w), op)
        want.append(cor)
    return want


# ------------------------------------------------------------------ letterbox
HSENT = 0xFDA5   # a NaN: no output half has this pattern


def fused_fits(shapes):
    buf = 64 + (3 * max(w for _, w in shapes) + 15) // 16 * 16 + 128
    return 2 * 256 + 32 + 4 * 3 * buf <= 227 * 1024


def expected_letterbox(s, out_h, out_w, k, compat, angle, out_ptr):
    """(Counter of the kernels rod_corrupt_letterbox_f16 launches, fused?, LowRes inside the kernel?, strip?)."""
    linear = True
    for h, w in s.shapes:
        nh, nw, _, _ = orc.letterbox_geometry(h, w, out_h, out_w)
        assert nh >= 1 and nw >= 1, ((h, w), out_h, out_w)
        if (nh, nw) == (h, w) or (h == 2 * nh and w == 2 * nw):
            linear = False
    fused = (out_w % 2 == 0 and out_ptr % 4 == 0 and linear and not angle and 3 <= k <= 31 and fused_fits(s.shapes))
    lowres, strip = lowres_expected(s)
    if fused:
        in_kernel = (all(sh in X2W or sh in LOWRES_IDENTITY for sh in s.shapes)
                     and all(o % 4 == 0 and p % 4 == 0 for o, p in zip(s.so, s.sp)) and s.src.data_ptr() % 4 == 0)
        want = collections.Counter({FUSED: 1})
        if not in_kernel:
            want += lowres
        return want, True, in_kernel, strip and not in_kernel
    blur = "filter2d_kernel" if angle else COPY if k == 1 else "blur_rows_kernel<9>" if k == 9 else "blur_rows_kernel<0>"
    want = collections.Counter({"noise_kernel<0>" if compat else "noise_kernel<1>": 1, UNFUSED: 1})
    want[blur] += 1
    return want + lowres, False, False, strip


_lb_want = {}
_geometry_checked = set()


def letterbox_want(cor, key, out_h, out_w, pad):
    """oracle letterbox of one corrupted image as uint16 bits; key (hashable) caches it, None: not cached."""
    if key is not None and key in _lb_want:
        return _lb_want[key]
    h, w = cor.shape[:2]
    if cv2_port.available() and (h, w, out_h, out_w) not in _geometry_checked:
        import cv2
        nh, nw, _, _ = orc.letterbox_geometry(h, w, out_h, out_w)
        img = image_of(h, w)
        assert np.array_equal(orc.resize_linear(img, nh, nw), cv2.resize(img, (nw, nh))), ("oracle != cv2", h, w, nh, nw)
        _geometry_checked.add((h, w, out_h, out_w))
    out = orc.letterbox_norm_f16(cor, out_h, out_w, pad).view(np.uint16)
    if key is not None:
        _lb_want[key] = out
    return out


LbCase = collections.namedtuple("LbCase", "name shapes ops out k pad src compat angle out_lead side_stream")


def lb_case(name, shapes, ops, out, k=9, pad=114, src=None, compat=False, angle=None, out_lead=0, side_stream=False):
    ops = [ops(i) for i in range(len(shapes))] if callable(ops) else list(ops)
    return LbCase(name, list(shapes), ops, out, k, pad, src or {}, compat, angle, out_lead, side_stream)


MIX = [(765, 1360), (96, 160), (97, 160), (66, 100), (67, 100), (64, 136), (65, 101), (33, 47), (20, 30), (66, 101)]
ALL_X2W = [(96, 160), (97, 160), (66, 100), (67, 100), (64, 136), (765, 1360), (5, 100), (1, 1)]
SMALL = [(3, 5), (5, 9), (7, 9), (20, 30), (33, 47), (3, 4)]


def i4(i):
    return i % 4


def letterbox_cases():
    mixed_ops = [3, 3, 1, 3, 2, 3, 0, 3]
    return [
        # downscales at 1360 -> 640 (lane_group 10), upscales, (1, w) / (h, 1) / (1, 1), w % 16, % 8, % 4, odd w
        lb_case("640-compat-dense", MIX + [(1, 40), (40, 1), (1, 1)], i4, (640, 640), compat=True),
        lb_case("320-philox-align4", MIX, i4, (320, 320), k=5, pad=0, src=dict(align=4), out_lead=2),
        # every shape exact-2x (odd and even h, a 1 x 1 identity): LowRes inside the fused kernel
        lb_case("lowres-in-kernel-philox", ALL_X2W, mixed_ops, (96, 98), k=31, pad=255,
                src=dict(pad=[0] * 7 + [1]), out_lead=8),
        lb_case("lowres-in-kernel-compat", ALL_X2W, [3, 1, 3, 2, 3, 0, 3, 3], (640, 640), k=3,
                src=dict(pad=[0] * 7 + [1]), compat=True),
        # ... and the same batch with the source base at +2: LowRes through the scratch (strip kernel)
        lb_case("lowres-scratch-srclead2", ALL_X2W, mixed_ops, (640, 640), compat=True, src=dict(pad=[0] * 7 + [1], lead=2)),
        lb_case("33x34-pitch1", MIX, i4, (33, 34), k=3, src=dict(align=16, pad=1)),
        lb_case("1x2-pitch4-lead16", [(3, 4), (3, 5), (7, 9), (5, 9)], [0, 1, 2, 3], (1, 2), src=dict(align=16, pad=4, lead=16),
                compat=True),
        lb_case("2x62-pitch16", [(1, 40), (5, 100), (3, 5), (33, 47)], [1, 2, 3, 1], (2, 62), k=5, pad=255,
                src=dict(align=16, pad=16), out_lead=2),
        lb_case("5x66-lead1", [(765, 1360), (66, 101), (97, 160), (1, 1)], [1, 3, 2, 0], (5, 66), pad=0,
                src=dict(align=16, lead=1), compat=True),
        lb_case("5x66-lead4-philox", [(765, 1360), (66, 101), (97, 160), (1, 1)], [1, 3, 1, 2], (5, 66), k=31,
                src=dict(align=16, lead=4)),
        # unfused: odd out_w, identity and exact-2x letterboxes, a general-angle kernel, k = 1
        lb_case("320x319-philox", MIX, i4, (320, 319)),
        lb_case("320x319-compat-pitch1", MIX, i4, (320, 319), k=31, src=dict(pad=1), compat=True),
        lb_case("identity-area2-philox", [(66, 100), (33, 47), (765, 1360), (65, 101)], [1, 1, 2, 3], (33, 50)),
        lb_case("identity-area2-compat", [(66, 100), (33, 47), (765, 1360), (65, 101)], [1, 3, 1, 2], (33, 50), pad=0,
                compat=True),
        lb_case("angle45", MIX, i4, (96, 98), angle=45),
        lb_case("k1", MIX, i4, (96, 98), k=1, pad=0),
        # batch sizes: 1, 129 (no stream fork on the unfused path), 300 (unsorted row order of the fused kernel)
        lb_case("n1-fused-philox", [(765, 1360)], [1], (640, 640)),
        lb_case("n1-fused-lowres", [(33, 47)], [3], (96, 98), k=31, compat=True),
        lb_case("n129-unfused", [SMALL[i % 6] for i in range(129)], i4, (320, 319)),
        lb_case("n300-fused-philox", [SMALL[i % 6] for i in range(300)], i4, (33, 34), out_lead=2),
        lb_case("n300-fused-compat", [SMALL[i % 6] for i in range(300)], lambda i: (i // 3) % 4, (33, 34), compat=True),
        # widest rows: 6373 pixels fit the fused kernel's buffers, 6374 do not (LowRes must still run once)
        lb_case("w6373-fused", [(8, 6373), (97, 160)], [3, 1], (640, 640)),
        lb_case("w6374-unfused", [(8, 6374), (97, 160)], [3, 1], (640, 640)),
        lb_case("side-stream", MIX, i4, (96, 98), side_stream=True),
    ]


LB_CASES = letterbox_cases()


def run_letterbox(torch, c, out_lead=None):
    """Runs case c with the output base at out_lead halves (default: the case's); returns (kernels, output bits, fused)."""
    out_lead = c.out_lead if out_lead is None else out_lead
    s = Source(torch, c.shapes, **c.src)
    n, (oh, ow) = len(c.shapes), c.out
    if c.angle:
        s.plan.set_blur_kernel(angle_kernel(c.k, c.angle))
    ops = torch.tensor(c.ops, dtype=torch.uint8, device="cuda")
    fields, field = s.fields(torch, c.compat)
    dev = None
    if not c.compat and 1 in c.ops:
        s.plan.set_gaussian_generator(1)   # the training path always uses Box-Muller
        dev = s.corrupt_on_device(torch, ops, None, c.k)
    cor = corrupted_want(s, c.ops, fields, c.k, c.angle, dev)
    size = n * 3 * oh * ow
    obuf = torch.full((out_lead + size + TAIL,), HSENT - 0x10000, dtype=torch.int16, device="cuda")
    out = obuf[out_lead:out_lead + size].view(torch.float16).view(n, 3, oh, ow)
    want_k, fused, in_kernel, strip = expected_letterbox(s, oh, ow, c.k, c.compat, c.angle, out.data_ptr())
    kw = dict(noise=field, sigma=SIGMA, k=c.k, factor=0.5, seed=SEED, first_image_index=FIRST, offset=OFFSET)
    host = {}
    if c.side_stream:
        st = torch.cuda.Stream()

        def call():
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                s.plan.corrupt_letterbox(s.src, ops, out, oh, ow, c.pad, **kw)
                host["out"] = obuf.cpu().numpy()
    else:
        def call():
            s.plan.corrupt_letterbox(s.src, ops, out, oh, ow, c.pad, **kw)

    got = launched(call)
    assert got == want_k, (c.name, out_lead, dict(got), dict(want_k))
    if not strip:
        want_n = (1 + (0 if in_kernel else s.plan.launches(3))) if fused else s.plan.launches(101)
        assert sum(got.values()) == want_n, (c.name, sum(got.values()), want_n)
    bits = (host["out"] if c.side_stream else obuf.cpu().numpy()).view(np.uint16)
    for i, ((h, w), op) in enumerate(zip(c.shapes, c.ops)):
        noisy = op == 1
        key = None if noisy else ((h, w), op, c.k, c.angle, c.out, c.pad)
        want = letterbox_want(cor[i], key, oh, ow, c.pad)
        g = bits[out_lead + i * 3 * oh * ow: out_lead + (i + 1) * 3 * oh * ow].reshape(3, oh, ow)
        bad = int((g != want).sum())
        assert bad == 0, (c.name, i, (h, w), op, f"{bad} halves differ")
    assert (bits[:out_lead] == HSENT).all() and (bits[out_lead + size:] == HSENT).all(), (c.name, "guard halves written")
    return got, bits[out_lead:out_lead + size].copy(), fused


def run_letterbox_case(torch, c):
    """Case c, and if it takes the fused path, the same call with the output base at +2 bytes (unfused path, same
    inputs): the two outputs must be bit-identical."""
    got, bits, fused = run_letterbox(torch, c)
    reached = [got]
    if fused:
        got1, bits1, fused1 = run_letterbox(torch, c, out_lead=1)
        assert not fused1 and got1[UNFUSED] == 1, (c.name, dict(got1))
        assert np.array_equal(bits, bits1), (c.name, "fused != unfused", int((bits != bits1).sum()))
        reached.append(got1)
    return reached


@gpu
@pytest.mark.parametrize("case", LB_CASES, ids=[c.name for c in LB_CASES])
def test_letterbox_paths(torch_, case):
    run_letterbox_case(torch_, case)


@gpu
def test_letterbox_paths_examples(torch_):
    """The selection spelled out: the 1360 x 765 mix is fused with a LowRes pre-pass, the exact-2x batch runs LowRes
    inside the kernel, rows of 6374 pixels go unfused with each LowRes list launched once, and a 2-byte aligned output
    takes the unfused path."""
    by = {c.name: c for c in LB_CASES}
    got = run_letterbox(torch_, by["640-compat-dense"])[0]
    assert got[FUSED] == 1 and got[UNFUSED] == 0 and len(got) > 1
    assert run_letterbox(torch_, by["lowres-in-kernel-philox"])[0] == {FUSED: 1}
    got = run_letterbox(torch_, by["w6374-unfused"])[0]
    assert got == {UNFUSED: 1, "noise_kernel<1>": 1, "blur_rows_kernel<9>": 1, "lowres_x2_kernel<128>": 1,
                   "lowres_x2h_kernel<16>": 1}, dict(got)
    got = run_letterbox(torch_, by["lowres-in-kernel-philox"], out_lead=1)[0]
    assert got[UNFUSED] == 1 and got[FUSED] == 0


# ------------------------------------------------------------------ CHW float32
FSENT = 0x7FA5A5A5   # a NaN: no output float has this pattern
CHW_SHAPES = [(4, 1), (3, 2), (2, 3), (3, 4), (4, 5), (3, 6), (2, 7), (3, 8), (4, 9), (5, 509), (3, 510), (5, 511),
              (2, 512), (5, 513), (2, 1021), (3, 1022), (4, 1023), (3, 1024), (2, 1025), (3, 2048)]
CHW_CASES = [("dense-philox", {}, False), ("dense-compat", {}, True),
             ("pitch1-lead1-philox", dict(align=1, pad=1, lead=1), False),
             ("pitch4-lead2-compat", dict(align=16, pad=4, lead=2), True),
             ("pitch16-lead16-philox", dict(align=16, pad=16, lead=16), False)]


def to_unit(cor):
    """torchvision's to_dtype_image: float(v) * fl(1/255) in float32, BGR -> RGB, HWC -> CHW."""
    return (cor[:, :, ::-1].astype(np.float32) * np.float32(1.0 / 255)).transpose(2, 0, 1)


def run_chw(torch, name, src, compat):
    s = Source(torch, CHW_SHAPES, **src)
    ops_h = [(i + (1 if compat else 0)) % 4 for i in range(len(CHW_SHAPES))]
    ops = torch.tensor(ops_h, dtype=torch.uint8, device="cuda")
    fields, field = s.fields(torch, compat)
    dev = s.corrupt_on_device(torch, ops, field, 9)   # the plan's own generator, as rod_corrupt_chw_f32 uses
    cor = corrupted_want(s, ops_h, fields, 9, None, dev)
    offs = s.plan.chw_offsets()
    lead = 64   # floats: keeps the 256-byte alignment the call requires
    obuf = torch.full((lead + offs[-1] + TAIL,), FSENT, dtype=torch.int32, device="cuda")
    out = obuf[lead:lead + offs[-1]].view(torch.float32)
    got = launched(lambda: s.plan.corrupt_chw_f32(s.src, ops, out, noise=field, sigma=SIGMA, k=9, factor=0.5, seed=SEED,
                                                  first_image_index=FIRST, offset=OFFSET))
    lowres, strip = lowres_expected(s)
    want_k = lowres + collections.Counter({"noise_kernel<0>" if compat else "noise_table_kernel<1, 1024, 2, 10>": 1,
                                           "blur_rows_kernel<9>": 1, "chw_f32_kernel": 1})
    assert got == want_k, (name, dict(got), dict(want_k))
    if not strip:
        assert sum(got.values()) == s.plan.launches(102), (name, sum(got.values()), s.plan.launches(102))
    host = obuf.cpu().numpy().view(np.uint32)
    covered = np.zeros(host.size, bool)
    for i, (h, w) in enumerate(CHW_SHAPES):
        a = lead + offs[i]
        g = host[a:a + 3 * h * w].reshape(3, h, w)
        want = to_unit(cor[i]).view(np.uint32)
        bad = int((g != want).sum())
        assert bad == 0, (name, i, (h, w), ops_h[i], f"{bad} floats differ")
        covered[a:a + 3 * h * w] = True
    bad = int((host[~covered] != FSENT).sum())
    assert bad == 0, (name, f"{bad} guard floats written")
    return got


@gpu
@pytest.mark.parametrize("case", CHW_CASES, ids=[c[0] for c in CHW_CASES])
def test_chw_paths(torch_, case):
    assert {h * w % 4 for h, w in CHW_SHAPES} == {0, 1, 2, 3}
    run_chw(torch_, *case)


# ------------------------------------------------------------------ restoration pairs
# (patch size, batch size, compat, calls on one plan)
RESTORATION_CASES = [(1, 130, False, 1), (2, 5, True, 2), (3, 1, False, 1), (7, 130, True, 1), (63, 5, False, 2),
                     (64, 1, True, 1), (65, 5, False, 1), (128, 5, True, 1), (255, 1, False, 1), (64, 130, False, 2)]


def run_restoration(torch, P, n, compat, calls):
    """n crops of P x P at every 16-byte phase of one frame (odd pitch, base at +3), flips and op-codes per call;
    several calls reuse the plan's inner plan.  Returns the kernels launched by every call."""
    from robust_object_detection_b200.batch import CorruptionPlan
    fh, fw = P + 37, P + 29
    pitch, lead = 3 * fw + 5, 3
    frame = image_of(fh, fw)
    hbuf = np.random.default_rng(P * 1000 + n).integers(0, 256, lead + fh * pitch + TAIL, dtype=np.uint8)
    hbuf[lead + np.arange(fh)[:, None] * pitch + np.arange(3 * fw)[None, :]] = frame.reshape(fh, 3 * fw)
    sbuf = torch.from_numpy(hbuf).cuda()
    yx = [((5 * i) % (fh - P + 1), (3 * i + i // 16) % (fw - P + 1)) for i in range(n)]
    offs = [y * pitch + 3 * x for y, x in yx]
    if n >= 16:
        assert {(lead + o) % 16 for o in offs} == set(range(16))
    plan = CorruptionPlan([(P, P)] * n, offs, [0] * n, src_pitches=[pitch] * n)
    stride = (3 * P * P + 255) // 256 * 256
    inner = types.SimpleNamespace(shapes=[(P, P)] * n, so=[i * stride for i in range(n)], sp=[3 * P] * n,
                                  do=[i * stride for i in range(n)], dp=[3 * P] * n, src=SCRATCH, dst=SCRATCH)
    lowres, _ = lowres_expected(inner)
    noise_k = "noise_kernel<0>" if compat else "noise_table_kernel<1, 1024, 2, 10>"
    want_inner = lowres + collections.Counter({COPY: 1, noise_k: 1, "blur_rows_kernel<9>": 1})
    size = n * 3 * P * P
    reached = []
    for call in range(calls):
        flips_h = [(i * 7 + call) % 3 == 0 for i in range(n)]
        ops_h = [(i + 2 * call + (0 if compat else 1)) % 4 for i in range(n)]
        patches = []
        for (y, x), f in zip(yx, flips_h):
            p = frame[y:y + P, x:x + P]
            patches.append(np.ascontiguousarray(p[:, ::-1] if f else p))
        fields = field = None
        if compat:
            fields = [np.random.default_rng(400 + 10 * call + i).normal(0, SIGMA, (P, P, 3)).astype(np.float32)
                      for i in range(n)]
            field = torch.from_numpy(np.stack(fields).reshape(-1)).cuda()
        ops = torch.tensor(ops_h, dtype=torch.uint8, device="cuda")
        dev = None
        if not compat:   # the corrupt() of a uniform plan of the host-cropped patches, generator of the outer plan
            uni = CorruptionPlan.uniform(n, P, P)
            psrc = torch.from_numpy(np.stack(patches)).cuda()
            pdst = torch.zeros_like(psrc)
            uni.corrupt(psrc, pdst, ops, sigma=SIGMA, k=9, factor=0.5, seed=SEED, first_image_index=FIRST, offset=OFFSET)
            dev = pdst.cpu().numpy()
        bufs = [torch.full((5 + size + TAIL,), FSENT, dtype=torch.int32, device="cuda") for _ in range(2)]
        cor_t, clean_t = (b[5:5 + size].view(torch.float32).view(n, 3, P, P) for b in bufs)
        flips = torch.tensor(flips_h, dtype=torch.uint8, device="cuda")
        names = trace(lambda: plan.restoration_pairs(sbuf[lead:], flips, ops, cor_t, clean_t, noise=field, sigma=SIGMA,
                                                     k=9, factor=0.5, seed=SEED, first_image_index=FIRST, offset=OFFSET))
        assert names[0] == "gather_patches_kernel" and names[-1] == "format_pairs_kernel", (P, n, call, names)
        assert collections.Counter(names[1:-1]) == want_inner, (P, n, call, names, dict(want_inner))
        reached.append(collections.Counter(names))
        hc, hk = (b.cpu().numpy().view(np.uint32) for b in bufs)
        for hb in (hc, hk):
            assert (hb[:5] == FSENT).all() and (hb[5 + size:] == FSENT).all(), (P, n, call, "guard floats written")
        for i, (p, op) in enumerate(zip(patches, ops_h)):
            if op == 0:
                c = p
            elif op == 1:
                c = orc.add_noise_field(p, fields[i]) if compat else dev[i]
            elif op == 2:
                c = orc.apply_motion_blur(p, 9, 0)
            else:
                c = orc.apply_lowres(p, 0.5)
            if dev is not None and op != 1:
                assert np.array_equal(dev[i], c), ("device corrupt() != oracle", P, i, op)
            wc = (c[:, :, ::-1].astype(np.float32) / np.float32(255)).transpose(2, 0, 1).view(np.uint32)
            wk = (p[:, :, ::-1].astype(np.float32) / np.float32(255)).transpose(2, 0, 1).view(np.uint32)
            gc = hc[5 + i * 3 * P * P: 5 + (i + 1) * 3 * P * P].reshape(3, P, P)
            gk = hk[5 + i * 3 * P * P: 5 + (i + 1) * 3 * P * P].reshape(3, P, P)
            assert np.array_equal(gk, wk), (P, n, call, i, "clean")
            assert np.array_equal(gc, wc), (P, n, call, i, op, int((gc != wc).sum()))
    return reached


@gpu
@pytest.mark.parametrize("case", RESTORATION_CASES, ids=[f"P{p}-n{n}-{'compat' if c else 'philox'}-x{k}"
                                                         for p, n, c, k in RESTORATION_CASES])
def test_restoration_paths(torch_, case):
    run_restoration(torch_, *case)


# the sizes of test_gpu_parity.py::test_restoration_resize_first_branch, plus a 1-row and a 1-column source
RESIZE_SIZES = [(40, 80, 64, 80), (100, 50, 100, 64), (30, 30, 64, 64), (64, 20, 64, 64), (63, 65, 64, 65), (7, 5, 256, 256),
                (1, 1, 3, 2), (200, 255, 256, 256), (97, 133, 97, 133), (120, 77, 333, 190), (1, 17, 5, 40), (17, 1, 40, 5)]


def run_resize(torch, h, w, nh, nw):
    from robust_object_detection_b200.batch import resize_linear_u8
    img = image_of(h, w)
    res = {}
    got = launched(lambda: res.setdefault("out", resize_linear_u8(img, nh, nw)))
    assert got == {"resize_linear_kernel": 1}, dict(got)
    want = orc.resize_linear(img, nh, nw)
    if cv2_port.available():
        import cv2
        assert np.array_equal(want, cv2.resize(img, (nw, nh))), ("oracle != cv2", h, w, nh, nw)
    assert np.array_equal(res["out"], want), (h, w, nh, nw)
    return got


@gpu
@pytest.mark.parametrize("size", RESIZE_SIZES, ids=["x".join(map(str, s)) for s in RESIZE_SIZES])
def test_resize_linear_path(torch_, size):
    run_resize(torch_, *size)


# ------------------------------------------------------------------ coverage
@gpu
def test_every_output_kernel_is_reached(torch_):
    """Runs the whole matrix (independent of test order and -k) and asserts that the output kernels it reaches are
    exactly OUTPUT_KERNELS; prints the number of cases that reached each."""
    reached = collections.Counter()

    def add(got):
        reached.update(k for k in set(got) if k in ALL_OUTPUT_KERNELS)

    for c in LB_CASES:
        for got in run_letterbox_case(torch_, c):
            add(got)
    for case in CHW_CASES:
        add(run_chw(torch_, *case))
    for case in RESTORATION_CASES:
        for got in run_restoration(torch_, *case):
            add(got)
    for size in RESIZE_SIZES:
        add(run_resize(torch_, *size))
    print("\ncases per output kernel:")
    for name in ALL_OUTPUT_KERNELS:
        print(f"  {reached[name]:5d}  {name}")
    assert sorted(reached) == ALL_OUTPUT_KERNELS, sorted(set(reached) ^ set(ALL_OUTPUT_KERNELS))
