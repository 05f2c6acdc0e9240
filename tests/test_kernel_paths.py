"""Which kernel serves which layout, for the u8 corruption ops (noise, blur, general-angle blur, LowRes).

The kernels of these ops are picked at run time from the image shapes, the row pitches and offsets and the base pointers
of the call.  Output checks alone do not show that a layout still reaches the kernel it was written for, so every case
here runs its call under torch.profiler, asserts the exact kernels it launched, and compares every output byte with the
oracle (Philox outputs with the restated stream) while the bytes the call must not write keep a sentinel: pitch padding,
gaps between images, the bytes in front of the base pointer, the tail of the buffer and the images an op-code masks.

KERNELS is the list of entry points of noise.cu, blur.cu, filter2d.cu and lowres.cu; a CPU test holds it against the
built library and test_every_kernel_is_reached runs the whole matrix and asserts that it reaches each of them.

LowRes selection (ensure_lowres_tables in plan.cu, launch_lowres_lists in lowres.cu), restated by expected_lowres():
every image lands in one tile list; one launch per non-empty list.
  family (shape, factor 0.5)                    list / kernel
  odd w, three x taps, regular y axis            X2I_CARRY (odd h) / X2I_EVEN (even h): lowres_x2i_kernel<true / false>
  odd w, three x taps, other y axes              X2G: lowres_x2g_kernel
  exact 2x in both axes, w % 4 == 0     (P)  \\  source rows (pitch | offset) not 4-aligned: X2_REST
  odd h up to ~2000, w % 4 == 0         (H)   > destination rows not 4-aligned: X2W8 (source rows 8-aligned, w % 8 == 0)
  odd h from ~2001, w % 4 == 0          (F)  /    or X2W4: lowres_x2w_kernel
                                                 else X2P / X2H / X2F by copy unit 16 / 8 / 4 (w and every offset and
                                                 pitch of the image a multiple of it): lowres_x2{p,h,f}_kernel<unit>
  other exact-2x widths (w % 4 != 0, FASTN y)    X2_REST: lowres_x2_kernel<128>
  anything else (factor != 0.5, w = 2 nw + 1 without three x taps, ...)   GENERIC: lowres_kernel
Base pointers: a source base that is not 4-aligned, or a destination base that is not 4-aligned while X2P / X2H / X2F
lists exist, replaces every band list (X2W, X2P, X2H, X2F) and X2_REST by ONE launch of lowres_x2_kernel<128> over all
exact-2x images.  Otherwise a staged list runs the kernel of the larger of its copy unit and the unit (src | dst) allows,
and X2W8 runs lowres_x2w_kernel<true> only when the source base is 8-aligned.
"""
import collections
import os
import re
import subprocess

import numpy as np
import pytest

from oracle import corruption_oracle as orc
from oracle import cv2_port
from tests.helpers import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "robust-object-detection_b200", "librod_b200.so")
gpu = pytest.mark.gpu

# ------------------------------------------------------------------ the kernel list
LOWRES_KERNELS = [
    "lowres_kernel", "lowres_x2_kernel<128>", "lowres_x2w_kernel<true>", "lowres_x2w_kernel<false>",
    "lowres_x2p_kernel<16>", "lowres_x2p_kernel<8>", "lowres_x2p_kernel<4>",
    "lowres_x2f_kernel<16>", "lowres_x2f_kernel<8>", "lowres_x2f_kernel<4>",
    "lowres_x2h_kernel<16>", "lowres_x2h_kernel<8>", "lowres_x2h_kernel<4>",
    "lowres_x2g_kernel", "lowres_x2i_kernel<true>", "lowres_x2i_kernel<false>",
]
KERNELS = {
    "noise.cu": ["noise_kernel<0>", "noise_kernel<1>", "noise_kernel<2>", "noise_kernel<3>",
                 "noise_table_kernel<1, 1024, 2, 7>", "noise_table_kernel<1, 1024, 2, 10>",
                 "noise_table_kernel<3, 1024, 2, 7>", "noise_table_kernel<3, 1024, 2, 10>"],
    "blur.cu": ["blur_rows_kernel<0>", "blur_rows_kernel<9>"],
    "filter2d.cu": ["filter2d_kernel"],
    "lowres.cu": LOWRES_KERNELS,
}
ALL_KERNELS = sorted(k for ks in KERNELS.values() for k in ks)
COPY = "noise_kernel<2>"   # NOISE_COPY: op-code 0 images of corrupt(), k = 1 blur, identity LowRes
X2 = "lowres_x2_kernel<128>"


def kernel_name(raw: str) -> str:
    """'void rod::lowres_x2w_kernel<(bool)1>(rod::LowresX2wParams)' -> 'lowres_x2w_kernel<true>'."""
    s = raw.strip()
    s = re.sub(r"\(bool\)1\b", "true", re.sub(r"\(bool\)0\b", "false", s))
    s = re.sub(r"\((?:unsigned )?int\)", "", s)
    if s.startswith("void "):
        s = s[5:]
    depth = 0
    for i, ch in enumerate(s):
        depth += (ch == "<") - (ch == ">")
        if ch == "(" and depth == 0:
            s = s[:i]
            break
    base, lt, args = s.partition("<")
    args = re.sub(r"\s*,\s*", ", ", args.strip())
    return base.split("::")[-1] + lt + args


def library_kernels(sources):
    """{source file: sorted kernel names (as in KERNELS)} of the entry points the built library holds for each of
    `sources` (cuobjdump -symbols, demangled with cu++filt)."""
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    bindir = os.path.dirname(os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"))   # the toolkit of csrc/Makefile
    dump = subprocess.check_output([os.path.join(bindir, "cuobjdump"), "-symbols", LIB], text=True)
    entries, ident = collections.defaultdict(list), None
    for line in dump.splitlines():
        m = re.match(r"\s*identifier\s*=\s*(\S+)", line)
        if m:
            ident = os.path.basename(m.group(1))
        elif "STO_ENTRY" in line and ident in sources:
            entries[ident].append(line.split()[-1])
    out = {}
    for ident in sources:
        assert entries[ident], f"no entry symbols of {ident} in {LIB}"
        names = subprocess.check_output([os.path.join(bindir, "cu++filt")], input="\n".join(entries[ident]) + "\n",
                                        text=True).split("\n")
        out[ident] = sorted(kernel_name(n) for n in names if n.strip())
    return out


def test_kernel_list_matches_library():
    """KERNELS holds every entry point of noise.cu, blur.cu, filter2d.cu and lowres.cu in the built library, and
    nothing else: a kernel added or removed there must be added to or removed from the matrix below."""
    for ident, got in library_kernels(KERNELS).items():
        want = KERNELS[ident]
        assert got == sorted(want), (ident, sorted(set(got) ^ set(want)))
    assert len(ALL_KERNELS) == 27


# ------------------------------------------------------------------ launch trace
def trace(fn):
    """Runs fn() under torch.profiler (CUDA activity only) and returns the kernels it launched (names as in KERNELS)
    in the order they started; copies and memsets are left out."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        if e.name.startswith(("Memcpy", "Memset")) or "(" not in e.name:   # kernels carry their parameter list
            continue
        names.append((e.time_range.start, kernel_name(e.name)))
    return [n for _, n in sorted(names, key=lambda t: t[0])]


def launched(fn):
    """The kernels fn() launched (names as in KERNELS, with multiplicity)."""
    return collections.Counter(trace(fn))


# ------------------------------------------------------------------ layouts
SENTINEL = 0xA5
TAIL = 64


class Layout:
    """Source and destination layout of one plan: per image a pitch padding and a 16-byte phase of its offset, and the
    byte lead of the plan's base pointer inside a larger buffer (buf[lead:])."""

    def __init__(self, spad=0, dpad=0, sphase=0, dphase=0, slead=0, dlead=0, mask=False):
        self.spad, self.dpad, self.sphase, self.dphase = spad, dpad, sphase, dphase
        self.slead, self.dlead, self.mask = slead, dlead, mask

    def __repr__(self):
        return (f"pad{self.spad}-{self.dpad}_ph{self.sphase}-{self.dphase}_lead{self.slead}-{self.dlead}"
                + ("_mask" if self.mask else ""))

    @staticmethod
    def _get(v, i):
        return v[i % len(v)] if isinstance(v, (list, tuple)) else v

    def offsets(self, shapes, pad, phase):
        offs, pitches, cur = [], [], 0
        for i, (h, w) in enumerate(shapes):
            p = 3 * w + self._get(pad, i)
            o = (cur + 15) // 16 * 16 + self._get(phase, i)
            offs.append(o)
            pitches.append(p)
            cur = o + (h - 1) * p + 3 * w + 16   # a gap of guard bytes before the next image
        return offs, pitches, cur


def image_of(h, w):
    return synth(h * 7919 + w, h, w)


def row_index(off, pitch, h, w):
    return off + np.arange(h)[:, None] * pitch + np.arange(3 * w)[None, :]


class Batch:
    """A plan over `shapes` laid out by `lay`, its source buffer (image bytes at the plan's offsets, random bytes in
    every gap) and a destination buffer filled with SENTINEL."""

    def __init__(self, torch, shapes, lay, opcode):
        from robust_object_detection_b200.batch import CorruptionPlan
        self.torch, self.shapes, self.lay = torch, list(shapes), lay
        self.so, self.sp, s_end = lay.offsets(shapes, lay.spad, lay.sphase)
        self.do, self.dp, d_end = lay.offsets(shapes, lay.dpad, lay.dphase)
        self.plan = CorruptionPlan(shapes, self.so, self.do, self.sp, self.dp)
        self.imgs = [image_of(h, w) for h, w in shapes]
        hsrc = np.random.default_rng(len(shapes) + s_end).integers(0, 256, lay.slead + s_end + TAIL, dtype=np.uint8)
        for img, o, p in zip(self.imgs, self.so, self.sp):
            h, w, _ = img.shape
            hsrc[row_index(lay.slead + o, p, h, w)] = img.reshape(h, 3 * w)
        self.sbuf = torch.from_numpy(hsrc).cuda()
        self.dbuf = torch.full((lay.dlead + d_end + TAIL,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.src, self.dst = self.sbuf[lay.slead:], self.dbuf[lay.dlead:]
        self.ops = [0 if (lay.mask and i % 3 == 1) else opcode for i in range(len(shapes))]
        self.opcodes = torch.tensor(self.ops, dtype=torch.uint8, device="cuda")

    def check(self, want, host=None, compare=None):
        """want[i]: the expected image i, or None where the destination must keep the sentinel."""
        host = self.dbuf.cpu().numpy() if host is None else host
        covered = np.zeros(host.size, bool)
        for i, ((h, w), o, p) in enumerate(zip(self.shapes, self.do, self.dp)):
            if want[i] is None:
                continue
            idx = row_index(self.lay.dlead + o, p, h, w)
            got = host[idx].reshape(h, w, 3)
            if compare is not None:
                compare(i, got, want[i])
            else:
                bad = int((got != want[i]).sum())
                assert bad == 0, f"image {i} {self.shapes[i]} ({self.lay}): {bad} bytes differ"
            covered[idx] = True
        bad = int((host[~covered] != SENTINEL).sum())
        assert bad == 0, f"{bad} guard bytes written ({self.lay})"


# ------------------------------------------------------------------ references (oracle, and cv2 where importable)
_want = {}


def reference(op, h, w, *params):
    key = (op, h, w) + params
    if key not in _want:
        img = image_of(h, w)
        if op == "lowres":
            out = orc.apply_lowres(img, params[0])
            if cv2_port.available():
                assert np.array_equal(out, cv2_port.lowres(img, params[0])), ("oracle != cv2", key)
        elif op == "blur":
            out = orc.apply_motion_blur(img, params[0], 0)
            # k * k >= 130: cv2.filter2D takes its DFT path, which the reference never meets at these k (not compared)
            if cv2_port.available() and params[0] ** 2 < orc.DFT_FILTER_ELEMS:
                assert np.array_equal(out, cv2_port.blur(img, params[0], 0)), ("oracle != cv2", key)
        elif op == "filter2d":
            kern = angle_kernel(*params)
            out = orc.apply_motion_blur(img, params[0], params[1], kernel=kern)
            if cv2_port.available():
                import cv2
                assert np.array_equal(out, cv2.filter2D(img, -1, kern)), ("oracle != cv2", key)
        else:
            raise ValueError(op)
        _want[key] = out
    return _want[key]


_golden_angles = None


def angle_kernel(k, angle):
    """The rotated k x k kernels recorded from the reference (tests/golden/golden_angles.npz)."""
    global _golden_angles
    if _golden_angles is None:
        _golden_angles = np.load(os.path.join(ROOT, "tests", "golden", "golden_angles.npz"))
    return _golden_angles[f"kernel_{k}_{angle}"]


# ------------------------------------------------------------------ LowRes: families and the selection model
# hand-classified shapes at factor 0.5 (the classes of the table in the module docstring); test_lowres_single_list
# checks each on a dense layout
FAMILY = {
    (32, 64): "P", (32, 40): "P", (32, 36): "P", (100, 248): "P", (2, 4): "P", (4, 8): "P",
    (33, 64): "H", (33, 40): "H", (33, 36): "H", (99, 248): "H",
    (2001, 16): "F", (2001, 8): "F", (2001, 12): "F", (2001, 248): "F",
    (2001, 5): "G", (65, 7): "I+", (65, 487): "I+", (66, 7): "I-", (66, 487): "I-",
    (2, 2): "R", (128, 130): "R", (3, 4): "R",
    (33, 4099): "GEN", (1, 3): "GEN",
}
STAGED = {"P": "lowres_x2p_kernel", "H": "lowres_x2h_kernel", "F": "lowres_x2f_kernel"}
FIXED = {"G": "lowres_x2g_kernel", "I+": "lowres_x2i_kernel<true>", "I-": "lowres_x2i_kernel<false>",
         "GEN": "lowres_kernel"}
UNITS = (16, 8, 4)


def lowres_list(fam, w, so, sp, do, dp):
    """The tile list of one image: a FIXED family, 'R' (X2_REST), 'W8' / 'W4', or (staged family, copy-unit class)."""
    if fam in FIXED or fam == "R":
        return fam
    if (sp | so) & 3:
        return "R"
    if (dp | do) & 3:
        return "W8" if ((sp | so) & 7) == 0 and w % 8 == 0 else "W4"
    a = sp | dp | so | do
    return (fam, 0 if w % 16 == 0 and a % 16 == 0 else (1 if w % 8 == 0 and a % 8 == 0 else 2))


def expected_lowres(b: Batch, factor=0.5, family=FAMILY):
    """(Counter of the kernels one LowRes call of batch b launches, whether the strip kernel replaced the band lists).
    b needs shapes, so / sp / do / dp and src / dst with data_ptr(); `family` classifies every shape."""
    if factor != 0.5:
        return collections.Counter({"lowres_kernel": 1}), False
    lists = {lowres_list(family[(h, w)], w, so, sp, do, dp)
             for (h, w), so, sp, do, dp in zip(b.shapes, b.so, b.sp, b.do, b.dp)}
    sbase, dbase = b.src.data_ptr(), b.dst.data_ptr()
    staged = [l for l in lists if isinstance(l, tuple)]
    banded = staged or "W8" in lists or "W4" in lists
    bands = banded and sbase % 4 == 0 and (not staged or dbase % 4 == 0)
    out = collections.Counter(FIXED[l] for l in lists if l in FIXED)
    if bands:
        base = sbase | dbase
        base_unit = 0 if base % 16 == 0 else (1 if base % 8 == 0 else 2)
        for fam, cls in staged:
            out[f"{STAGED[fam]}<{UNITS[max(cls, base_unit)]}>"] += 1
        if "W8" in lists:
            out["lowres_x2w_kernel<true>" if sbase % 8 == 0 else "lowres_x2w_kernel<false>"] += 1
        if "W4" in lists:
            out["lowres_x2w_kernel<false>"] += 1
        if "R" in lists:
            out[X2] += 1
    elif banded or "R" in lists:
        out[X2] += 1
    return out, banded and not bands


def run_lowres(torch, shapes, lay, factor=0.5):
    b = Batch(torch, shapes, lay, 3)
    got = launched(lambda: b.plan.lowres(b.src, b.dst, factor, opcodes=b.opcodes))
    want, strip = expected_lowres(b, factor)
    assert got == want, (shapes, lay, dict(got), dict(want))
    if not strip:
        assert sum(got.values()) == b.plan.launches(3), (sum(got.values()), b.plan.launches(3))
    else:
        assert sum(got.values()) < b.plan.launches(3)
    b.check([reference("lowres", h, w, factor) if op == 3 else None for (h, w), op in zip(shapes, b.ops)])
    return got


# every family and list of the table in one plan (the 2001-row shapes narrow)
MIXED = [(32, 64), (32, 40), (32, 36), (100, 248), (33, 64), (33, 40), (33, 36), (99, 248), (2001, 16), (2001, 8),
         (2001, 12), (2001, 5), (65, 7), (66, 7), (65, 487), (2, 2), (128, 130), (3, 4), (33, 4099), (1, 3), (2, 4)]
# ... and with every fourth destination row one byte longer: the X2W lists join in
MIXED_W = Layout(dpad=[0, 0, 0, 1])
PITCH_SHAPES = [(32, 64), (100, 248), (33, 64), (2001, 16), (2001, 8), (65, 7), (128, 130), (1, 3), (4, 8)]
PADS = (0, 1, 4, 8, 16)
LEADS = (0, 1, 2, 4, 8)


def lowres_cases():
    """(id, shapes, layout, factor) of the LowRes matrix."""
    cases = [(f"dense-{h}x{w}", [(h, w)], Layout(), 0.5) for h, w in FAMILY]
    for h, w in [(32, 64), (32, 36), (33, 64), (2001, 16), (2001, 12), (100, 248)]:
        cases.append((f"dpitch+1-{h}x{w}", [(h, w)], Layout(dpad=1), 0.5))     # X2W: odd destination pitch
        cases.append((f"doff+2-{h}x{w}", [(h, w)], Layout(dphase=2), 0.5))     # X2W: destination offset 2 mod 4
    for f in (0.3, 0.75, 1.0 / 3):
        cases.append((f"factor{f:.3f}", [(64, 64), (33, 47), (2, 3)], Layout(mask=True), f))
    for sl in LEADS:
        for dl in LEADS:
            cases.append((f"lead{sl}-{dl}", MIXED, Layout(slead=sl, dlead=dl, dpad=MIXED_W.dpad, mask=(sl == dl)), 0.5))
    for i, sp in enumerate(PADS):
        for j, dp in enumerate(PADS):
            lay = Layout(spad=sp, dpad=dp, sphase=[(4 * k + sp) % 16 for k in range(4)],
                         dphase=[(8 * k + 3 * dp) % 16 for k in range(3)], mask=(i + j) % 4 == 0)
            cases.append((f"pitch{sp}-{dp}", PITCH_SHAPES, lay, 0.5))
    return cases


LOWRES_CASES = lowres_cases()


@gpu
@pytest.mark.parametrize("case", LOWRES_CASES, ids=[c[0] for c in LOWRES_CASES])
def test_lowres_layouts(torch_, case):
    _, shapes, lay, factor = case
    run_lowres(torch_, shapes, lay, factor)


@gpu
def test_lowres_examples(torch_):
    """The base-pointer substitutions spelled out: a class-16 X2P list with a source base at +8 runs the 8-byte kernel;
    a source base at +1 runs the strip kernel for every exact-2x image, the odd-width kernels still run; a
    destination base at +2 with packed lists present takes the strip kernel too, and so does the identity factor's
    copy."""
    got = run_lowres(torch_, [(32, 64)], Layout(slead=8))
    assert got == {"lowres_x2p_kernel<8>": 1}
    got = run_lowres(torch_, MIXED, Layout(slead=1, dpad=MIXED_W.dpad))
    assert got == {X2: 1, "lowres_x2g_kernel": 1, "lowres_x2i_kernel<true>": 1, "lowres_x2i_kernel<false>": 1,
                   "lowres_kernel": 1}
    got = run_lowres(torch_, [(32, 64), (32, 36)], Layout(dlead=2))
    assert got == {X2: 1}
    got = run_lowres(torch_, [(32, 64)], Layout(dpad=1, slead=4))
    assert got == {"lowres_x2w_kernel<false>": 1}
    b = Batch(torch_, [(32, 64), (7, 5)], Layout(slead=1, dlead=3), 3)
    assert launched(lambda: b.plan.lowres(b.src, b.dst, 1.0)) == {COPY: 1}
    b.check([b.imgs[0], b.imgs[1]])


@gpu
def test_lowres_many_lists_on_a_side_stream(torch_):
    """One call over every list forks onto the plan's two streams and joins back into the caller's: the output read
    on the caller's (non-default) stream, with no synchronisation in between, is complete."""
    b = Batch(torch_, MIXED, MIXED_W, 3)
    s = torch_.cuda.Stream()
    host = {}

    def call():
        s.wait_stream(torch_.cuda.current_stream())
        with torch_.cuda.stream(s):
            b.plan.lowres(b.src, b.dst, 0.5)
            host["out"] = b.dbuf.cpu().numpy()

    got = launched(call)
    assert got == expected_lowres(b)[0] and sum(got.values()) == b.plan.launches(3) >= 10
    b.check([reference("lowres", h, w, 0.5) for h, w in MIXED], host=host["out"])


# ------------------------------------------------------------------ blur, filter2d, noise
OP_SHAPES = [(5, 3), (9, 13), (3, 1), (7, 2), (1, 16), (17, 100), (40, 129), (6, 6)]
OP_LAYOUTS = [
    Layout(),
    Layout(spad=1, sphase=[0, 5, 11]),
    Layout(spad=4, dpad=8, slead=4, dphase=[8, 0]),
    Layout(spad=16, dpad=1, dlead=1, mask=True),
    Layout(spad=8, dpad=16, slead=8, dlead=2, sphase=[3, 7], dphase=[9, 1]),
    Layout(dpad=4, slead=1, sphase=[2, 6], mask=True),
    Layout(spad=1, dpad=1, slead=5, dlead=5, sphase=[1, 2, 3], dphase=[1, 2, 3]),   # equal 16-byte phases
]


def blur_cases():
    return [(k, lay) for k in (9, 3, 5, 31, 1) for lay in OP_LAYOUTS]


def filter2d_cases():
    return [((k, a), lay) for k, a in ((9, 45), (11, 100), (3, 45), (5, 60), (7, 33)) for lay in OP_LAYOUTS[:5]]


def run_blur(torch, k, lay):
    b = Batch(torch, OP_SHAPES, lay, 2)
    got = launched(lambda: b.plan.blur(b.src, b.dst, k=k, opcodes=b.opcodes))
    assert got == {COPY if k == 1 else ("blur_rows_kernel<9>" if k == 9 else "blur_rows_kernel<0>"): 1}, dict(got)
    b.check([reference("blur", h, w, k) if op == 2 else None for (h, w), op in zip(OP_SHAPES, b.ops)])
    return got


def run_filter2d(torch, ka, lay):
    k, angle = ka
    b = Batch(torch, OP_SHAPES, lay, 2)
    b.plan.set_blur_kernel(angle_kernel(k, angle))
    got = launched(lambda: b.plan.blur(b.src, b.dst, k=k, opcodes=b.opcodes))
    assert got == {"filter2d_kernel": 1}, dict(got)
    b.check([reference("filter2d", h, w, k, angle) if op == 2 else None for (h, w), op in zip(OP_SHAPES, b.ops)])
    return got


BLUR_CASES = blur_cases()
F2D_CASES = filter2d_cases()


@gpu
@pytest.mark.parametrize("case", BLUR_CASES, ids=[f"k{k}-{lay}" for k, lay in BLUR_CASES])
def test_blur_layouts(torch_, case):
    run_blur(torch_, *case)


@gpu
@pytest.mark.parametrize("case", F2D_CASES, ids=[f"k{k}a{a}-{lay}" for (k, a), lay in F2D_CASES])
def test_filter2d_layouts(torch_, case):
    run_filter2d(torch_, *case)


NOISE_GENERATORS = {"table": (0, "noise_table_kernel<1, 1024, 2, 10>", "noise_table_kernel<3, 1024, 2, 10>"),
                    "table7": (2, "noise_table_kernel<1, 1024, 2, 7>", "noise_table_kernel<3, 1024, 2, 7>"),
                    "boxmuller": (1, "noise_kernel<1>", "noise_kernel<3>")}
SEED, FIRST, OFFSET, SIGMA = 0x5EED0123456789AB, 11, 5, 15.0


def philox_want(gen, i, img):
    return orc.philox_noise_field(img.size, SIGMA, SEED, FIRST + i, OFFSET,
                                  generator={"table": "auto", "table7": "table7", "boxmuller": "boxmuller"}[gen])


def run_philox(torch, gen, lay):
    b = Batch(torch, OP_SHAPES, lay, 1)
    b.plan.set_gaussian_generator(NOISE_GENERATORS[gen][0])
    got = launched(lambda: b.plan.noise(b.src, b.dst, None, SIGMA, SEED, FIRST, OFFSET, opcodes=b.opcodes))
    assert got == {NOISE_GENERATORS[gen][1]: 1}, dict(got)
    want = [orc.add_philox_noise(img, philox_want(gen, i, img)) if op == 1 else None
            for i, (img, op) in enumerate(zip(b.imgs, b.ops))]

    def close(i, got_i, want_i):   # Box-Muller: float32 kernel vs float64 restatement, a byte may move by one
        d = np.abs(got_i.astype(int) - want_i)
        assert d.max() <= 1 and (d != 0).sum() <= 1 + 1e-3 * d.size, (i, int((d != 0).sum()))

    b.check(want, compare=close if gen == "boxmuller" else None)
    return got


def run_compat(torch, lay, field_lead):
    """Compat noise from a device field (one float32 per element, images back to back in plan order) that starts
    `field_lead` floats into its buffer."""
    b = Batch(torch, OP_SHAPES, lay, 1)
    fields = [np.random.default_rng(900 + i).normal(0, SIGMA, img.shape).astype(np.float32)
              for i, img in enumerate(b.imgs)]
    fbuf = torch.from_numpy(np.concatenate([np.zeros(field_lead, np.float32)] + [f.reshape(-1) for f in fields])).cuda()
    got = launched(lambda: b.plan.noise(b.src, b.dst, fbuf[field_lead:], SIGMA, opcodes=b.opcodes))
    assert got == {"noise_kernel<0>": 1}, dict(got)
    b.check([orc.add_noise_field(img, f) if op == 1 else None for img, f, op in zip(b.imgs, fields, b.ops)])
    return got


def run_field(torch, gen, field_lead):
    """noise_field into a float32 buffer at a lead of `field_lead` floats; the floats around it keep a sentinel."""
    from robust_object_detection_b200.batch import CorruptionPlan
    lay = OP_LAYOUTS[field_lead % len(OP_LAYOUTS)]
    so, sp, _ = lay.offsets(OP_SHAPES, lay.spad, lay.sphase)
    do, dp, _ = lay.offsets(OP_SHAPES, lay.dpad, lay.dphase)
    plan = CorruptionPlan(OP_SHAPES, so, do, sp, dp)
    plan.set_gaussian_generator(NOISE_GENERATORS[gen][0])
    n = plan.payload_bytes
    fbuf = torch.full((field_lead + n + 16,), -1234.5, dtype=torch.float32, device="cuda")
    got = launched(lambda: plan.noise_field(fbuf[field_lead:], SIGMA, SEED, FIRST, OFFSET))
    assert got == {NOISE_GENERATORS[gen][2]: 1}, dict(got)
    host = fbuf.cpu().numpy()
    assert (host[:field_lead] == -1234.5).all() and (host[field_lead + n:] == -1234.5).all()
    e = field_lead
    for i, (h, w) in enumerate(OP_SHAPES):
        want = philox_want(gen, i, image_of(h, w))
        f = host[e:e + want.size].astype(np.float64)
        if gen == "boxmuller":
            assert np.abs(f - want).max() < 2e-3, (gen, i)
        else:
            assert np.array_equal(f, want), (gen, i)
        e += want.size
    return got


NOISE_CASES = ([("philox", g, lay) for g in NOISE_GENERATORS for lay in OP_LAYOUTS]
               + [("compat", lay, j % 2) for j, lay in enumerate(OP_LAYOUTS)]
               + [("field", g, lead) for g in NOISE_GENERATORS for lead in (0, 1, 3)])


def run_noise(torch, case):
    kind, a, b = case
    return {"philox": run_philox, "compat": run_compat, "field": run_field}[kind](torch, a, b)


@gpu
@pytest.mark.parametrize("case", NOISE_CASES, ids=[f"{k}-{a}-{b}" for k, a, b in NOISE_CASES])
def test_noise_layouts(torch_, case):
    run_noise(torch_, case)


# ------------------------------------------------------------------ corrupt(): every op in one call
CORRUPT_SHAPES = [(32, 64), (33, 40), (65, 7), (2001, 8), (128, 130), (1, 3), (32, 36), (66, 7), (3, 4), (2, 2),
                  (99, 248), (2001, 5)]
CORRUPT_CASES = [(Layout(), False), (Layout(spad=4, dpad=1, dlead=1, sphase=[4, 0, 12]), True),
                 (Layout(spad=16, dpad=8, slead=8, dlead=4), False)]


def run_corrupt(torch, lay, compat):
    """corrupt() with op-codes 0..3: op-code 0 images are copied by noise_kernel<2>, the others get their op."""
    b = Batch(torch, CORRUPT_SHAPES, lay, 0)
    ops = [i % 4 for i in range(len(CORRUPT_SHAPES))]
    b.ops = ops
    b.opcodes = torch.tensor(ops, dtype=torch.uint8, device="cuda")
    fields = [np.random.default_rng(700 + i).normal(0, SIGMA, img.shape).astype(np.float32) for i, img in enumerate(b.imgs)]
    field = torch.from_numpy(np.concatenate([f.reshape(-1) for f in fields])).cuda() if compat else None
    b.plan.set_gaussian_generator(0)
    got = launched(lambda: b.plan.corrupt(b.src, b.dst, b.opcodes, noise=field, sigma=SIGMA, k=9, factor=0.5,
                                          seed=SEED, first_image_index=FIRST, offset=OFFSET))
    want_k = expected_lowres(b)[0] + collections.Counter(
        {COPY: 1, "blur_rows_kernel<9>": 1, ("noise_kernel<0>" if compat else "noise_table_kernel<1, 1024, 2, 10>"): 1})
    assert got == want_k, (dict(got), dict(want_k))
    want = []
    for i, ((h, w), img, op) in enumerate(zip(CORRUPT_SHAPES, b.imgs, ops)):
        if op == 0:
            want.append(img)
        elif op == 1:
            want.append(orc.add_noise_field(img, fields[i]) if compat else orc.add_philox_noise(img, philox_want("table", i, img)))
        elif op == 2:
            want.append(reference("blur", h, w, 9))
        else:
            want.append(reference("lowres", h, w, 0.5))
    b.check(want)
    return got


@gpu
@pytest.mark.parametrize("case", CORRUPT_CASES, ids=[f"{lay}-{'compat' if c else 'philox'}" for lay, c in CORRUPT_CASES])
def test_corrupt_layouts(torch_, case):
    run_corrupt(torch_, *case)


# ------------------------------------------------------------------ coverage
@gpu
def test_every_kernel_is_reached(torch_):
    """Runs the whole matrix (independent of test order and -k) and asserts that the kernels it reaches are exactly
    KERNELS; prints the number of cases that reached each."""
    reached = collections.Counter()

    def add(got):
        reached.update(set(got))

    for _, shapes, lay, factor in LOWRES_CASES:
        add(run_lowres(torch_, shapes, lay, factor))
    for k, lay in BLUR_CASES:
        add(run_blur(torch_, k, lay))
    for ka, lay in F2D_CASES:
        add(run_filter2d(torch_, ka, lay))
    for case in NOISE_CASES:
        add(run_noise(torch_, case))
    for lay, compat in CORRUPT_CASES:
        add(run_corrupt(torch_, lay, compat))
    print("\ncases per kernel:")
    for name in ALL_KERNELS:
        print(f"  {reached[name]:5d}  {name}")
    assert sorted(reached) == ALL_KERNELS, sorted(set(reached) ^ set(ALL_KERNELS))


@pytest.fixture(scope="module")
def torch_():
    import torch
    assert torch.cuda.is_available()
    return torch
