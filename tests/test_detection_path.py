"""The Faster R-CNN loader path (train_frcnn_augmented.py:61-67): RandomCorruption(0.5) + ToImage + ToDtype(float32,
scale=True) per item, against rod_corrupt_chw_f32 / training.DetectionCorruptionBatcher / torch.ops.rod.corrupt_chw.

CPU tests pin what the device path relies on (torchvision's arithmetic, PIL vs OpenCV decoding, the RNG order, the output
layout); GPU tests compare tensors exactly."""
import io
import os
import random

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "robust-object-detection_b200", "librod_b200.so")

cv2 = pytest.importorskip("cv2")
torch = pytest.importorskip("torch")
tv2 = pytest.importorskip("torchvision.transforms.v2")
from PIL import Image, ImageFile  # noqa: E402

from oracle import cv2_port  # noqa: E402

# frames of the reference-pipeline test: the VisDrone-like sizes of the issue plus widths 1..9 (all four W % 4)
SHAPES = [(765, 1360), (1050, 1400), (1078, 1916), (1079, 1917), (765, 1361)] + [(5 + 3 * w, w) for w in range(1, 10)]


@pytest.fixture(scope="module")
def built():
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    return LIB


def _frame(seed, h, w):
    """Smooth RGB content with noise on top (JPEG-friendly, not constant)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // max(w - 1, 1)), (yy * 255 // max(h - 1, 1)), ((xx + yy) * 7) % 256], -1)
    return np.clip(base + rng.integers(-20, 21, (h, w, 3)), 0, 255).astype(np.uint8)


class RefRandomCorruption:
    """augmentations.py:60-74 over the live OpenCV / NumPy calls (oracle/cv2_port.py)."""

    def __init__(self, p=0.5):
        self.p = p

    def __call__(self, img):
        if random.random() > self.p:
            return img
        img_bgr = cv2.cvtColor(np.array(img), cv2.COLOR_RGB2BGR)
        out = cv2_port.OPS[random.choice(["noise", "blur", "lowres"])](img_bgr)
        return Image.fromarray(cv2.cvtColor(out, cv2.COLOR_BGR2RGB))


def _reference_transform():
    return tv2.Compose([RefRandomCorruption(0.5), tv2.ToImage(), tv2.ToDtype(torch.float32, scale=True)])


def _reference(pils, seed):
    random.seed(seed)
    np.random.seed(seed)
    t = _reference_transform()
    return [t(im).to("cuda") for im in pils]


def _seed_with_all_ops(n, p=0.5):
    from robust_object_detection_b200.batch import draw_decisions
    for s in range(1000):
        random.seed(s)
        if set(draw_decisions(n, gate="pil", p=p).tolist()) == {0, 1, 2, 3}:
            return s
    raise AssertionError("no seed draws all four op-codes")


def _write_files(d):
    """Writes the file mix of the from-files test into d; returns the paths."""
    files = []
    for i, (h, w) in enumerate([(120, 161), (97, 64), (33, 5), (64, 200)]):
        ok, buf = cv2.imencode(".jpg", _frame(10 + i, h, w)[:, :, ::-1], [cv2.IMWRITE_JPEG_QUALITY, 95])
        files.append((f"base{i}.jpg", buf.tobytes()))
    ok, buf = cv2.imencode(".jpg", cv2.cvtColor(_frame(20, 70, 90), cv2.COLOR_RGB2GRAY), [cv2.IMWRITE_JPEG_QUALITY, 95])
    files.append(("grey.jpg", buf.tobytes()))
    ok, buf = cv2.imencode(".jpg", _frame(21, 80, 110)[:, :, ::-1], [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    files.append(("progressive.jpg", buf.tobytes()))
    ok, buf = cv2.imencode(".png", _frame(22, 50, 77)[:, :, ::-1])
    files.append(("frame.png", buf.tobytes()))
    files.append(("exif6.jpg", _exif6_jpeg()))
    ok, buf = cv2.imencode(".jpg", _frame(23, 96, 128)[:, :, ::-1], [cv2.IMWRITE_JPEG_QUALITY, 95])
    files.append(("truncated.jpg", buf.tobytes()[: len(buf) * 3 // 5]))
    paths = []
    for name, data in files:
        p = os.path.join(d, name)
        with open(p, "wb") as f:
            f.write(data)
        paths.append(p)
    return paths


def _exif6_jpeg():
    """A 40x64 (h x w) JPEG with EXIF orientation 6, written by PIL."""
    exif = Image.Exif()
    exif[0x0112] = 6
    buf = io.BytesIO()
    Image.fromarray(_frame(30, 40, 64)).save(buf, format="JPEG", exif=exif, quality=90)
    return buf.getvalue()


def _chw_rule(shapes):
    """The documented layout of rod_corrupt_chw_f32's output (include/rod_b200.h): blocks of 3*H*W floats in plan order,
    each starting at a multiple of 64 floats; the last entry is the total."""
    offs = [0]
    for h, w in shapes:
        offs.append(offs[-1] + (3 * h * w + 63) // 64 * 64)
    return offs


# ------------------------------------------------------------------------------------------------------------ CPU tests
def test_to_dtype_is_the_float32_product():
    """ToDtype(float32, scale=True) = fl(float(v) * fl(1/255)) for all 256 values: what chw_f32_kernel computes."""
    v = torch.arange(256, dtype=torch.uint8).view(1, 1, 256)
    got = tv2.functional.to_dtype(v, torch.float32, scale=True).view(-1).numpy()
    want = np.arange(256, dtype=np.float32) * np.float32(1.0 / 255)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # ... which is not the correctly rounded quotient for every v (restoration.cu's table is not this one)
    assert not np.array_equal(got, np.arange(256, dtype=np.float32) / np.float32(255))


def test_pil_decode_equals_reversed_cv2_imdecode(tmp_path):
    """For every JPEG the device decoder is given in the GPU tests (baseline q95 and greyscale), PIL's RGB reading is
    OpenCV's BGR reading reversed, so the device decoder (cv2.imread's pixels) stands in for PIL's decode."""
    n = 0
    for p in _write_files(str(tmp_path)):
        name = os.path.basename(p)
        if not (name.startswith("base") or name == "grey.jpg"):
            continue
        data = open(p, "rb").read()
        pil = np.asarray(Image.open(p).convert("RGB"))
        cv = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(pil, cv[:, :, ::-1]), name
        n += 1
    assert n == 5


def test_exif_orientation_pil_keeps_cv2_rotates():
    """PIL does not apply EXIF orientation, cv2.imdecode does: files with one must be read with PIL on this path."""
    data = _exif6_jpeg()
    assert np.asarray(Image.open(io.BytesIO(data)).convert("RGB")).shape == (40, 64, 3)
    assert cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR).shape == (64, 40, 3)


def test_batched_draw_order_equals_per_item_loop():
    """Decisions of the whole batch first, then the noise fields in image order = the reference's per-item
    interleaving (`random` and `np.random` are independent streams)."""
    from robust_object_detection_b200.batch import draw_decisions
    shapes = [(3 + i % 4, 2 + i % 5) for i in range(40)]
    random.seed(5)
    np.random.seed(5)
    want_ops, want_fields = [], []
    for h, w in shapes:
        if random.random() > 0.5:
            want_ops.append(0)
            continue
        name = random.choice(["noise", "blur", "lowres"])
        want_ops.append(1 + ["noise", "blur", "lowres"].index(name))
        if name == "noise":
            want_fields.append(np.random.normal(0, 15, (h, w, 3)).astype(np.float32))
    random.seed(5)
    np.random.seed(5)
    ops = draw_decisions(len(shapes), gate="pil", p=0.5)
    fields = [np.random.normal(0, 15, shapes[i] + (3,)).astype(np.float32) for i in np.flatnonzero(ops == 1)]
    assert ops.tolist() == want_ops and {1, 2, 3} <= set(want_ops)
    assert len(fields) == len(want_fields) and all(np.array_equal(a, b) for a, b in zip(fields, want_fields))


def test_chw_offset_rule_aligned_and_disjoint(built):
    """Every image block starts 256-byte aligned, blocks do not overlap and hold 3*H*W floats; the strides of
    torch.ops.rod.corrupt_chw's fake implementation follow the same rule."""
    from torch._subclasses.fake_tensor import FakeTensorMode
    import robust_object_detection_b200.torch_ops  # noqa: F401
    rng = np.random.default_rng(0)
    shapes = [(int(h), int(w)) for h, w in rng.integers(1, 300, (200, 2))] + SHAPES
    offs = _chw_rule(shapes)
    for i, (h, w) in enumerate(shapes):
        assert (offs[i] * 4) % 256 == 0
        assert offs[i] + 3 * h * w <= offs[i + 1] < offs[i] + 3 * h * w + 64
    with FakeTensorMode():
        for h, w in [(765, 1360), (7, 3), (8, 8)]:
            x = torch.empty((3, h, w, 3), dtype=torch.uint8, device="cuda")
            y = torch.ops.rod.corrupt_chw(x, torch.empty(3, dtype=torch.uint8, device="cuda"), 15.0, 9, 0.5, 0, 0)
            assert y.shape == (3, 3, h, w) and y.dtype == torch.float32
            assert y.stride() == (_chw_rule([(h, w)])[1], h * w, w, 1)


# ------------------------------------------------------------------------------------------------------------ GPU tests
def _batcher(**kw):
    from robust_object_detection_b200.training import DetectionCorruptionBatcher
    return DetectionCorruptionBatcher(**kw)


def _torch_conversion(bgr_u8):
    """[H,W,3] BGR uint8 (CUDA) -> what ToImage + ToDtype(float32, scale=True) make of its RGB version."""
    return bgr_u8.permute(2, 0, 1).flip(0).float().mul_(1 / 255)


@pytest.mark.gpu
def test_reference_pipeline_equality_compat(built):
    pils = [Image.fromarray(_frame(i, h, w)) for i, (h, w) in enumerate(SHAPES)]
    seed = _seed_with_all_ops(len(pils))
    want = _reference(pils, seed)
    random.seed(seed)
    np.random.seed(seed)
    b = _batcher(p=0.5, noise="compat")
    got = b(pils)
    assert set(b.last_ops.tolist()) == {0, 1, 2, 3}
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.is_cuda and g.dtype == torch.float32 and g.shape == w.shape, i
        assert torch.equal(g, w), (i, SHAPES[i], int(b.last_ops[i]))
    # both global streams advanced exactly as the reference's did
    after = (random.random(), np.random.random())
    _reference(pils, seed)
    assert (random.random(), np.random.random()) == after


@pytest.mark.gpu
def test_philox_mode_equals_corrupt_then_conversion_and_ignores_grouping(built):
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = SHAPES[4:] + [(300, 401), (64, 64)]
    rgb = [_frame(40 + i, h, w) for i, (h, w) in enumerate(shapes)]
    seed = _seed_with_all_ops(len(rgb))
    random.seed(seed)
    b = _batcher(p=0.5, noise="philox", seed=11)
    got = b(rgb)
    ops = b.last_ops
    assert set(ops.tolist()) == {0, 1, 2, 3}
    plan = CorruptionPlan.ragged(shapes)
    src = torch.from_numpy(plan.pack([np.ascontiguousarray(a[:, :, ::-1]) for a in rgb])).cuda()
    dst = torch.empty_like(src)
    plan.corrupt(src, dst, torch.from_numpy(ops).cuda(), seed=11)
    for i, ((h, w), off) in enumerate(zip(shapes, plan.dst_offsets)):
        assert torch.equal(got[i], _torch_conversion(dst[off:off + 3 * h * w].view(h, w, 3))), i
    # split into batches of 3, 1 and the rest: same tensors (Philox keyed by the running image index)
    random.seed(seed)
    b2 = _batcher(p=0.5, noise="philox", seed=11)
    parts = [rgb[:3], rgb[3:4], rgb[4:]]
    split = [t for out in b2.run(parts) for t in out]
    assert all(torch.equal(a, c) for a, c in zip(got, split)) and len(split) == len(got)


@pytest.mark.gpu
def test_from_files_equals_reference_pipeline(built, tmp_path, monkeypatch):
    from robust_object_detection_b200.jpeg import probe
    monkeypatch.setattr(ImageFile, "LOAD_TRUNCATED_IMAGES", True)
    paths = _write_files(str(tmp_path))
    by_name = {os.path.basename(p): p for p in paths}
    assert probe(open(by_name["base0.jpg"], "rb").read()) is not None  # the device decoder is exercised
    pils = [Image.open(p).convert("RGB") for p in paths]
    assert pils[paths.index(by_name["exif6.jpg"])].size == (64, 40)
    for seed in range(3):  # a few draws so that the fallback files meet several op-codes
        want = _reference(pils, seed)
        random.seed(seed)
        np.random.seed(seed)
        b = _batcher(p=0.5, noise="compat", io_threads=4)
        got = b(paths)
        for i, (g, w) in enumerate(zip(got, want)):
            assert torch.equal(g, w), (seed, os.path.basename(paths[i]), int(b.last_ops[i]))
        random.seed(seed)
        np.random.seed(seed)
        got_bytes = _batcher(p=0.5, noise="compat")([open(p, "rb").read() for p in paths])
        assert all(torch.equal(g, w) for g, w in zip(got_bytes, want))


@pytest.mark.gpu
def test_guard_values_and_pitched_sources(built):
    from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
    big_h, big_w = 90, 203
    frame = torch.from_numpy(_frame(50, big_h, big_w)).cuda()
    crops = [(0, 0, 90, 203), (1, 1, 40, 61), (3, 2, 17, 7), (5, 5, 30, 1), (2, 7, 25, 130), (0, 3, 11, 9), (7, 11, 33, 5),
             (4, 13, 20, 64)]
    shapes = [(h, w) for _, _, h, w in crops]
    n = len(crops)
    seed = _seed_with_all_ops(n)
    random.seed(seed)
    ops = torch.from_numpy(draw_decisions(n, gate="pil", p=0.5)).cuda()
    pitched = CorruptionPlan(shapes, [3 * (y * big_w + x) for y, x, _, _ in crops], CorruptionPlan.ragged(shapes).dst_offsets,
                             src_pitches=[3 * big_w] * n)
    dense = CorruptionPlan.ragged(shapes)
    src_dense = torch.zeros(dense.src_bytes, dtype=torch.uint8, device="cuda")
    for (y, x, h, w), off in zip(crops, dense.src_offsets):
        src_dense[off:off + 3 * h * w] = frame[y:y + h, x:x + w].reshape(-1)
    assert pitched.chw_offsets() == dense.chw_offsets() == _chw_rule(shapes)
    total = dense.chw_offsets()[-1]
    outs = []
    for plan, s in ((pitched, frame.reshape(-1)), (dense, src_dense)):
        out = torch.empty(total + 64, dtype=torch.float32, device="cuda")
        out.view(torch.int32).fill_(0x7FC0DEAD)
        plan.corrupt_chw_f32(s, ops, out, seed=3)
        outs.append(out)
    offs = dense.chw_offsets()
    for out in outs:
        bits = out.view(torch.int32)
        for i, (h, w) in enumerate(shapes):
            assert (bits[offs[i] + 3 * h * w:offs[i + 1]] == 0x7FC0DEAD).all(), i
        assert (bits[total:] == 0x7FC0DEAD).all()
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    # and the images are the conversion of corrupt()
    dst = torch.empty_like(src_dense)
    dense.corrupt(src_dense, dst, ops, seed=3)
    for (h, w), o, d in zip(shapes, offs, dense.dst_offsets):
        assert torch.equal(outs[1][o:o + 3 * h * w].view(3, h, w), _torch_conversion(dst[d:d + 3 * h * w].view(h, w, 3)))


@pytest.mark.gpu
def test_full_size_batch(built):
    from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
    n, h, w = 256, 765, 1360
    base = torch.from_numpy(np.stack([_frame(60 + i, h, w)[:, :, ::-1] for i in range(4)])).cuda()
    src = base.repeat(n // 4, 1, 1, 1).contiguous()
    random.seed(7)
    ops = draw_decisions(n, gate="pil", p=0.5)
    assert set(ops.tolist()) == {0, 1, 2, 3}
    ops_d = torch.from_numpy(ops).cuda()
    plan = CorruptionPlan.uniform(n, h, w)
    out = torch.empty(plan.chw_offsets()[-1], dtype=torch.float32, device="cuda")
    plan.corrupt_chw_f32(src, ops_d, out, seed=9)
    dst = torch.empty_like(src)
    plan.corrupt(src, dst, ops_d, seed=9)
    stride = plan.chw_offsets()[1]
    got = torch.as_strided(out, (n, 3, h, w), (stride, h * w, w, 1))
    for lo in range(0, n, 32):
        want = dst[lo:lo + 32].permute(0, 3, 1, 2).flip(1).float().mul_(1 / 255)
        assert torch.equal(got[lo:lo + 32], want), lo


@pytest.mark.gpu
def test_dataloader_collate_and_torch_op(built):
    from torch.utils.data import DataLoader
    import robust_object_detection_b200.torch_ops  # noqa: F401
    from robust_object_detection_b200.batch import CorruptionPlan

    class Dataset:  # COCODetectionDataset's shape: (PIL image, target), transforms optional
        def __init__(self, transforms=None):
            self.transforms = transforms
            self.shapes = [(48, 64), (31, 45), (60, 17), (48, 64), (9, 7), (33, 50), (20, 20)]

        def __len__(self):
            return len(self.shapes)

        def __getitem__(self, i):
            img = Image.fromarray(_frame(70 + i, *self.shapes[i]))
            target = {"boxes": torch.tensor([[0.0, 0.0, 4.0, 4.0]]), "image_id": i}
            return (self.transforms(img) if self.transforms else img), target

    seed = 3
    random.seed(seed)
    np.random.seed(seed)
    ref = DataLoader(Dataset(_reference_transform()), batch_size=2, shuffle=False, num_workers=0,
                     collate_fn=lambda b: tuple(zip(*b)))
    want = [([im.to("cuda") for im in images], targets) for images, targets in ref]
    random.seed(seed)
    np.random.seed(seed)
    b = _batcher(p=0.5)
    got = list(DataLoader(Dataset(), batch_size=2, shuffle=False, num_workers=0, collate_fn=b.collate))
    assert len(got) == len(want)
    for (gi, gt), (wi, wt) in zip(got, want):
        assert isinstance(gi, tuple) and isinstance(gt, tuple) and len(gi) == len(wi)
        assert [t["image_id"] for t in gt] == [t["image_id"] for t in wt]
        for a, c in zip(gi, wi):
            assert a.is_cuda and a.to("cuda") is a and torch.equal(a, c)
    # torch.ops.rod.corrupt_chw on a uniform batch
    n, h, w = 5, 37, 53
    x = torch.from_numpy(np.stack([_frame(80 + i, h, w) for i in range(n)])).cuda()
    ops = torch.tensor([0, 1, 2, 3, 1], dtype=torch.uint8, device="cuda")
    y = torch.ops.rod.corrupt_chw(x, ops, 15.0, 9, 0.5, 4, 2)
    dst = torch.empty_like(x)
    CorruptionPlan.uniform(n, h, w).corrupt(x, dst, ops, seed=4, first_image_index=2)
    assert y.shape == (n, 3, h, w) and torch.equal(y, dst.permute(0, 3, 1, 2).flip(1).float().mul_(1 / 255))
