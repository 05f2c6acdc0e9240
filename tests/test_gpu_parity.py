"""GPU parity tests: the sm_100a kernels, called through the C ABI (ctypes -> librod_b200.so),
against (a) golden vectors recorded from the unmodified reference and (b) the numpy oracle on
the same seeded inputs.  Bit-exact for blur, lowres, compat noise and the letterbox output;
Philox noise is checked against its restated stream (float tolerance 2e-3 on the field) and
statistically (SURVEY 8d config 1b)."""
import random
import sys
import types

import os

import numpy as np
import pytest

from oracle import corruption_oracle as orc
from tests.helpers import SMALL_SHAPES, sha, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def aug():
    import torch
    assert torch.cuda.is_available()
    from robust_object_detection_b200 import augmentations
    augmentations.set_noise_mode("compat")
    return augmentations


@pytest.fixture(scope="module")
def torch_():
    import torch
    return torch


# ------------------------------------------------------------------ per-image drop-in functions
@pytest.mark.parametrize("kind", ["uniform", "binary"])
def test_small_shapes_vs_golden(aug, golden_small, kind):
    for i, (h, w) in enumerate(SMALL_SHAPES):
        tag = f"{kind}_{h}x{w}"
        img = golden_small[f"in_{tag}"]
        assert np.array_equal(aug.apply_motion_blur(img, 9, 0), golden_small[f"blur9_{tag}"]), tag
        assert np.array_equal(aug.apply_motion_blur(img, 5, 0), golden_small[f"blur5_{tag}"]), tag
        assert np.array_equal(aug.apply_lowres(img, 0.5), golden_small[f"lowres_{tag}"]), tag
        np.random.seed(7 + i)
        assert np.array_equal(aug.apply_noise(img, 15), golden_small[f"noise_{tag}"]), tag


def test_strided_crop_factors_rails(aug, golden_small):
    crop = golden_small["in_crop_base"][5:53, 7:91]
    assert not crop.flags["C_CONTIGUOUS"]
    out = aug.apply_motion_blur(crop, 9, 0)
    assert out.flags["C_CONTIGUOUS"] and np.array_equal(out, golden_small["blur9_crop"])
    assert np.array_equal(aug.apply_lowres(crop, 0.5), golden_small["lowres_crop"])
    img = golden_small["in_factor"]
    for f in (0.25, 0.3, 0.75):
        assert np.array_equal(aug.apply_lowres(img, f), golden_small[f"lowres_f{f}"]), f
    np.random.seed(11)
    assert np.array_equal(aug.apply_noise(np.full((32, 40, 3), 128, np.uint8), 15), golden_small["noise_const128"])
    np.random.seed(12)
    assert np.array_equal(aug.apply_noise(golden_small["in_rails"], 15), golden_small["noise_rails"])
    # inputs are never mutated; flipped views are accepted
    before = crop.copy()
    aug.apply_lowres(crop[:, ::-1], 0.5)
    assert np.array_equal(crop, before)


def test_big_cases_sha(aug, golden_hashes):
    for name, g in golden_hashes["big"].items():
        img = synth(g["seed"], g["h"], g["w"])
        assert sha(aug.apply_motion_blur(img, 9, 0)) == g["blur9"], name
        assert sha(aug.apply_lowres(img, 0.5)) == g["lowres"], name
        np.random.seed(42)
        assert sha(aug.apply_noise(img, 15)) == g["noise_seed42"], name


def test_noise_sequence_config1(aug, golden_hashes):
    """BASELINE.json configs[0] at full size: all 64 sequential apply_noise calls after one np.random.seed(42), against the
    sha256 of the unmodified reference's 64 outputs."""
    g = golden_hashes["noise_sequence"]
    assert len(g["sha"]) == 64
    np.random.seed(g["seed"])
    for i, want in enumerate(g["sha"]):
        assert sha(aug.apply_noise(synth(g["first_image_seed"] + i, 765, 1360), 15)) == want, i


@pytest.mark.parametrize("k", [1, 3, 7, 9, 13, 21, 31])
def test_blur_kernel_sizes_vs_oracle(aug, k):
    for n, (h, w) in enumerate([(5, 3), (9, 13), (40, 129), (31, 1361), (64, 700)]):
        img = synth(800 + n, h, w)
        assert np.array_equal(aug.apply_motion_blur(img, k, 0), orc.apply_motion_blur(img, k, 0)), (k, h, w)


def test_lowres_shapes_and_factors_vs_oracle(aug):
    shapes = [(1, 1), (2, 2), (3, 7), (65, 255), (70, 257), (128, 130), (360, 480), (361, 481), (100, 2000), (33, 4099)]
    for n, (h, w) in enumerate(shapes):
        img = synth(900 + n, h, w)
        for f in (0.5, 0.25, 1 / 3, 0.6, 0.9, 1.0):
            assert np.array_equal(aug.apply_lowres(img, f), orc.apply_lowres(img, f)), (h, w, f)


def test_motion_blur_general_angles(aug, torch_):
    """SURVEY 8f rank 3: apply_motion_blur at angles != 0 (2-D float kernel, cv2.filter2D semantics incl. the
    non-FMA scalar tail of each row) against outputs recorded from the unmodified reference."""
    import json
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    g = np.load(os.path.join(here, "golden_angles.npz"))
    meta = json.load(open(os.path.join(here, "golden_angles.json")))
    for k, ang in meta["cases"]:
        assert np.array_equal(aug._motion_blur_kernel(k, ang), g[f"kernel_{k}_{ang}"]), (k, ang)
        for i, (h, w) in enumerate(meta["shapes"]):
            for kind in ("uniform", "binary"):
                got = aug.apply_motion_blur(synth(300 + i, h, w, kind), k, ang)
                assert np.array_equal(got, g[f"out_{k}_{ang}_{kind}_{h}x{w}"]), (k, ang, h, w, kind)
        for name, seed, h, w in meta["big"]:
            assert sha(aug.apply_motion_blur(synth(seed, h, w), k, ang)) == meta["sha"][f"{k}_{ang}_{name}"], (k, ang, name)
    # the angle-0 box is back after a general kernel was used on the same cached plan
    img = synth(300, 33, 47)
    aug.apply_motion_blur(img, 9, 45)
    assert np.array_equal(aug.apply_motion_blur(img, 9, 0), orc.apply_motion_blur(img, 9, 0))
    # device-resident ragged batch with op-code masking
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(48, 129), (31, 100), (33, 47)]
    imgs = [synth(300 + i, h, w) for i, (h, w) in zip((6, 5, 4), shapes)]
    plan = CorruptionPlan.ragged(shapes)
    plan.set_blur_kernel(g["kernel_9_45"])
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    dst = torch_.full_like(src, 5)
    plan.blur(src, dst, k=9, opcodes=torch_.tensor([2, 0, 2], dtype=torch_.uint8, device="cuda"))
    outs = plan.unpack(dst.cpu().numpy())
    assert np.array_equal(outs[0], g["out_9_45_uniform_48x129"]) and np.array_equal(outs[2], g["out_9_45_uniform_33x47"])
    assert (outs[1] == 5).all()


def test_unsupported_parameters_raise(aug):
    img = synth(1, 16, 16)
    with pytest.raises(NotImplementedError):
        aug.apply_motion_blur(img, 13, 30)  # 169 kernel elements: OpenCV's DFT path, not reproducible bit-exactly
    with pytest.raises(NotImplementedError):
        aug.apply_motion_blur(img, 4, 0)
    with pytest.raises(NotImplementedError):
        aug.apply_lowres(img, 1.5)
    with pytest.raises(NotImplementedError):
        aug.apply_lowres(synth(2, 64, 64), 0.05)  # > 8 area taps: outside the exact-parity domain
    # C ABI argument checks of the newer entry points: status codes, never a crash
    from robust_object_detection_b200 import _native as N
    from robust_object_detection_b200.batch import CorruptionPlan
    plan = CorruptionPlan.uniform(1, 16, 16)
    assert N.lib().rod_plan_set_gaussian_generator(plan._h, 7) == N.ROD_ERR_INVALID_ARG
    assert N.lib().rod_plan_set_gaussian_generator(None, 0) == N.ROD_ERR_INVALID_ARG
    import ctypes
    pos, has, cached = ctypes.c_int32(700), ctypes.c_int32(0), ctypes.c_double(0.0)
    key = np.zeros(624, np.uint32)
    out = np.zeros(4, np.float32)
    assert N.lib().rod_numpy_legacy_normal_f32(key.ctypes.data, ctypes.byref(pos), ctypes.byref(has), ctypes.byref(cached),
                                               1.0, 4, out.ctypes.data, 1) == N.ROD_ERR_INVALID_ARG   # pos > 624
    with pytest.raises(NotImplementedError):
        import torch
        big = torch.zeros((1, 16, 16, 3), dtype=torch.uint8, device="cuda")
        plan.noise(big, big.clone(), None, 5000.0)   # Philox sigma beyond int16 offsets


# ------------------------------------------------------------------ random apply + adapters
def test_random_corruption_streams(aug, golden_hashes):
    g = golden_hashes["random_corruption"]
    random.seed(g["py_seed"])
    np.random.seed(g["np_seed"])
    img = synth(g["img_seed"], g["h"], g["w"])
    assert [sha(aug._apply_random_corruption(img)) for _ in g["sha"]] == g["sha"]


def test_pil_transform(aug, golden_hashes):
    from PIL import Image
    g = golden_hashes["pil_transform"]
    random.seed(g["py_seed"])
    np.random.seed(g["np_seed"])
    pil = Image.fromarray(synth(g["img_seed"], g["h"], g["w"]))
    t = aug.RandomCorruption(p=0.5)
    outs = [t(pil) for _ in g["sha"]]
    assert [sha(np.array(o)) for o in outs] == g["sha"]
    random.seed(1)
    skipped = [o for o in (aug.RandomCorruption(p=0.0)(pil) for _ in range(4))]
    assert all(o is pil for o in skipped)  # the same object comes back when the gate skips


def test_ultralytics_patch_with_stub_module(aug, golden_hashes, monkeypatch):
    calls = []

    class Albumentations:
        def __call__(self, labels):
            calls.append(labels["img"].shape)
            return labels

    pkg = types.ModuleType("ultralytics")
    data = types.ModuleType("ultralytics.data")
    augment = types.ModuleType("ultralytics.data.augment")
    augment.Albumentations = Albumentations
    pkg.data, data.augment = data, augment
    for name, mod in (("ultralytics", pkg), ("ultralytics.data", data), ("ultralytics.data.augment", augment)):
        monkeypatch.setitem(sys.modules, name, mod)
    aug.patch_ultralytics_augmentations()
    img = synth(31, 64, 64)
    random.seed(42)
    np.random.seed(42)
    got = [Albumentations()({"img": img})["img"] for _ in range(16)]
    random.seed(42)
    np.random.seed(42)
    want = []
    for op in golden_hashes["decisions"]["ultralytics"][:16]:
        # the oracle consumes random.random()/random.choice itself; replay with the same seeds
        r = random.random()
        want.append(orc.apply_random_corruption(img) if r < 0.5 else img)
    assert len(calls) == 16
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    assert [0 if a is img else 1 for a in got] == [1 if o else 0 for o in golden_hashes["decisions"]["ultralytics"][:16]]


# ------------------------------------------------------------------ Philox mode
def test_philox_field_and_fused_output(torch_):
    """Both Gaussian generators of Philox mode against their restated streams: the table generator (default at
    3 <= sigma <= 20; on Philox4x32-10 or, selectable, -7) is integer arithmetic and matches exactly; Box-Muller (forced
    per plan, or sigma outside that range) within float tolerance."""
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(37, 53), (64, 64), (31, 45)]
    plan = CorruptionPlan.ragged(shapes)
    imgs = [synth(50 + i, h, w) for i, (h, w) in enumerate(shapes)]
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    seed, first, off = 0x1234567890ABCDEF, 5, 3
    for generator, sigma in (("table", 15.0), ("table", 4.5), ("table", 3.0), ("table", 20.0), ("table7", 15.0),
                             ("boxmuller", 15.0), ("auto-boxmuller", 40.0), ("auto-boxmuller", 1.0), ("auto-boxmuller", 0.5)):
        plan.set_gaussian_generator({"boxmuller": 1, "table7": 2}.get(generator, 0))
        dst = torch_.zeros_like(src)
        field = torch_.zeros(plan.payload_bytes, dtype=torch_.float32, device="cuda")
        plan.noise_field(field, sigma, seed, first, off)
        plan.noise(src, dst, None, sigma, seed, first, off)
        f = field.cpu().numpy()
        outs = plan.unpack(dst.cpu().numpy())
        e = 0
        for i, (img, (h, w)) in enumerate(zip(imgs, shapes)):
            n = 3 * h * w
            if generator in ("table", "table7"):
                want = orc.philox_noise_field(n, sigma, seed, first + i, off,     # auto -> table
                                              generator="table7" if generator == "table7" else "auto")
                assert np.array_equal(f[e:e + n].astype(np.float64), want), (generator, sigma, i)
                assert np.array_equal(outs[i], orc.add_philox_noise(img, want)), (generator, sigma, i)
            else:
                want = orc.philox_noise_field(n, sigma, seed, first + i, off, generator="boxmuller")
                assert np.max(np.abs(f[e:e + n] - want)) < max(2e-3 * sigma / 15.0, 2e-5), (generator, sigma, i)
                # the kernel adds the field it reports: clamp(v + floor(noise), 0, 255); the dumped field is the
                # fp32-rounded product, the kernel floors the unrounded one, so a byte may differ only where noise
                # is within an ulp of an integer
                assert (outs[i] != orc.add_philox_noise(img, f[e:e + n])).mean() < 1e-4, (generator, i)
                assert np.abs(outs[i].astype(int) - orc.add_philox_noise(img, want)).max() <= 1 and \
                    (outs[i] != orc.add_philox_noise(img, want)).mean() < 1e-3, (generator, i)
            e += n
        # compat path on the dumped field (device-resident supplied-noise mode) agrees up to the reference's
        # float32 rounding of v + noise
        dst2 = torch_.zeros_like(src)
        plan.noise(src, dst2, field, sigma)
        assert (dst != dst2).float().mean().item() < 1e-4
    plan.set_gaussian_generator(0)


def test_philox_table_full_size_and_unaligned_spans(torch_):
    """The table generator at BASELINE size (vector path, all work-item shapes) and on pitched rows / odd widths (the
    element-wise path): bit-exact against the restated stream (integer arithmetic on both sides)."""
    from robust_object_detection_b200.batch import CorruptionPlan
    h, w = 765, 1360
    plan = CorruptionPlan.uniform(2, h, w)
    img = np.stack([synth(1234, h, w), synth(1235, h, w)])
    src = torch_.from_numpy(img).cuda()
    dst = torch_.empty_like(src)
    plan.noise(src, dst, None, 15.0, seed=0xC0FFEE, first_image_index=3)
    out = dst.cpu().numpy()
    for i in range(2):
        want = orc.philox_noise_field(img[i].size, 15.0, 0xC0FFEE, 3 + i)
        assert np.array_equal(out[i], orc.add_philox_noise(img[i], want)), i
    # odd width + pitched source rows: spans that start off a group boundary / off 16-byte alignment
    hh, ww = 45, 61
    big = synth(77, hh + 4, ww + 6)
    crop = big[2:2 + hh, 3:3 + ww]
    from robust_object_detection_b200 import augmentations as aug
    aug.set_noise_mode("philox", seed=31)
    try:
        got = aug.apply_noise(crop, 15.0)
    finally:
        aug.set_noise_mode("compat")
    want = orc.philox_noise_field(crop.size, 15.0, 31, 0)
    assert np.array_equal(got, orc.add_philox_noise(np.ascontiguousarray(crop), want))


def test_philox_table_pitched_batch_guard_bytes(torch_):
    """Table generator on a ragged batch with pitched source AND destination rows (every span is a row piece, most of
    them off 16-byte alignment and off a Philox group boundary) plus op-code masking: image bytes bit-exact against
    the restated stream, pitch padding / gaps / masked images untouched."""
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(37, 53), (64, 64), (31, 45), (3, 5), (1, 1), (90, 1366), (2, 6000)]
    imgs = [synth(8100 + i, h, w) for i, (h, w) in enumerate(shapes)]
    sp = [3 * w + 20 for h, w in shapes]
    dp = [3 * w + 9 for h, w in shapes]
    so = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, w), q in zip(shapes, sp)])])
    do = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, w), q in zip(shapes, dp)])])
    plan = CorruptionPlan(shapes, so[:-1], do[:-1], src_pitches=sp, dst_pitches=dp)
    hsrc = np.full(int(so[-1]), 0xAB, np.uint8)
    for img, o, q in zip(imgs, so, sp):
        h, w, _ = img.shape
        hsrc[o:o + h * q].reshape(h, q)[:, :3 * w] = img.reshape(h, 3 * w)
    src = torch_.from_numpy(hsrc).cuda()
    dst = torch_.full((int(do[-1]),), 7, dtype=torch_.uint8, device="cuda")
    ops = torch_.tensor([1, 1, 0, 1, 1, 1, 1], dtype=torch_.uint8, device="cuda")
    plan.noise(src, dst, None, 15.0, seed=77, first_image_index=10, opcodes=ops)
    hdst = dst.cpu().numpy()
    covered = np.zeros(hdst.size, bool)
    for i, (img, o, q) in enumerate(zip(imgs, do, dp)):
        h, w, _ = img.shape
        rows = hdst[o:o + h * q].reshape(h, q)
        if i == 2:
            assert (rows == 7).all()           # op-code 0: not a noise image
            continue
        want = orc.add_philox_noise(img, orc.philox_noise_field(img.size, 15.0, 77, 10 + i))
        assert np.array_equal(rows[:, :3 * w].reshape(h, w, 3), want), (i, shapes[i])
        cov = covered[o:o + h * q].reshape(h, q)
        cov[:, :3 * w] = True
    assert (hdst[~covered] == 7).all()         # padding, gaps between images, the masked image


def test_philox_statistics_and_reproducibility(torch_):
    from robust_object_detection_b200.batch import CorruptionPlan
    h, w = 765, 1360
    plan = CorruptionPlan.uniform(2, h, w)
    img = np.stack([synth(1000, h, w), np.full((h, w, 3), 128, np.uint8)])
    src = torch_.from_numpy(img).cuda()
    dst = torch_.empty_like(src)
    plan.noise(src, dst, None, 15.0, seed=42)
    out = dst.cpu().numpy().astype(np.int32)
    d0 = out[0] - img[0]
    mid = (img[0] >= 70) & (img[0] <= 185)
    # 1.4 M mid-range samples: standard error of the mean is 15/sqrt(n) = 0.013 -> 4 sigma
    assert abs(d0[mid].mean() + 0.5) < 0.05
    assert abs(d0[mid].std() - 15.0) < 0.05
    # clipping fractions against the reference's own numpy draw on the same image (binomial noise ~1e-4)
    np.random.seed(1)
    ref = orc.apply_noise(img[0], 15)
    assert abs((out[0] == 0).mean() - (ref == 0).mean()) < 6e-4
    assert abs((out[0] == 255).mean() - (ref == 255).mean()) < 6e-4
    assert 0.020 < ((out[0] == 0) & (img[0] > 0)).mean() + (img[0] == 0).mean() * 0.5 < 0.029
    d1 = out[1] - 128
    assert abs(d1.mean() + 0.5) < 0.035 and abs(d1.std() - 15.0) < 0.03
    # chi-square of the residual histogram on the constant image against N(0, 15^2) bins
    from scipy import stats
    edges = np.arange(-60, 62)
    hist, _ = np.histogram(d1, bins=edges)
    # d1 = trunc(128 + z) - 128 = floor(z) for |z| < 128
    p = np.diff(stats.norm.cdf(edges, scale=15.0))
    chi = ((hist - p * d1.size) ** 2 / (p * d1.size)).sum()
    assert chi < 2.0 * len(p), chi
    # same (seed, image index) -> identical; different seed or index -> uncorrelated
    dst2 = torch_.empty_like(src)
    plan.noise(src, dst2, None, 15.0, seed=42)
    assert torch_.equal(dst, dst2)
    plan.noise(src, dst2, None, 15.0, seed=43)
    d2 = dst2.cpu().numpy()[1].astype(np.int32) - 128
    assert abs(np.corrcoef(d1.ravel(), d2.ravel())[0, 1]) < 0.01
    # image-index keyed: image 1 of this batch == image 0 of a batch that starts at index 1
    plan1 = CorruptionPlan.uniform(1, h, w)
    d3 = torch_.empty_like(src[1:])
    plan1.noise(src[1:].contiguous(), d3, None, 15.0, seed=42, first_image_index=1)
    assert torch_.equal(d3[0], dst[1])


# ------------------------------------------------------------------ device-resident batches
def test_uniform_batch_all_ops(torch_):
    from robust_object_detection_b200.batch import CorruptionPlan
    n, h, w = 6, 765, 1360
    plan = CorruptionPlan.uniform(n, h, w)
    imgs = np.stack([synth(2000 + i, h, w) for i in range(n)])
    src = torch_.from_numpy(imgs).cuda()
    dst = torch_.empty_like(src)
    plan.blur(src, dst)
    out = dst.cpu().numpy()
    for i in range(n):
        assert np.array_equal(out[i], orc.apply_motion_blur(imgs[i], 9, 0)), i
    plan.lowres(src, dst)
    out = dst.cpu().numpy()
    for i in range(n):
        assert np.array_equal(out[i], orc.apply_lowres(imgs[i], 0.5)), i
    # op-codes: untouched images keep their previous bytes in dst
    dst.fill_(7)
    ops = torch_.tensor([2, 0, 2, 3, 1, 0], dtype=torch_.uint8, device="cuda")
    plan.blur(src, dst, opcodes=ops)
    out = dst.cpu().numpy()
    assert np.array_equal(out[0], orc.apply_motion_blur(imgs[0], 9, 0)) and (out[1] == 7).all() and (out[3] == 7).all()
    plan.corrupt(src, dst, ops, seed=9)
    out = dst.cpu().numpy()
    assert np.array_equal(out[1], imgs[1]) and np.array_equal(out[5], imgs[5])
    assert np.array_equal(out[2], orc.apply_motion_blur(imgs[2], 9, 0))
    assert np.array_equal(out[3], orc.apply_lowres(imgs[3], 0.5))
    fld = orc.philox_noise_field(imgs[4].size, 15.0, 9, 4)   # table generator: integer-valued, exact
    assert np.mean(out[4] != orc.add_philox_noise(imgs[4], fld)) < 1e-6


CONFIG3_SHAPES = [(765, 1360), (1050, 1400), (788, 1400), (1078, 1916), (1080, 1920), (1500, 2000), (540, 960),
                  (360, 480), (765, 1361), (1079, 1917), (1499, 1999)]


def test_ragged_mixed_resolution_batch(torch_):
    from robust_object_detection_b200.batch import CorruptionPlan
    rng = np.random.default_rng(3000)
    shapes = [CONFIG3_SHAPES[i] for i in rng.integers(0, len(CONFIG3_SHAPES), 14)] + CONFIG3_SHAPES[-3:]
    plan = CorruptionPlan.ragged(shapes)
    imgs = [synth(3100 + i, h, w) for i, (h, w) in enumerate(shapes)]
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    dst = torch_.zeros_like(src)
    plan.lowres(src, dst)
    for i, (img, out) in enumerate(zip(imgs, plan.unpack(dst.cpu().numpy()))):
        mism = int((out != orc.apply_lowres(img, 0.5)).sum())
        assert mism == 0, (i, shapes[i], mism)
    plan.blur(src, dst)
    for i, (img, out) in enumerate(zip(imgs, plan.unpack(dst.cpu().numpy()))):
        assert np.array_equal(out, orc.apply_motion_blur(img, 9, 0)), (i, shapes[i])
    # packed compat noise over the ragged batch (odd sizes: unaligned float field offsets)
    np.random.seed(5)
    fields = [orc.draw_noise_field(img.shape, 15) for img in imgs]
    nz = torch_.from_numpy(np.concatenate([f.reshape(-1) for f in fields])).cuda()
    plan.noise(src, dst, nz, 15.0)
    for i, (img, out) in enumerate(zip(imgs, plan.unpack(dst.cpu().numpy()))):
        assert np.array_equal(out, orc.add_noise_field(img, fields[i])), (i, shapes[i])


def test_lowres_marching_kernel_alignments(torch_):
    """The band kernels on rows at 4- and 8-byte phases: images packed at 4-byte granularity (their destination rows
    stay 4-byte aligned, so the exact-2x images go to lowres_x2p_kernel / lowres_x2h_kernel with 8- or 4-byte copy
    units, not to lowres_x2w_kernel), widths with a two-pixel last chunk, pitched rows, and a source base that is not
    4-byte aligned (the strip kernel lowres_x2_kernel takes every exact-2x image).  (2001, 1360) selects
    lowres_x2f_kernel and (2001, 1361) lowres_x2g_kernel.  tests/test_kernel_paths.py traces which kernel each layout
    reaches, lowres_x2w_kernel included."""
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(765, 1360), (360, 480), (100, 8), (9, 4), (2, 4), (5, 12), (64, 64), (65, 128), (131, 36), (201, 1400),
              (97, 1916), (540, 960), (33, 2000), (40, 20), (77, 1364), (1080, 1920), (1050, 1400), (41, 44),
              (98, 1916), (6, 244), (4, 248), (10, 1204), (12, 1448),   # rows at 4- / 8-byte phases, last strips of one (two-pixel) chunk
              (2001, 1360), (2001, 1361)]
    imgs = [synth(4200 + i, h, w) for i, (h, w) in enumerate(shapes)]
    want = [orc.apply_lowres(im, 0.5) for im in imgs]
    for align in (4, 256):
        plan = CorruptionPlan.ragged(shapes, align=align)
        packed = plan.pack(imgs)
        for lead in (0, 1):
            buf = torch_.zeros(lead + plan.src_bytes, dtype=torch_.uint8, device="cuda")
            src = buf[lead:]
            src.copy_(torch_.from_numpy(packed))
            dst = torch_.zeros(plan.dst_bytes, dtype=torch_.uint8, device="cuda")
            plan.lowres(src, dst)
            for i, out in enumerate(plan.unpack(dst.cpu().numpy())):
                assert np.array_equal(out, want[i]), (align, lead, i, shapes[i])
    # pitched source and destination rows (crop-like views)
    sp = [3 * w + 20 for h, w in shapes]
    dp = [3 * w + 8 for h, w in shapes]
    so = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, w), q in zip(shapes, sp)])])
    do = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, w), q in zip(shapes, dp)])])
    plan = CorruptionPlan(shapes, so[:-1], do[:-1], src_pitches=sp, dst_pitches=dp)
    hsrc = np.full(int(so[-1]), 0xAB, np.uint8)
    for img, o, q in zip(imgs, so, sp):
        h, w, _ = img.shape
        hsrc[o:o + h * q].reshape(h, q)[:, :3 * w] = img.reshape(h, 3 * w)
    src = torch_.from_numpy(hsrc).cuda()
    dst = torch_.full((int(do[-1]),), 7, dtype=torch_.uint8, device="cuda")
    plan.lowres(src, dst)
    hdst = dst.cpu().numpy()
    for i, (img, o, q) in enumerate(zip(imgs, do, dp)):
        h, w, _ = img.shape
        rows = hdst[o:o + h * q].reshape(h, q)
        assert np.array_equal(rows[:, :3 * w].reshape(h, w, 3), want[i]), (i, shapes[i])
        assert (rows[:, 3 * w:] == 7).all(), i  # pitch padding untouched
    # many bands per image and op-code masking
    plan = CorruptionPlan.uniform(3, 765, 1360)
    src = torch_.from_numpy(np.stack([imgs[0]] * 3)).cuda()
    dst = torch_.full_like(src, 9)
    plan.lowres(src, dst, opcodes=torch_.tensor([3, 0, 3], dtype=torch_.uint8, device="cuda"))
    out = dst.cpu().numpy()
    assert np.array_equal(out[0], want[0]) and np.array_equal(out[2], want[0]) and (out[1] == 9).all()


def test_spawned_dataloader_workers(aug):
    """The process model of INTEGRATION.md section 2: DataLoader-style workers started with the SPAWN method each
    initialise CUDA on their own and run the per-image hook; every worker's outputs equal what the oracle gives for the
    same seeds (random / np.random streams are per process, as in the reference's workers)."""
    import multiprocessing as mp
    from tests.helpers import spawn_worker_corrupt
    jobs = [(101, 97, 133), (202, 120, 200), (303, 64, 64), (404, 81, 90)]
    with mp.get_context("spawn").Pool(2) as pool:
        results = dict(pool.map(spawn_worker_corrupt, jobs))
    for seed, h, w in jobs:
        img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        random.seed(seed)
        np.random.seed(seed)
        want = [orc.apply_op(img, 1 + ("noise", "blur", "lowres").index(random.choice(["noise", "blur", "lowres"])))
                for _ in range(4)]
        assert [o.tobytes() for o in want] == results[seed], seed


def test_dataloader_workers_fork_and_spawn(aug, torch_):
    """A real torch.utils.data.DataLoader(num_workers=2) around the per-image hook, under both start methods
    (train_yolo_augmented.py:33 runs the hook in 8 DataLoader workers).  spawn: every worker owns a CUDA context and
    the outputs equal the oracle's for the same seeds.  fork: this process has used CUDA, so a forked worker cannot --
    the drop-in raises a RuntimeError naming the fix (not a raw CUDA error); the DataLoader re-raises it here."""
    from torch.utils.data import DataLoader
    from tests.helpers import CorruptDataset
    aug.apply_lowres(synth(1, 8, 8), 0.5)       # this process owns a CUDA context now
    jobs = [(501, 97, 133), (502, 120, 200), (503, 64, 64), (504, 81, 90), (505, 33, 47), (506, 40, 56)]
    got = {}
    for seed, data in DataLoader(CorruptDataset(jobs), batch_size=None, num_workers=2, multiprocessing_context="spawn"):
        got[int(seed)] = data
    for seed, h, w in jobs:
        img = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        random.seed(seed)
        np.random.seed(seed)
        op = 1 + ("noise", "blur", "lowres").index(random.choice(["noise", "blur", "lowres"]))
        assert got[seed] == orc.apply_op(img, op).tobytes(), seed
    with pytest.raises(RuntimeError, match="spawn"):
        for _ in DataLoader(CorruptDataset(jobs), batch_size=None, num_workers=2, multiprocessing_context="fork"):
            pass


def test_threads_sharing_shapes(aug):
    """The per-image functions are re-entrant (SURVEY 8b): threads corrupting same-shaped images concurrently -- they
    share the cached plan, its staging buffers and, for the two blur variants, its installed kernel -- all get the
    reference's bytes."""
    import threading
    img = [synth(7000 + i, 120, 200) for i in range(4)]
    want = {"blur": [orc.apply_motion_blur(x, 9, 0) for x in img], "lowres": [orc.apply_lowres(x, 0.5) for x in img],
            "blur5": [orc.apply_motion_blur(x, 5, 0) for x in img]}
    kern = aug._motion_blur_kernel(5, 45.0)
    want["blur45"] = [orc.apply_motion_blur(x, 5, 45.0, kernel=kern) for x in img]
    errors = []

    def work(t):
        try:
            for it in range(25):
                i = (t + it) % 4
                for name, fn in (("blur", lambda x: aug.apply_motion_blur(x, 9, 0)), ("lowres", lambda x: aug.apply_lowres(x, 0.5)),
                                 ("blur45", lambda x: aug.apply_motion_blur(x, 5, 45.0)), ("blur5", lambda x: aug.apply_motion_blur(x, 5, 0))):
                    if not np.array_equal(fn(img[i]), want[name][i]):
                        errors.append((t, it, name))
        except Exception as e:  # noqa: BLE001
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=work, args=(t,)) for t in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors[:5]


def test_apply_host_non_monotonic_plan(torch_):
    """rod_apply_host on plans whose images are NOT laid out in increasing order (reversed and shuffled offsets, which
    rod_plan_create accepts): the host upload must cover every image, not the span between the first and last descriptor."""
    from robust_object_detection_b200 import _native as N
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(37, 53), (64, 64), (31, 45), (20, 100)]
    sizes = [3 * h * w for h, w in shapes]
    imgs = [synth(8300 + i, h, w) for i, (h, w) in enumerate(shapes)]
    for order in ([3, 2, 1, 0], [2, 0, 3, 1]):
        offs = [0] * 4
        cur = 0
        for i in order:                      # image i sits at the position `order` gives it
            offs[i] = cur
            cur += (sizes[i] + 255) // 256 * 256
        plan = CorruptionPlan(shapes, offs, offs)
        src = np.full(cur, 0xEE, np.uint8)
        for i in range(4):
            src[offs[i]:offs[i] + sizes[i]] = imgs[i].reshape(-1)
        for op, fn in ((N.OP_BLUR, lambda x: orc.apply_motion_blur(x, 9, 0)), (N.OP_LOWRES, lambda x: orc.apply_lowres(x, 0.5))):
            dst = np.zeros(cur, np.uint8)
            plan.apply_host(op, src, dst)
            for i, (h, w) in enumerate(shapes):
                assert np.array_equal(dst[offs[i]:offs[i] + sizes[i]].reshape(h, w, 3), fn(imgs[i])), (order, op, i)


def test_torch_library_ops_parity(torch_):
    """The torch.library layer (torch.ops.rod.*) on CUDA uint8 tensors, current stream, against the oracle."""
    import robust_object_detection_b200.torch_ops  # noqa: F401
    rod = torch_.ops.rod
    n, h, w = 5, 97, 133
    imgs = np.stack([synth(8400 + i, h, w) for i in range(n)])
    x = torch_.from_numpy(imgs).cuda()
    assert np.array_equal(rod.blur(x, 9, 0.0).cpu().numpy(), np.stack([orc.apply_motion_blur(i, 9, 0) for i in imgs]))
    assert np.array_equal(rod.lowres(x, 0.5).cpu().numpy(), np.stack([orc.apply_lowres(i, 0.5) for i in imgs]))
    assert np.array_equal(rod.lowres(x[0], 0.5).cpu().numpy(), orc.apply_lowres(imgs[0], 0.5))          # [H,W,3] form
    kern = orc_kernel = None
    from robust_object_detection_b200.augmentations import _motion_blur_kernel
    kern = _motion_blur_kernel(5, 60.0)
    assert np.array_equal(rod.blur(x, 5, 60.0).cpu().numpy(), np.stack([orc.apply_motion_blur(i, 5, 60.0, kernel=kern) for i in imgs]))
    assert np.array_equal(rod.blur(x, 9, 0.0).cpu().numpy(), np.stack([orc.apply_motion_blur(i, 9, 0) for i in imgs]))  # back to the box
    np.random.seed(5)
    field = np.random.normal(0, 15, imgs.shape).astype(np.float32)
    got = rod.noise(x, 15.0, 0, 0, torch_.from_numpy(field).cuda()).cpu().numpy()
    assert np.array_equal(got, np.stack([orc.add_noise_field(i, f) for i, f in zip(imgs, field)]))
    got = rod.noise(x, 15.0, 77, 3).cpu().numpy()                                                  # Philox mode
    for i in range(n):
        assert np.array_equal(got[i], orc.add_philox_noise(imgs[i], orc.philox_noise_field(imgs[i].size, 15.0, 77, 3 + i)))
    ops = np.array([0, 1, 2, 3, 2], np.uint8)
    got = rod.corrupt_batch(x, torch_.from_numpy(ops).cuda(), 15.0, 9, 0.5, 9, 100).cpu().numpy()
    assert np.array_equal(got[0], imgs[0]) and np.array_equal(got[2], orc.apply_motion_blur(imgs[2], 9, 0))
    assert np.array_equal(got[3], orc.apply_lowres(imgs[3], 0.5)) and np.array_equal(got[4], orc.apply_motion_blur(imgs[4], 9, 0))
    assert np.array_equal(got[1], orc.add_philox_noise(imgs[1], orc.philox_noise_field(imgs[1].size, 15.0, 9, 101)))
    f16 = rod.corrupt_letterbox(x, torch_.from_numpy(ops).cuda(), 64, 96, 114, 15.0, 9, 0.5, 9, 100)
    assert f16.shape == (n, 3, 64, 96) and f16.dtype == torch_.float16
    assert np.array_equal(f16[2].cpu().numpy(), orc.letterbox_norm_f16(orc.apply_motion_blur(imgs[2], 9, 0), 64, 96))
    assert np.array_equal(f16[0].cpu().numpy(), orc.letterbox_norm_f16(imgs[0], 64, 96))
    # stream semantics: the ops run on the current stream
    s = torch_.cuda.Stream()
    with torch_.cuda.stream(s):
        y = rod.lowres(x, 0.5)
    s.synchronize()
    assert np.array_equal(y.cpu().numpy(), np.stack([orc.apply_lowres(i, 0.5) for i in imgs]))
    with pytest.raises(Exception):
        rod.blur(x.cpu(), 9, 0.0)


def test_letterbox_vs_cv2_primitive_golden(torch_):
    """The fused corrupt + letterbox kernel with every image clean, against the vectors built from live cv2.resize +
    cv2.copyMakeBorder (tests/golden/golden_letterbox.json): the formatting stage is pinned to OpenCV primitives, not only
    to the builder's NumPy restatement."""
    import json
    from robust_object_detection_b200.batch import CorruptionPlan
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_letterbox.json")))
    for seed, h, w, oh, ow in g["cases"]:
        img = synth(seed, h, w)
        plan = CorruptionPlan.uniform(1, h, w)
        src = torch_.from_numpy(img[None]).cuda()
        out = torch_.zeros((1, 3, oh, ow), dtype=torch_.float16, device="cuda")
        plan.corrupt_letterbox(src, torch_.zeros(1, dtype=torch_.uint8, device="cuda"), out, oh, ow, 114)
        assert sha(out[0].cpu().numpy()) == g["sha"][f"{seed}_{h}x{w}_{oh}x{ow}"], (h, w, oh, ow)


def test_noise_prewarm_then_first_launch_in_graph(torch_):
    """rod_noise_prewarm: after it, the FIRST Philox launch with a new sigma does no allocation / blocking copy and can
    be captured in a CUDA graph."""
    from robust_object_detection_b200.batch import CorruptionPlan
    sigma = 7.625                                        # not used by any other test in this process
    n, h, w = 3, 64, 80
    plan = CorruptionPlan.uniform(n, h, w)
    imgs = np.stack([synth(8500 + i, h, w) for i in range(n)])
    src = torch_.from_numpy(imgs).cuda()
    dst = torch_.zeros_like(src)
    plan.blur(src, dst)                                  # (warm-up of unrelated lazy state)
    CorruptionPlan.prewarm_noise(sigma)
    torch_.cuda.synchronize()
    g = torch_.cuda.CUDAGraph()
    with torch_.cuda.graph(g):
        plan.noise(src, dst, None, sigma, seed=11)
    g.replay()
    torch_.cuda.synchronize()
    out = dst.cpu().numpy()
    for i in range(n):
        assert np.array_equal(out[i], orc.add_philox_noise(imgs[i], orc.philox_noise_field(imgs[i].size, sigma, 11, i)))


def test_cuda_graph_capture_and_replay(torch_):
    """The device-resident entry points are stream-ordered (memset of the work counter + kernels): a corrupt_batch and a
    corrupt_letterbox call captured into a CUDA graph (after one eager call: resize tables, the noise quantile table and
    the auxiliary streams are created on first use) replay to the same bytes on new input contents."""
    from robust_object_detection_b200.batch import CorruptionPlan
    n, h, w = 6, 360, 480
    plan = CorruptionPlan.uniform(n, h, w)
    ops = torch_.tensor([1, 2, 3, 0, 2, 1], dtype=torch_.uint8, device="cuda")
    src = torch_.from_numpy(np.stack([synth(9500 + i, h, w) for i in range(n)])).cuda()
    dst = torch_.zeros_like(src)
    f16 = torch_.zeros((n, 3, 160, 160), dtype=torch_.float16, device="cuda")
    plan.corrupt(src, dst, ops, seed=5)                       # eager warm-up
    plan.corrupt_letterbox(src, ops, f16, 160, 160, 114, seed=5)
    torch_.cuda.synchronize()
    g = torch_.cuda.CUDAGraph()
    with torch_.cuda.graph(g):
        plan.corrupt(src, dst, ops, seed=5)
        plan.corrupt_letterbox(src, ops, f16, 160, 160, 114, seed=5)
    for rep in range(2):
        new = np.stack([synth(9600 + 10 * rep + i, h, w) for i in range(n)])
        src.copy_(torch_.from_numpy(new).cuda())
        dst.zero_()
        f16.zero_()
        g.replay()
        torch_.cuda.synchronize()
        got, got16 = dst.cpu().numpy(), f16.cpu().numpy()
        want = torch_.zeros_like(src)
        want16 = torch_.zeros_like(f16)
        plan.corrupt(src, want, ops, seed=5)
        plan.corrupt_letterbox(src, ops, want16, 160, 160, 114, seed=5)
        assert np.array_equal(got, want.cpu().numpy()) and np.array_equal(got16, want16.cpu().numpy()), rep
        assert np.array_equal(got[1], orc.apply_motion_blur(new[1], 9, 0)) and np.array_equal(got[2], orc.apply_lowres(new[2], 0.5))
        assert np.array_equal(got[3], new[3])


def test_very_wide_rows(aug):
    """Rows far wider than any VisDrone frame (panoramas): the blur kernel keeps a whole row per warp in shared memory and
    drops to fewer warps per CTA when 8 rows no longer fit; the other kernels tile in x.  Bit-exact vs the oracle."""
    for h, w in [(3, 12000), (2, 30001), (5, 9500)]:
        img = synth(9900 + h, h, w)
        assert np.array_equal(aug.apply_motion_blur(img, 9, 0), orc.apply_motion_blur(img, 9, 0)), (h, w)
        assert np.array_equal(aug.apply_motion_blur(img, 5, 0), orc.apply_motion_blur(img, 5, 0)), (h, w)
        assert np.array_equal(aug.apply_lowres(img, 0.5), orc.apply_lowres(img, 0.5)), (h, w)
        np.random.seed(3)
        got = aug.apply_noise(img, 15)
        np.random.seed(3)
        assert np.array_equal(got, orc.apply_noise(img, 15)), (h, w)


def test_full_size_config2_batch_by_replication(torch_):
    """BASELINE config 2 at full size (256 x 765x1360): 8 distinct images repeated 32 times; every
    replica must equal the oracle's output for its source image (bit-exact)."""
    from robust_object_detection_b200.batch import CorruptionPlan
    n, h, w = 256, 765, 1360
    base = np.stack([synth(2000 + i, h, w) for i in range(8)])
    src = torch_.from_numpy(base).cuda().repeat(32, 1, 1, 1).contiguous()
    dst = torch_.empty_like(src)
    plan = CorruptionPlan.uniform(n, h, w)
    for op, fn in (("blur", lambda im: orc.apply_motion_blur(im, 9, 0)), ("lowres", lambda im: orc.apply_lowres(im, 0.5))):
        getattr(plan, op)(src, dst)
        want = torch_.from_numpy(np.stack([fn(im) for im in base])).cuda()
        assert torch_.equal(dst.view(32, 8, h, w, 3), want.unsqueeze(0).expand(32, -1, -1, -1, -1)), op


def test_full_size_config3_mixed_256_by_replication(torch_):
    """BASELINE config 3 at full size: 256 mixed-resolution images (the 11 shapes of bench.py's draw, incl. the
    odd-dimension variants) in one ragged batch -- one seeded image per shape, replicated according to the draw; every
    replica must equal the oracle's fused LowRes output for its source image (0 mismatching bytes)."""
    from robust_object_detection_b200.batch import CorruptionPlan
    rng = np.random.default_rng(3000)
    idx = rng.integers(0, len(CONFIG3_SHAPES), 256)
    shapes = [CONFIG3_SHAPES[i] for i in idx]
    plan = CorruptionPlan.ragged(shapes)
    base = [synth(3300 + k, h, w) for k, (h, w) in enumerate(CONFIG3_SHAPES)]
    want = [torch_.from_numpy(orc.apply_lowres(b, 0.5)).cuda() for b in base]
    dev = [torch_.from_numpy(b).cuda() for b in base]
    src = torch_.zeros(plan.src_bytes, dtype=torch_.uint8, device="cuda")
    for i, k in enumerate(idx):
        h, w = shapes[i]
        src[plan.src_offsets[i]:plan.src_offsets[i] + 3 * h * w] = dev[k].reshape(-1)
    dst = torch_.zeros_like(src)
    plan.lowres(src, dst)
    assert len(set(int(k) for k in idx)) == len(CONFIG3_SHAPES)
    for i, k in enumerate(idx):
        h, w = shapes[i]
        got = dst[plan.dst_offsets[i]:plan.dst_offsets[i] + 3 * h * w].view(h, w, 3)
        mism = int((got != want[k]).sum().item())
        assert mism == 0, (i, shapes[i], mism)


def test_config5_batch16_seed42(torch_):
    """BASELINE config 5 as one case: batch 16 of 765x1360 frames, decisions drawn on the host with random.seed(42) in
    the reference's order (random() < 0.5, then random.choice: golden 'ultralytics' stream), fused corrupt + letterbox 640
    + normalise -> fp16 NCHW.  Non-noise images are bit-exact against oracle corruption + letterbox (itself pinned to the
    cv2-primitive golden); noise images (Box-Muller Philox on this path) against the restated stream up to its float
    tolerance."""
    from robust_object_detection_b200.batch import CorruptionPlan, draw_decisions
    n, h, w = 16, 765, 1360
    random.seed(42)
    ops_host = draw_decisions(n)
    assert [int(o) for o in ops_host] == [0, 2, 1, 0, 0, 0, 2, 1, 3, 0, 0, 0, 0, 2, 0, 0]     # SURVEY section 4
    imgs = np.stack([synth(5200 + i, h, w) for i in range(n)])
    plan = CorruptionPlan.uniform(n, h, w)
    src = torch_.from_numpy(imgs).cuda()
    out = torch_.zeros((n, 3, 640, 640), dtype=torch_.float16, device="cuda")
    plan.corrupt_letterbox(src, torch_.from_numpy(ops_host).cuda(), out, 640, 640, 114, seed=42)
    got = out.cpu().numpy()
    for i in range(n):
        if ops_host[i] == 1:
            cor = orc.add_philox_noise(imgs[i], orc.philox_noise_field(imgs[i].size, 15.0, 42, i, generator="boxmuller"))
            want = orc.letterbox_norm_f16(cor, 640, 640, 114).astype(np.float32)
            assert np.mean(np.abs(got[i].astype(np.float32) - want) > 1e-6) < 2e-3, i
        else:
            want = orc.letterbox_norm_f16(orc.apply_op(imgs[i], int(ops_host[i])), 640, 640, 114)
            assert np.array_equal(got[i], want), (i, int(ops_host[i]))
    assert np.all(got[:, :, :140, :] == np.float16(114 / 255)) and np.all(got[:, :, 500:, :] == np.float16(114 / 255))


def test_full_size_config4_testset_by_replication_and_sharding(torch_):
    """BASELINE config 4 at full size: 1610 VisDrone-shaped images (8 real frame sizes, same draw as bench.py) in one
    ragged device-resident batch, the three corruptions of the test-set build.  Parity at this size rests on properties
    that do not need 1610 oracle runs: (1) replication -- one distinct image per frame size, so every output must equal
    the oracle's output for that size's image (blur, LowRes: bit-exact); (2) Philox noise is keyed by the global image
    index -- three images are checked against the restated stream, and corrupting the batch as two image-index shards
    (what two ranks would do, sharding.py) must give the same bytes as one batch; (3) image-index sharding of the other
    two ops likewise."""
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.sharding import shard_range
    pool = [(765, 1360), (1050, 1400), (788, 1400), (1078, 1916), (1080, 1920), (1500, 2000), (540, 960), (360, 480)]
    kinds = np.random.default_rng(4000).integers(0, 8, 1610)
    shapes = [pool[i] for i in kinds]
    base = [synth(9000 + i, h, w) for i, (h, w) in enumerate(pool)]
    dbase = [torch_.from_numpy(b.reshape(-1)).cuda() for b in base]
    plan = CorruptionPlan.ragged(shapes)
    src = torch_.zeros(plan.src_bytes, dtype=torch_.uint8, device="cuda")
    for off, k in zip(plan.src_offsets, kinds):
        src[off:off + dbase[k].numel()] = dbase[k]
    dst = torch_.empty_like(src)

    def image(buf, i):
        h, w = shapes[i]
        return buf[plan.dst_offsets[i]:plan.dst_offsets[i] + 3 * h * w]

    full = {}
    for op, fn in (("blur", lambda im: orc.apply_motion_blur(im, 9, 0)), ("lowres", lambda im: orc.apply_lowres(im, 0.5))):
        dst.zero_()
        getattr(plan, op)(src, dst)
        want = [torch_.from_numpy(fn(b).reshape(-1)).cuda() for b in base]
        assert all(torch_.equal(image(dst, i), want[kinds[i]]) for i in range(1610)), op
        full[op] = dst.clone()
    dst.zero_()
    plan.noise(src, dst, None, 15.0, seed=42, first_image_index=0)
    for i in (0, 807, 1609):
        h, w = shapes[i]
        fld = orc.philox_noise_field(3 * h * w, 15.0, 42, i)
        assert np.array_equal(image(dst, i).cpu().numpy().reshape(h, w, 3), orc.add_philox_noise(base[kinds[i]], fld)), i
    full["noise"] = dst.clone()
    # the same work as two image-index shards (each shard: its own plan over its own images, global Philox index)
    for rank in range(2):
        lo, hi = shard_range(1610, rank, 2)
        sp = CorruptionPlan.ragged(shapes[lo:hi])
        b0 = plan.src_offsets[lo]
        ssrc = src[b0:b0 + sp.src_bytes]
        sdst = torch_.empty_like(ssrc)
        for op in ("blur", "lowres", "noise"):
            sdst.zero_()
            if op == "noise":
                sp.noise(ssrc, sdst, None, 15.0, seed=42, first_image_index=lo)
            else:
                getattr(sp, op)(ssrc, sdst)
            for j in (0, (hi - lo) // 2, hi - lo - 1):
                h, w = shapes[lo + j]
                got = sdst[sp.dst_offsets[j]:sp.dst_offsets[j] + 3 * h * w]
                assert torch_.equal(got, image(full[op], lo + j)), (rank, op, j)
            assert torch_.equal(sdst[:sp.dst_offsets[-1]], full[op][b0:b0 + sp.dst_offsets[-1]]), (rank, op)


@pytest.mark.parametrize("ow", [640, 639])
def test_letterbox_fused_training_path(torch_, ow):
    # the (640, 640) source is an identity letterbox at 640 x 640 and 639 is odd: both widths take the unfused path
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(765, 1360)] * 5 + [(720, 1280), (360, 480), (640, 640), (1079, 1917)]
    plan = CorruptionPlan.ragged(shapes)
    imgs = [synth(5000 + i, h, w) for i, (h, w) in enumerate(shapes)]
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    ops_host = np.array([0, 2, 3, 2, 0, 3, 2, 0, 3], dtype=np.uint8)
    ops = torch_.from_numpy(ops_host).cuda()
    out = torch_.empty((len(shapes), 3, 640, ow), dtype=torch_.float16, device="cuda")
    plan.corrupt_letterbox(src, ops, out, 640, ow, 114, seed=1)
    got = out.cpu().numpy()
    for i, img in enumerate(imgs):
        want = orc.letterbox_norm_f16(orc.apply_op(img, int(ops_host[i])), 640, ow, 114)
        assert np.array_equal(got[i], want), (i, shapes[i])


@pytest.mark.parametrize("ow", [320, 319])
def test_fused_letterbox_kernel_paths(torch_, ow):
    """fused_letterbox2_kernel (every shape a plain linear letterbox): 16-byte-aligned rows (cp.async staging), odd widths
    (32-bit / byte staging, Philox groups straddling rows), supplied noise field, another blur size, and a pitched
    source; all against the oracle, bit-exact except Philox noise (statistical mode).  An odd output width runs the same
    cases on the unfused path."""
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(765, 1360), (765, 1360), (540, 960), (333, 517), (401, 1001), (1079, 1917), (360, 480), (765, 1360)]
    ops_host = np.array([1, 2, 3, 2, 1, 0, 1, 0], dtype=np.uint8)
    imgs = [synth(5100 + i, h, w) for i, (h, w) in enumerate(shapes)]
    plan = CorruptionPlan.ragged(shapes)
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    ops = torch_.from_numpy(ops_host).cuda()
    out = torch_.empty((len(shapes), 3, 320, ow), dtype=torch_.float16, device="cuda")
    # (a) compat noise (supplied field), k = 9
    np.random.seed(33)
    fields = [orc.draw_noise_field(im.shape, 15) for im in imgs]
    nz = torch_.from_numpy(np.concatenate([f.reshape(-1) for f in fields])).cuda()
    plan.corrupt_letterbox(src, ops, out, 320, ow, 114, noise=nz)
    got = out.cpu().numpy()
    for i, img in enumerate(imgs):
        op = int(ops_host[i])
        cor = orc.add_noise_field(img, fields[i]) if op == 1 else orc.apply_op(img, op)
        assert np.array_equal(got[i], orc.letterbox_norm_f16(cor, 320, ow, 114)), (i, shapes[i], op)
    # (b) Philox noise keyed by a global index offset, blur k = 5
    plan.corrupt_letterbox(src, ops, out, 320, ow, 114, k=5, seed=77, first_image_index=1000)
    got = out.cpu().numpy()
    for i, img in enumerate(imgs):
        op = int(ops_host[i])
        if op == 1:
            want = orc.letterbox_norm_f16(orc.add_philox_noise(img, orc.philox_noise_field(img.size, 15.0, 77, 1000 + i, generator="boxmuller")), 320, ow, 114)
            assert np.mean(got[i] != want) < 2e-3, (i, shapes[i])
        else:
            cor = orc.apply_motion_blur(img, 5, 0) if op == 2 else orc.apply_op(img, op)
            assert np.array_equal(got[i], orc.letterbox_norm_f16(cor, 320, ow, 114)), (i, shapes[i], op)
    # (c) pitched source rows
    sp = [3 * w + 12 for h, w in shapes]
    so = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, w), q in zip(shapes, sp)])])
    planp = CorruptionPlan(shapes, so[:-1], plan.dst_offsets, src_pitches=sp)
    hsrc = np.full(int(so[-1]), 0xAB, np.uint8)
    for img, o, q in zip(imgs, so, sp):
        h, w, _ = img.shape
        hsrc[o:o + h * q].reshape(h, q)[:, :3 * w] = img.reshape(h, 3 * w)
    ops2 = torch_.from_numpy(np.array([2, 0, 3, 2, 0, 2, 3, 0], dtype=np.uint8)).cuda()
    planp.corrupt_letterbox(torch_.from_numpy(hsrc).cuda(), ops2, out, 320, ow, 114)
    got = out.cpu().numpy()
    for i, img in enumerate(imgs):
        want = orc.letterbox_norm_f16(orc.apply_op(img, int(ops2[i].item())), 320, ow, 114)
        assert np.array_equal(got[i], want), (i, shapes[i])


@pytest.mark.parametrize("oh, ow", [(640, 640), (320, 416), (96, 96), (96, 97)])
def test_fused_letterbox_lowres_in_kernel(torch_, oh, ow):
    """Every shape exact-2x (w % 4 == 0): the LowRes rows are produced inside fused_letterbox2_kernel too (no scratch);
    odd and even heights, a width with a two-pixel last chunk, several output sizes; an odd output width takes the
    unfused path."""
    from robust_object_detection_b200.batch import CorruptionPlan
    shapes = [(765, 1360), (540, 960), (360, 480), (1080, 1920), (1050, 1400), (97, 1916), (131, 36), (765, 1360)]
    ops_host = np.array([3, 3, 3, 3, 3, 3, 3, 2], dtype=np.uint8)
    imgs = [synth(5200 + i, h, w) for i, (h, w) in enumerate(shapes)]
    plan = CorruptionPlan.ragged(shapes)
    src = torch_.from_numpy(plan.pack(imgs)).cuda()
    ops = torch_.from_numpy(ops_host).cuda()
    want_cor = [orc.apply_op(im, int(o)) for im, o in zip(imgs, ops_host)]
    out = torch_.empty((len(shapes), 3, oh, ow), dtype=torch_.float16, device="cuda")
    plan.corrupt_letterbox(src, ops, out, oh, ow, 114)
    got = out.cpu().numpy()
    for i in range(len(shapes)):
        assert np.array_equal(got[i], orc.letterbox_norm_f16(want_cor[i], oh, ow, 114)), (i, shapes[i], oh, ow)


def test_apply_host_chunked_pipeline(torch_):
    """Host-buffer entry point with enough payload for several H2D/kernel/D2H chunks."""
    from robust_object_detection_b200 import _native as N
    from robust_object_detection_b200.batch import CorruptionPlan
    n, h, w = 40, 765, 1360
    imgs = np.stack([synth(2000 + (i % 4), h, w) for i in range(n)])
    plan = CorruptionPlan.uniform(n, h, w)
    dst = np.zeros_like(imgs)
    plan.apply_host(N.OP_BLUR, imgs, dst)
    want = [orc.apply_motion_blur(imgs[i], 9, 0) for i in range(4)]
    for i in range(n):
        assert np.array_equal(dst[i], want[i % 4]), i
    plan.apply_host(N.OP_LOWRES, imgs, dst)
    want = [orc.apply_lowres(imgs[i], 0.5) for i in range(4)]
    for i in range(n):
        assert np.array_equal(dst[i], want[i % 4]), i


def test_restoration_pairs_fused(torch_):
    """SURVEY 8f rank 4: RestorationDataset.__getitem__ on device (crop view -> flip -> corrupt -> RGB f32 CHW / 255 for
    the corrupted input and the clean target), decisions drawn in the reference's RNG order."""
    from robust_object_detection_b200.batch import CorruptionPlan, draw_restoration_decisions
    size = 64
    shapes = [(120, 200), (97, 133), (64, 64), (300, 180), (81, 90), (200, 201)]
    imgs = [synth(5000 + i, h, w) for i, (h, w) in enumerate(shapes)]
    base = CorruptionPlan.ragged(shapes)  # only used to pack the full images into one device buffer
    src = torch_.from_numpy(base.pack(imgs)).cuda()
    random.seed(2)
    dec = [draw_restoration_decisions(h, w, size, is_train=(i != 2)) for i, (h, w) in enumerate(shapes)]
    offs = [base.src_offsets[i] + y * 3 * shapes[i][1] + 3 * x for i, (y, x, _, _) in enumerate(dec)]
    plan = CorruptionPlan([(size, size)] * len(shapes), offs, [0] * len(shapes), src_pitches=[3 * w for _, w in shapes])
    flips = torch_.tensor([int(f) for _, _, f, _ in dec], dtype=torch_.uint8, device="cuda")
    ops = torch_.tensor([o for _, _, _, o in dec], dtype=torch_.uint8, device="cuda")
    np.random.seed(21)
    fields = [orc.draw_noise_field((size, size, 3), 15) for _ in shapes]
    nz = torch_.from_numpy(np.stack(fields).reshape(-1)).cuda()
    corrupted = torch_.zeros((len(shapes), 3, size, size), dtype=torch_.float32, device="cuda")
    clean = torch_.zeros_like(corrupted)
    plan.restoration_pairs(src, flips, ops, corrupted, clean, noise=nz)
    assert {o for _, _, _, o in dec} == {1, 2, 3} and any(f for _, _, f, _ in dec)
    for i, (img, (y, x, flip, op)) in enumerate(zip(imgs, dec)):
        patch = img[y:y + size, x:x + size]
        if flip:
            patch = patch[:, ::-1]
        patch = np.ascontiguousarray(patch)
        cor = {1: lambda p: orc.add_noise_field(p, fields[i]), 2: lambda p: orc.apply_motion_blur(p, 9, 0),
               3: lambda p: orc.apply_lowres(p, 0.5)}[op](patch)
        want_clean = (patch[:, :, ::-1].astype(np.float32) / 255.0).transpose(2, 0, 1)
        want_cor = (cor[:, :, ::-1].astype(np.float32) / 255.0).transpose(2, 0, 1)
        assert np.array_equal(clean[i].cpu().numpy(), want_clean), i
        assert np.array_equal(corrupted[i].cpu().numpy(), want_cor), (i, op)


def test_restoration_pair_batcher_host_level(torch_):
    """training.RestorationPairBatcher: host frames in, (corrupted, clean) float32 batches on the device out, equal to the
    reference dataset's per-item arithmetic (train_restoration.py:104-129 restated with the oracle) under the same
    random / np.random seeds -- train mode (random crop, flip) and validation mode (centre crop)."""
    from robust_object_detection_b200.training import RestorationPairBatcher
    P = 64
    shapes = [(120, 200), (97, 133), (64, 64), (300, 180), (81, 90), (200, 201), (765, 1360), (70, 64)]
    frames = [synth(5600 + i, h, w) for i, (h, w) in enumerate(shapes)]
    for is_train in (True, False):
        random.seed(8)
        np.random.seed(9)
        batcher = RestorationPairBatcher(patch_size=P, is_train=is_train)
        got = [batcher(frames[:5]), batcher(frames[5:])]
        cor = np.concatenate([g[0].cpu().numpy() for g in got])
        clean = np.concatenate([g[1].cpu().numpy() for g in got])
        random.seed(8)
        np.random.seed(9)
        ops_seen = set()
        for i, img in enumerate(frames):
            h, w = img.shape[:2]
            if is_train:
                y, x = random.randint(0, h - P), random.randint(0, w - P)
                patch = img[y:y + P, x:x + P]
                if random.random() > 0.5:
                    patch = patch[:, ::-1]
            else:
                patch = img[(h - P) // 2:(h - P) // 2 + P, (w - P) // 2:(w - P) // 2 + P]
            patch = np.ascontiguousarray(patch)
            op = 1 + ("noise", "blur", "lowres").index(random.choice(["noise", "blur", "lowres"]))
            ops_seen.add(op)
            c = orc.apply_op(patch, op)   # noise: np.random.normal on the global stream, like the reference
            assert np.array_equal(clean[i], (patch[:, :, ::-1].astype(np.float32) / 255.0).transpose(2, 0, 1)), (is_train, i)
            assert np.array_equal(cor[i], (c[:, :, ::-1].astype(np.float32) / 255.0).transpose(2, 0, 1)), (is_train, i, op)
        assert ops_seen == {1, 2, 3}


def test_restoration_resize_first_branch(torch_):
    """Frames smaller than the patch (train_restoration.py:79-81, 88-90): rod_resize_linear_u8 against live
    cv2.resize(INTER_LINEAR) for enlargements in one or both axes, and RestorationPairBatcher on such frames against the
    pairs of the unmodified RestorationDataset (golden_restoration_small.npz; compat noise: bit-exact)."""
    import cv2
    from robust_object_detection_b200.batch import resize_linear_u8
    from robust_object_detection_b200.training import RestorationPairBatcher
    for i, (h, w, nh, nw) in enumerate([(40, 80, 64, 80), (100, 50, 100, 64), (30, 30, 64, 64), (64, 20, 64, 64), (63, 65, 64, 65),
                                        (7, 5, 256, 256), (1, 1, 3, 2), (200, 255, 256, 256), (97, 133, 97, 133), (120, 77, 333, 190)]):
        img = synth(5300 + i, h, w)
        want = img if (nh, nw) == (h, w) else cv2.resize(img, (nw, nh))
        assert np.array_equal(resize_linear_u8(img, nh, nw), want), (h, w, nh, nw)
    with pytest.raises(NotImplementedError):
        resize_linear_u8(synth(1, 40, 80), 20, 80)   # reductions are not this entry point's job
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_restoration_small.npz"))
    small = [(40, 80), (100, 50), (30, 30), (64, 20), (70, 64), (63, 65)]
    frames = [synth(5100 + i, h, w) for i, (h, w) in enumerate(small)]
    for is_train in (True, False):
        random.seed(4)
        np.random.seed(41)
        tag = "train" if is_train else "val"
        pairs = RestorationPairBatcher(patch_size=64, is_train=is_train)
        for i, fr in enumerate(frames):   # one frame per call: the reference draws crop / flip / op / noise per item, in this order
            cor, clean = pairs([fr])
            assert np.array_equal(clean[0].cpu().numpy(), g[f"{tag}_clean_{i}"]), (tag, i)
            assert np.array_equal(cor[0].cpu().numpy(), g[f"{tag}_cor_{i}"]), (tag, i, pairs.last_decisions)


def test_training_batcher_pinned_pipeline(torch_):
    """SURVEY 8f rank 2: main-process hook -- pinned staging + copy stream + corrupt_letterbox, decisions in the
    reference's RNG order, Philox keyed by the running global image index (independent of batching)."""
    from robust_object_detection_b200.training import CorruptionBatcher
    shapes = [(765, 1360), (540, 960), (360, 480), (333, 517)]
    frames = [synth(6000 + i, *shapes[i % 4]) for i in range(12)]
    batches = [frames[0:4], frames[4:7], frames[7:12]]
    random.seed(42)
    want_ops = orc.draw_decisions(12, gate="ultralytics")
    random.seed(42)
    b = CorruptionBatcher(out_hw=(160, 160), seed=9)
    outs, ops = [], []
    for x in b.run(batches):
        outs.append(x.cpu().numpy())
        ops.extend(b.last_ops.tolist())
    assert ops == list(want_ops) and len(set(ops)) == 4
    got = np.concatenate(outs)
    for i, (img, op) in enumerate(zip(frames, ops)):
        if op == 1:
            cor = orc.add_philox_noise(img, orc.philox_noise_field(img.size, 15.0, 9, i, generator="boxmuller"))
        else:
            cor = orc.apply_op(img, op)
        want = orc.letterbox_norm_f16(cor, 160, 160)
        if op == 1:
            assert np.mean(got[i] != want) < 2e-3, i   # sin/cos/log approximations at truncation boundaries
        else:
            assert np.array_equal(got[i], want), (i, op)
    # same frames, different batching, same result (global image index keys the noise)
    random.seed(42)
    b2 = CorruptionBatcher(out_hw=(160, 160), seed=9)
    got2 = np.concatenate([x.cpu().numpy() for x in b2.run([frames[0:6], frames[6:12]])])
    assert np.array_equal(got, got2)


@pytest.mark.parametrize("is_train", [True, False])
def test_restoration_pairs_vs_reference_dataset_gpu(torch_, is_train):
    """The fused device path against pairs produced by the unmodified RestorationDataset (golden_restoration.npz)."""
    from robust_object_detection_b200.batch import CorruptionPlan
    from tests.test_oracle_golden import RESTORATION_SHAPES, restoration_inputs
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_restoration.npz"))
    frames, dec, fields = restoration_inputs(is_train)
    base = CorruptionPlan.ragged(RESTORATION_SHAPES)
    src = torch_.from_numpy(base.pack(frames)).cuda()
    offs = [base.src_offsets[i] + y * 3 * RESTORATION_SHAPES[i][1] + 3 * x for i, (y, x, _, _) in enumerate(dec)]
    n = len(frames)
    plan = CorruptionPlan([(64, 64)] * n, offs, [0] * n, src_pitches=[3 * w for _, w in RESTORATION_SHAPES])
    flips = torch_.tensor([int(f) for _, _, f, _ in dec], dtype=torch_.uint8, device="cuda")
    ops = torch_.tensor([o for _, _, _, o in dec], dtype=torch_.uint8, device="cuda")
    nz = torch_.from_numpy(np.stack(fields).reshape(-1)).cuda()
    cor = torch_.zeros((n, 3, 64, 64), dtype=torch_.float32, device="cuda")
    clean = torch_.zeros_like(cor)
    plan.restoration_pairs(src, flips, ops, cor, clean, noise=nz)
    tag = "train" if is_train else "val"
    for i in range(n):
        assert np.array_equal(clean[i].cpu().numpy(), g[f"{tag}_clean_{i}"]), i
        assert np.array_equal(cor[i].cpu().numpy(), g[f"{tag}_cor_{i}"]), (i, dec[i])


def test_build_corrupted_testsets_drop_in(tmp_path, monkeypatch):
    """Row a9 end to end: the drop-in batch driver on a synthetic YOLO + COCO tree of JPEG files.  Every output file must
    be byte-identical to what the reference loop produces: same cv2 codec, same glob order, same np.random stream for
    Test_Noise (expected bytes are computed here with the oracle + cv2.imwrite in the same order)."""
    import cv2
    from robust_object_detection_b200 import build_corrupted_testsets as drv
    shapes = [(120, 200), (97, 133), (64, 64), (300, 180), (81, 90), (200, 202), (765, 1360)]
    for tree in ("yolo", "coco"):
        img_dir = tmp_path / tree / "images" / "val"
        img_dir.mkdir(parents=True)
        for i, (h, w) in enumerate(shapes):
            # smooth-ish content so the JPEG round trip is not pure noise
            base = cv2.GaussianBlur(synth(7000 + i, h, w), (0, 0), 2.0)
            cv2.imwrite(str(img_dir / f"frame_{i:03d}.jpg"), base)
        (img_dir / "broken.jpg").write_bytes(b"not a jpeg")          # unreadable: skipped, consumes no RNG
        (img_dir / "frame_png.png").write_bytes(cv2.imencode(".png", synth(7100, 50, 70))[1].tobytes())
    (tmp_path / "yolo" / "labels" / "val").mkdir(parents=True)
    for i in range(len(shapes)):
        (tmp_path / "yolo" / "labels" / "val" / f"frame_{i:03d}.txt").write_text(f"0 0.5 0.5 0.1 0.{i + 1}\n")
    (tmp_path / "coco" / "annotations").mkdir(parents=True)
    (tmp_path / "coco" / "annotations" / "instances_val.json").write_text('{"images": [], "annotations": []}')
    monkeypatch.setattr(drv, "YOLO_SRC", tmp_path / "yolo")
    monkeypatch.setattr(drv, "COCO_SRC", tmp_path / "coco")
    monkeypatch.setattr(drv, "OUT_ROOT", tmp_path / "out")
    monkeypatch.setattr(drv, "BATCH_BYTES", 20 << 20)  # several GPU batches
    drv.main()

    # expected: the reference loop (build_corrupted_testsets.py:169-173, :85-166) restated with the oracle
    np.random.seed(42)
    ops = {"Test_Clean": 0, "Test_Noise": 1, "Test_Blur": 2, "Test_LowRes": 3}
    n_files = 0
    for tree, sub in (("yolo", "yolo6"), ("coco", "coco6")):
        for v in ["Test_Clean", "Test_Noise", "Test_Blur", "Test_LowRes"]:
            dst = tmp_path / "out" / sub / v
            for p in (tmp_path / tree / "images" / "val").glob("*.*"):
                img = cv2.imread(str(p))
                if img is None:
                    assert not (dst / "images" / "val" / p.name).exists()
                    continue
                want = orc.apply_op(img, ops[v])
                ok, enc = cv2.imencode(p.suffix, want)
                assert ok and (dst / "images" / "val" / p.name).read_bytes() == enc.tobytes(), (tree, v, p.name)
                n_files += 1
            if tree == "yolo":
                assert (dst / "data.yaml").read_text().startswith(f"path: {dst.as_posix()}")
                assert sorted(q.name for q in (dst / "labels" / "val").glob("*.txt")) == [f"frame_{i:03d}.txt" for i in range(len(shapes))]
            else:
                assert (dst / "annotations" / "instances_val.json").read_text() == '{"images": [], "annotations": []}'
    assert n_files == 2 * 4 * (len(shapes) + 1)


@pytest.mark.parametrize("noise_mode", ["philox", "compat"])
def test_build_corrupted_testsets_sharded_equals_single(tmp_path, monkeypatch, noise_mode):
    """BASELINE configs[3] with files: two ranks (run here one after the other through the SHARD knob, which stands for
    torchrun's RANK / WORLD_SIZE) write, between them, exactly the files one process writes -- byte for byte, in both
    noise modes (Philox is keyed by the position in the glob list; the serial compat stream belongs to rank 0)."""
    import cv2
    from robust_object_detection_b200 import build_corrupted_testsets as drv
    shapes = [(120, 200), (97, 133), (64, 64), (300, 180), (81, 90), (200, 202), (240, 320), (33, 47), (150, 150)]
    img_dir = tmp_path / "yolo" / "images" / "val"
    img_dir.mkdir(parents=True)
    for i, (h, w) in enumerate(shapes):
        cv2.imwrite(str(img_dir / f"frame_{i:03d}.jpg"), cv2.GaussianBlur(synth(7300 + i, h, w), (0, 0), 1.5))
    (img_dir / "broken.jpg").write_bytes(b"not a jpeg")   # unreadable files must not shift the Philox keys of the others
    (tmp_path / "yolo" / "labels" / "val").mkdir(parents=True)
    (tmp_path / "yolo" / "labels" / "val" / "frame_000.txt").write_text("0 0.5 0.5 0.1 0.1\n")
    monkeypatch.setattr(drv, "YOLO_SRC", tmp_path / "yolo")
    monkeypatch.setattr(drv, "NOISE_MODE", noise_mode)
    monkeypatch.setattr(drv, "BATCH_BYTES", 20 << 20)   # the readahead counts 6 MB per file: four files per batch
    trees = {}
    for name, shards in (("single", [None]), ("sharded", [(1, 2), (0, 2)])):
        monkeypatch.setattr(drv, "OUT_ROOT", tmp_path / name)
        for shard in shards:
            monkeypatch.setattr(drv, "SHARD", shard)
            drv.set_seed(drv.SEED)
            drv.build_yolo_testsets()
        files = {}
        for q in sorted((tmp_path / name).rglob("*")):
            if q.is_file():
                files[str(q.relative_to(tmp_path / name))] = q.read_bytes()
        trees[name] = files
    assert len(trees["single"]) == 4 * (len(shapes) + 2)   # images + label + data.yaml per variant
    assert trees["single"].keys() == trees["sharded"].keys()
    for k, v in trees["single"].items():
        if k.endswith("data.yaml"):
            continue   # carries the absolute output root
        assert trees["sharded"][k] == v, k


def test_random_shapes_stress(torch_):
    """120 random shapes (1..320 x 1..420, biased to the kernels' corner cases: w % 4, w % 8, odd sizes, tiny images) in
    ragged batches with 4-byte packing: blur, lowres and compat noise against the oracle, bit-exact."""
    from robust_object_detection_b200.batch import CorruptionPlan
    rng = np.random.default_rng(20240)
    shapes = []
    for i in range(120):
        h = int(rng.integers(1, 321))
        w = int(rng.integers(1, 421))
        if i % 3 == 0:
            w = max(4, w & ~3)          # exact-2x width, w % 4 == 0: the warp-marching kernel
        if i % 9 == 0:
            w = max(8, w & ~7)          # 8-byte-aligned rows
        if i % 10 == 1:
            h, w = int(rng.integers(1, 6)), int(rng.integers(1, 12))
        shapes.append((h, w))
    imgs = [synth(9000 + i, h, w, "binary" if i % 5 == 0 else "uniform") for i, (h, w) in enumerate(shapes)]
    for lo in range(0, len(shapes), 40):
        sh, im = shapes[lo:lo + 40], imgs[lo:lo + 40]
        plan = CorruptionPlan.ragged(sh, align=4)
        src = torch_.from_numpy(plan.pack(im)).cuda()
        dst = torch_.zeros(plan.dst_bytes, dtype=torch_.uint8, device="cuda")
        plan.blur(src, dst)
        for i, out in enumerate(plan.unpack(dst.cpu().numpy())):
            assert np.array_equal(out, orc.apply_motion_blur(im[i], 9, 0)), ("blur", sh[i])
        plan.lowres(src, dst)
        for i, out in enumerate(plan.unpack(dst.cpu().numpy())):
            assert np.array_equal(out, orc.apply_lowres(im[i], 0.5)), ("lowres", sh[i])
        np.random.seed(lo)
        fields = [orc.draw_noise_field(x.shape, 15) for x in im]
        plan.noise(src, dst, torch_.from_numpy(np.concatenate([f.reshape(-1) for f in fields])).cuda(), 15.0)
        for i, out in enumerate(plan.unpack(dst.cpu().numpy())):
            assert np.array_equal(out, orc.add_noise_field(im[i], fields[i])), ("noise", sh[i])


def test_fused_letterbox_random_stress(torch_):
    """Random shapes / ops / output sizes through corrupt_letterbox (fused kernel with in-kernel LowRes for the all-even
    batch, scratch pre-pass for the mixed batch, unfused fallback when a letterbox degenerates), vs the oracle."""
    from robust_object_detection_b200.batch import CorruptionPlan
    rng = np.random.default_rng(777)
    for trial in range(6):
        n = 10
        even = trial % 2 == 0
        shapes = []
        for i in range(n):
            h, w = int(rng.integers(8, 260)), int(rng.integers(8, 340))
            if even:
                w = max(8, w & ~3)
            shapes.append((h, w))
        ops_host = rng.integers(0, 4, n).astype(np.uint8)
        ops_host[ops_host == 1] = 2 if trial % 3 else 1   # compat noise only in some trials
        oh, ow = [(96, 96), (128, 160), (64, 200)][trial % 3]
        imgs = [synth(9500 + 16 * trial + i, h, w) for i, (h, w) in enumerate(shapes)]
        plan = CorruptionPlan.ragged(shapes, align=4 if trial % 2 else 256)
        src = torch_.from_numpy(plan.pack(imgs)).cuda()
        np.random.seed(trial)
        fields = [orc.draw_noise_field(im.shape, 15) for im in imgs]
        nz = torch_.from_numpy(np.concatenate([f.reshape(-1) for f in fields])).cuda()
        out = torch_.empty((n, 3, oh, ow), dtype=torch_.float16, device="cuda")
        plan.corrupt_letterbox(src, torch_.from_numpy(ops_host).cuda(), out, oh, ow, 114, noise=nz)
        got = out.cpu().numpy()
        for i, img in enumerate(imgs):
            op = int(ops_host[i])
            cor = orc.add_noise_field(img, fields[i]) if op == 1 else orc.apply_op(img, op)
            assert np.array_equal(got[i], orc.letterbox_norm_f16(cor, oh, ow, 114)), (trial, i, shapes[i], op)


def test_jpeg_encoder_matches_cv2(torch_):
    """SURVEY 8f rank 1: the device JPEG encoder (rod_jpeg_encode) against cv2.imencode, byte for byte: a ragged batch of
    sizes that are not multiples of 8 / 16 (libjpeg's dummy blocks), uniform noise (long streams, 0xFF stuffing), smooth
    and constant content, a pitched layout, and the BASELINE frame size."""
    import cv2
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegEncoder
    shapes = [(16, 16), (8, 8), (1, 1), (37, 53), (64, 48), (17, 33), (100, 9), (9, 100), (120, 200), (97, 133), (38, 40),
              (765, 1360), (360, 480), (540, 960)]
    imgs = []
    for i, (h, w) in enumerate(shapes):
        kind = i % 4
        if kind == 0 or h * w > 100000:
            imgs.append(synth(9000 + i, h, w))
        elif kind == 1:
            imgs.append(cv2.GaussianBlur(synth(9100 + i, h, w), (0, 0), 2.5))
        elif kind == 2:
            imgs.append(np.full((h, w, 3), 255 if i % 8 == 2 else 0, np.uint8))
        else:
            imgs.append((synth(9200 + i, h, w) > 127).astype(np.uint8) * 255)
    plan = CorruptionPlan.ragged(shapes)
    dev = torch_.from_numpy(plan.pack(imgs)).cuda()
    enc = JpegEncoder(shapes, plan.src_offsets)
    for rep in range(2):   # a second run reuses the zeroed stream buffers
        files = enc.encode(dev)
        for i, (img, got) in enumerate(zip(imgs, files)):
            want = cv2.imencode(".jpg", img)[1].tobytes()
            assert got is not None and got == want, (rep, i, shapes[i], None if got is None else len(got), len(want))
    # pitched rows
    pitches = [3 * w + 5 for _, w in shapes]
    offs = np.concatenate([[0], np.cumsum([(h * q + 255) // 256 * 256 for (h, _), q in zip(shapes, pitches)])])
    host = np.full(int(offs[-1]), 0xAB, np.uint8)
    for img, o, q in zip(imgs, offs, pitches):
        h, w, _ = img.shape
        host[o:o + h * q].reshape(h, q)[:, :3 * w] = img.reshape(h, 3 * w)
    files = JpegEncoder(shapes, offs[:-1], pitches).encode(torch_.from_numpy(host).cuda())
    for i, (img, got) in enumerate(zip(imgs, files)):
        assert got == cv2.imencode(".jpg", img)[1].tobytes(), (i, shapes[i])


def test_jpeg_encoder_matches_golden(torch_):
    """The device JPEG encoder against the cv2.imencode hashes recorded in the build container (golden_jpeg.json)."""
    import hashlib
    import json
    import cv2
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegEncoder
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_jpeg.json")))
    imgs = []
    for seed, h, w, kind in g["cases"]:
        img = synth(seed, h, w)
        if kind == "smooth":
            img = cv2.GaussianBlur(img, (0, 0), 2.5)
        elif kind == "binary":
            img = (img > 127).astype(np.uint8) * 255
        imgs.append(img)
    shapes = [(h, w) for _, h, w, _ in g["cases"]]
    plan = CorruptionPlan.ragged(shapes)
    files = JpegEncoder(shapes, plan.src_offsets).encode(torch_.from_numpy(plan.pack(imgs)).cuda())
    for (seed, h, w, kind), f in zip(g["cases"], files):
        assert f is not None and hashlib.sha256(f).hexdigest() == g["sha"][f"{seed}_{h}x{w}_{kind}"], (seed, h, w, kind)


def test_jpeg_encoder_random_shapes_stress(torch_):
    """Device JPEG encoder on random shapes (1 .. 260 pixels per side, plus a few large odd ones) and content types, as one
    ragged batch, against cv2.imencode."""
    import cv2
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegEncoder
    rng = np.random.default_rng(77)
    shapes = [(int(rng.integers(1, 261)), int(rng.integers(1, 261))) for _ in range(40)] + [(1079, 1917), (1499, 1999), (15, 2001), (2001, 17)]
    imgs = []
    for i, (h, w) in enumerate(shapes):
        base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        kind = i % 3
        imgs.append(base if kind == 0 else cv2.GaussianBlur(base, (0, 0), 1.5 + (i % 5)) if kind == 1 else (base // 64) * 85)
    plan = CorruptionPlan.ragged(shapes)
    files = JpegEncoder(shapes, plan.src_offsets).encode(torch_.from_numpy(plan.pack(imgs)).cuda())
    for i, (img, got) in enumerate(zip(imgs, files)):
        want = cv2.imencode(".jpg", img)[1].tobytes()
        assert got is not None and got == want, (i, shapes[i], None if got is None else len(got), len(want))


def test_jpeg_decoder_matches_cv2(torch_):
    """Device JPEG decoder (row f1, the reading side: scripts/build_corrupted_testsets.py:109) on one ragged batch: files
    of many sizes, qualities and contents decode to the pixels of cv2.imdecode, straight into the layout of a CorruptionPlan;
    files of other layouts are reported per image and leave their slot untouched."""
    import cv2
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegDecoder, probe
    rng = np.random.default_rng(99)
    shapes = [(int(rng.integers(1, 261)), int(rng.integers(5, 261))) for _ in range(40)] + [(765, 1360), (1079, 1917), (1500, 2000), (15, 2001), (2001, 17)]
    files, want = [], []
    for i, (h, w) in enumerate(shapes):
        base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        kind = i % 3
        img = base if kind == 0 else cv2.GaussianBlur(base, (0, 0), 1.5 + (i % 5)) if kind == 1 else (base // 64) * 85
        params = [[], [cv2.IMWRITE_JPEG_QUALITY, int(rng.integers(10, 101))], [cv2.IMWRITE_JPEG_OPTIMIZE, 1]][(i // 3) % 3]
        if i % 7 == 4:     # 4:2:2, 4:4:4 and greyscale files among the 4:2:0 ones
            params = params + [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422]
        elif i % 7 == 5:
            params = params + [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]
        elif i % 7 == 6:
            img = np.ascontiguousarray(img[:, :, 1])
        if i % 4 == 1:     # restart markers (intervals of 1 .. 9 MCUs)
            params = params + [cv2.IMWRITE_JPEG_RST_INTERVAL, 1 + i % 9]
        enc = cv2.imencode(".jpg", img, params)[1]
        files.append(enc.tobytes())
        want.append(cv2.imdecode(enc, cv2.IMREAD_COLOR))
    odd = {3: cv2.imencode(".jpg", want[3], [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes(), 7: b"not a jpeg",
           11: cv2.imencode(".png", want[11])[1].tobytes(), 40: files[40][:len(files[40]) // 2]}
    for i, f in odd.items():
        files[i] = f
    sizes = [probe(f) for f in files]
    # probe() reads the header only: the file cut off inside its scan (40) is found out by the decoder's constructor
    assert all((sizes[i] is None) == (i in odd and i != 40) for i in range(len(files)))
    assert all(sizes[i] == shapes[i] for i in range(len(files)) if i not in odd)
    plan = CorruptionPlan.ragged(shapes)
    dec = JpegDecoder(files, plan.src_offsets, host_threads=4)
    assert dec.shapes == [None if i == 40 else sz for i, sz in enumerate(sizes)]
    pix = torch_.full((plan.src_bytes + 64,), 0xA5, dtype=torch_.uint8, device="cuda")
    dec.decode(pix)
    st = dec.status()
    assert [int(s) for s in st] == [0 if i not in odd else (12 if i == 3 else 13 if i == 40 else 11) for i in range(len(files))]
    got = pix.cpu().numpy()
    assert (got[plan.src_bytes:] == 0xA5).all()
    for i, ((h, w), off) in enumerate(zip(shapes, plan.src_offsets)):
        g = got[off:off + 3 * h * w].reshape(h, w, 3)
        if i in odd:
            assert (g == 0xA5).all(), i
        else:
            assert np.array_equal(g, want[i]), (i, shapes[i])
    # a stream that breaks off inside the entropy-coded data but still ends in EOI: reported by the device, not decoded
    bad = bytearray(files[0])
    scan = bytes(bad).index(b"\xff\xda")
    cut = bytes(bad[:scan + 14 + (len(bad) - scan) // 3]) + b"\xff\xd9"
    dec2 = JpegDecoder([cut, files[1]], [0, 3 * shapes[0][0] * shapes[0][1]])
    if dec2.shapes[0] is not None:
        pix2 = torch_.zeros(3 * (shapes[0][0] * shapes[0][1] + shapes[1][0] * shapes[1][1]), dtype=torch_.uint8, device="cuda")
        dec2.decode(pix2)
        st2 = dec2.status()
        assert int(st2[0]) in (1, 2) and int(st2[1]) == 0
        off = 3 * shapes[0][0] * shapes[0][1]
        assert np.array_equal(pix2.cpu().numpy()[off:].reshape(shapes[1][0], shapes[1][1], 3), want[1])


def test_jpeg_decoder_pitched_destination_guard_bytes(torch_):
    """The decoder writes image rows at the pitches it is given and nothing else: rows of a pitched destination keep their
    guard bytes (odd pitches: the colour kernel's 2-byte stores must fall back to byte stores on odd addresses)."""
    import cv2
    from robust_object_detection_b200.jpeg import JpegDecoder
    rng = np.random.default_rng(5)
    shapes, pads = [(37, 53), (64, 129), (9, 200), (120, 77)], [7, 0, 1, 32]
    files, want, offs, pitches, cur = [], [], [], [], 3
    for (h, w), pad in zip(shapes, pads):
        enc = cv2.imencode(".jpg", cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 1.2))[1]
        files.append(enc.tobytes())
        want.append(cv2.imdecode(enc, cv2.IMREAD_COLOR))
        offs.append(cur)
        pitches.append(3 * w + pad)
        cur += h * (3 * w + pad) + 5
    pix = torch_.full((cur + 16,), 0x5A, dtype=torch_.uint8, device="cuda")
    dec = JpegDecoder(files, offs, pitches)
    dec.decode(pix)
    assert (dec.status() == 0).all()
    got = pix.cpu().numpy()
    mask = np.ones(got.size, bool)
    for (h, w), off, pitch, img in zip(shapes, offs, pitches, want):
        rows = got[off:off + h * pitch].reshape(h, pitch)
        assert np.array_equal(rows[:, :3 * w].reshape(h, w, 3), img), (h, w)
        m = mask[off:off + h * pitch].reshape(h, pitch)
        m[:, :3 * w] = False
    assert (got[mask] == 0x5A).all()


def test_file_batcher_equals_frame_batcher(torch_, tmp_path):
    """FileCorruptionBatcher (JPEG files -> device decoder -> fused corrupt + letterbox) gives the tensor CorruptionBatcher
    gives for the cv2.imread frames of the same files, under the same random seed -- including a PNG and a progressive
    JPEG, which go through the host codec, and a file passed as bytes."""
    import random
    import cv2
    from robust_object_detection_b200.training import CorruptionBatcher, FileCorruptionBatcher
    rng = np.random.default_rng(12)
    shapes = [(765, 1360), (540, 960), (360, 480), (97, 133), (300, 180), (788, 1400)]
    paths = []
    for i, (h, w) in enumerate(shapes):
        img = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 1.0 + i % 3)
        p = tmp_path / (f"f{i}.png" if i == 3 else f"f{i}.jpg")
        cv2.imwrite(str(p), img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1] if i == 4 else [])
        paths.append(str(p))
    frames = [cv2.imread(p) for p in paths]
    batches = [paths[:3], paths[3:], [open(paths[0], "rb").read(), paths[5]]]
    frame_batches = [frames[:3], frames[3:], [frames[0], frames[5]]]
    random.seed(42)
    want = [x.cpu().numpy() for x in CorruptionBatcher(out_hw=(160, 160), seed=9).run(frame_batches)]
    random.seed(42)
    fb = FileCorruptionBatcher(out_hw=(160, 160), seed=9, io_threads=4)
    got = [x.cpu().numpy() for x in fb.run(batches)]
    assert len(got) == 3 and all(np.array_equal(g, w) for g, w in zip(got, want))
    random.seed(42)
    assert np.array_equal(FileCorruptionBatcher(out_hw=(160, 160), seed=9)(batches[0]).cpu().numpy(), want[0])
    with pytest.raises(IOError):
        fb([b"not an image"])


def test_restoration_pairs_from_files(torch_, tmp_path):
    """RestorationPairBatcher.from_files (files -> device JPEG decoder -> crops on the device) equals the batcher on the
    cv2.imread frames under the same seeds, incl. a frame smaller than the patch (resize-first branch) and a PNG."""
    import random
    import cv2
    from robust_object_detection_b200.training import RestorationPairBatcher
    rng = np.random.default_rng(13)
    shapes = [(300, 400), (765, 1360), (200, 180), (97, 300), (256, 256), (540, 960)]
    paths = []
    for i, (h, w) in enumerate(shapes):
        p = tmp_path / (f"r{i}.png" if i == 4 else f"r{i}.jpg")
        cv2.imwrite(str(p), cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (0, 0), 1.5))
        paths.append(str(p))
    frames = [cv2.imread(p) for p in paths]
    for is_train in (True, False):
        for noise in ("compat", "philox"):
            random.seed(7)
            np.random.seed(7)
            a = RestorationPairBatcher(patch_size=256, is_train=is_train, noise=noise, seed=3)
            want = a(frames)
            random.seed(7)
            np.random.seed(7)
            b = RestorationPairBatcher(patch_size=256, is_train=is_train, noise=noise, seed=3)
            got = b.from_files(paths)
            assert a.last_decisions == b.last_decisions
            assert torch_.equal(got[0], want[0]) and torch_.equal(got[1], want[1]), (is_train, noise)


def test_jpeg_decoder_matches_golden(torch_):
    """Device JPEG decoder against the files and pixel hashes recorded in the build container (golden_jpegdec.json)."""
    import base64
    import hashlib
    import json
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegDecoder
    g = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_jpegdec.json")))
    files = [base64.b64decode(c["file_b64"]) for c in g["cases"]]
    shapes = [tuple(c["shape"][:2]) for c in g["cases"]]
    plan = CorruptionPlan.ragged(shapes)
    dec = JpegDecoder(files, plan.src_offsets)
    assert dec.shapes == shapes
    pix = torch_.empty(plan.src_bytes, dtype=torch_.uint8, device="cuda")
    dec.decode(pix)
    assert (dec.status() == 0).all()
    got = pix.cpu().numpy()
    for c, (h, w), off in zip(g["cases"], shapes, plan.src_offsets):
        assert hashlib.sha256(got[off:off + 3 * h * w].tobytes()).hexdigest() == c["pixels_sha256"], c["name"]


def test_jpeg_codec_full_size_config4_round_trip(torch_):
    """Both halves of the device JPEG codec at the size of BASELINE config 4: 1610 VisDrone-shaped frames (8 frame sizes,
    same draw as bench.py) in one ragged batch are encoded on the device, the 1610 files are decoded back on the device.
    Parity at this size by replication: one distinct frame per size, so every file must equal cv2.imencode's file for that
    frame and every decoded frame cv2.imdecode's pixels of it (8 host codec runs instead of 1610)."""
    import cv2
    from robust_object_detection_b200.batch import CorruptionPlan
    from robust_object_detection_b200.jpeg import JpegDecoder, JpegEncoder
    pool = [(765, 1360), (1050, 1400), (788, 1400), (1078, 1916), (1080, 1920), (1500, 2000), (540, 960), (360, 480)]
    kinds = np.random.default_rng(4000).integers(0, 8, 1610)
    shapes = [pool[i] for i in kinds]
    base = [cv2.GaussianBlur(synth(9100 + i, h, w), (0, 0), 2.0) for i, (h, w) in enumerate(pool)]
    want_files = [cv2.imencode(".jpg", b)[1] for b in base]
    want_pixels = [torch_.from_numpy(cv2.imdecode(f, cv2.IMREAD_COLOR).reshape(-1)).cuda() for f in want_files]
    dbase = [torch_.from_numpy(b.reshape(-1)).cuda() for b in base]
    plan = CorruptionPlan.ragged(shapes)
    src = torch_.zeros(plan.src_bytes, dtype=torch_.uint8, device="cuda")
    for off, k in zip(plan.src_offsets, kinds):
        src[off:off + dbase[k].numel()] = dbase[k]
    files = JpegEncoder(shapes, plan.src_offsets).encode(src)
    for i in range(1610):
        assert files[i] is not None and files[i] == want_files[kinds[i]].tobytes(), i
    back = torch_.empty_like(src)
    dec = JpegDecoder(files, plan.src_offsets, host_threads=16)
    assert dec.shapes == shapes
    dec.decode(back)
    assert (dec.status() == 0).all()
    for i, (off, k) in enumerate(zip(plan.src_offsets, kinds)):
        assert torch_.equal(back[off:off + want_pixels[k].numel()], want_pixels[k]), i
