"""The device draw of compat noise (csrc/legacy_rng.cu, augmentations.legacy_normal_f32_device) against NumPy's legacy
stream.  CPU: the jump polynomials and a sequential replay of the chunked algorithm (tests/emu/legacy_rng_replay.cpp,
built with g++ from the kernels' rod_mt.h), and the float32 guard that decides which values the host recomputes.  GPU:
fields and the full generator state against np.random itself."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "emu", "legacy_rng_replay.cpp")
N_WORDS, STRIDE, MAX_CHUNKS = 624, 128, 256  # legacy_rng.cu kStride / kMaxChunks

u32p, i32p, dp, f32p, u64p = (ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_int32),
                              ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint64))


@pytest.fixture(scope="module")
def rep(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    out = str(tmp_path_factory.mktemp("mt") / "libreplay.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-frounding-math", "-shared", "-fPIC",
                           "-o", out, SRC])
    lib = ctypes.CDLL(out)
    lib.replay_jump.argtypes = [u32p, ctypes.c_uint64, u32p, ctypes.c_int, u32p]
    lib.replay_table_row.argtypes = [ctypes.c_int, ctypes.c_int, u64p]
    lib.replay_normal.argtypes = [u32p, i32p, i32p, dp, ctypes.c_double, ctypes.c_uint64, f32p, ctypes.c_int, ctypes.c_int]
    lib.replay_guard.argtypes = [u32p, ctypes.c_uint64, ctypes.c_double, u64p, u64p]
    lib.replay_log.argtypes = [dp, dp, ctypes.c_uint64]
    lib.replay_guard_ok.argtypes = [ctypes.c_double]
    return lib


def _p(a, t):
    return a.ctypes.data_as(ctypes.POINTER(t))


def _block_after(key, blocks):
    """Block `blocks` of the raw word stream from block 0 = key, by sequential generation in NumPy's own MT19937."""
    bg = np.random.MT19937()
    bg.state = {"bit_generator": "MT19937", "state": {"key": key.copy(), "pos": 624}}
    left = 624 * blocks
    while left:
        k = min(left, 1 << 22)
        bg.random_raw(k)
        left -= k
    return np.array(bg.state["state"]["key"], dtype=np.uint32)


def _key(seed):
    return np.array(np.random.RandomState(seed).get_state()[1], dtype=np.uint32)


# ------------------------------------------------------------------------------------------------ CPU
def test_characteristic_polynomial_degree(rep):
    assert rep.replay_phi_degree() == 19937


@pytest.mark.parametrize("blocks", [1, STRIDE, MAX_CHUNKS * STRIDE - STRIDE])
def test_jump_equals_sequential_generation(rep, blocks):
    """The window at distance `blocks` blocks is exact but for the low 31 bits of its word 0; a chunk start (jump to the
    block before, generate one) is the exact block, key[0] included.  The largest distance is the last table row's."""
    for seed in (0, 7, 12345):
        key = _key(seed)
        want = _block_after(key, blocks)
        window, block = np.zeros(624, np.uint32), np.zeros(624, np.uint32)
        rep.replay_jump(_p(key, ctypes.c_uint32), 624 * blocks, _p(window, ctypes.c_uint32), blocks, _p(block, ctypes.c_uint32))
        assert np.array_equal(window[1:], want[1:]) and (window[0] >> 31) == (want[0] >> 31), (seed, blocks)
        assert np.array_equal(block, want), (seed, blocks)


def test_table_rows_are_the_chunk_distances(rep):
    """Row c of the table (built by chaining multiplications) reaches the same block as a direct jump."""
    key = _key(3)
    row = np.zeros(312, np.uint64)
    for c in (1, 2, 5):
        rep.replay_table_row(STRIDE, c, _p(row, ctypes.c_uint64))
        direct, block = np.zeros(624, np.uint32), np.zeros(624, np.uint32)
        rep.replay_jump(_p(key, ctypes.c_uint32), 624 * (c * STRIDE - 1), _p(direct, ctypes.c_uint32), c * STRIDE, _p(block, ctypes.c_uint32))
        assert np.array_equal(block, _block_after(key, c * STRIDE))


def _replay(rep, sigma, n, stride=STRIDE, max_chunks=MAX_CHUNKS):
    st = np.random.get_state(legacy=True)
    key = np.array(st[1], dtype=np.uint32)
    pos, has, cached = ctypes.c_int32(int(st[2])), ctypes.c_int32(int(st[3])), ctypes.c_double(float(st[4]))
    out = np.full(max(n, 1), np.nan, np.float32)
    rep.replay_normal(_p(key, ctypes.c_uint32), ctypes.byref(pos), ctypes.byref(has), ctypes.byref(cached), float(sigma), n,
                      _p(out, ctypes.c_float), stride, max_chunks)
    return out[:n], ("MT19937", key, pos.value, has.value, cached.value)


def _same_state(a, b):
    return a[0] == b[0] and np.array_equal(np.asarray(a[1]), np.asarray(b[1])) and a[2:] == b[2:]


SIZES = [0, 1, 2, 3, 623, 624, 625, 5001, 6000]
ENTRY = ["seed", "pos1", "pos623", "pos624", "gauss"]


def _enter(kind, seed):
    """Entry states: fresh seed (pos 624), pos 1 / 623 within the key, and a cached Gaussian."""
    np.random.seed(seed)
    if kind in ("pos1", "pos623"):
        np.random.random_sample(1)  # a fresh block
        st = list(np.random.get_state(legacy=True))
        st[2] = 1 if kind == "pos1" else 623
        np.random.set_state(tuple(st))
    elif kind == "pos624":
        np.random.random_sample(312)  # 624 words: the key is used up
    elif kind == "gauss":
        np.random.standard_normal(3)


@pytest.mark.parametrize("sigma", [15.0, 2.5, 0.0])
@pytest.mark.parametrize("kind", ENTRY)
def test_replay_matches_numpy(rep, sigma, kind):
    for n in SIZES:
        _enter(kind, 100 + n)
        before = np.random.get_state(legacy=True)
        got, state = _replay(rep, sigma, n)
        np.random.set_state(before)
        want = np.random.normal(0, sigma, n).astype(np.float32)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (kind, n, sigma)
        assert _same_state(state, np.random.get_state(legacy=True)), (kind, n, sigma)


@pytest.mark.parametrize("stride,max_chunks", [(2, 3), (2, 256), (3, 1)])
def test_replay_small_chunks_and_rounds(rep, stride, max_chunks):
    """Chunks of 2-3 blocks and 1-3 chunks per round: candidates straddle chunk ends (a chunk owns the candidates that
    start in it) and most calls take several rounds."""
    for kind in ENTRY:
        for n in (1, 625, 2001, 4000, 30001):
            _enter(kind, 7 * n)
            before = np.random.get_state(legacy=True)
            got, state = _replay(rep, 15.0, n, stride, max_chunks)
            np.random.set_state(before)
            want = np.random.normal(0, 15.0, n).astype(np.float32)
            assert np.array_equal(got, want), (kind, n, stride, max_chunks)
            assert _same_state(state, np.random.get_state(legacy=True)), (kind, n, stride, max_chunks)


@pytest.mark.parametrize("sigma", [15.0, 2.5, 1e-3])
def test_guard_flags_every_value_a_two_ulp_log_changes(rep, sigma):
    """Over the stream: a log() 1 or 2 ulps off changes no unflagged output, and some values are flagged."""
    changed, flagged = ctypes.c_uint64(), ctypes.c_uint64()
    missed = rep.replay_guard(_p(_key(11), ctypes.c_uint32), 1 << 22, sigma, ctypes.byref(changed), ctypes.byref(flagged))
    assert missed == 0
    assert changed.value <= flagged.value and flagged.value > 0


def test_guard_near_float_rounding_boundaries(rep):
    """Such changes are rare on the stream, so also directly: doubles within 2^-49 relative of a float32 rounding
    boundary (the most a 2-ulp log error moves an output) are flagged; a double equal to a float32 is not."""
    rng = np.random.default_rng(4)
    vals = np.concatenate([rng.normal(0, 15, 2000), rng.normal(0, 1e-3, 200), [1e-42, 3e38, -3.4e38]]).astype(np.float32)
    for v in vals:
        up = np.nextafter(v, np.float32(np.inf))
        mid = (float(v) + float(up)) / 2.0  # the boundary between v and its neighbour
        for rel in (0.0, 2.0 ** -52, -(2.0 ** -52), 2.0 ** -49, -(2.0 ** -49)):
            assert rep.replay_guard_ok(mid * (1.0 + rel)) == 0, (v, rel)
        if np.isfinite(v) and abs(float(v)) > 1e-37:
            assert rep.replay_guard_ok(float(v)) == 1, v


# ------------------------------------------------------------------------------------------------ GPU
def _device_draw(sigma, total, spans, guard=np.float32(-777.25)):
    import torch
    from robust_object_detection_b200 import augmentations as aug
    out = torch.full((total,), float(guard), dtype=torch.float32, device="cuda")
    fix = aug.legacy_normal_f32_device(sigma, out, spans)
    return out.cpu().numpy(), fix


def _check_device(sigma, spans, total, guard=np.float32(-777.25)):
    from robust_object_detection_b200 import augmentations as aug  # noqa: F401
    before = np.random.get_state(legacy=True)
    got, fix = _device_draw(sigma, total, spans, guard)
    after = np.random.get_state(legacy=True)
    np.random.set_state(before)
    n = sum(c for _, c in spans)
    want = np.random.normal(0, sigma, n).astype(np.float32)
    assert _same_state(after, np.random.get_state(legacy=True))
    mask = np.zeros(total, bool)
    k = 0
    for o, c in spans:
        assert np.array_equal(got[o:o + c].view(np.uint32), want[k:k + c].view(np.uint32)), (o, c)
        mask[o:o + c] = True
        k += c
    assert (got[~mask] == guard).all()  # nothing written between segments
    return fix


@pytest.mark.gpu
@pytest.mark.parametrize("sigma", [15.0, 2.5, 0.0])
@pytest.mark.parametrize("kind", ENTRY)
def test_device_sizes_and_states(sigma, kind):
    for n in SIZES + [10 ** 5 + 1]:
        _enter(kind, 100 + n)
        _check_device(sigma, [(3, n)], n + 7)
        _enter(kind, 200 + n)
        a = n // 3
        _check_device(sigma, [(0, a), (a + 5, 0), (a + 5, n - a)], n + 9)  # a gap, an empty span


@pytest.mark.gpu
def test_device_full_fields_and_rounds():
    """One 1360x765x3 field; 16 of them as 16 segments in one call (more than one round: a round covers 256 x 128
    blocks); the stream continues exactly afterwards; the host fix-ups occur and are right."""
    f = 1360 * 765 * 3
    np.random.seed(42)
    _check_device(15.0, [(0, f)], f)
    np.random.standard_normal(1)  # a cached Gaussian
    spans = [(i * (f + 64), f) for i in range(16)]
    fix = _check_device(15.0, spans, 16 * (f + 64))
    assert fix > 0
    np.random.random(3)
    _check_device(15.0, [(1, 5)], 8)


@pytest.mark.gpu
def test_device_interleaved_consumers():
    from robust_object_detection_b200 import augmentations as aug  # noqa: F401
    np.random.seed(5)
    for step in range(12):
        np.random.random(step)
        np.random.randint(0, 1000, step * 3 + 1)
        if step % 3 == 0:
            np.random.standard_normal(1)
        _check_device(15.0 if step % 2 else 2.5, [(0, 997 * step + 1), (997 * step + 50, 3 + step)], 997 * step + 60 + step)


@pytest.mark.gpu
def test_device_arguments_and_negative_sigma():
    import torch
    from robust_object_detection_b200 import augmentations as aug
    out = torch.zeros(16, dtype=torch.float32, device="cuda")
    np.random.seed(1)
    before = np.random.get_state(legacy=True)
    with pytest.raises(ValueError):
        aug.legacy_normal_f32_device(-1.0, out, [(0, 4)])
    assert _same_state(before, np.random.get_state(legacy=True))
    with pytest.raises(ValueError):
        aug.legacy_normal_f32_device(15.0, out, [(8, 4), (0, 4)])  # unsorted
    with pytest.raises(ValueError):
        aug.legacy_normal_f32_device(15.0, out, [(0, 6), (4, 4)])  # overlapping
    with pytest.raises(ValueError):
        aug.legacy_normal_f32_device(15.0, out, [(10, 8)])  # outside
    assert _same_state(before, np.random.get_state(legacy=True))
    assert aug.legacy_normal_f32_device(15.0, out, []) == 0
    assert _same_state(before, np.random.get_state(legacy=True))


@pytest.mark.gpu
def test_device_log_within_guard_bound(rep):
    """CUDA's double log() against libm's over 2^24 r2 values of the generator: at most 2 ulps apart (the guard's bound)."""
    import torch
    np.random.seed(9)
    d = np.random.random_sample(2 * 22_000_000)  # the doubles the polar method turns into x1, x2 (~78.5 % accepted)
    x = 2.0 * d - 1.0
    r2 = x[0::2] * x[0::2] + x[1::2] * x[1::2]
    r2 = r2[(r2 < 1.0) & (r2 != 0.0)][:1 << 24]
    assert r2.size == 1 << 24
    host = np.empty_like(r2)
    rep.replay_log(_p(r2, ctypes.c_double), _p(host, ctypes.c_double), r2.size)
    dev = torch.log(torch.from_numpy(r2).cuda()).cpu().numpy()
    ulps = np.abs(dev.view(np.int64) - host.view(np.int64))
    assert ulps.max() <= 2, int(ulps.max())
