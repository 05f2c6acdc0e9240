"""Progressive JPEG files through the device decoder (csrc/rod_jpegdec.h decode_prog_segment, csrc/jpegdec.cu).

CPU: a sequential replay of the decoder (tests/emu/jpegdec_progressive_replay.cpp, built with g++ from the product's
headers: parser, scan levels, the four progressive MCU decoders, the baseline IDCT / colour functions) against
cv2.imdecode on files written by OpenCV and PIL, and on files a small progressive writer in the same harness re-encodes
under other scan scripts; the files that must be reported; the probe contract.  GPU: a ragged mixed batch against
cv2.imdecode."""
import ctypes
import io
import os
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "emu", "jpegdec_progressive_replay.cpp")
LIB = os.path.join(ROOT, "robust-object-detection_b200", "librod_b200.so")

cv2 = pytest.importorskip("cv2")


@pytest.fixture(scope="module")
def rep(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    out = str(tmp_path_factory.mktemp("progjpeg") / "libreplay.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, SRC])
    lib = ctypes.CDLL(out)
    vp = ctypes.c_void_p
    lib.replay_decode.argtypes = [vp, ctypes.c_long, vp, ctypes.c_long, vp, ctypes.c_int]
    lib.replay_write.argtypes = [vp, ctypes.c_long, vp, ctypes.c_int, vp, ctypes.c_long]
    lib.replay_write.restype = ctypes.c_long
    return lib


@pytest.fixture(scope="module")
def built():
    if not os.path.exists(LIB):
        import __graft_entry__ as g
        g.build()
    return LIB


def _decode(rep, data, poison=1):
    """(status, HWC BGR pixels or None, progressive?) of the replayed device decoder."""
    buf = np.frombuffer(bytes(data), np.uint8)
    hw = np.zeros(3, np.int32)
    out = np.zeros(3 * 2048 * 2048, np.uint8)
    rc = rep.replay_decode(buf.ctypes.data, buf.size, out.ctypes.data, out.size, hw.ctypes.data, poison)
    img = out[:hw[0] * hw[1] * 3].reshape(hw[0], hw[1], 3).copy() if rc == 0 else None
    return rc, img, bool(hw[2])


def _write(rep, baseline, script):
    """The coefficients of `baseline` re-encoded as a progressive file under `script` (rows of 10 ints)."""
    buf = np.frombuffer(bytes(baseline), np.uint8)
    s = np.ascontiguousarray(np.array(script, np.int32).reshape(-1, 10))
    out = np.zeros(len(buf) * 16 + (1 << 20), np.uint8)   # (fixed-length codes: larger than the input)
    n = rep.replay_write(buf.ctypes.data, buf.size, s.ctypes.data, len(s), out.ctypes.data, out.size)
    assert n > 0, n
    return out[:n].tobytes()


def _imdecode(data):
    return cv2.imdecode(np.frombuffer(bytes(data), np.uint8), cv2.IMREAD_COLOR)


def _content(rng, h, w, kind):
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        img = cv2.GaussianBlur(img, (0, 0), 2.0)
    elif kind == 2:
        img[:] = rng.integers(0, 256, 3, dtype=np.uint8)
    elif kind == 3:
        img = cv2.GaussianBlur(img, (0, 0), 0.7)
    return img


LAYOUTS = {"420": [], "422": [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422],
           "444": [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444], "grey": []}


def _cv2_pair(img, layout, params):
    """(progressive file, its baseline twin) as OpenCV writes them."""
    if layout == "grey":
        img = np.ascontiguousarray(img[:, :, 0])
    p = list(params) + LAYOUTS[layout]
    prog = cv2.imencode(".jpg", img, p + [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    base = cv2.imencode(".jpg", img, p)[1].tobytes()
    return prog, base


def _sos_positions(data):
    """Byte offsets of the SOS markers of a file (walking the segments and the entropy-coded data)."""
    out, i = [], 2
    while i + 4 <= len(data):
        m = data[i + 1]
        if m == 0xD9:
            break
        L = (data[i + 2] << 8) | data[i + 3]
        if m != 0xDA:
            i += 2 + L
            continue
        out.append(i)
        i += 2 + L
        while i + 1 < len(data) and not (data[i] == 0xFF and data[i + 1] not in (0x00, 0xFF) and not 0xD0 <= data[i + 1] <= 0xD7):
            i += 1
    return out


# scan scripts: rows (ncomp, comp0, comp1, comp2, Ss, Se, Ah, Al, table slot, restart interval)
def _script(kind, ncomp):
    dc_all = [ncomp, 0, 1, 2] if ncomp == 3 else [1, 0, 0, 0]
    chroma = [1, 2] if ncomp == 3 else []
    if kind == "spectral":     # spectral selection only: Ah = Al = 0 everywhere
        rows = [dc_all + [0, 0, 0, 0, 0, 0], [1, 0, 0, 0, 1, 5, 0, 0, 0, 0], [1, 0, 0, 0, 6, 63, 0, 0, 1, 0]]
        rows += [[1, c, 0, 0, 1, 63, 0, 0, c % 2, 0] for c in chroma]
    elif kind == "deep":       # successive approximation from Al = 3 down to 0 for DC and AC
        rows = [dc_all + [0, 0, 0, 3, 0, 0]] + [[1, c, 0, 0, 1, 63, 0, 3, 1, 0] for c in [0] + chroma]
        for ah in (3, 2, 1):
            rows.append(dc_all + [0, 0, ah, ah - 1, 0, 0])
            rows += [[1, c, 0, 0, 1, 63, ah, ah - 1, 1, 0] for c in [0] + chroma]
    elif kind == "bands":      # one DC scan per component, chroma first; the luma AC split into four bands
        rows = [[1, c, 0, 0, 0, 0, 0, 0, 0, 0] for c in chroma[::-1] + [0]]
        rows += [[1, c, 0, 0, 1, 63, 0, 1, 1, 0] for c in chroma]
        rows += [[1, 0, 0, 0, a, b, 0, 0, 0, 0] for a, b in ((1, 2), (3, 9), (10, 30), (31, 63))]
        rows += [[1, c, 0, 0, 1, 63, 1, 0, 1, 0] for c in chroma]
    else:                      # "restart": restart intervals in non-interleaved scans, table slots 2 and 3
        rows = [dc_all + [0, 0, 0, 1, 2, 2], [1, 0, 0, 0, 1, 63, 0, 1, 3, 5]]
        rows += [[1, c, 0, 0, 1, 63, 0, 0, 2 + c % 2, c + 1] for c in chroma]
        rows += [dc_all + [0, 0, 1, 0, 0, 3], [1, 0, 0, 0, 1, 63, 1, 0, 3, 7]]
    return rows


SCRIPTS = ("spectral", "deep", "bands", "restart")


# ------------------------------------------------------------------------------------------------------------ CPU tests
def test_replay_matches_cv2_on_cv2_files(rep):
    """OpenCV's progressive files: every size of the baseline decoder's small grid (heights from 1, widths from 5), three
    VisDrone frame sizes, 4:2:0 / 4:2:2 / 4:4:4 / greyscale, qualities 5..100, restart intervals 1..9.  The pixels equal
    cv2.imdecode's of the file and of its baseline twin; coefficient blocks no scan reaches are poisoned first and must
    not show (the colour stage never reads them)."""
    rng = np.random.default_rng(21)
    cases = [(h, w) for h in (1, 2, 3, 7, 8, 9, 15, 16, 17, 31, 33) for w in (5, 6, 7, 8, 9, 15, 16, 17, 18, 31, 32, 33, 47, 65)]
    cases += [(765, 1360), (1078, 1916), (540, 960)]
    for i, (h, w) in enumerate(cases):
        layout = ("420", "422", "444", "grey")[i % 4]
        params = [cv2.IMWRITE_JPEG_QUALITY, int((5, 40, 75, 95, 100)[(i // 4) % 5])]
        if i % 3 == 1:
            params += [cv2.IMWRITE_JPEG_RST_INTERVAL, 1 + i % 9]
        prog, base = _cv2_pair(_content(rng, h, w, i % 4), layout, params)
        rc, got, is_prog = _decode(rep, prog)
        assert rc == 0 and is_prog, (h, w, layout, params, rc)
        want = _imdecode(prog)
        assert np.array_equal(got, want), (h, w, layout, params)
        assert np.array_equal(want, _imdecode(base)), (h, w, layout, params)


def test_replay_matches_cv2_on_pil_files(rep):
    """PIL's progressive writer, with and without optimised tables, 4:2:0 / 4:4:4 / greyscale, small and odd sizes."""
    from PIL import Image
    rng = np.random.default_rng(22)
    for i, (h, w) in enumerate([(1, 9), (5, 33), (17, 18), (97, 133), (240, 321), (765, 1360)]):
        for optimize in (False, True):
            for mode, sub in (("RGB", 2), ("RGB", 0), ("L", 0)):
                arr = _content(rng, h, w, 1 + i % 3)
                im = Image.fromarray(arr if mode == "RGB" else arr[:, :, 0])
                buf = io.BytesIO()
                im.save(buf, "JPEG", progressive=True, optimize=optimize, quality=int(rng.integers(40, 96)), subsampling=sub)
                data = buf.getvalue()
                rc, got, is_prog = _decode(rep, data)
                assert rc == 0 and is_prog, (h, w, optimize, mode, rc)
                assert np.array_equal(got, _imdecode(data)), (h, w, optimize, mode)


def test_written_scripts_match_cv2(rep):
    """Scan scripts OpenCV and PIL never write, re-encoded from baseline files by the harness's writer: spectral
    selection only; DC and AC successive approximation from Al = 3; one DC scan per component, chroma first, luma AC in
    four bands; restart intervals in non-interleaved scans with table slots 2 and 3.  cv2.imdecode of every written file
    equals that of the baseline file (the writer is right), and so does the replayed decoder."""
    rng = np.random.default_rng(23)
    n = 0
    for i, (h, w) in enumerate([(1, 5), (9, 17), (33, 47), (120, 161), (765, 1360)]):
        for layout in ("420", "422", "444", "grey"):
            _, base = _cv2_pair(_content(rng, h, w, 1 + (i + n) % 3), layout, [cv2.IMWRITE_JPEG_QUALITY, 90])
            want = _imdecode(base)
            for kind in SCRIPTS:
                f = _write(rep, base, _script(kind, 1 if layout == "grey" else 3))
                assert np.array_equal(_imdecode(f), want), (h, w, layout, kind)
                rc, got, is_prog = _decode(rep, f)
                assert rc == 0 and is_prog and np.array_equal(got, want), (h, w, layout, kind, rc)
                n += 1
    assert n == 80


def _default_prog(seed=30, h=64, w=96):
    rng = np.random.default_rng(seed)
    return cv2.imencode(".jpg", _content(rng, h, w, 3), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()


def test_reported_files(rep):
    """Files the decoder must report, never approximate: 12 for a file cut after its sixth scan (coefficient bits left
    unknown: libjpeg would block-smooth), a bogus progression (Ah not the previous Al), a DQT that redefines a table in
    use between scans; 1 / 2 / 13 for corrupt or truncated data in a refinement scan."""
    f = _default_prog()
    sos = _sos_positions(f)
    assert len(sos) == 10
    assert _decode(rep, f)[0] == 0
    assert _decode(rep, f[:sos[6]] + b"\xff\xd9")[0] == 12
    bogus = bytearray(f)
    ahal = sos[5] + 2 + ((f[sos[5] + 2] << 8) | f[sos[5] + 3]) - 1   # the Ah / Al byte of scan 6 (luma 1..63, 2 -> 1)
    assert bogus[ahal] == 0x21
    bogus[ahal] = 0x32
    assert _decode(rep, bytes(bogus))[0] == 12
    i, dqt = 2, None
    while dqt is None:
        L = (f[i + 2] << 8) | f[i + 3]
        if f[i + 1] == 0xDB:
            dqt = f[i:i + 2 + L]
        i += 2 + L
    assert _decode(rep, f[:sos[1]] + dqt + f[sos[1]:])[0] == 12
    # the last scan (luma refinement 1 -> 0): its data overwritten / cut short
    last = sos[9] + 2 + ((f[sos[9] + 2] << 8) | f[sos[9] + 3])
    bad = bytearray(f)
    bad[last:len(f) - 2] = bytes([0xFE]) * (len(f) - 2 - last)
    assert _decode(rep, bytes(bad))[0] in (1, 2)
    assert _decode(rep, f[:last + (len(f) - last) // 3] + b"\xff\xd9")[0] in (1, 2)
    assert _decode(rep, f[:last + (len(f) - last) // 3])[0] == 13


def test_probe_contract(built):
    """probe(f) keeps its contract (None for a progressive file); probe(f, progressive=True) is the frame size; a
    progressive file the decoder must report stays None either way."""
    from robust_object_detection_b200.jpeg import probe, sizes_of
    f = _default_prog(31, 57, 203)
    assert probe(f) is None
    assert probe(f, progressive=True) == (57, 203)
    sos = _sos_positions(f)
    assert probe(f[:sos[6]] + b"\xff\xd9", progressive=True) is None
    base = cv2.imencode(".jpg", np.zeros((8, 9, 3), np.uint8))[1].tobytes()
    assert sizes_of([base, f], progressive=True) == [(8, 9), (57, 203)]
    assert sizes_of([base, f]) == [(8, 9), None]


# ------------------------------------------------------------------------------------------------------------ GPU tests
def _is_progressive(data):
    i = 2
    while i + 4 <= len(data) and data[i] == 0xFF:
        if data[i + 1] == 0xC2:
            return True
        if data[i + 1] == 0xDA:
            return False
        i += 2 + ((data[i + 2] << 8) | data[i + 3])
    return False


@pytest.mark.gpu
def test_ragged_mixed_batch_matches_cv2(rep, built):
    """One batch of baseline and progressive files of random shapes and layouts (OpenCV, PIL, the four written scripts)
    plus files the decoder reports, decoded into a pitched destination with guard bytes: pixels equal cv2.imdecode's,
    reported slots and guard bytes keep their fill, and the trace shows the progressive Huffman kernel ran."""
    import torch
    from PIL import Image
    from robust_object_detection_b200.jpeg import JpegDecoder
    rng = np.random.default_rng(40)
    files = []
    for i in range(48):
        h, w = int(rng.integers(1, 400)), int(rng.integers(5, 600))
        layout = ("420", "422", "444", "grey")[i % 4]
        params = [cv2.IMWRITE_JPEG_QUALITY, int(rng.integers(20, 101))]
        if i % 5 == 0:
            params += [cv2.IMWRITE_JPEG_RST_INTERVAL, int(rng.integers(1, 10))]
        prog, base = _cv2_pair(_content(rng, h, w, i % 4), layout, params)
        files.append(prog if i % 2 == 0 else base)
        if i % 6 == 1:
            buf = io.BytesIO()
            Image.fromarray(_content(rng, h, w, 1)).save(buf, "JPEG", progressive=True, optimize=bool(i % 4 == 1))
            files.append(buf.getvalue())
        if i % 8 == 3:
            files.append(_write(rep, base, _script(SCRIPTS[(i // 8) % 4], 1 if layout == "grey" else 3)))
    _, base = _cv2_pair(_content(rng, 765, 1360, 3), "420", [cv2.IMWRITE_JPEG_QUALITY, 95])
    files += [_write(rep, base, _script(k, 3)) for k in SCRIPTS]
    f = _default_prog()
    reported = {len(files): 12, len(files) + 1: 11}
    files += [f[:_sos_positions(f)[6]] + b"\xff\xd9", cv2.imencode(".png", np.zeros((9, 9, 3), np.uint8))[1].tobytes()]
    want = [_imdecode(d) if i not in reported else None for i, d in enumerate(files)]
    assert sum(_is_progressive(d) for d in files) >= 30 and sum(not _is_progressive(d) for d in files) >= 20
    shapes = [(w_.shape[0], w_.shape[1]) if w_ is not None else (9, 9) for w_ in want]
    offs, pitches, cur = [], [], 5
    for (h, w) in shapes:
        offs.append(cur)
        pitches.append(3 * w + int(rng.integers(0, 9)))
        cur += h * pitches[-1] + int(rng.integers(0, 40))
    pix = torch.full((cur + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    dec = JpegDecoder(files, offs, pitches, host_threads=4, progressive=True)
    assert [int(s) for s in dec.host_status] == [reported.get(i, 0) for i in range(len(files))]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        dec.decode(pix)
        st = dec.status()
        torch.cuda.synchronize()
    assert [int(s) for s in st] == [reported.get(i, 0) for i in range(len(files))]
    names = {e.name for e in prof.events()}
    assert any("jpegdec_prog_kernel" in n for n in names), sorted(names)
    assert any("jpegdec_write_kernel" in n for n in names)
    got = pix.cpu().numpy()
    mask = np.ones(got.size, bool)
    for i, ((h, w), off, pitch) in enumerate(zip(shapes, offs, pitches)):
        if i in reported:
            continue
        rows = got[off:off + h * pitch].reshape(h, pitch)
        assert np.array_equal(rows[:, :3 * w].reshape(h, w, 3), want[i]), (i, h, w, _is_progressive(files[i]))
        mask[off:off + h * pitch].reshape(h, pitch)[:, :3 * w] = False
    assert (got[mask] == 0x5A).all()
