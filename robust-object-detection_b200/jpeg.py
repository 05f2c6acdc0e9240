"""Device-side JPEG encoding whose files equal cv2.imwrite's byte for byte, and device-side JPEG decoding whose pixels
equal cv2.imread's (SURVEY 8f rank 1): baseline files, and with progressive=True progressive ones.

`cv2.imwrite(str(dst_img_dir / img_path.name), out)` (scripts/build_corrupted_testsets.py:124, :164) is the last step of
the test-set build; with the corruption on the GPU it is what the build spends its time in.  JpegEncoder encodes a
device-resident batch (HWC BGR uint8, the layout of a CorruptionPlan) with rod_jpeg_encode: OpenCV 4.13's own parameters
(libjpeg-turbo defaults: YCbCr 4:2:0, quality 95, standard Huffman tables, islow DCT), its own header bytes (taken from
cv2.imencode on the host, per image size) and entropy-coded data that is bit-identical to libjpeg-turbo's.  No CPU
fallback inside: an image whose stream does not fit its device buffer comes back as None and the caller decides."""
from __future__ import annotations

import ctypes
import threading
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N
from .batch import _ptr, _stream_handle

_HEADER_TEMPLATE = None
_TLS = threading.local()   # per-thread ring of three page-locked download buffers, grow-only (pinning costs ~0.3 s per GB)


def _download_buffer(nbytes: int):
    """The next buffer of the calling thread's ring.  Views handed out by encode(copy=False) stay valid until the third
    following encode() call on the same thread."""
    import torch
    ring = getattr(_TLS, "ring", None)
    if ring is None:
        ring = _TLS.ring = [None, None, None]
        _TLS.turn = 0
    _TLS.turn = (_TLS.turn + 1) % 3
    t = ring[_TLS.turn]
    if t is None or t.numel() < nbytes:
        t = ring[_TLS.turn] = torch.empty(max(int(nbytes) * 5 // 4, 1 << 20), dtype=torch.uint8).pin_memory()
    return t


def _header_template() -> bytes:
    """SOI .. SOS as OpenCV writes them with its default parameters (the tables do not depend on the image size)."""
    global _HEADER_TEMPLATE
    if _HEADER_TEMPLATE is None:
        import cv2
        ok, buf = cv2.imencode(".jpg", np.zeros((16, 16, 3), np.uint8))
        if not ok:
            raise RuntimeError("cv2.imencode failed")
        b = buf.tobytes()
        i = 2
        while True:
            if b[i] != 0xFF:
                raise RuntimeError("unexpected JPEG header layout")
            seg = (b[i + 2] << 8) | b[i + 3]
            if b[i + 1] == 0xDA:
                _HEADER_TEMPLATE = b[:i + 2 + seg]
                break
            i += 2 + seg
    return _HEADER_TEMPLATE


def header_for(h: int, w: int) -> bytes:
    """The template with the frame size of SOF0 set to h x w."""
    t = bytearray(_header_template())
    i = 2
    while t[i + 1] != 0xC0:
        i += 2 + ((t[i + 2] << 8) | t[i + 3])
    t[i + 5:i + 9] = bytes([h >> 8, h & 255, w >> 8, w & 255])
    return bytes(t)


class JpegEncoder:
    """Encoder for one batch layout: images of `shapes` at byte `offsets` (row pitch 3 * w unless `pitches` is given)."""

    def __init__(self, shapes: Sequence[Tuple[int, int]], offsets: Sequence[int], pitches: Optional[Sequence[int]] = None):
        N.require_device()
        n = len(shapes)
        descs = (N.ImageDesc * n)()
        for i, (h, w) in enumerate(shapes):
            descs[i].src_offset = descs[i].dst_offset = int(offsets[i])
            descs[i].height, descs[i].width = int(h), int(w)
            descs[i].src_pitch = descs[i].dst_pitch = int(pitches[i]) if pitches is not None else 3 * int(w)
        hdr = _header_template()
        hbuf = (ctypes.c_uint8 * len(hdr)).from_buffer_copy(hdr)
        handle = ctypes.c_void_p()
        N.check(N.lib().rod_jpeg_create(descs, n, hbuf, len(hdr), ctypes.byref(handle)), "rod_jpeg_create")
        self._h = handle
        self.shapes = [(int(h), int(w)) for h, w in shapes]
        self.n_images = n
        self._off = [int(N.lib().rod_jpeg_stream_offset(handle, i)) for i in range(n + 1)]

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                N.lib().rod_jpeg_destroy(h)
            except Exception:
                pass
            self._h = None

    def encode(self, pixels, stream=None, copy: bool = True) -> List[Optional[object]]:
        """pixels: CUDA uint8 tensor holding the batch.  Returns one complete JPEG file per image -- `bytes`, or with
        copy=False a (header bytes, uint8 array view into a page-locked buffer) pair that is valid until the third following
        encode() call of this thread -- and None where the encoded stream did not fit its device buffer."""
        st = _stream_handle(stream)
        N.check(N.lib().rod_jpeg_encode(self._h, _ptr(pixels), st), "rod_jpeg_encode")
        hbuf = _download_buffer(self._off[-1])
        lens = np.zeros(self.n_images, dtype=np.uint32)
        N.check(N.lib().rod_jpeg_download(self._h, hbuf.data_ptr(), lens.ctypes.data, st), "rod_jpeg_download")
        host = hbuf.numpy()
        out: List[Optional[object]] = []
        for i, (h, w) in enumerate(self.shapes):
            n = int(lens[i])
            if n == 0xFFFFFFFF:
                out.append(None)
            elif copy:
                out.append(header_for(h, w) + host[self._off[i]:self._off[i] + n].tobytes())
            else:
                out.append((header_for(h, w), host[self._off[i]:self._off[i] + n]))
        return out


def _formats(progressive: bool) -> int:
    return N.JPEGDEC_BASELINE | (N.JPEGDEC_PROGRESSIVE if progressive else 0)


def probe(data, progressive: bool = False) -> Optional[Tuple[int, int]]:
    """(height, width) when the device decoder takes this JPEG file (bytes-like), else None (host codec).  Progressive
    files count only with progressive=True (the file is then walked to its end: every scan is checked)."""
    buf = np.frombuffer(data, dtype=np.uint8)
    h, w = ctypes.c_int(), ctypes.c_int()
    rc = N.lib().rod_jpegdec_probe_ex(buf.ctypes.data, buf.size, _formats(progressive), ctypes.byref(h), ctypes.byref(w))
    return (h.value, w.value) if rc == N.ROD_OK else None


class JpegDecoder:
    """Decoder for one batch of JPEG files: `cv2.imread` (scripts/build_corrupted_testsets.py:109, :149) for a device-resident
    batch.  files: bytes-like objects (whole files); image i is written as HWC BGR uint8 at byte offsets[i] of the tensor
    given to decode(), row pitch 3 * width unless `pitches` says otherwise -- the layout of a CorruptionPlan built from
    `shapes`.  The constructor does the host work (markers, Huffman tables, scans copied without their byte stuffing into
    page-locked memory, on `host_threads` threads); `shapes[i]` is (h, w), or None where the device decoder does not take
    the file (it takes baseline 4:2:0 / 4:2:2 / 4:4:4 / greyscale files, with or without restart markers, and with
    progressive=True progressive files of the same layouts whose scans refine every coefficient to the last bit -- the
    pixels of their baseline twin, as cv2.imread and PIL give them; not: EXIF rotation, CMYK, arithmetic coding, not a
    JPEG ...): the caller reads those with the host codec.  No CPU decoding inside."""

    def __init__(self, files: Sequence, offsets: Sequence[int], pitches: Optional[Sequence[int]] = None, host_threads: int = 8,
                 progressive: bool = False):
        N.require_device()
        n = len(files)
        self._bufs = [np.frombuffer(f, dtype=np.uint8) for f in files]   # keeps the file bytes alive for create()
        ptrs = (ctypes.c_void_p * n)(*[b.ctypes.data for b in self._bufs])
        lens = (ctypes.c_uint64 * n)(*[b.size for b in self._bufs])
        offs = (ctypes.c_uint64 * n)(*[int(o) for o in offsets])
        pit = (ctypes.c_int64 * n)(*[int(q) for q in pitches]) if pitches is not None else None
        handle = ctypes.c_void_p()
        N.check(N.lib().rod_jpegdec_create_ex(ptrs, lens, n, offs, pit, int(host_threads), _formats(progressive), ctypes.byref(handle)),
                "rod_jpegdec_create_ex")
        self._h = handle
        self._bufs = None   # the scans were copied
        self.n_images = n
        st = np.zeros(n, np.int32)
        hh, ww = np.zeros(n, np.int32), np.zeros(n, np.int32)
        N.check(N.lib().rod_jpegdec_host_status(handle, st.ctypes.data, hh.ctypes.data, ww.ctypes.data), "rod_jpegdec_host_status")
        self.host_status = st
        self.shapes: List[Optional[Tuple[int, int]]] = [(int(h), int(w)) if s == 0 else None for s, h, w in zip(st, hh, ww)]

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                N.lib().rod_jpegdec_destroy(h)
            except Exception:
                pass
            self._h = None

    def decode(self, pixels, stream=None) -> None:
        """On `stream` (default: torch's current stream): pixels (CUDA uint8 tensor) receives the images.  Returns when the
        Huffman stage has synchronised (a few host round trips); IDCT and colour conversion are still in flight."""
        N.check(N.lib().rod_jpegdec_decode(self._h, _ptr(pixels), _stream_handle(stream)), "rod_jpegdec_decode")

    def status(self, stream=None) -> np.ndarray:
        """Waits for the stream.  Per image 0: decoded; 1 / 2: corrupt / truncated entropy-coded data (pixels undefined:
        read the file with the host codec); >= 10: the constructor's verdict (not decodable on the device)."""
        st = np.zeros(self.n_images, np.int32)
        N.check(N.lib().rod_jpegdec_status(self._h, st.ctypes.data, _stream_handle(stream)), "rod_jpegdec_status")
        return st


def sizes_of(files: Sequence, progressive: bool = False) -> List[Optional[Tuple[int, int]]]:
    """probe() for a list of files."""
    return [probe(f, progressive) for f in files]
