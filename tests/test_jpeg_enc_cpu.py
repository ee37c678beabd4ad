"""Host half of the device JPEG encoder (no GPU): the header bytes equal cv2.imencode's up to the end of SOS, the output bound holds on
the worst cases, out-of-scope requests are refused with a reason, the frozen corpus digests equal live cv2, and the bindings."""
import ctypes as C
import hashlib
import importlib.util
import os
import struct

import numpy as np
import pytest

import yolo_fastest_b200 as yf
from yolo_fastest_b200 import _lib
from yolo_fastest_b200.detector import jpeg_encode_layout

cv2 = pytest.importorskip("cv2")
HERE = os.path.dirname(os.path.abspath(__file__))
S420, S422, S444 = cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444


def _maker():
    spec = importlib.util.spec_from_file_location("make_golden_jpeg_enc", os.path.join(HERE, "golden", "make_golden_jpeg_enc.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _imencode(img, q, s):
    return cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s])[1].tobytes()


def _sos_end(b):
    i = 2
    while True:
        m, L = b[i + 1], struct.unpack(">H", b[i + 2:i + 4])[0]
        if m == 0xDA:
            return i + 2 + L
        i += 2 + L


def test_sampling_constants_are_cv2s():
    assert (_lib.JPEG_SAMPLING_420, _lib.JPEG_SAMPLING_422, _lib.JPEG_SAMPLING_444) == (S420, S422, S444)


def test_header_equals_cv2_prefix():
    rng = np.random.default_rng(5)
    frames = {(h, w): rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((1, 1), (16384, 8), (8, 16384), (37, 53))}
    for q in range(1, 101):
        for s in (S420, S422, S444):
            for (h, w), img in frames.items():
                if (h, w) in ((16384, 8), (8, 16384)) and q % 9:        # the tall and wide frames at every 9th quality
                    continue
                want = _imencode(img, q, s)
                assert yf.jpeg_encode_header(h, w, q, s) == want[:_sos_end(want)], (h, w, q, hex(s))


def test_bound_holds_on_worst_cases():
    rng = np.random.default_rng(9)
    cases = []
    for h, w in ((1, 1), (8, 8), (17, 33), (127, 255)):
        cases.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))                     # noise: long codes, dense 0xFF bytes
        y, x = np.mgrid[0:h, 0:w]
        cases.append(np.where(((x + y) % 2)[:, :, None] == 1, 255, 0).astype(np.uint8).repeat(3, 2))   # checkerboard
        cases.append(np.where((x % 3 == 0)[:, :, None], 255, 0).astype(np.uint8).repeat(3, 2))         # stripes
    for img in cases:
        for s in (S420, S422, S444):
            n = len(_imencode(img, 100, s))
            assert yf.jpeg_encode_bound(img.shape[0], img.shape[1], s) >= n, (img.shape, hex(s), n)
    b = yf.jpeg_encode_bound(1080, 1920, S420)
    assert 1920 * 1080 * 3 < b < 8 * 1920 * 1080 * 3                   # what a caller has to allocate per 1080p file


def test_refusals_name_their_reason():
    lib = yf.lib()
    buf = np.zeros(1024, np.uint8)
    for q in (0, 101, -5):
        with pytest.raises(yf.YfError, match="quality %d outside" % q):
            yf.jpeg_encode_header(8, 8, q, S420)
    for s in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, 0x121111, 0, 0x221112):
        with pytest.raises(yf.YfError, match="sampling factor 0x%x is not supported" % s):
            yf.jpeg_encode_header(8, 8, 95, s)
        with pytest.raises(yf.YfError, match="sampling factor"):
            yf.jpeg_encode_bound(8, 8, s)
    for h, w in ((0, 8), (8, 0), (16385, 8), (8, 16385)):
        with pytest.raises(yf.YfError, match="size %dx%d outside" % (h, w)):
            yf.jpeg_encode_bound(h, w, S420)
        with pytest.raises(yf.YfError, match="size %dx%d outside" % (h, w)):
            yf.jpeg_encode_header(h, w, 95, S420)
    assert lib.yf_jpeg_encode_header(8, 8, 95, S420, buf.ctypes.data, 622) == -1
    assert "623 bytes" in lib.yf_last_error(None).decode()
    ok = np.zeros((4, 4, 3), np.uint8)
    with pytest.raises(yf.YfError, match="frame 1 is a gray"):
        jpeg_encode_layout([ok, np.zeros((4, 4), np.uint8)], 95, S420)
    with pytest.raises(yf.YfError, match="frame 2 is 16385x4"):
        jpeg_encode_layout([ok, ok, np.zeros((16385, 4, 3), np.uint8)], 95, S420)
    with pytest.raises(yf.YfError, match="frame 0 has shape"):
        jpeg_encode_layout([np.zeros((4, 4, 4), np.uint8)], 95, S420)
    with pytest.raises(yf.YfError, match="quality 0"):
        jpeg_encode_layout([ok], 0, S420)
    with pytest.raises(yf.YfError, match="sampling factor"):
        jpeg_encode_layout([ok], 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)


def test_golden_equals_live_cv2():
    """Guards against cv2 drift: the frozen digests are what this cv2 writes (the GPU tests compare with both)."""
    m = _maker()
    g = np.load(os.path.join(HERE, "golden", "jpeg_enc.npz"))
    rows = m.recipes()
    assert len(rows) == len(g["h"]) and int(g["seed"]) == m.SEED
    assert os.path.getsize(os.path.join(HERE, "golden", "jpeg_enc.npz")) < 256 * 1024
    classes = set()
    for i, (h, w, c, q, s) in enumerate(rows):
        assert (h, w, c, q, s) == (g["h"][i], g["w"][i], g["content"][i], g["quality"][i], g["sampling"][i]), i
        data = _imencode(m.frame(m.SEED, i, h, w, c), q, s)
        assert len(data) == g["length"][i] and hashlib.sha256(data).hexdigest() == str(g["sha256"][i]), i
        if h <= 32 and w <= 32:
            classes.add((h % 16, w % 16, s))
    assert len(classes) == 16 * 16 * 3
    assert set(g["quality"].tolist()) == {1, 2, 10, 50, 75, 90, 95, 100}


def test_symbols_bound():
    l = yf.lib()
    P = C.c_void_p
    assert l.yf_jpeg_encode_bound.argtypes == [C.c_int, C.c_int, C.c_int] and l.yf_jpeg_encode_bound.restype == C.c_int64
    assert l.yf_jpeg_encode_header.argtypes == [C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int64]
    assert l.yf_encode_jpeg.argtypes == [P, P, C.c_int, P, P, P, C.c_int, C.c_int, P, P, C.c_int64, P, P]
    assert l.yf_encode_host_jpeg.argtypes == [P, P, C.c_int64, C.c_int, P, P, P, C.c_int, C.c_int, P, C.c_int64, P, P]
    for name in ("yf_jpeg_encode_header", "yf_encode_jpeg", "yf_encode_host_jpeg"):
        assert getattr(l, name).restype == C.c_int
    for name in ("yf_jpeg_encode_bound", "yf_jpeg_encode_header", "yf_encode_jpeg", "yf_encode_host_jpeg"):
        assert name in {s[0] for s in _lib.SYMBOLS}
    assert l.yf_encode_jpeg(None, None, 1, None, None, None, 95, S420, None, None, 0, None, None) == -1
    assert l.yf_encode_host_jpeg(None, None, 0, 1, None, None, None, 95, S420, None, 0, None, None) == -1
