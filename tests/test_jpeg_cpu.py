"""Header parser of the device JPEG decoder (yf_jpeg_probe, host only) and its corpus: every supported corpus file is taken with its
size, every unsupported kind is turned down with a reason that names it, truncations and seeded header mutations fail cleanly, and
the frozen cv2 output of the corpus still equals live cv2.imdecode."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

import yolo_fastest_b200 as yf
from yolo_fastest_b200 import _lib
from yolo_fastest_b200.detector import jpeg_layout

HERE = os.path.dirname(os.path.abspath(__file__))
JDIR = os.path.join(HERE, "golden", "jpeg")
IMAGES = os.path.join(HERE, "golden", "images")


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _probe(data):
    """-> (rc, h, w, reason)"""
    buf = np.frombuffer(data, np.uint8)
    h, w = C.c_int32(-7), C.c_int32(-7)
    rc = yf.lib().yf_jpeg_probe(buf.ctypes.data if buf.size else None, buf.size, C.byref(h), C.byref(w))
    return rc, h.value, w.value, yf.lib().yf_last_error(None).decode()


def _corpus():
    return sorted(n for n in os.listdir(JDIR) if not n.startswith("reject_"))


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(HERE, "golden", "jpeg.npz"))


def _segments(b):
    out, i = [], 2
    while True:
        m, L = b[i + 1], struct.unpack(">H", b[i + 2:i + 4])[0]
        out.append((m, i, i + 2 + L))
        if m == 0xDA:
            return out
        i += 2 + L


def test_probe_takes_every_supported_file(golden):
    names = _corpus()
    assert len(names) >= 60
    for n in names:
        rc, h, w, why = _probe(_read(os.path.join(JDIR, n)))
        assert rc == 0, (n, why)
        assert (h, w) == golden[n].shape[:2], n
    for n in sorted(os.listdir(IMAGES)):
        assert yf.jpeg_probe(_read(os.path.join(IMAGES, n))) == (512, 640), n


def _patched_sof(b, marker=None, precision=None):
    b = bytearray(b)
    for m, s, e in _segments(bytes(b)):
        if m in (0xC0, 0xC1):
            if marker is not None:
                b[s + 1] = marker
            if precision is not None:
                b[s + 4] = precision
    return bytes(b)


def _bare_sof(ncomp):
    comps = b"".join(bytes([c + 1, 0x11, 0]) for c in range(ncomp))
    sof = bytes([8]) + struct.pack(">HH", 16, 16) + bytes([ncomp]) + comps
    return b"\xff\xd8" + b"\xff\xc0" + struct.pack(">H", len(sof) + 2) + sof + b"\xff\xd9"


def _rgb_ids(b):
    """drop the JFIF marker and name the components 'R', 'G', 'B' (libjpeg then reads the file as RGB)"""
    b = bytearray(b)
    segs = _segments(bytes(b))
    for m, s, e in segs:
        if m == 0xC0:
            for c in range(3):
                b[s + 10 + 3 * c] = b"RGB"[c]
        if m == 0xDA:
            for c in range(3):
                b[s + 5 + 2 * c] = b"RGB"[c]
    app0 = [(s, e) for m, s, e in segs if m == 0xE0]
    for s, e in reversed(app0):
        del b[s:e]
    return bytes(b)


def _two_scans(b):
    """append a second copy of the SOS segment and its scan after the first scan"""
    sos = [(s, e) for m, s, e in _segments(b) if m == 0xDA][0]
    body = b[sos[0]:]
    assert body.endswith(b"\xff\xd9")
    return b[:-2] + body


def test_probe_rejects_every_unsupported_kind():
    base = _read(os.path.join(JDIR, "420_37x53_nodht_q80.jpg"))
    cases = {
        "reject_progressive.jpg": "progressive", "reject_411.jpg": "sampling factors 4x1", "reject_440.jpg": "sampling factors 1x2",
        "reject_exif_orientation6.jpg": "EXIF orientation 6", "reject_adobe_rgb.jpg": "Adobe marker with transform 0",
        "reject_png.png": "not a JPEG",
    }
    for n, want in cases.items():
        rc, _, _, why = _probe(_read(os.path.join(JDIR, n)))
        assert rc == -1 and want in why, (n, why)
    made = [
        (_patched_sof(base, marker=0xC9), "arithmetic"), (_patched_sof(base, marker=0xC3), "lossless"),
        (_patched_sof(base, marker=0xC5), "hierarchical"), (_patched_sof(base, precision=12), "12-bit"),
        (_bare_sof(4), "CMYK"), (_bare_sof(2), "2-component"), (_rgb_ids(base), "component IDs 'R', 'G', 'B'"),
        (_two_scans(base), "more than one scan"), (b"GIF89a" + bytes(64), "not a JPEG"), (b"", "not a JPEG"),
    ]
    for data, want in made:
        rc, _, _, why = _probe(data)
        assert rc == -1 and want in why, (want, why)


def test_probe_fails_cleanly_on_every_header_prefix():
    """Every prefix that ends before the scan data is turned down; a prefix that ends inside the scan is taken (the device decoder
    marks such a file corrupt), and none crashes."""
    for n in ("gray_127x255_q100.jpg", "420_37x53_rst3_q75.jpg", "422_64x48_opt_q85.jpg"):
        b = _read(os.path.join(JDIR, n))
        scan = _segments(b)[-1][2]
        for k in range(len(b)):
            rc, h, w, why = _probe(b[:k])
            if k < scan:
                assert rc == -1 and why, (n, k)
            else:
                assert rc in (0, -1), (n, k)


def test_probe_survives_header_mutations():
    """A few thousand seeded single-byte mutations of the headers of corpus files: YF_ERR_ARG or a size in range, never a crash."""
    rng = np.random.default_rng(7)
    names = _corpus()
    taken = 0
    for i in range(3000):
        b = bytearray(_read(os.path.join(JDIR, names[i % len(names)])))
        scan = _segments(bytes(b))[-1][2]
        pos = int(rng.integers(0, scan))
        b[pos] = int(rng.integers(0, 256))
        rc, h, w, why = _probe(bytes(b))
        assert rc in (0, -1)
        if rc == 0:
            taken += 1
            assert 1 <= h <= 16384 and 1 <= w <= 16384
        else:
            assert why
    assert 0 < taken < 3000


def test_layout_names_the_file_not_taken():
    good = _read(os.path.join(JDIR, "gray_8x8_q100.jpg"))
    with pytest.raises(yf.YfError, match="file 2: progressive"):
        jpeg_layout([good, good, _read(os.path.join(JDIR, "reject_progressive.jpg"))])
    files, off, ln, foff, Ho, Wo, fbytes = jpeg_layout([good, _read(os.path.join(JDIR, "420_17x33_const_q90.jpg"))])
    assert list(off) == [0, len(good)] and list(Ho) == [8, 17] and list(Wo) == [8, 33]
    assert foff[1] % 16 == 0 and foff[1] >= 8 * 8 * 3 and fbytes == foff[1] + 17 * 33 * 3
    assert files.size == len(good) + ln[1]


def test_golden_equals_live_cv2(golden):
    """Guards against cv2 drift: the frozen decodes are what this cv2 returns (the GPU tests compare with both)."""
    cv2 = pytest.importorskip("cv2")
    for n in _corpus():
        got = cv2.imdecode(np.fromfile(os.path.join(JDIR, n), np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(got, golden[n]), n
    assert sum(os.path.getsize(os.path.join(JDIR, n)) for n in os.listdir(JDIR)) + os.path.getsize(
        os.path.join(HERE, "golden", "jpeg.npz")) < 2 * 1024 * 1024


def test_nodht_files_use_the_standard_tables(golden):
    """cv2 decodes a file without DHT segments with the T.81 K.3 tables: putting back the DHT segments of a file cv2 wrote with its
    default (standard) tables gives the same decode."""
    cv2 = pytest.importorskip("cv2")
    checked = 0
    for n in _corpus():
        if "nodht" not in n:
            continue
        b = _read(os.path.join(JDIR, n))
        assert all(m != 0xC4 for m, _, _ in _segments(b)), n
        donor = _read(os.path.join(JDIR, ("gray" if n.startswith("gray") else "420") + "_17x33_const_q90.jpg"))
        dht = b"".join(donor[s:e] for m, s, e in _segments(donor) if m == 0xC4)
        back = cv2.imdecode(np.frombuffer(b[:2] + dht + b[2:], np.uint8), cv2.IMREAD_COLOR)
        assert np.array_equal(back, golden[n]), n
        checked += 1
    assert checked >= 5


def test_symbols_bound():
    l = yf.lib()
    P = C.c_void_p
    assert l.yf_jpeg_probe.argtypes == [P, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    assert l.yf_decode_jpeg.argtypes == [P, P, C.c_int64, C.c_int, P, P, P, P, C.c_int64, P, P]
    assert l.yf_detect_host_jpeg.argtypes == [P, P, C.c_int64, C.c_int, P, P, P, C.POINTER(_lib.YfPostParams), P, P, P, P, P]
    for name in ("yf_jpeg_probe", "yf_decode_jpeg", "yf_detect_host_jpeg"):
        assert getattr(l, name).restype == C.c_int
        assert name in {s[0] for s in _lib.SYMBOLS}
    assert l.yf_decode_jpeg(None, None, 0, 1, None, None, None, None, 0, None, None) == -1
    assert l.yf_detect_host_jpeg(None, None, 0, 1, None, None, None, None, None, None, None, None, None) == -1
