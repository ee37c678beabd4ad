"""Corpus of the device JPEG decoder (run where cv2 is importable):
    python tests/golden/make_golden_jpeg.py
Writes small files made with cv2.imencode (seeded) to tests/golden/jpeg/ and, for every file the decoder takes, what
cv2.imdecode(buf, IMREAD_COLOR) returns to tests/golden/jpeg.npz (key = file name). Files named reject_* are kinds the decoder's
header parser turns down; the npz has no entry for them.

Accepted files cover gray, 4:4:4, 4:2:2 and 4:2:0; every partial-MCU edge of a 16x16 MCU (sizes 1x1 .. 127x255); quality 5, 50, 90
and 100; uniform noise at quality 100 (clamping, range-limit wrap, dense 0xFF00 stuffing); constant images (DC-only blocks); restart
intervals 0, 1 and 3; optimised Huffman tables; and files whose DHT segments were removed (decoded with the standard tables)."""
import os
import struct

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
DIR = os.path.join(HERE, "jpeg")
KINDS = {"gray": None, "444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
         "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420}
SIZES = [(1, 1), (1, 17), (15, 1), (8, 8), (17, 33), (37, 53), (64, 48), (127, 255)]
QUALITIES = [5, 50, 90, 100]


def segments(b):
    """(marker, start, end) of every marker segment between SOI and SOS (SOS included, its scan not)."""
    out, i = [], 2
    while True:
        m = b[i + 1]
        L = struct.unpack(">H", b[i + 2:i + 4])[0]
        out.append((m, i, i + 2 + L))
        if m == 0xDA:
            return out
        i += 2 + L


def without(b, markers):
    keep, last = bytearray(b[:2]), 2
    for m, s, e in segments(b):
        if m not in markers:
            keep += b[s:e]
        last = e
    return bytes(keep + b[last:])


def with_segment(b, marker, payload):
    """insert a segment right after SOI"""
    return b[:2] + bytes([0xFF, marker]) + struct.pack(">H", len(payload) + 2) + payload + b[2:]


def image(rng, h, w, chans, mode):
    if mode == "noise":
        return rng.integers(0, 256, (h, w, chans), dtype=np.uint8)
    if mode == "const":
        return np.full((h, w, chans), rng.integers(0, 256), dtype=np.uint8)
    y, x = np.mgrid[0:h, 0:w]
    base = np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) * 7) % 256], -1)[:, :, :chans]
    return np.clip(base + rng.integers(-20, 21, (h, w, chans)), 0, 255).astype(np.uint8)


def encode(img, kind, quality, rst=0, optimize=False, progressive=False, sampling=None):
    params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize),
              cv2.IMWRITE_JPEG_PROGRESSIVE, int(progressive)]
    if kind != "gray":
        params += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sampling or KINDS[kind]]
    ok, buf = cv2.imencode(".jpg", img[:, :, 0] if kind == "gray" else img, params)
    assert ok
    return buf.tobytes()


def exif_orientation(o):
    """APP1 payload: Exif header + a little-endian TIFF with one IFD0 entry, Orientation (0x0112) SHORT = o"""
    tiff = b"II" + struct.pack("<HI", 42, 8) + struct.pack("<H", 1) + struct.pack("<HHIHH", 0x0112, 3, 1, o, 0) + struct.pack("<I", 0)
    return b"Exif\0\0" + tiff


def build():
    rng = np.random.default_rng(2024)
    files = {}
    for kind in KINDS:
        ch = 1 if kind == "gray" else 3
        for i, (h, w) in enumerate(SIZES):
            q = QUALITIES[i % 4]
            files["%s_%dx%d_q%d.jpg" % (kind, h, w, q)] = encode(image(rng, h, w, ch, "smooth"), kind, q)
        for h, w in ((37, 53), (127, 255)):
            files["%s_%dx%d_noise_q100.jpg" % (kind, h, w)] = encode(image(rng, h, w, ch, "noise"), kind, 100)
        files["%s_17x33_const_q90.jpg" % kind] = encode(image(rng, 17, 33, ch, "const"), kind, 90)
        for rst in (1, 3):
            files["%s_37x53_rst%d_q75.jpg" % (kind, rst)] = encode(image(rng, 37, 53, ch, "smooth"), kind, 75, rst=rst)
        files["%s_64x48_opt_q85.jpg" % kind] = encode(image(rng, 64, 48, ch, "smooth"), kind, 85, optimize=True)
        files["%s_37x53_nodht_q80.jpg" % kind] = without(encode(image(rng, 37, 53, ch, "smooth"), kind, 80), {0xC4})
    files["420_33x47_rst3_nodht_q60.jpg"] = without(encode(image(rng, 33, 47, 3, "smooth"), "420", 60, rst=3), {0xC4})
    # kinds the decoder turns down
    base = encode(image(rng, 24, 40, 3, "smooth"), "420", 90)
    rej = {
        "reject_progressive.jpg": encode(image(rng, 24, 40, 3, "smooth"), "420", 90, progressive=True),
        "reject_411.jpg": encode(image(rng, 24, 40, 3, "smooth"), "444", 90, sampling=cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411),
        "reject_440.jpg": encode(image(rng, 24, 40, 3, "smooth"), "444", 90, sampling=cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440),
        "reject_exif_orientation6.jpg": with_segment(base, 0xE1, exif_orientation(6)),
        "reject_adobe_rgb.jpg": with_segment(without(base, {0xE0}), 0xEE, b"Adobe" + struct.pack(">HHHB", 100, 0, 0, 0)),
    }
    ok, png = cv2.imencode(".png", image(rng, 24, 40, 3, "smooth"))
    rej["reject_png.png"] = png.tobytes()
    files.update(rej)
    return files


def main():
    files = build()
    os.makedirs(DIR, exist_ok=True)
    for old in os.listdir(DIR):
        os.remove(os.path.join(DIR, old))
    out = {"cv2_version": np.array(cv2.__version__)}
    for name, data in sorted(files.items()):
        with open(os.path.join(DIR, name), "wb") as f:
            f.write(data)
        if not name.startswith("reject_"):
            img = cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR)
            assert img is not None, name
            out[name] = img
    np.savez_compressed(os.path.join(HERE, "jpeg.npz"), **out)
    total = sum(len(d) for d in files.values()) + os.path.getsize(os.path.join(HERE, "jpeg.npz"))
    print("wrote %d files to %s and %s; %d bytes in all" % (len(files), DIR, os.path.join(HERE, "jpeg.npz"), total))


if __name__ == "__main__":
    main()
