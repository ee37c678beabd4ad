"""Corpus of the device JPEG encoder (run where cv2 is importable):
    python tests/golden/make_golden_jpeg_enc.py
Writes tests/golden/jpeg_enc.npz: the seed, one recipe per case (h, w, content, quality, sampling) and, for each case, the length and
SHA-256 digest of cv2.imencode(".jpg", frame, [IMWRITE_JPEG_QUALITY, q, IMWRITE_JPEG_SAMPLING_FACTOR, s]). The frames are not stored:
frame(seed, case, ...) regenerates them, so the file stays small.

Cases: every (h mod 16, w mod 16) edge class of a 16x16 MCU at sizes 1 .. 32, in each of 4:2:0, 4:2:2 and 4:4:4; sizes near 127x255;
qualities 1, 2, 10, 50, 75, 90, 95 and 100; constant, gradient and seeded noise frames; and the 20 shipped images."""
import hashlib
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
IMAGES = os.path.join(HERE, "images")
SEED = 2026
QUALITIES = [1, 2, 10, 50, 75, 90, 95, 100]
SAMPLINGS = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444]
CONST, GRADIENT, NOISE, SHIPPED = 0, 1, 2, 3           # content codes; SHIPPED + k is the k-th shipped image (sorted names)


def shipped_names():
    return sorted(os.listdir(IMAGES))


def frame(seed, case, h, w, content):
    """The BGR uint8 frame [h, w, 3] of one case."""
    if content >= SHIPPED:
        return cv2.imread(os.path.join(IMAGES, shipped_names()[content - SHIPPED]))
    rng = np.random.default_rng([seed, case])
    if content == CONST:
        return np.broadcast_to(rng.integers(0, 256, 3, dtype=np.uint8), (h, w, 3)).copy()
    if content == NOISE:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    y, x = np.mgrid[0:h, 0:w]
    base = np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), ((x + y) * 7) % 256], -1)
    return np.clip(base + rng.integers(-20, 21, (h, w, 3)), 0, 255).astype(np.uint8)


def encode(img, quality, sampling):
    ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, int(quality), cv2.IMWRITE_JPEG_SAMPLING_FACTOR, int(sampling)])
    assert ok
    return buf.tobytes()


def recipes():
    """-> rows (h, w, content, quality, sampling)"""
    rows = []
    n = 0
    for s in SAMPLINGS:
        for hm in range(16):
            for wm in range(16):
                h = hm + 16 if hm == 0 or (hm + wm) % 2 else hm         # 1 .. 32: both MCU-row counts for most classes
                w = wm + 16 if wm == 0 or (hm * wm) % 3 == 1 else wm
                rows.append((h, w, (CONST, GRADIENT, NOISE)[n % 3], QUALITIES[n % len(QUALITIES)], s))
                n += 1
    for s in SAMPLINGS:
        for h, w in ((127, 255), (128, 256), (126, 254), (127, 256), (33, 33), (1, 1)):
            rows.append((h, w, NOISE, 100, s))
            rows.append((h, w, GRADIENT, 75, s))
    for k in range(len(shipped_names())):
        rows.append((512, 640, SHIPPED + k, (95, 90, 50, 100)[k % 4], SAMPLINGS[k % 3]))
    return rows


def main():
    rows = recipes()
    lens, digests = [], []
    for i, (h, w, c, q, s) in enumerate(rows):
        data = encode(frame(SEED, i, h, w, c), q, s)
        lens.append(len(data))
        digests.append(hashlib.sha256(data).hexdigest())
    r = np.array(rows, np.int64)
    np.savez_compressed(os.path.join(HERE, "jpeg_enc.npz"), seed=np.int64(SEED), h=r[:, 0], w=r[:, 1], content=r[:, 2],
                        quality=r[:, 3], sampling=r[:, 4], length=np.array(lens, np.int64), sha256=np.array(digests),
                        cv2_version=np.array(cv2.__version__))
    print("wrote %d cases to %s" % (len(rows), os.path.join(HERE, "jpeg_enc.npz")))


if __name__ == "__main__":
    main()
