"""Freeze cv2's own outputs for the mixed-size / colour pre-processing tests (run where cv2 is importable):
    python tests/golden/make_golden_frames.py
Writes tests/golden/frames.npz: small BGR frames of odd sizes with, for each, the target size and
  gray: cv2.resize(cv2.cvtColor(frame, BGR2GRAY), (W, H))      - detect.py:107-122, single-channel network
  rgb:  cv2.resize(frame, (W, H))[:, :, ::-1].transpose(2, 0, 1) - detect.py:107-122, 3-channel network
(the resize is skipped when the sizes agree, as in the reference)."""
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
rng = np.random.default_rng(17)
out = {"cv2_version": np.array(cv2.__version__)}
cases = [(1, 1, 32, 32), (1, 37, 32, 64), (29, 1, 64, 32), (13, 57, 32, 96), (61, 43, 64, 64), (97, 131, 64, 96), (48, 64, 96, 128),
         (64, 96, 64, 96), (35, 210, 32, 64), (120, 7, 64, 32)]
for i, (Ho, Wo, H, W) in enumerate(cases):
    frame = rng.integers(0, 256, (Ho, Wo, 3), dtype=np.uint8)
    same = (Ho, Wo) == (H, W)
    g = cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)
    c = frame if same else cv2.resize(frame, (W, H))
    out["f%d_bgr" % i] = frame
    out["f%d_gray" % i] = g if same else cv2.resize(g, (W, H))
    out["f%d_rgb" % i] = np.ascontiguousarray(c[:, :, ::-1].transpose(2, 0, 1))
np.savez_compressed(os.path.join(HERE, "frames.npz"), **out)
print("wrote", os.path.join(HERE, "frames.npz"), os.path.getsize(os.path.join(HERE, "frames.npz")), "bytes")
