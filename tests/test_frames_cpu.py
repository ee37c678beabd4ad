"""Mixed-size / colour pre-processing without a GPU: the colour oracle (pre_process_rgb) against cv2, frozen and live; the host
packing of frame lists (offsets, alignment, rejection of bad frames); the bound C entry points."""
import os

import numpy as np
import pytest
import torch

from oracle import preprocess_oracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "frames.npz"))


def pre_process_rgb(bgr, H, W):
    """Colour oracle, detect.py:107-122 for a 3-channel network: uint8 [Ho, Wo, 3] BGR -> uint8 [3, H, W] R, G, B planes. cv2.resize
    of a 3-channel uint8 image is the oracle's resize_linear applied to each channel on its own (same taps, same fixed-point
    steps); then the reference's [:, :, ::-1] and HWC -> CHW. The resize is skipped when the sizes agree, as in the reference.
    Pinned against cv2 below (live, and frozen in tests/golden/frames.npz); tests/test_frames_gpu.py imports it from here."""
    planes = [bgr[:, :, c] for c in (2, 1, 0)]
    return np.stack([p if p.shape == (H, W) else po.resize_linear(p, H, W) for p in planes])


def _cases():
    i = 0
    while "f%d_bgr" % i in GOLD:
        yield i, GOLD["f%d_bgr" % i], GOLD["f%d_gray" % i], GOLD["f%d_rgb" % i]
        i += 1


def test_oracles_match_frozen_cv2():
    n = 0
    for i, frame, gray, rgb in _cases():
        H, W = gray.shape
        assert rgb.shape == (3, H, W)
        got = pre_process_rgb(frame, H, W)
        assert got.dtype == np.uint8 and np.array_equal(got, rgb), "rgb case %d" % i          # bit-exact
        assert np.array_equal(po.pre_process(frame, H, W), gray), "gray case %d" % i
        n += 1
    assert n >= 8


def test_rgb_oracle_matches_live_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(23)
    for (Ho, Wo, H, W) in [(512, 640, 256, 320), (333, 517, 256, 320), (1080, 1920, 512, 640), (128, 160, 512, 640),
                           (481, 639, 256, 320), (256, 320, 256, 320), (1, 1, 32, 32), (5, 1, 64, 96), (1, 9, 32, 64)]:
        frame = rng.integers(0, 256, (Ho, Wo, 3), dtype=np.uint8)
        c = frame if (Ho, Wo) == (H, W) else cv2.resize(frame, (W, H))
        want = c[:, :, ::-1].transpose(2, 0, 1)
        assert np.array_equal(pre_process_rgb(frame, H, W), want), (Ho, Wo, H, W)
    # the identity taps (c0 = 2048, c1 = 0) give the identity, as skipping the resize does
    frame = rng.integers(0, 256, (64, 96, 3), dtype=np.uint8)
    assert np.array_equal(po.resize_linear(frame[:, :, 1], 64, 96), frame[:, :, 1])


def test_frame_layout_offsets_and_packing():
    from yolo_fastest_b200.detector import FRAME_ALIGN, frame_layout, pack_frames
    rng = np.random.default_rng(5)
    base = rng.integers(0, 256, (40, 30, 3), dtype=np.uint8)
    frames = [rng.integers(0, 256, (7, 5, 3), dtype=np.uint8), base[::2, ::3],                 # a strided view
              torch.from_numpy(rng.integers(0, 256, (3, 11, 3), dtype=np.uint8)), rng.integers(0, 256, (1, 1, 3), dtype=np.uint8)]
    off, Ho, Wo, nbytes = frame_layout(frames)
    assert off.dtype == np.int64 and Ho.dtype == np.int32 and Wo.dtype == np.int32
    assert list(Ho) == [7, 20, 3, 1] and list(Wo) == [5, 10, 11, 1]
    assert off[0] == 0 and all(o % FRAME_ALIGN == 0 for o in off)
    sizes = Ho.astype(np.int64) * Wo * 3
    assert all(off[b] + sizes[b] <= off[b + 1] for b in range(3))                               # disjoint, in order
    assert all(off[b + 1] - (off[b] + sizes[b]) < FRAME_ALIGN for b in range(3))                # no more padding than alignment needs
    assert nbytes == off[-1] + sizes[-1]
    buf = np.full(nbytes, 77, np.uint8)
    pack_frames(frames, buf, off)
    for f, o, s in zip(frames, off, sizes):
        a = f.numpy() if isinstance(f, torch.Tensor) else f
        assert np.array_equal(buf[o:o + s].reshape(a.shape), a)


@pytest.mark.parametrize("bad", [
    [], (), "frame", None,
    [np.zeros((4, 4, 3), np.float32)], [torch.zeros((4, 4, 3))],            # not uint8
    [np.zeros((4, 4), np.uint8)], [np.zeros((4, 4, 4), np.uint8)], [np.zeros((2, 4, 4, 3), np.uint8)],   # not [h, w, 3]
    [np.zeros((0, 4, 3), np.uint8)], [np.zeros((4, 0, 3), np.uint8)], [np.zeros((16385, 1, 3), np.uint8)],   # outside [1, 16384]
    [np.zeros((4, 4, 3), np.uint8), [[0, 0, 0]]],                             # a plain list is not a frame
])
def test_frame_layout_rejects_bad_frames(bad):
    import yolo_fastest_b200 as yf
    from yolo_fastest_b200.detector import frame_layout
    with pytest.raises(yf.YfError):
        frame_layout(bad)


def test_largest_side_accepted():
    from yolo_fastest_b200.detector import frame_layout
    off, Ho, Wo, nbytes = frame_layout([np.zeros((1, 16384, 3), np.uint8), np.zeros((16384, 1, 3), np.uint8)])
    assert list(Wo) == [16384, 1] and list(Ho) == [1, 16384] and nbytes == off[1] + 16384 * 3


def test_frames_symbols_bound():
    from yolo_fastest_b200 import _lib
    l = _lib.lib()
    names = [s[0] for s in _lib.SYMBOLS]
    for name, nargs in (("yf_preprocess_frames", 8), ("yf_detect_host_frames", 12)):
        assert name in names
        fn = getattr(l, name)
        assert fn.restype is not None and len(fn.argtypes) == nargs
    assert _lib.lib().yf_detect_host_frames.argtypes[2] is __import__("ctypes").c_int64
