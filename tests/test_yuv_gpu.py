"""YUV 4:2:0 frames on the device (yf_yuv420_to_bgr / yf_preprocess_yuv420 / yf_detect_yuv420) against live cv2: the BGR frames byte for
byte, the network input byte for byte what pre_process_frames makes of cv2's BGR frames, and detections equal to detect_frames of
them, for NV12 and I420, host and cuda frames, cv2's single-array form and pitched plane tuples, gray and colour networks."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import yolo_fastest_b200 as yf
from conftest import rows_equal
from oracle import yuv_oracle as yo
from test_frames_gpu import _colour_detector, _gray_detector, colour_ckpt  # noqa: F401  (colour_ckpt is a fixture)

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
IMAGES = os.path.join(HERE, "golden", "images")
FMTS = ["nv12", "i420"]
CODE = {"nv12": "COLOR_YUV2BGR_NV12", "i420": "COLOR_YUV2BGR_I420"}


def _cv2():
    return pytest.importorskip("cv2")


def _bgr(frame, fmt):
    """cv2.cvtColor of a frame in cv2's form (numpy, or a tensor brought to the host)"""
    a = frame.cpu().numpy() if isinstance(frame, torch.Tensor) else frame
    return _cv2().cvtColor(np.ascontiguousarray(a), getattr(_cv2(), CODE[fmt]))


def _random(rng, h, w):
    return rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)


def _sweep_sizes():
    return [(h, 34) for h in range(2, 1025, 2)] + [(6, w) for w in range(2, 1025, 2)] + [(512, 640), (1080, 1920), (16384, 2), (2, 16384)]


def _check_bgr(det, frames, want, what):
    got = det.yuv_to_bgr(frames[0], frames[1])
    assert len(got) == len(want)
    for b, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and np.array_equal(g.cpu().numpy(), w), "%s: frame %d of size %s" % (what, b, w.shape[:2])


@pytest.mark.parametrize("fmt", FMTS)
def test_to_bgr_sweep(fmt):
    """Every even height 2..1024 at width 34, every even width 2..1024 at height 6, 512x640, 1080x1920, 16384x2 and 2x16384: host
    frames, and the same frames as cuda tensors, against cv2.cvtColor."""
    rng = np.random.default_rng(41)
    det = _gray_detector("256x320")
    sizes = _sweep_sizes()
    for i0 in range(0, len(sizes), 128):
        frames = [_random(rng, h, w) for h, w in sizes[i0:i0 + 128]]
        want = [_bgr(f, fmt) for f in frames]
        _check_bgr(det, (frames, fmt), want, "%s host" % fmt)
        _check_bgr(det, ([torch.from_numpy(f).cuda() for f in frames], fmt), want, "%s cuda" % fmt)


def _surface(rng, h, w, fmt, surf_h, pitch, offset=0):
    """A decoder-style surface on the device: luma rows of `pitch` bytes, chroma after `surf_h` rows (NV12: interleaved UV of the same
    pitch; I420: U and V in allocations of their own, pitch pitch / 2), planes starting `offset` bytes into their allocations.
    -> (plane tuple, the frame in cv2's form on the host)"""
    frame = _random(rng, h, w)
    Y, U, V = yo.planes(frame, fmt)

    def plane(rows, cols, p, data, total_rows):
        buf = torch.from_numpy(rng.integers(0, 256, offset + total_rows * p, dtype=np.uint8)).cuda()
        t = buf[offset:offset + rows * p].view(rows, p)[:, :cols]
        t.copy_(torch.from_numpy(np.ascontiguousarray(data)))
        return t, buf
    if fmt == "nv12":
        buf = torch.from_numpy(rng.integers(0, 256, offset + (surf_h + surf_h // 2) * pitch, dtype=np.uint8)).cuda()
        s = buf[offset:offset + (surf_h + surf_h // 2) * pitch].view(surf_h + surf_h // 2, pitch)
        s[:h, :w] = torch.from_numpy(np.ascontiguousarray(Y))
        s[surf_h:surf_h + h // 2, :w] = torch.from_numpy(np.ascontiguousarray(frame[h:]))
        return (s[:h, :w], s[surf_h:surf_h + h // 2, :w]), frame
    y, _ = plane(h, w, pitch, Y, surf_h)
    u, _ = plane(h // 2, w // 2, pitch // 2, U, surf_h // 2)
    v, _ = plane(h // 2, w // 2, pitch // 2, V, surf_h // 2)
    return (y, u, v), frame


def _pre_want(det, frames, fmt):
    return det.pre_process_frames([_bgr(f, fmt) for f in frames]).cpu().numpy()


@pytest.mark.parametrize("fmt", FMTS)
def test_pitched_tuples_and_odd_offsets(fmt, colour_ckpt):  # noqa: F811
    """1080p planes of a 1088-row surface with a 2048-byte pitch (staged), the same at odd byte offsets and odd pitches (byte loads),
    and a mixed batch of both forms: conversion and pre-processing, gray and colour."""
    rng = np.random.default_rng(43)
    cases = [(1080, 1920, 1088, 2048, 0), (1080, 1920, 1088, 2048, 1), (480, 640, 480, 641, 3), (34, 50, 36, 51, 1), (2, 2, 2, 3, 1)]
    tuples, frames = zip(*[_surface(rng, h, w, fmt, sh, p, o) for h, w, sh, p, o in cases])
    want = [_bgr(f, fmt) for f in frames]
    det = _gray_detector("512x640")
    _check_bgr(det, (list(tuples), fmt), want, "%s tuples" % fmt)
    mixed = list(tuples) + [torch.from_numpy(f).cuda() for f in frames]
    _check_bgr(det, (mixed, fmt), want + want, "%s mixed forms" % fmt)
    for d in (det, _gray_detector("256x320"), _colour_detector(colour_ckpt, "256x320")):
        got = d.pre_process_yuv(mixed, fmt).cpu().numpy()
        assert np.array_equal(got, _pre_want(d, frames + frames, fmt)), (fmt, d.input_shape)


@pytest.mark.parametrize("fmt", FMTS)
def test_descriptors_of_cuda_frames(fmt):
    """Cuda frames are read in place: offsets from the lowest plane address, nbytes up to the highest plane end."""
    rng = np.random.default_rng(47)
    (t, frame) = _surface(rng, 1080, 1920, fmt, 1088, 2048, 5)
    cv2form = torch.from_numpy(_random(rng, 4, 8)).cuda()
    desc, on_dev, base, nbytes = yf.yuv_layout([t, cv2form], fmt)
    assert on_dev and base == min([p.data_ptr() for p in t] + [cv2form.data_ptr()])
    d = desc[0]
    assert (d["h"], d["w"], d["y_pitch"]) == (1080, 1920, 2048) and d["y_off"] == t[0].data_ptr() - base
    assert d["u_off"] == t[1].data_ptr() - base and d["c_step"] == (2 if fmt == "nv12" else 1)
    assert d["v_off"] == (d["u_off"] + 1 if fmt == "nv12" else t[2].data_ptr() - base)
    assert d["c_pitch"] == (2048 if fmt == "nv12" else 1024)
    e = desc[1]
    assert e["y_off"] == cv2form.data_ptr() - base and e["u_off"] == e["y_off"] + 32 and e["y_pitch"] == 8
    ends = [p.data_ptr() + (p.shape[0] - 1) * p.stride(0) + p.shape[1] for p in t] + [cv2form.data_ptr() + cv2form.numel()]
    assert nbytes == max(ends) - base


@pytest.mark.parametrize("res", ["256x320", "512x640"])
def test_pre_process_sweep(res, colour_ckpt):  # noqa: F811
    """pre_process_yuv == pre_process_frames of cv2's BGR frames on the sweep's sizes, gray networks at both sizes and a colour network,
    NV12 and I420, host frames and cuda frames."""
    rng = np.random.default_rng(53)
    dets = [_gray_detector(res)] + ([_colour_detector(colour_ckpt, res)] if res == "256x320" else [])
    sizes = _sweep_sizes()
    for fmt in FMTS:
        for i0 in range(0, len(sizes), 128):
            frames = [_random(rng, h, w) for h, w in sizes[i0:i0 + 128]]
            for det in dets:
                want = _pre_want(det, frames, fmt)
                assert np.array_equal(det.pre_process_yuv(frames, fmt).cpu().numpy(), want), (fmt, res, i0)
                cuda = [torch.from_numpy(f).cuda() for f in frames]
                assert np.array_equal(det.pre_process_yuv(cuda, fmt).cpu().numpy(), want), (fmt, res, i0, "cuda")


def test_chunks():
    """300 frames of mixed sizes: two descriptor chunks, each writing its own frames."""
    rng = np.random.default_rng(59)
    det = _gray_detector("256x320")
    sizes = [(2 * (3 + b % 11), 2 * (4 + b % 13)) for b in range(300)]
    for fmt in FMTS:
        frames = [_random(rng, h, w) for h, w in sizes]
        _check_bgr(det, (frames, fmt), [_bgr(f, fmt) for f in frames], "%s 300 frames" % fmt)
        assert np.array_equal(det.pre_process_yuv(frames, fmt).cpu().numpy(), _pre_want(det, frames, fmt))


def _shipped_yuv(fmt, sizes=None):
    """The 20 shipped images (optionally resized) as cv2.cvtColor(BGR2YUV_I420) makes them, in `fmt`; -> (yuv frames, cv2's BGR)"""
    cv2 = _cv2()
    out = []
    for i, n in enumerate(sorted(os.listdir(IMAGES))):
        img = cv2.imread(os.path.join(IMAGES, n))
        if sizes:
            h, w = sizes[i % len(sizes)]
            img = cv2.resize(img, (w, h))
        i420 = cv2.cvtColor(img, cv2.COLOR_BGR2YUV_I420)
        out.append(i420 if fmt == "i420" else yo.from_planes(*yo.planes(i420, "i420"), "nv12"))
    return out, [_bgr(f, fmt) for f in out]


def _rows_match(want, got):
    assert len(want) == len(got)
    for w, g in zip(want, got):
        rows_equal(w, g)
    assert sum(len(r) for r in got) > 0


@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("res", ["256x320", "512x640"])
def test_detect_shipped_images(fmt, res):
    det = _gray_detector(res)
    frames, bgr = _shipped_yuv(fmt)
    want = det.detect_frames(bgr)
    _rows_match(want, det.detect_yuv(frames, fmt))
    _rows_match(want, det.detect_yuv([torch.from_numpy(f).cuda() for f in frames], fmt))


@pytest.mark.parametrize("fmt", FMTS)
def test_detect_colour_network(fmt, colour_ckpt):  # noqa: F811
    det = _colour_detector(colour_ckpt, "256x320")
    frames, bgr = _shipped_yuv(fmt)
    _rows_match(det.detect_frames(bgr), det.detect_yuv([torch.from_numpy(f).cuda() for f in frames], fmt))


@pytest.mark.parametrize("fmt", FMTS)
def test_detect_mixed_sizes_adjusted(fmt):
    """1080p, 720p and 640x512 frames in one batch, boxes mapped back to each frame (adjust=True), and the raw rows too."""
    det = _gray_detector("512x640")
    frames, bgr = _shipped_yuv(fmt, [(1080, 1920), (720, 1280), (512, 640)])
    _rows_match(det.detect_frames(bgr, adjust=True), det.detect_yuv(frames, fmt, adjust=True))
    raw_w, raw_g = det.detect_frames(bgr, raw=True), det.detect_yuv(frames, fmt, raw=True)
    assert all(np.array_equal(a, b) for a, b in zip(raw_w, raw_g))


@pytest.mark.parametrize("fmt", FMTS)
def test_detect_on_a_side_stream_from_surfaces(fmt):
    """Pitched device surfaces, detection enqueued on a non-default stream."""
    rng = np.random.default_rng(61)
    det = _gray_detector("512x640")
    frames, bgr = _shipped_yuv(fmt, [(1080, 1920), (512, 640)])
    surf = []
    for f in frames:
        h, w = f.shape[0] * 2 // 3, f.shape[1]
        t, _ = _surface(rng, h, w, fmt, h + 8 if h == 1080 else h, w + 128)
        Y, U, V = yo.planes(f, fmt)
        t[0].copy_(torch.from_numpy(np.ascontiguousarray(Y)))
        if fmt == "nv12":
            t[1].copy_(torch.from_numpy(np.ascontiguousarray(f[h:])))
        else:
            t[1].copy_(torch.from_numpy(np.ascontiguousarray(U)))
            t[2].copy_(torch.from_numpy(np.ascontiguousarray(V)))
        surf.append(t)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = det.detect_yuv(surf, fmt)
    _rows_match(det.detect_frames(bgr), got)


def test_overflow_rerun():
    det = _gray_detector("256x320")
    frames, _ = _shipped_yuv("nv12")
    full = det.detect_yuv(frames)
    assert max(len(r) for r in full) > 1
    assert det.detect_yuv(frames, max_det=1) == full              # nothing cut: run again with room for every detection


def test_refused_frames_launch_nothing():
    det = _gray_detector("256x320")
    ctx = det.model.context(det.device, 256, 320, 4)
    n0 = ctx.launch_count()
    good = torch.zeros((6, 8), dtype=torch.uint8, device="cuda")
    bad_inputs = [
        ([good, torch.zeros((6, 5), dtype=torch.uint8, device="cuda")], "nv12"),           # odd width
        ([good, np.zeros((6, 8), np.uint8)], "nv12"),                                       # host and device mixed
        ([good], "p010"),                                                                   # not a format
        ([(torch.zeros((4, 8), dtype=torch.uint8, device="cuda"), torch.zeros((2, 6), dtype=torch.uint8, device="cuda"))], "nv12"),
        ([torch.zeros((8, 12), dtype=torch.uint8, device="cuda").t()], "nv12"),             # columns not adjacent
    ]
    for frames, fmt in bad_inputs:
        for call in (det.yuv_to_bgr, det.pre_process_yuv, det.detect_yuv):
            with pytest.raises(yf.YfError):
                call(frames, fmt)
    # the C entry points refuse a descriptor outside the buffer, and a batch beyond max_batch, with nothing enqueued
    desc, _, base, nbytes = yf.yuv_layout([good], "nv12")
    lib = yf.lib()
    out = torch.empty((ctx.max_batch + 1, 256, 320), dtype=torch.uint8, device="cuda")
    assert lib.yf_preprocess_yuv420(ctx.handle, base, nbytes - 1, 1, desc.ctypes.data, out.data_ptr(), None) == -1
    assert "frame 0: V plane" in lib.yf_last_error(ctx.handle).decode()
    many = np.repeat(desc, ctx.max_batch + 1)
    assert lib.yf_preprocess_yuv420(ctx.handle, base, nbytes, many.size, many.ctypes.data, out.data_ptr(), None) == -1
    p = det.post_process._params(yf._lib.MODE_DETECT, 8)
    dets = torch.empty((1, 8, 56), dtype=torch.uint8, device="cuda")
    cnt = torch.empty((1,), dtype=torch.int32, device="cuda")
    assert lib.yf_detect_yuv420(ctx.handle, base, nbytes - 1, 1, desc.ctypes.data, C.byref(p), dets.data_ptr(), cnt.data_ptr(),
                                None, None) == -1
    foff = np.zeros(1, np.int64)
    assert lib.yf_yuv420_to_bgr(ctx.handle, base, nbytes, 1, desc.ctypes.data, out.data_ptr(), foff.ctypes.data, 4 * 8 * 3 - 1, None) == -1
    assert ctx.launch_count() == n0
    assert lib.yf_preprocess_yuv420(ctx.handle, base, nbytes, 1, desc.ctypes.data, out.data_ptr(), None) == 0
    torch.cuda.synchronize()
    assert ctx.launch_count() == n0 + 1
