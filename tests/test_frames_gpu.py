"""Mixed-size frame batches and colour networks (yf_preprocess_frames / yf_detect_host_frames) against the CPU oracle: bit-exact
bytes for every source width and height up to 1024, ragged and chunked batches, the byte-load fallback, and detections equal to
the oracle pre-processing followed by detect_batch."""
import ctypes as C
import logging
import os

import numpy as np
import pytest
import torch

import yolo_fastest_b200 as yf
from conftest import rows_equal
from oracle import preprocess_oracle as po
from test_frames_cpu import pre_process_rgb

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
IMAGES = os.path.join(HERE, "golden", "images")
RES = ["256x320", "512x640"]


def _gray_detector(res):
    return yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(HERE, "golden", "weights", "yolo_fastest_%s.pth" % res), yf.config_for(res), None)


@pytest.fixture(scope="module")
def colour_ckpt(tmp_path_factory):
    from test_forward_gpu import _three_channel_sd

    class G:                                            # what _three_channel_sd needs of the session's gold fixture
        @staticmethod
        def sd(name):
            return torch.load(os.path.join(HERE, "golden", "weights", name + ".pth"), map_location="cpu")
    path = str(tmp_path_factory.mktemp("rgb") / "rgb.pth")
    torch.save(_three_channel_sd(G), path)
    return path


def _colour_detector(path, res, logger=None):
    cfg = yf.config_for(res)
    io = cfg["io_params"]
    io["input_channel"] = 3
    io["input_shape"] = io["input_shape"][0:2] + [3]
    io["conf_thre"] = 0.3
    return yf.Detect_YOLO(torch.device("cuda:0"), path, cfg, logger)


def _oracle(det, frame):
    H, W, chans = det.input_shape
    return po.pre_process(frame, H, W) if chans == 1 else pre_process_rgb(frame, H, W)


def _check_bytes(det, frames, what):
    got = det.pre_process_frames(frames).cpu().numpy()
    assert got.shape[0] == len(frames)
    for b, f in enumerate(frames):
        f = f.cpu().numpy() if isinstance(f, torch.Tensor) else f
        assert np.array_equal(got[b], _oracle(det, f)), "%s: frame %d of size %dx%d" % (what, b, f.shape[0], f.shape[1])


def _scale_rows(rows, h, w, H, W):
    """adjust_coord's arithmetic with the frame's own size (detect.py:131-139)"""
    if [h, w] == [H, W]:
        return rows
    sh, sw = h / H, w / W
    return [[round(r[0] * sw), round(r[1] * sh), round(r[2] * sw), round(r[3] * sh)] + list(r[4:]) for r in rows]


@pytest.mark.parametrize("res", RES)
def test_tap_sweep_every_source_size_to_1024(res, colour_ckpt):
    """Every source height and every source width in [1, 1024], through the gray and the colour instantiation: the in-kernel taps
    must equal the oracle's (and so prep_taps / cv2's) for each of them. The other side of each frame is small and varies, so both
    the staged and the byte-load forms are exercised."""
    rng = np.random.default_rng(101)
    sizes = [(n, 1 + n % 8) for n in range(1, 1025)] + [(1 + n % 5, n) for n in range(1, 1025)]
    for det in (_gray_detector(res), _colour_detector(colour_ckpt, res)):
        for i0 in range(0, len(sizes), 64):
            frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes[i0:i0 + 64]]
            _check_bytes(det, frames, "%s in_ch=%d sweep" % (res, det.input_shape[2]))


@pytest.mark.parametrize("res", RES)
def test_mixed_sizes_one_batch(res, colour_ckpt):
    """The sizes of test_preprocess_gpu plus degenerate ones (1x1, 1xN, Nx1), widths not divisible by 4, and a 3x16384 frame too
    wide to stage in shared memory (byte-load fallback) in ONE batch; host frames and cuda frames."""
    rng = np.random.default_rng(7)
    for det in (_gray_detector(res), _colour_detector(colour_ckpt, res)):
        H, W = det.input_shape[0:2]
        sizes = [(512, 640), (480, 640), (333, 517), (128, 160), (1080, 1920), (H, W), (1, 1), (1, 301), (257, 1), (7, 13), (3, 16384),
                 (45, 62), (99, 101)]
        frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
        frames += [np.full((100, 200, 3), 0, np.uint8), np.full((77, 33, 3), 255, np.uint8)]
        _check_bytes(det, frames, "%s in_ch=%d host" % (res, det.input_shape[2]))
        dev = [torch.from_numpy(f).cuda() for f in frames[::-1]]
        _check_bytes(det, dev, "%s in_ch=%d cuda" % (res, det.input_shape[2]))


def test_unaligned_offsets(colour_ckpt):
    """Frames at odd byte offsets of a device buffer (rows not 4-byte aligned) take the byte-load form and stay exact."""
    rng = np.random.default_rng(9)
    for det in (_gray_detector("256x320"), _colour_detector(colour_ckpt, "256x320")):
        H, W, chans = det.input_shape
        sizes = [(512, 640), (64, 80), (333, 517), (256, 320)]
        frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
        off = np.array([1, 983043, 983043 + 15360 + 6, 983043 + 15360 + 6 + 516483 + 1], np.int64)
        Ho = np.array([h for h, _ in sizes], np.int32)
        Wo = np.array([w for _, w in sizes], np.int32)
        buf = np.zeros(int(off[-1]) + 256 * 320 * 3 + 3, np.uint8)
        for f, o in zip(frames, off):
            buf[o:o + f.size] = f.reshape(-1)
        d = torch.from_numpy(buf).cuda()
        ctx = det.model.context(det.device, H, W, len(frames))
        out = torch.empty((len(frames), H, W) if chans == 1 else (len(frames), 3, H, W), dtype=torch.uint8, device="cuda")
        yf._lib.check(yf.lib().yf_preprocess_frames(ctx.handle, d.data_ptr(), len(frames), off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data,
                                                    out.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)), ctx.handle)
        got = out.cpu().numpy()
        for b, f in enumerate(frames):
            assert np.array_equal(got[b], _oracle(det, f)), (chans, b)


def test_chunk_boundary():
    """More than 512 frames: the descriptors go to the kernel in chunks of 512, the output of each chunk at its own place."""
    rng = np.random.default_rng(13)
    det = _gray_detector("256x320")
    frames = [rng.integers(0, 256, (17 + b % 5, 20 + 4 * (b % 3) + (b % 2), 3), dtype=np.uint8) for b in range(600)]
    _check_bytes(det, frames, "600 frames")


@pytest.mark.parametrize("res", RES)
def test_equal_sizes_match_preprocess_bgr(res):
    rng = np.random.default_rng(3)
    det = _gray_detector(res)
    H, W = det.input_shape[0:2]
    for (B, Ho, Wo) in [(5, 512, 640), (3, 480, 640), (2, 333, 517), (2, 128, 160), (1, 1080, 1920), (4, H, W)]:
        frames = rng.integers(0, 256, (B, Ho, Wo, 3), dtype=np.uint8)
        a = det.pre_process_batch(frames)
        b = det.pre_process_frames(list(frames))
        assert torch.equal(a, b), (res, B, Ho, Wo)


def _shipped_mixed():
    """The 20 shipped images (512x640), some of them resized on the host to other sizes."""
    cv2 = pytest.importorskip("cv2")
    names = sorted(os.listdir(IMAGES))
    other = [None, (480, 600), (333, 517), (1080, 1920), (256, 320)]
    frames = []
    for i, n in enumerate(names):
        img = cv2.imread(os.path.join(IMAGES, n))
        size = other[i % len(other)]
        frames.append(img if size is None else cv2.resize(img, (size[1], size[0])))
    return frames


def _want_rows(det, frames):
    H, W = det.input_shape[0:2]
    u8 = np.stack([_oracle(det, f) for f in frames])
    rows = det.detect_batch(u8)
    return [_scale_rows(r, f.shape[0], f.shape[1], H, W) for r, f in zip(rows, frames)]


@pytest.mark.parametrize("res", RES)
def test_shipped_images_mixed_sizes(res):
    det = _gray_detector(res)
    frames = _shipped_mixed()
    got = det.detect_frames(frames)
    want = _want_rows(det, frames)
    for w, g in zip(want, got):
        rows_equal(w, g)
    assert sum(len(r) for r in got) > 0


def test_colour_network(colour_ckpt):
    """A 3-channel network: detect_frames == oracle RGB planes -> detect_batch, and == the per-file path of batch_detect
    (pre_process -> model -> postprocess_batch -> adjust_coord) on frames of origin_img_shape."""
    det = _colour_detector(colour_ckpt, "256x320")
    frames = _shipped_mixed()
    got = det.detect_frames(frames)
    for w, g in zip(_want_rows(det, frames), got):
        rows_equal(w, g)
    assert sum(len(r) for r in got) > 0
    names = sorted(os.listdir(IMAGES))
    import cv2
    orig = [cv2.imread(os.path.join(IMAGES, n)) for n in names]
    got = det.detect_frames(orig)
    with torch.no_grad():                               # fp32 input at batch 1: other forward kernels, heads equal within 1e-4
        for n, g in zip(names, got):
            img, _ = det.pre_process(os.path.join(IMAGES, n))
            want = det.post_process.postprocess_batch(det.model(img))[0]
            det.adjust_coord(want)
            rows_equal(want, g, conf_tol=1e-4)


@pytest.mark.parametrize("kind", ["gray", "colour"])
def test_mixed_size_folder(kind, tmp_path, colour_ckpt):
    """batch_detect_batched on a folder of mixed sizes (or any folder, for a colour network): every result file, one log line per
    image, and each image's detect / no-target flag that of detect_frames."""
    cv2 = pytest.importorskip("cv2")
    src = tmp_path / "in"
    src.mkdir()
    for n, f in zip(sorted(os.listdir(IMAGES)), _shipped_mixed()):
        cv2.imwrite(str(src / (os.path.splitext(n)[0] + ".png")), f)
    records = []

    class Hd(logging.Handler):
        def emit(self, r):
            records.append(r.getMessage())
    logger = logging.getLogger("yf-test-frames-" + kind)
    logger.setLevel(logging.INFO)
    logger.addHandler(Hd())
    det = _gray_detector("256x320") if kind == "gray" else _colour_detector(colour_ckpt, "256x320")
    det.logger = logger
    out = tmp_path / "out"
    out.mkdir()
    det.batch_detect_batched(str(src), str(out), batch_size=8)
    names = os.listdir(str(src))
    assert sorted(os.listdir(str(out))) == sorted("result_" + n for n in names)
    assert len(records) == len(names) + 1 and records[-1].startswith("detect avg_time:")
    rows = det.detect_frames([cv2.imread(str(src / n)) for n in names])
    for n, r in zip(names, rows):
        line = [x for x in records if x.startswith("image_name:%s " % n)]
        assert len(line) == 1
        assert ("no targets" in line[0]) == (len(r) == 0), n
    assert any(len(r) for r in rows)


def test_overflow_rerun_and_bad_input():
    det = _gray_detector("256x320")
    frames = _shipped_mixed()
    full = det.detect_frames(frames)
    assert max(len(r) for r in full) > 1
    assert det.detect_frames(frames, max_det=1) == full                         # nothing cut: the batch is run again with room
    for bad in ([], [np.zeros((8, 8, 3), np.float32)], [np.zeros((8, 8), np.uint8)], [np.zeros((8, 8, 4), np.uint8)],
                [np.zeros((16385, 1, 3), np.uint8)], [torch.zeros((8, 8, 3), dtype=torch.uint8, device="cuda")]):
        with pytest.raises(yf.YfError):
            det.detect_frames(bad)
    with pytest.raises(yf.YfError):
        det.pre_process_frames([np.zeros((8, 8, 3), np.uint8), torch.zeros((8, 8, 3), dtype=torch.uint8, device="cuda")])
    with pytest.raises(yf.YfError):
        det.pre_process_frames([np.zeros((0, 8, 3), np.uint8)])
    # the C entry points check every descriptor themselves
    ctx = det.model.context(det.device, 256, 320, 2)
    buf = torch.zeros(1000, dtype=torch.uint8, device="cuda")
    out = torch.empty((4, 256, 320), dtype=torch.uint8, device="cuda")
    lib = yf.lib()

    def pre(B, off, Ho, Wo):
        off, Ho, Wo = np.array(off, np.int64), np.array(Ho, np.int32), np.array(Wo, np.int32)
        return lib.yf_preprocess_frames(ctx.handle, buf.data_ptr(), B, off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data, out.data_ptr(), None)
    assert pre(1, [0], [10], [10]) == 0
    torch.cuda.synchronize()
    assert pre(ctx.max_batch + 1, [0] * (ctx.max_batch + 1), [1] * (ctx.max_batch + 1), [1] * (ctx.max_batch + 1)) == -1
    assert pre(1, [0], [0], [10]) == -1 and pre(1, [0], [10], [16385]) == -1 and pre(1, [-1], [10], [10]) == -1
    pin_out = torch.empty((1, 8, 56), dtype=torch.uint8).pin_memory()
    cnt = torch.empty((1,), dtype=torch.int32).pin_memory()
    host = np.zeros(300, np.uint8)
    p = det.post_process._params(yf._lib.MODE_DETECT, 8)

    def det_host(nbytes, off, Ho, Wo):
        off, Ho, Wo = np.array(off, np.int64), np.array(Ho, np.int32), np.array(Wo, np.int32)
        return lib.yf_detect_host_frames(ctx.handle, host.ctypes.data, nbytes, 1, off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data,
                                         C.byref(p), pin_out.data_ptr(), cnt.data_ptr(), None, None)
    assert det_host(300, [0], [10], [10]) == 0
    assert det_host(299, [0], [10], [10]) == -1 and det_host(300, [1], [10], [10]) == -1
    assert "outside" in lib.yf_last_error(ctx.handle).decode()
