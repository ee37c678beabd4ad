"""Device JPEG encoder (yf_encode_jpeg / yf_encode_host_jpeg, Detect_YOLO.encode_jpeg) against cv2.imencode: byte-equal files for the
whole corpus, large and extreme sizes, a batch of more than one descriptor chunk, mixed sizes, host and device frames and decode_jpeg
output; the round trip through the device decoder; refusals with nothing launched; the host entry point's output cap; and the batched
file driver's result files and log lines unchanged when it encodes on the device."""
import hashlib
import importlib.util
import logging
import os
import shutil

import numpy as np
import pytest
import torch

import yolo_fastest_b200 as yf

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
IMAGES = os.path.join(HERE, "golden", "images")
JDIR = os.path.join(HERE, "golden", "jpeg")
cv2 = pytest.importorskip("cv2")
S420, S422, S444 = cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444


def _det(res="512x640"):
    return yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(HERE, "golden", "weights", "yolo_fastest_%s.pth" % res), yf.config_for(res), None)


def _imencode(img, q=95, s=S420):
    return cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s])[1].tobytes()


def _maker():
    spec = importlib.util.spec_from_file_location("make_golden_jpeg_enc", os.path.join(HERE, "golden", "make_golden_jpeg_enc.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _shipped():
    return [cv2.imread(os.path.join(IMAGES, n)) for n in sorted(os.listdir(IMAGES))]


def _smooth(rng, h, w):
    img = cv2.GaussianBlur(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), (7, 7), 3)
    return np.clip(img.astype(np.int16) + rng.integers(-12, 13, (h, w, 3)), 0, 255).astype(np.uint8)


def test_corpus_byte_equal():
    """Every corpus case, one call per (quality, sampling) with the frames' sizes mixed; host frames and the same frames on the device."""
    m = _maker()
    g = np.load(os.path.join(HERE, "golden", "jpeg_enc.npz"))
    det = _det()
    groups = {}
    for i, (h, w, c, q, s) in enumerate(m.recipes()):
        groups.setdefault((q, s), []).append((i, m.frame(m.SEED, i, h, w, c)))
    for (q, s), cases in groups.items():
        frames = [f for _, f in cases]
        for on_dev in (False, True):
            got = det.encode_jpeg([torch.from_numpy(f).cuda() for f in frames] if on_dev else frames, quality=q, sampling=s)
            for (i, f), data in zip(cases, got):
                assert hashlib.sha256(data).hexdigest() == str(g["sha256"][i]), (i, q, hex(s), on_dev)
                assert data == _imencode(f, q, s), (i, q, hex(s), on_dev)


def test_large_and_extreme_sizes():
    rng = np.random.default_rng(4)
    det = _det()
    cases = [(_smooth(rng, 1080, 1920), s, 95) for s in (S420, S422, S444)]
    cases += [(_smooth(rng, 3000, 4000), S420, 90), (rng.integers(0, 256, (16384, 8, 3), dtype=np.uint8), S444, 100),
              (rng.integers(0, 256, (8, 16384, 3), dtype=np.uint8), S420, 100)]
    for img, s, q in cases:
        assert det.encode_jpeg([img], quality=q, sampling=s)[0] == _imencode(img, q, s), (img.shape, hex(s))


def test_odd_block_counts_alone():
    """One 4:4:4 frame whose block count is odd (3 * mcux * mcuy with both MCU counts odd), alone in its call, on the host and the
    device entry point: the workspace parts after the coefficients then start at odd multiples of 8 bytes unless they are aligned."""
    rng = np.random.default_rng(21)
    det = _det()
    for h, w in ((8, 8), (1, 1), (33, 33), (37, 53), (17, 9)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        want = _imencode(img, 90, S444)
        assert det.encode_jpeg([img], quality=90, sampling=S444) == [want], (h, w)
        assert det.encode_jpeg([torch.from_numpy(img).cuda()], quality=90, sampling=S444) == [want], (h, w)


def test_more_than_one_chunk_and_launches():
    """300 frames of mixed sizes: two chunks of 256, 4 kernels each (the host entry point adds one packing kernel a chunk)."""
    rng = np.random.default_rng(8)
    frames = [_smooth(rng, int(rng.integers(1, 80)), int(rng.integers(1, 80))) for _ in range(300)]
    det = _det()
    ctx = det.model.context(det.device, 512, 640, 1)
    want = [_imencode(f) for f in frames]
    n0 = ctx.launch_count()
    assert det.encode_jpeg([torch.from_numpy(f).cuda() for f in frames]) == want
    assert ctx.launch_count() - n0 == 4 * 2
    n0 = ctx.launch_count()
    assert det.encode_jpeg(frames) == want
    assert ctx.launch_count() - n0 == 5 * 2


def test_decoder_output_fed_back_and_round_trip():
    det = _det()
    rng = np.random.default_rng(12)
    frames = _shipped()[:6] + [_smooth(rng, 37, 53), rng.integers(0, 256, (33, 17, 3), dtype=np.uint8)]
    for s in (S420, S422, S444):
        for q in (50, 95):
            files = det.encode_jpeg(frames, quality=q, sampling=s)
            assert files == [_imencode(f, q, s) for f in frames]
            back = det.decode_jpeg(files)                  # cuda frames: the decoder's output, straight back into the encoder
            for f, b, data in zip(frames, back, files):
                ref = cv2.imdecode(np.frombuffer(_imencode(f, q, s), np.uint8), cv2.IMREAD_COLOR)
                assert np.array_equal(b.cpu().numpy(), ref)
            again = det.encode_jpeg(back, quality=q, sampling=s)
            assert again == [_imencode(b.cpu().numpy(), q, s) for b in back]
    # a non-contiguous cuda view is taken too
    f = torch.from_numpy(_shipped()[0]).cuda()
    view = f[10:300:2, 5:400]
    assert det.encode_jpeg([view])[0] == _imencode(view.cpu().numpy())


def test_bad_arguments_launch_nothing():
    det = _det()
    ctx = det.model.context(det.device, 512, 640, 1)
    ok = np.zeros((16, 16, 3), np.uint8)
    n0 = ctx.launch_count()
    bad = [
        (dict(frames=[ok, np.zeros((16, 16), np.uint8)]), "frame 1 is a gray"),
        (dict(frames=[ok, ok, np.zeros((16385, 2, 3), np.uint8)]), "frame 2 is 16385x2"),
        (dict(frames=[ok, np.zeros((4, 4, 3), np.float32)]), "frame 1 is float32"),
        (dict(frames=[ok], quality=0), "quality 0"),
        (dict(frames=[ok], quality=101), "quality 101"),
        (dict(frames=[ok], sampling=cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411), "sampling factor"),
        (dict(frames=[ok, torch.from_numpy(ok).cuda()]), "all on the host or all on the device"),
        (dict(frames=[]), "non-empty"),
    ]
    for kw, msg in bad:
        with pytest.raises(yf.YfError, match=msg):
            det.encode_jpeg(**kw)
    # the C entry point refuses an output buffer without room for the bound, before anything runs
    l = yf.lib()
    dev = torch.from_numpy(ok).cuda()
    out = torch.empty((1000,), dtype=torch.uint8, device="cuda")
    lens = torch.empty((1,), dtype=torch.int64, device="cuda")
    foff, h, w, oo = np.zeros(1, np.int64), np.full(1, 16, np.int32), np.full(1, 16, np.int32), np.zeros(1, np.int64)
    rc = l.yf_encode_jpeg(ctx.handle, dev.data_ptr(), 1, foff.ctypes.data, h.ctypes.data, w.ctypes.data, 95, S420, out.data_ptr(),
                          oo.ctypes.data, out.numel(), lens.data_ptr(), None)
    assert rc == -1 and "outside the 1000-byte output buffer" in l.yf_last_error(ctx.handle).decode()
    assert ctx.launch_count() == n0


def test_host_entry_cap_too_small():
    det = _det()
    ctx = det.model.context(det.device, 512, 640, 1)
    frames = _shipped()[:3]
    want = [_imencode(f) for f in frames]
    off, Ho, Wo, nbytes = yf.frame_layout(frames)
    buf = np.zeros(nbytes, np.uint8)
    for f, o in zip(frames, off):
        buf[int(o):int(o) + f.size] = f.reshape(-1)
    total = sum(map(len, want))
    l = yf.lib()
    out = np.full(total + 64, 0xAB, np.uint8)
    ln = np.zeros(3, np.int64)
    rc = l.yf_encode_host_jpeg(ctx.handle, buf.ctypes.data, nbytes, 3, off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data, 95, S420,
                               out.ctypes.data, total - 1, ln.ctypes.data, None)
    assert rc == -1 and "take %d bytes" % total in l.yf_last_error(ctx.handle).decode()
    assert (out == 0xAB).all() and list(ln) == [len(x) for x in want]
    rc = l.yf_encode_host_jpeg(ctx.handle, buf.ctypes.data, nbytes, 3, off.ctypes.data, Ho.ctypes.data, Wo.ctypes.data, 95, S420,
                               out.ctypes.data, total, ln.ctypes.data, None)
    assert rc == 0 and out[:total].tobytes() == b"".join(want) and (out[total:] == 0xAB).all()


def _run_driver(det, src, out, batch_size):
    records = []

    class Hd(logging.Handler):
        def emit(self, r):
            records.append(r.getMessage())
    logger = logging.getLogger("yf-test-jpeg-enc-%s" % out)
    logger.setLevel(logging.INFO)
    logger.addHandler(Hd())
    det.logger = logger
    os.makedirs(out)
    det.batch_detect_batched(src, out, batch_size=batch_size)
    return records


def _strip_times(line):
    return line.split(", infer time:")[0] if line.startswith("image_name:") else "avg"


def _same_dirs(a, b):
    assert sorted(os.listdir(a)) == sorted(os.listdir(b))
    for n in os.listdir(a):
        with open(os.path.join(a, n), "rb") as x, open(os.path.join(b, n), "rb") as y:
            assert x.read() == y.read(), n


def test_batch_driver_output_unchanged(tmp_path, monkeypatch):
    """40 shipped files at batch 32 (extensions .jpg and .JPG): the first batch's results are encoded on the device, the last 8 are
    written by cv2.imwrite; result files and log lines equal a run that writes everything with cv2.imwrite."""
    det = _det()
    src = str(tmp_path / "in")
    os.makedirs(src)
    for i, n in enumerate((sorted(os.listdir(IMAGES)) * 2)[:40]):
        shutil.copy(os.path.join(IMAGES, n), os.path.join(src, "%02d_%s" % (i, n if i % 3 else n[:-4] + ".JPG")))
    calls = []
    real = det.encode_jpeg
    monkeypatch.setattr(det, "encode_jpeg", lambda frames, *a, **k: calls.append(len(frames)) or real(frames, *a, **k))
    monkeypatch.setattr(det, "JPEG_ENCODE_MIN_BATCH", 32)
    new = _run_driver(det, src, str(tmp_path / "new"), 32)
    assert calls == [32]
    monkeypatch.setattr(det, "JPEG_ENCODE_MIN_BATCH", 10 ** 9)
    old = _run_driver(det, src, str(tmp_path / "old"), 32)
    assert calls == [32]
    assert [_strip_times(x) for x in new] == [_strip_times(x) for x in old] and len(new) == 41
    _same_dirs(str(tmp_path / "old"), str(tmp_path / "new"))


def test_batch_driver_png_stays_with_cv2(tmp_path, monkeypatch):
    """JPEGs, a progressive JPEG and a PNG in one folder, every batch eligible: the JPEG results are encoded on the device, the PNG
    result is still a PNG written by cv2; everything equals a run without device encoding."""
    det = _det()
    monkeypatch.setattr(det, "JPEG_MIN_BATCH", 1)
    src = tmp_path / "in"
    src.mkdir()
    for n in sorted(os.listdir(IMAGES))[:6]:
        shutil.copy(os.path.join(IMAGES, n), str(src))
    shutil.copy(os.path.join(JDIR, "reject_progressive.jpg"), str(src))
    shutil.copy(os.path.join(JDIR, "reject_png.png"), str(src))
    calls = []
    real = det.encode_jpeg
    monkeypatch.setattr(det, "encode_jpeg", lambda frames, *a, **k: calls.append(len(frames)) or real(frames, *a, **k))
    monkeypatch.setattr(det, "JPEG_ENCODE_MIN_BATCH", 1)
    new = _run_driver(det, str(src), str(tmp_path / "new"), 3)
    assert sum(calls) == 7 and len(new) == 9
    with open(str(tmp_path / "new" / "result_reject_png.png"), "rb") as f:
        assert f.read(8) == b"\x89PNG\r\n\x1a\n"
    monkeypatch.setattr(det, "JPEG_ENCODE_MIN_BATCH", 10 ** 9)
    old = _run_driver(det, str(src), str(tmp_path / "old"), 3)
    assert [_strip_times(x) for x in new] == [_strip_times(x) for x in old]
    _same_dirs(str(tmp_path / "old"), str(tmp_path / "new"))
