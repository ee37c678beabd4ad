"""Device JPEG decoder (yf_decode_jpeg / yf_detect_host_jpeg) against cv2: byte-equal frames for the whole corpus, the shipped images,
a batch of more than one descriptor chunk and large generated files; detect_jpeg rows equal to detect_frames(cv2.imread ...); the
batched file driver's output unchanged; unsupported and corrupt files reported by index."""
import logging
import os
import shutil

import numpy as np
import pytest
import torch

import yolo_fastest_b200 as yf
from yolo_fastest_b200 import detector
from conftest import rows_equal

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
JDIR = os.path.join(HERE, "golden", "jpeg")
IMAGES = os.path.join(HERE, "golden", "images")
cv2 = pytest.importorskip("cv2")


def _det(res="512x640"):
    return yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(HERE, "golden", "weights", "yolo_fastest_%s.pth" % res), yf.config_for(res), None)


def _shipped():
    return [os.path.join(IMAGES, n) for n in sorted(os.listdir(IMAGES))]


def _corpus():
    return [os.path.join(JDIR, n) for n in sorted(os.listdir(JDIR)) if not n.startswith("reject_")]


def _imdecode(path_or_bytes):
    b = np.fromfile(path_or_bytes, np.uint8) if isinstance(path_or_bytes, str) else np.frombuffer(path_or_bytes, np.uint8)
    return cv2.imdecode(b, cv2.IMREAD_COLOR)


def test_corpus_and_shipped_images_byte_equal():
    det = _det()
    golden = np.load(os.path.join(HERE, "golden", "jpeg.npz"))
    files = _corpus() + _shipped()
    n0 = det.model.context(det.device, 512, 640, len(files)).launch_count()
    got = det.decode_jpeg(files)
    assert det.model._ctx.launch_count() - n0 == 3          # one chunk: entropy, IDCT, colour
    for f, g in zip(files, got):
        g = g.cpu().numpy()
        assert np.array_equal(g, _imdecode(f)), f
        n = os.path.basename(f)
        if n in golden:
            assert np.array_equal(g, golden[n]), n


def test_more_than_one_chunk():
    det = _det()
    files = (_corpus() * 5)[:300]
    n0 = det.model.context(det.device, 512, 640, len(files)).launch_count()
    got = det.decode_jpeg(files)
    assert det.model._ctx.launch_count() - n0 == 3 * 2        # bounded by the chunk count (256 files a chunk)
    for f, g in zip(files, got):
        assert np.array_equal(g.cpu().numpy(), _imdecode(f)), f


def test_large_generated_files():
    rng = np.random.default_rng(3)
    cases = [((1080, 1920, 3), cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420), ((1080, 1920, 3), cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422),
             ((3000, 4000), None), ((8, 16384), None)]
    datas = []
    for shape, sf in cases:
        img = cv2.GaussianBlur(rng.integers(0, 256, shape, dtype=np.uint8), (7, 7), 3)
        img = np.clip(img.astype(np.int16) + rng.integers(-12, 13, shape), 0, 255).astype(np.uint8)
        params = [cv2.IMWRITE_JPEG_QUALITY, 92] + ([cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf] if sf else [])
        ok, buf = cv2.imencode(".jpg", img, params)
        datas.append(buf.tobytes())
    got = _det().decode_jpeg(datas)
    for d, g in zip(datas, got):
        assert np.array_equal(g.cpu().numpy(), _imdecode(d)), g.shape


@pytest.mark.parametrize("res", ["256x320", "512x640"])
def test_detect_jpeg_equals_detect_frames(res):
    det = _det(res)
    files = _shipped()
    want = det.detect_frames([cv2.imread(f) for f in files])
    got = det.detect_jpeg(files)
    assert any(len(r) for r in want)
    for w, g in zip(want, got):
        rows_equal(w, g)
    assert det.detect_jpeg(files, max_det=1) == got            # the overflow rerun, nothing cut


def test_detect_jpeg_colour_network(tmp_path):
    from test_frames_gpu import _colour_detector
    from test_forward_gpu import _three_channel_sd

    class G:
        @staticmethod
        def sd(name):
            return torch.load(os.path.join(HERE, "golden", "weights", name + ".pth"), map_location="cpu")
    path = str(tmp_path / "rgb.pth")
    torch.save(_three_channel_sd(G), path)
    det = _colour_detector(path, "256x320")
    rng = np.random.default_rng(11)
    datas = []
    for i, f in enumerate(_shipped()[:8]):
        g = cv2.imread(f)
        tint = np.clip(g.astype(np.int16) + rng.integers(-40, 41, (1, 1, 3)), 0, 255).astype(np.uint8)
        sf = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444][i % 3]
        ok, buf = cv2.imencode(".jpg", tint[: 300 + 20 * i, : 500 + 7 * i], [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf])
        datas.append(buf.tobytes())
    want = det.detect_frames([_imdecode(d) for d in datas])
    got = det.detect_jpeg(datas)
    assert any(len(r) for r in want)
    for w, g in zip(want, got):
        rows_equal(w, g)


def _run_driver(det, src, out, batch_size):
    records = []

    class Hd(logging.Handler):
        def emit(self, r):
            records.append(r.getMessage())
    logger = logging.getLogger("yf-test-jpeg-%s" % out)
    logger.setLevel(logging.INFO)
    logger.addHandler(Hd())
    det.logger = logger
    os.makedirs(out)
    det.batch_detect_batched(src, out, batch_size=batch_size)
    return records


def _strip_times(line):
    return line.split(", infer time:")[0] if line.startswith("image_name:") else "avg"


def test_batch_driver_output_unchanged(tmp_path, monkeypatch):
    """40 files at batch 32: the first batch is decoded on the device, the last 8 files on the host (below JPEG_MIN_BATCH); the
    result files and log lines equal those of the host decoder for every file."""
    det = _det()
    src = str(tmp_path / "in")
    os.makedirs(src)
    for i, f in enumerate((_shipped() * 2)[:40]):
        shutil.copy(f, os.path.join(src, "%02d_%s" % (i, os.path.basename(f))))
    calls = []
    real = det._detect_jpeg
    monkeypatch.setattr(det, "_detect_jpeg", lambda *a: calls.append(len(a[1])) or real(*a))
    new = _run_driver(det, src, str(tmp_path / "new"), 32)
    assert calls == [32]

    def reject(data):
        raise yf.YfError("rejected for the comparison")
    monkeypatch.setattr(detector, "jpeg_probe", reject)
    old = _run_driver(det, src, str(tmp_path / "old"), 32)
    assert calls == [32]
    assert [_strip_times(x) for x in new] == [_strip_times(x) for x in old] and len(new) == 41
    for n in os.listdir(str(tmp_path / "old")):
        with open(os.path.join(str(tmp_path / "old"), n), "rb") as a, open(os.path.join(str(tmp_path / "new"), n), "rb") as b:
            assert a.read() == b.read(), n


def test_batch_driver_mixed_folder(tmp_path, monkeypatch):
    """JPEGs, a progressive JPEG and a PNG in one folder: batches of JPEGs go to the device, the others to cv2.imread."""
    det = _det()
    monkeypatch.setattr(det, "JPEG_MIN_BATCH", 1)
    src = tmp_path / "in"
    src.mkdir()
    for f in _shipped()[:6]:
        shutil.copy(f, str(src))
    shutil.copy(os.path.join(JDIR, "reject_progressive.jpg"), str(src))
    shutil.copy(os.path.join(JDIR, "reject_png.png"), str(src))
    records = _run_driver(det, str(src), str(tmp_path / "out"), 3)
    assert len(records) == 9 and len(os.listdir(str(tmp_path / "out"))) == 8


def test_unsupported_file_named_and_nothing_launched():
    det = _det()
    files = _shipped()[:3] + [os.path.join(JDIR, "reject_progressive.jpg")]
    ctx = det.model.context(det.device, 512, 640, len(files))
    n0 = ctx.launch_count()
    with pytest.raises(yf.YfError, match="file 3: progressive"):
        det.detect_jpeg(files)
    with pytest.raises(yf.YfError, match="file 3: progressive"):
        det.decode_jpeg(files)
    assert ctx.launch_count() == n0


def test_truncated_scan_sets_the_corrupt_bit():
    """Once, without repeats: a file cut inside its scan. The decoder reads only the file's bytes, marks it, and the call raises."""
    det = _det()
    good = open(_shipped()[0], "rb").read()
    cut = good[: len(good) // 2]
    with pytest.raises(yf.YfError, match="file 1: corrupt"):
        det.detect_jpeg([good, cut])
    assert np.array_equal(det.decode_jpeg([good])[0].cpu().numpy(), _imdecode(good))
