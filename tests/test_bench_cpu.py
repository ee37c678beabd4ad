"""bench.py's host side: the --dump-outputs file format (dump_outputs) and the argument check of --steps."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench
from yolo_fastest_b200 import _lib

from conftest import ROOT


def _slab(counts, max_det):
    """A detect_device result: records 0..min(count, max_det) of image b set, every other byte 0xFF (unset memory)."""
    raw = np.full((len(counts), max_det, 56), 0xFF, np.uint8)
    recs = raw.view(_lib.DET_DTYPE).reshape(len(counts), max_det)
    for b, c in enumerate(counts):
        for k in range(min(c, max_det)):
            recs[b, k] = (10 * b + k, 1.5, 20.25, 30.0, 0.75 - 0.01 * k, 0.5, k % 3, b * max_det + k)
    status = torch.zeros(len(counts), dtype=torch.int32)
    status[1] = 2
    return torch.from_numpy(raw), torch.tensor(counts, dtype=torch.int32), status


def test_dump_outputs_format(tmp_path):
    out, counts, status = _slab([0, 2, 6], 4)
    bench.dump_outputs(str(tmp_path), out, counts, status)
    got = {n: np.load(tmp_path / (n + ".npy")) for n in ("detections", "counts", "status", "image_index")}
    assert sorted(os.listdir(tmp_path)) == ["counts.npy", "detections.npy", "image_index.npy", "status.npy"]
    assert all(a.dtype == np.float64 for a in got.values())
    d = got["detections"]
    assert d.shape == (3, 4, 8)
    assert not d[0].any() and not d[1, 2:].any()                 # slots without a record are 0, not the unset bytes
    assert d[1, 1].tolist() == [11.0, 1.5, 20.25, 30.0, 0.74, 0.5, 1.0, 5.0]
    assert d[2, :, 0].tolist() == [20.0, 21.0, 22.0, 23.0]        # count 6 > max_det 4: the slab's 4 records
    assert got["counts"].tolist() == [0.0, 2.0, 6.0] and got["status"].tolist() == [0.0, 2.0, 0.0]
    assert got["image_index"].tolist() == [0.0, 1.0, 2.0]


def test_dump_outputs_sample_is_bounded_and_fixed(tmp_path, monkeypatch):
    out, counts, status = _slab([1] * 50, 2)
    per_image = 8 * (2 * 8 + 3)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 7 * per_image)
    idx = []
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), out, counts, status)
        assert sum(os.path.getsize(tmp_path / run / f) - 128 for f in os.listdir(tmp_path / run)) <= 7 * per_image   # 128: .npy header
        idx.append(np.load(tmp_path / run / "image_index.npy"))
        d = np.load(tmp_path / run / "detections.npy")
        assert d.shape == (7, 2, 8) and d[:, 0, 0].tolist() == (10 * idx[-1]).tolist()
    assert idx[0].tolist() == idx[1].tolist() and len(set(idx[0])) == 7 and list(idx[0]) == sorted(idx[0])


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
