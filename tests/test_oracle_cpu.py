"""The oracle against the golden vectors frozen from the reference (tests/golden/make_golden.py) and
against the facts the reference publishes.  CPU only."""
import contextlib
import os

import numpy as np
import torch

from oracle import yolo_oracle as O
from yolo_fastest_b200 import COCO_ANCHORS, config_for

from conftest import rows_equal

# The golden heads were frozen by CPU runs at 8 threads. oneDNN's fp32 convolutions split their reduction by the thread count (at 12 or
# 16 threads the sums run in another order; at 1 thread ATen runs the 1x1 convolutions outside oneDNN), so the bit-identity checks
# reproduce the goldens at that count whatever the host's core count.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def _golden_threads():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(n)


def _io(res):
    return config_for(res)["io_params"]


def test_forward_matches_golden_heads(gold):
    for res in ("256x320", "512x640"):
        g = gold.res[res]
        sd = gold.sd("yolo_fastest_" + res)
        n = min(4, len(g["u8"]))
        x = torch.cat([O.preprocess_gray(u) for u in g["u8"][:n]], 0)
        hl, hs = O.forward(sd, x)
        # batched oneDNN kernels may pick another blocking than the batch-1 run that made the goldens
        assert torch.allclose(hl, torch.from_numpy(g["head_large"][:n]), rtol=1e-5, atol=1e-5)
        assert torch.allclose(hs, torch.from_numpy(g["head_small"][:n]), rtol=1e-5, atol=1e-5)
        # one image at batch 1, exactly as the golden script ran it: bit-identical
        with _golden_threads():
            h1 = O.forward(sd, x[:1])
        assert torch.equal(h1[0][0], torch.from_numpy(g["head_large"][0]))
        assert torch.equal(h1[1][0], torch.from_numpy(g["head_small"][0]))


def test_forward_synthetic_golden(gold):
    for res in ("256x320",):
        g = gold.res[res]
        io = _io(res)
        H, W = io["input_shape"][0:2]
        gen = torch.Generator().manual_seed(int(g["syn_seed"]))
        u8 = torch.randint(0, 256, (2, H, W), generator=gen, dtype=torch.uint8).numpy()
        x = torch.cat([O.preprocess_gray(s) for s in u8], 0)
        hl, hs = O.forward(gold.sd("yolo_fastest_" + res), x)
        assert torch.allclose(hl, torch.from_numpy(g["syn_head_large"]), rtol=1e-5, atol=1e-5)
        assert torch.allclose(hs, torch.from_numpy(g["syn_head_small"]), rtol=1e-5, atol=1e-5)


def test_decode_and_nms_match_golden(gold):
    for res in ("256x320", "512x640"):
        g = gold.res[res]
        io = _io(res)
        for i in range(len(g["head_large"])):
            pred = (g["head_large"][i:i + 1], g["head_small"][i:i + 1])
            dec = O.decode_box(pred, io["anchors"], io["input_shape"], io["conf_thre"], io["num_anchors"], io["num_cls"])
            rows_equal(g["decoded_%02d" % i], dec, conf_tol=0)
            kept = O.detect_postprocess(pred, io["anchors"], io["input_shape"], io["conf_thre"], io["nms_thre"],
                                        io["num_anchors"], io["num_cls"])
            rows_equal(g["kept_%02d" % i], kept, conf_tol=0)
            adj = [list(r) for r in kept]
            if res == "256x320":
                O.adjust_coord(adj, io["input_shape"], io["origin_img_shape"])
            rows_equal(g["kept_adj_%02d" % i], adj, conf_tol=0)


def test_published_detect_flags(gold):
    """test_result/*/笔记本cpu(python)_test_result/cpu-test.log: every 256x320 image has targets; at 512x640
    only noCloud_2m_4359.jpg has none."""
    g1, g2 = gold.res["256x320"], gold.res["512x640"]
    assert g1["has_targets"].all()
    names = [str(n) for n in g2["names"]]
    assert [n for n, f in zip(names, g2["has_targets"]) if not f] == ["noCloud_2m_4359.jpg"]
    for res, g in (("256x320", g1), ("512x640", g2)):
        for i in range(20):
            assert (len(g["kept_%02d" % i]) > 0) == bool(g["has_targets"][i])


def test_example_boxes_from_survey(gold):
    """SURVEY.md §4: 256x320, Cloud_2m_4093.jpg keeps [132,112,169,132] conf .9836 and [69,69,98,100] conf .9114, class 2."""
    g = gold.res["256x320"]
    i = [str(n) for n in g["names"]].index("Cloud_2m_4093.jpg")
    k = g["kept_%02d" % i]
    assert [[int(v) for v in r[:4]] for r in k] == [[132, 112, 169, 132], [69, 69, 98, 100]]
    assert abs(k[0][4] - 0.9836) < 1e-4 and abs(k[1][4] - 0.9114) < 1e-4 and int(k[0][6]) == 2 and int(k[1][6]) == 2


def test_validation_flavour_matches_golden(gold):
    for res in ("256x320", "512x640"):
        g = gold.res[res]
        io = _io(res)
        for i in range(len(g["head_large"])):
            heads = (torch.from_numpy(g["head_large"][i:i + 1]), torch.from_numpy(g["head_small"][i:i + 1]))
            v = torch.cat([O.val_decode(heads[h], io["anchors"][h], io["num_cls"], io["input_shape"]) for h in range(2)], 1)
            out = O.val_nms(v, io["num_cls"], io["conf_thre"], io["nms_thre"])[0]
            want = g["val_%02d" % i]
            if len(want) == 0:
                assert out is None
            else:
                assert np.array_equal(out.numpy(), want)


def test_stress_golden(gold):
    g = gold.stress
    for b in range(2):
        pred = (g["head_large"][b:b + 1], g["head_small"][b:b + 1])
        kept = O.detect_postprocess(pred, COCO_ANCHORS, [416, 416, 1], 0.001, 0.2, 3, 80)
        rows_equal(g["kept_%02d" % b], kept, conf_tol=0)


def test_nms_properties():
    rng = np.random.default_rng(3)
    for n in (0, 1, 2, 17, 200):
        xy = rng.integers(0, 300, size=(n, 2))
        wh = rng.integers(0, 80, size=(n, 2))          # zero-area boxes included
        conf = np.sort(rng.random(n))[::-1]
        rows = [[int(x), int(y), int(x + w), int(y + h), float(c), 0.5, 0] for (x, y), (w, h), c in zip(xy, wh, conf)]
        kept = O.nms(rows, 0.2)
        assert O.nms(kept, 0.2) == kept                                     # idempotent
        assert all(kept[i][4] >= kept[i + 1][4] for i in range(len(kept) - 1))
        for i in range(len(kept)):                                          # no kept pair overlaps above the threshold
            for j in range(i + 1, len(kept)):
                assert not (O.cal_iou(kept[j], kept[i]) > 0.2)
        if n:
            assert kept[0] == rows[0]
    # empty union: NaN never suppresses (YOLO_ncnn.cpp:212,221-234)
    z = [[5, 5, 5, 5, 0.9, 0.5, 0], [5, 5, 5, 5, 0.8, 0.5, 0]]
    assert O.nms(z, 0.2) == z


def test_decode_overflow_domain():
    """|logit| > 709 raises OverflowError exactly like the reference's math.exp (detect.py:25,63-64)."""
    hl = np.zeros((1, 24, 2, 2), np.float32)
    hs = np.zeros((1, 24, 1, 1), np.float32)
    hl[0, 4, 0, 0] = -800.0
    try:
        O.decode_box((hl, hs), [[[1, 1]] * 3] * 2, [32, 32, 1], 0.5, 3, 3)
        raised = False
    except OverflowError:
        raised = True
    assert raised


def test_lite_oracle_matches_reference_golden(gold):
    """oracle.forward_lite against the unmodified reference's YoloFastest_lite outputs (tests/golden/make_golden_lite.py)."""
    g = np.load(os.path.join(gold.dir, "golden_lite.npz"))
    sd = O.lite_state_dict(gold.sd("yolo_fastest_256x320"))
    assert sd["head_5.weight"].shape == (72, 128, 1, 1) and sd["head_4.weight"].shape == (72, 96, 1, 1)
    for tag in ("a", "b"):
        B, H, W = (int(v) for v in g["shape_" + tag])
        x = (torch.randint(0, 256, (B, 1, H, W), generator=torch.Generator().manual_seed(int(g["seed"]))).float() - 128.0) / 255.0
        with _golden_threads():
            head = O.forward_lite(sd, x)
        assert torch.equal(head, torch.from_numpy(g["head_" + tag]))
