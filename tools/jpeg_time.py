"""Times the device JPEG decoder (profiles/r04_jpeg.txt):
    python tools/jpeg_time.py [--out FILE] [--reps 15]

1. decode kernel time per 256 files and per stage (torch.profiler, CUDA activities), the shipped 640x512 gray images cycled and
   1920x1080 4:2:0 colour files, for both thread mappings of the entropy kernel (one file per warp, one file per lane);
2. end to end, files in host memory -> detections at 640x512, batch 256: detect_jpeg, host cv2.imdecode on one thread +
   detect_frames, host cv2.imdecode over a thread pool of every host core + detect_frames;
3. batch-1 latency of detect_jpeg against cv2.imdecode + detect_frames;
4. batch_detect_batched wall time on 1024 files (the shipped images under distinct names) with the device decoder and with the host
   decoder (jpeg_probe made to turn every file down), at batch 8 and 32.
Arms alternate within one process; the wall times are medians, the kernel times means over the profiled calls. The card's name and power limit are read in the same run."""
import argparse
import logging
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import yolo_fastest_b200 as yf  # noqa: E402
from yolo_fastest_b200 import detector  # noqa: E402

IMAGES = os.path.join(ROOT, "tests", "golden", "images")
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def med(xs):
    return statistics.median(xs)


def host_decode(datas, pool=None):
    f = lambda d: cv2.imdecode(np.frombuffer(d, np.uint8), cv2.IMREAD_COLOR)  # noqa: E731
    return list(pool.map(f, datas)) if pool else [f(d) for d in datas]


def kernel_times(det, datas, fpw, reps):
    """per-stage device time (ms) of one decode call, from torch.profiler over `reps` calls"""
    from torch.profiler import ProfilerActivity, profile
    os.environ["YF_JPEG_FILES_PER_WARP"] = str(fpw)
    det.decode_jpeg(datas)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            det.decode_jpeg(datas)
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        for k in ("jpeg_entropy_kernel", "jpeg_idct_kernel", "jpeg_color_kernel"):
            if k in e.name:
                tot[k] = tot.get(k, 0.0) + e.device_time_total / 1000.0
    return {k: v / reps for k, v in tot.items()}


def call_ms(fn, reps):
    out = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1000)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file (default: stdout only)")
    ap.add_argument("--reps", type=int, default=15)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say("card: %s" % q.stdout.strip().splitlines()[0])
    say("host cores: %d, cv2 %s, torch %s" % (os.cpu_count(), cv2.__version__, torch.__version__))
    det = yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(ROOT, "tests", "golden", "weights", "yolo_fastest_512x640.pth"),
                         yf.config_for("512x640"), None)
    shipped = [open(os.path.join(IMAGES, n), "rb").read() for n in sorted(os.listdir(IMAGES))]
    gray256 = [shipped[i % len(shipped)] for i in range(256)]
    rng = np.random.default_rng(1)
    colour = []
    for i in range(16):
        img = cv2.GaussianBlur(rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8), (9, 9), 4)
        ok, buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420])
        colour.append(buf.tobytes())
    colour256 = [colour[i % 16] for i in range(256)]
    det.model.context(det.device, 512, 640, 256)
    for d in (gray256[:4], colour256[:4]):                 # the device output is cv2's before anything is timed
        for g, f in zip(det.decode_jpeg(d), d):
            assert np.array_equal(g.cpu().numpy(), cv2.imdecode(np.frombuffer(f, np.uint8), cv2.IMREAD_COLOR))

    say("\n1. decode kernels, ms per call of 256 files (torch.profiler, mean of %d calls; file bytes: gray %.1f MB, colour %.1f MB)"
        % (a.reps, sum(map(len, gray256)) / 1e6, sum(map(len, colour256)) / 1e6))
    say("%-28s %-18s %10s %10s %10s %10s" % ("files", "entropy mapping", "entropy", "idct", "colour", "sum"))
    for name, datas in (("shipped 640x512 gray", gray256), ("1920x1080 4:2:0 colour", colour256)):
        for fpw, label in ((1, "1 file / warp"), (32, "1 file / lane")):
            t = kernel_times(det, datas, fpw, a.reps)
            e, i, c = t.get("jpeg_entropy_kernel", 0), t.get("jpeg_idct_kernel", 0), t.get("jpeg_color_kernel", 0)
            say("%-28s %-18s %10.3f %10.3f %10.3f %10.3f" % (name, label, e, i, c, e + i + c))
    os.environ.pop("YF_JPEG_FILES_PER_WARP", None)

    say("\n2. end to end, 256 shipped files in host memory -> detections (640x512), ms per batch, median of %d, arms alternating" % a.reps)
    pool = ThreadPoolExecutor(os.cpu_count())
    arms = {
        "detect_jpeg (device decode)": lambda: det.detect_jpeg(gray256),
        "cv2.imdecode 1 thread + detect_frames": lambda: det.detect_frames(host_decode(gray256)),
        "cv2.imdecode %d threads + detect_frames" % os.cpu_count(): lambda: det.detect_frames(host_decode(gray256, pool)),
    }
    want = det.detect_frames(host_decode(gray256))
    assert det.detect_jpeg(gray256) == want
    times = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, fn in arms.items():
            times[k] += call_ms(fn, 1)
    for k, v in times.items():
        say("  %-42s %9.2f ms  %8.0f img/s" % (k, med(v), 256 / med(v) * 1000))

    say("\n3. batch-1 latency, one shipped file, ms, median of %d" % (4 * a.reps))
    one = shipped[:1]
    arms1 = {"detect_jpeg": lambda: det.detect_jpeg(one), "cv2.imdecode + detect_frames": lambda: det.detect_frames(host_decode(one))}
    t1 = {k: [] for k in arms1}
    for k, fn in arms1.items():
        fn()
    for _ in range(4 * a.reps):
        for k, fn in arms1.items():
            t1[k] += call_ms(fn, 1)
    for k, v in t1.items():
        say("  %-42s %9.3f ms" % (k, med(v)))

    say("\n4. batch_detect_batched on 1024 files (shipped images, distinct names), wall seconds, median of 3, arms alternating")
    tmp = tempfile.mkdtemp()
    try:
        src = os.path.join(tmp, "in")
        os.makedirs(src)
        names = sorted(os.listdir(IMAGES))
        for i in range(1024):
            shutil.copy(os.path.join(IMAGES, names[i % 20]), os.path.join(src, "%04d_%s" % (i, names[i % 20])))
        det.logger = logging.getLogger("jpeg_time")
        probe = detector.jpeg_probe

        def reject(data):
            raise yf.YfError("host decoder arm")

        def run(bs, device):
            detector.jpeg_probe = probe if device else reject
            det.JPEG_MIN_BATCH = 1 if device else yf.Detect_YOLO.JPEG_MIN_BATCH      # the device arm decodes every batch on the device
            out = os.path.join(tmp, "out")
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(out)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            det.batch_detect_batched(src, out, batch_size=bs)
            torch.cuda.synchronize()
            return time.perf_counter() - t0
        for bs in (8, 32):
            res = {"device": [], "host": []}
            run(bs, True), run(bs, False)
            for _ in range(3):
                res["device"].append(run(bs, True))
                res["host"].append(run(bs, False))
            say("  batch %2d: device decode %.2f s (%.0f img/s), cv2.imread %.2f s (%.0f img/s)"
                % (bs, med(res["device"]), 1024 / med(res["device"]), med(res["host"]), 1024 / med(res["host"])))
        detector.jpeg_probe = probe
        det.JPEG_MIN_BATCH = yf.Detect_YOLO.JPEG_MIN_BATCH
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
