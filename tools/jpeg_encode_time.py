"""Times the device JPEG encoder (profiles/r05_jpeg_encode.txt):
    python tools/jpeg_encode_time.py [--out FILE] [--reps 11]

1. encode kernel time per call of 256 cuda frames, per kernel (torch.profiler, CUDA activities): the shipped 640x512 images at q95
   4:2:0, smooth 1920x1080 frames at q95 4:2:0, and 640x512 uniform noise at q100 4:4:4 (the worst case for code lengths and 0xFF
   stuffing);
2. end to end, 256 shipped 640x512 frames in host memory -> 256 bytes objects: encode_jpeg, cv2.imencode on one thread,
   cv2.imencode over a thread pool of every host core;
3. batch-1 latency: encode_jpeg of one shipped frame against cv2.imencode;
4. batch_detect_batched wall time on 1024 files (the shipped images under distinct names) with device encoding on
   (JPEG_ENCODE_MIN_BATCH 1) and off (every result through cv2.imwrite), at batch 4, 8 and 32, and where the wall time goes: reading
   the files, cv2.imread, drawing the boxes, encode_jpeg, writing the encoded bytes, cv2.imwrite (encode + write), and the rest
   (device decode + detection, logging, Python).
Arms alternate within one process; wall times are medians, kernel times means over the profiled calls. Every arm's output is checked
against cv2 before it is timed. The card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import builtins
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
KERNELS = ("jpeg_enc_dct_kernel", "jpeg_enc_len_kernel", "jpeg_enc_emit_kernel", "jpeg_enc_stuff_kernel")
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def med(xs):
    return statistics.median(xs)


def imencode(f, q=95, s=cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420):
    return cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s])[1].tobytes()


def kernel_times(det, frames, q, s, reps):
    """per-kernel device time (ms) of one encode_jpeg call on cuda frames, from torch.profiler over `reps` calls"""
    from torch.profiler import ProfilerActivity, profile
    det.encode_jpeg(frames, quality=q, sampling=s)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            det.encode_jpeg(frames, quality=q, sampling=s)
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        for k in KERNELS:
            if k in e.name:
                tot[k] = tot.get(k, 0.0) + e.device_time_total / 1000.0
    return {k: v / reps for k, v in tot.items()}


def call_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1000


class Buckets:
    """Wall time of the driver's host steps, by wrapping the calls it makes (restored by close())."""

    def __init__(self, det):
        self.t = {}
        self.det = det
        self.saved = (detector.plot_one_box, cv2.imread, cv2.imwrite, det.encode_jpeg)
        det.encode_jpeg = self.timed("encode_jpeg", det.encode_jpeg)
        detector.plot_one_box = self.timed("draw boxes", detector.plot_one_box)
        cv2.imread = self.timed("cv2.imread", cv2.imread)
        cv2.imwrite = self.timed("cv2.imwrite", cv2.imwrite)
        b = self

        class TimedFile:
            def __init__(self, path, mode="r", *a, **k):
                self.key = "write encoded bytes" if "w" in mode else "read files"
                t0 = time.perf_counter()
                self.f = builtins.open(path, mode, *a, **k)
                b.add(self.key, time.perf_counter() - t0)

            def __enter__(self):
                self.t0 = time.perf_counter()
                return self.f

            def __exit__(self, *exc):
                self.f.close()
                b.add(self.key, time.perf_counter() - self.t0)
        detector.open = TimedFile

    def add(self, k, dt):
        self.t[k] = self.t.get(k, 0.0) + dt

    def timed(self, k, fn):
        def w(*a, **kw):
            t0 = time.perf_counter()
            try:
                return fn(*a, **kw)
            finally:
                self.add(k, time.perf_counter() - t0)
        return w

    def close(self):
        detector.plot_one_box, cv2.imread, cv2.imwrite, self.det.encode_jpeg = self.saved
        del detector.open


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file (default: stdout only)")
    ap.add_argument("--reps", type=int, default=11)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say("card: %s" % q.stdout.strip().splitlines()[0])
    say("host cores: %d, cv2 %s, torch %s" % (os.cpu_count(), cv2.__version__, torch.__version__))
    det = yf.Detect_YOLO(torch.device("cuda:0"), os.path.join(ROOT, "tests", "golden", "weights", "yolo_fastest_512x640.pth"),
                         yf.config_for("512x640"), None)
    S420, S444 = cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444
    shipped = [cv2.imread(os.path.join(IMAGES, n)) for n in sorted(os.listdir(IMAGES))]
    ship256 = [shipped[i % len(shipped)] for i in range(256)]
    rng = np.random.default_rng(1)
    hd = [cv2.GaussianBlur(rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8), (9, 9), 4) for _ in range(16)]
    noise = [rng.integers(0, 256, (512, 640, 3), dtype=np.uint8) for _ in range(16)]
    sets = [("shipped 640x512, q95 4:2:0", ship256, 95, S420), ("1920x1080 smooth, q95 4:2:0", [hd[i % 16] for i in range(256)], 95, S420),
            ("640x512 noise, q100 4:4:4", [noise[i % 16] for i in range(256)], 100, S444)]
    for name, frames, qq, s in sets:                 # the device output is cv2's before anything is timed
        idx = list(range(0, 256, 37))
        got = det.encode_jpeg([torch.from_numpy(frames[i]).cuda() for i in idx], quality=qq, sampling=s)
        assert got == [imencode(frames[i], qq, s) for i in idx], name

    say("\n1. encode kernels, ms per call of 256 cuda frames (torch.profiler, mean of %d calls)" % a.reps)
    say("%-30s %10s %10s %10s %10s %10s %12s" % ("frames", "dct", "len+scan", "emit", "stuff", "sum", "output MB"))
    for name, frames, qq, s in sets:
        dev = [torch.from_numpy(f).cuda() for f in frames]
        t = kernel_times(det, dev, qq, s, a.reps)
        mb = sum(len(imencode(frames[i], qq, s)) for i in range(16)) * 16 / 1e6
        v = [t.get(k, 0.0) for k in KERNELS]
        say("%-30s %10.3f %10.3f %10.3f %10.3f %10.3f %12.1f" % (name, *v, sum(v), mb))
        del dev

    say("\n2. end to end, 256 shipped 640x512 frames in host memory -> 256 bytes objects (q95 4:2:0), ms per batch, median of %d, "
        "arms alternating" % a.reps)
    pool = ThreadPoolExecutor(os.cpu_count())
    arms = {
        "encode_jpeg (device)": lambda: det.encode_jpeg(ship256),
        "cv2.imencode 1 thread": lambda: [imencode(f) for f in ship256],
        "cv2.imencode %d threads" % os.cpu_count(): lambda: list(pool.map(imencode, ship256)),
    }
    want = arms["cv2.imencode 1 thread"]()
    for k, fn in arms.items():
        assert fn() == want, k
    times = {k: [] for k in arms}
    for _ in range(a.reps):
        for k, fn in arms.items():
            times[k].append(call_ms(fn))
    for k, v in times.items():
        say("  %-42s %9.2f ms  %8.0f img/s" % (k, med(v), 256 / med(v) * 1000))

    say("\n3. batch-1 latency, one shipped 640x512 frame, ms, median of %d" % (4 * a.reps))
    one = shipped[:1]
    arms1 = {"encode_jpeg": lambda: det.encode_jpeg(one), "cv2.imencode": lambda: [imencode(f) for f in one]}
    t1 = {k: [] for k in arms1}
    for k, fn in arms1.items():
        assert fn() == [imencode(one[0])], k
    for _ in range(4 * a.reps):
        for k, fn in arms1.items():
            t1[k].append(call_ms(fn))
    for k, v in t1.items():
        say("  %-42s %9.3f ms" % (k, med(v)))

    say("\n4. batch_detect_batched on 1024 files (shipped images, distinct names), wall seconds, median of 3, arms alternating; the "
        "device decoder as configured (JPEG_MIN_BATCH %d). Shares of the wall time (median run of each arm):" % det.JPEG_MIN_BATCH)
    tmp = tempfile.mkdtemp()
    try:
        src = os.path.join(tmp, "in")
        os.makedirs(src)
        names = sorted(os.listdir(IMAGES))
        for i in range(1024):
            shutil.copy(os.path.join(IMAGES, names[i % 20]), os.path.join(src, "%04d_%s" % (i, names[i % 20])))
        det.logger = logging.getLogger("jpeg_encode_time")

        def run(bs, device):
            det.JPEG_ENCODE_MIN_BATCH = 1 if device else 10 ** 9
            out = os.path.join(tmp, "out_%s" % device)
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(out)
            b = Buckets(det)
            try:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                det.batch_detect_batched(src, out, batch_size=bs)
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
            finally:
                b.close()
            return wall, b.t

        run(32, True), run(32, False)
        a_out, b_out = os.path.join(tmp, "out_True"), os.path.join(tmp, "out_False")
        for n in os.listdir(b_out):                       # both arms wrote the same files
            assert open(os.path.join(a_out, n), "rb").read() == open(os.path.join(b_out, n), "rb").read(), n
        for bs in (4, 8, 32):
            res = {True: [], False: []}
            run(bs, True), run(bs, False)
            for _ in range(3):
                res[True].append(run(bs, True))
                res[False].append(run(bs, False))
            walls = {k: med([w for w, _ in v]) for k, v in res.items()}
            say("  batch %2d: device encode %.2f s (%.0f img/s), cv2.imwrite %.2f s (%.0f img/s)"
                % (bs, walls[True], 1024 / walls[True], walls[False], 1024 / walls[False]))
            for arm in (True, False):
                wall, parts = sorted(res[arm], key=lambda x: x[0])[1]
                rest = wall - sum(parts.values())
                say("    %-14s " % ("device encode" if arm else "cv2.imwrite") +
                    ", ".join("%s %.0f%%" % (k, 100 * v / wall) for k, v in sorted(parts.items(), key=lambda x: -x[1])) +
                    ", rest (decode + detect, logging, Python) %.0f%%" % (100 * rest / wall))
        det.JPEG_ENCODE_MIN_BATCH = yf.Detect_YOLO.JPEG_ENCODE_MIN_BATCH
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
