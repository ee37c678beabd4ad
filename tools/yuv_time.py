"""Times the YUV 4:2:0 path (profiles/r06_yuv.txt):
    python tools/yuv_time.py [--out FILE] [--reps 21]

1. kernel time of one call on 256 NV12 cuda frames (CUDA events around the call; the input alternates between two sets of 256 frames,
   so consecutive calls do not read from L2 what the previous one left there):
   - the fused pre-processing (yf_preprocess_yuv420) for 640x512 frames to a gray 640x512 and 320x256 network and to a colour 320x256
     network, and for 1920x1080 frames to a gray 640x512 network;
   - yf_preprocess_frames on the same frames already converted to BGR;
   - the conversion alone (yf_yuv420_to_bgr);
2. end to end, 256 frames to detection rows (host clock around calls that end in a synchronisation), 640x512 and 1920x1080 frames, gray
   640x512 network: detect_yuv from cuda NV12 frames, against the path without it: the frames copied to the host, cv2.cvtColor per
   frame, detect_frames.
Arms alternate within one process and report medians. Every arm's output is checked against cv2 before it is timed. The card's name,
power limit and maximum SM clock are read in the same run."""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import yolo_fastest_b200 as yf  # noqa: E402
from oracle import yuv_oracle as yo  # noqa: E402

IMAGES = os.path.join(ROOT, "tests", "golden", "images")
B = 256
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def detector(res, colour=False):
    path = os.path.join(ROOT, "tests", "golden", "weights", "yolo_fastest_%s.pth" % res)
    cfg = yf.config_for(res)
    if colour:                                           # the colour network of the tests: the gray checkpoint's stem widened to 3 planes
        from test_forward_gpu import _three_channel_sd

        class G:
            @staticmethod
            def sd(name):
                return torch.load(os.path.join(ROOT, "tests", "golden", "weights", name + ".pth"), map_location="cpu")
        path = os.path.join(os.environ.get("TMPDIR", "/tmp"), "yf_yuv_time_rgb.pth")
        torch.save(_three_channel_sd(G), path)
        io = cfg["io_params"]
        io["input_channel"] = 3
        io["input_shape"] = io["input_shape"][0:2] + [3]
    return yf.Detect_YOLO(torch.device("cuda:0"), path, cfg, None)


def nv12_frames(h, w):
    """B host NV12 frames in cv2's form: the shipped images resized to h x w, through cv2's BGR2YUV_I420"""
    imgs = [cv2.resize(cv2.imread(os.path.join(IMAGES, n)), (w, h)) for n in sorted(os.listdir(IMAGES))]
    out = []
    for i in range(B):
        i420 = cv2.cvtColor(imgs[i % len(imgs)], cv2.COLOR_BGR2YUV_I420)
        out.append(yo.from_planes(*yo.planes(i420, "i420"), "nv12"))
    return out


class DeviceSet:
    """B cuda NV12 frames in one allocation and their BGR frames (cv2's conversion) in another, with the C descriptors of both"""

    def __init__(self, frames):
        h, w = frames[0].shape[0] * 2 // 3, frames[0].shape[1]
        self.yuv = torch.from_numpy(np.stack(frames)).cuda()
        self.desc, _, self.base, self.nbytes = yf.yuv_layout(list(self.yuv), "nv12")
        self.bgr_host = [cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in frames]
        self.bgr = torch.from_numpy(np.stack(self.bgr_host)).cuda()
        self.off = np.arange(B, dtype=np.int64) * h * w * 3
        self.Ho, self.Wo = np.full(B, h, np.int32), np.full(B, w, np.int32)


def event_ms(fn, sets, reps):
    """median device time of fn(set) over reps calls, the sets taken in turn"""
    ts = []
    for r in range(reps):
        s = sets[r % len(sets)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(s)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def kernels(reps):
    lib = yf.lib()
    say("1. kernels, ms per call of %d NV12 cuda frames (CUDA events, median of %d calls alternating between two input sets of %d "
        "frames)" % (B, reps, B))
    say("%-40s %12s %16s %12s %9s" % ("frames -> network input", "fused yuv", "frames from BGR", "yuv_to_bgr", "NV12 MB"))
    cache = {}
    for (fh, fw), res, colour in [((512, 640), "512x640", False), ((512, 640), "256x320", False), ((512, 640), "256x320", True),
                                  ((1080, 1920), "512x640", False)]:
        if (fh, fw) not in cache:
            hf = nv12_frames(fh, fw)
            cache = {(fh, fw): [DeviceSet(hf), DeviceSet(hf)]}
        sets = cache[(fh, fw)]
        det = detector(res, colour)
        H, W, ch = det.input_shape
        ctx = det.model.context(det.device, H, W, B)
        out = torch.empty((B, ch, H, W), dtype=torch.uint8, device="cuda")
        bgr_out = torch.empty((B * fh * fw * 3,), dtype=torch.uint8, device="cuda")
        s0 = sets[0]
        # outputs against cv2 before timing
        want = det.pre_process_frames(s0.bgr_host).cpu().numpy()
        got = det.pre_process_yuv(list(s0.yuv), "nv12").cpu().numpy()
        assert np.array_equal(got.reshape(want.shape), want), "fused pre-processing differs from cv2 + pre_process_frames"
        bgr = det.yuv_to_bgr(list(s0.yuv), "nv12")
        assert all(np.array_equal(g.cpu().numpy(), w) for g, w in zip(bgr, s0.bgr_host)), "yuv_to_bgr differs from cv2"

        def fused(s):
            yf._lib.check(lib.yf_preprocess_yuv420(ctx.handle, s.base, s.nbytes, B, s.desc.ctypes.data, out.data_ptr(), None), ctx.handle)

        def frames(s):
            yf._lib.check(lib.yf_preprocess_frames(ctx.handle, s.bgr.data_ptr(), B, s.off.ctypes.data, s.Ho.ctypes.data, s.Wo.ctypes.data,
                                                   out.data_ptr(), None), ctx.handle)

        def conv(s):
            yf._lib.check(lib.yf_yuv420_to_bgr(ctx.handle, s.base, s.nbytes, B, s.desc.ctypes.data, bgr_out.data_ptr(), s.off.ctypes.data,
                                               bgr_out.numel(), None), ctx.handle)
        for fn in (fused, frames, conv):                 # warm-up of every shape
            fn(sets[0])
            fn(sets[1])
        torch.cuda.synchronize()
        t = {fn: [] for fn in (fused, frames, conv)}
        for _ in range(3):                               # arms alternate
            for fn in (fused, frames, conv):
                t[fn].append(event_ms(fn, sets, reps))
        what = "%dx%d -> %s %dx%d" % (fw, fh, "colour" if colour else "gray", W, H)
        say("%-40s %12.3f %16.3f %12.3f %9.1f" % (what, statistics.median(t[fused]), statistics.median(t[frames]),
                                                  statistics.median(t[conv]), s0.nbytes / 1e6))
        del det, ctx
    say()


def end_to_end(reps):
    say("2. end to end, %d frames -> detection rows, gray 640x512 network, ms per batch (host clock around synchronised calls, median "
        "of %d, arms alternating)" % (B, reps))
    det = detector("512x640")
    for fh, fw in [(512, 640), (1080, 1920)]:
        hf = nv12_frames(fh, fw)
        dev = [torch.from_numpy(f).cuda() for f in hf]

        def device_path():
            return det.detect_yuv(dev, "nv12")

        def host_path():
            host = [f.cpu().numpy() for f in dev]
            return det.detect_frames([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in host])
        a, b = device_path(), host_path()
        assert a == b and sum(len(r) for r in a) > 0, "detect_yuv rows differ from cv2.cvtColor + detect_frames"
        t = {device_path: [], host_path: []}
        for _ in range(reps):
            for fn in (device_path, host_path):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                t[fn].append((time.perf_counter() - t0) * 1e3)
        for fn, name in ((device_path, "detect_yuv, cuda NV12 frames"), (host_path, "to host + cv2.cvtColor + detect_frames")):
            m = statistics.median(t[fn])
            say("  %4dx%-4d %-44s %9.2f ms %8.0f img/s" % (fw, fh, name, m, B / m * 1e3))
    say()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report to this file (default: stdout only)")
    ap.add_argument("--reps", type=int, default=21)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/yuv_time.py measures on the GPU and found none")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    say("# tools/yuv_time.py (YUV 4:2:0 frames on the device, DESIGN.md §5.9); one run, all arms in one process")
    say("card: %s" % (q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "not read (nvidia-smi failed)"))
    say("host cores: %d, cv2 %s, torch %s" % (os.cpu_count(), cv2.__version__, torch.__version__))
    say()
    kernels(args.reps)
    end_to_end(args.reps)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
