"""Device time of the frame pre-processing kernels: yf_preprocess_bgr (host tap table, one size per call) against
yf_preprocess_frames (taps computed in the kernel, sizes free), measured in the same process with CUDA events, the two arms
alternating, after warm-up, on frame batches larger than the 126 MB L2.

    python tools/prep_frames_time.py [--reps 30] [--out FILE]     (GPU box)

(a) 256 uniform 512x640 BGR frames -> gray 512x640 and 256x320, old vs new kernel
(b) the colour output ([B, 3, H, W] R, G, B planes) of the same frames
(c) a ragged batch of 256 frames cycling 512x640, 480x640, 333x517, 1080x1920, 128x160: new kernel in one call vs the old one
    called once per size (each call with a new size rebuilds and uploads its tap table)
(d) end to end from host frames: detect_bgr_batch(np.stack(frames)) vs detect_frames(frames), host clock around the call
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__  # noqa: E402

__graft_entry__.build()
import yolo_fastest_b200 as yf  # noqa: E402
from yolo_fastest_b200 import _lib  # noqa: E402

LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        q = "power limit not readable (%s)" % e
    return "%s, %s" % (name, q)


def timed(fn, reps):
    """median / min device ms of fn() over `reps` event-bracketed calls"""
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def ab(name, arms, reps, nbytes):
    """arms: [(label, fn)]; warm-up, then `reps` rounds alternating the arms; prints median / min and the ratio to the first arm"""
    for _, fn in arms:
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    res = {label: [] for label, _ in arms}
    for _ in range(reps):
        for label, fn in arms:
            res[label] += timed(fn, 1)
    base = float(np.median(res[arms[0][0]]))
    for label, _ in arms:
        med, lo = float(np.median(res[label])), float(np.min(res[label]))
        say("  %-44s median %8.3f ms  min %8.3f ms  %6.0f GB/s  x%.3f" % (name + " " + label, med, lo, nbytes / med / 1e6, med / base))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = yf.lib()
    dev = torch.device("cuda:0")
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)      # noqa: E731
    say("prep_frames_time: %s; torch %s; %d reps per arm, alternating" % (card(), torch.__version__, args.reps))
    B, Ho, Wo = 256, 512, 640
    rng = np.random.default_rng(1)
    uni = torch.from_numpy(rng.integers(0, 256, (B, Ho, Wo, 3), dtype=np.uint8)).to(dev)        # 251.7 MB > L2
    fb = Ho * Wo * 3
    off = np.arange(B, dtype=np.int64) * fb
    Hs, Ws = np.full(B, Ho, np.int32), np.full(B, Wo, np.int32)

    say("(a) uniform %d x %dx%d BGR frames -> gray: yf_preprocess_bgr vs yf_preprocess_frames" % (B, Ho, Wo))
    for (H, W) in ((512, 640), (256, 320)):
        ctx = _lib.Ctx(0, 1, 3, 3, B, H, W)
        out_old = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        out_new = torch.empty_like(out_old)
        old = lambda: _lib.check(lib.yf_preprocess_bgr(ctx.handle, uni.data_ptr(), B, Ho, Wo, out_old.data_ptr(), stream()), ctx.handle)  # noqa: E731
        new = lambda: _lib.check(lib.yf_preprocess_frames(ctx.handle, uni.data_ptr(), B, off.ctypes.data, Hs.ctypes.data, Ws.ctypes.data,  # noqa: E731
                                                          out_new.data_ptr(), stream()), ctx.handle)
        ab("-> %dx%d" % (H, W), [("yf_preprocess_bgr", old), ("yf_preprocess_frames", new)], args.reps, B * fb + out_old.numel())
        torch.cuda.synchronize()
        say("    outputs equal: %s" % bool(torch.equal(out_old, out_new)))
        ctx.close()

    say("(b) the same frames -> colour planes [B, 3, H, W] (yf_preprocess_frames, in_ch = 3)")
    for (H, W) in ((512, 640), (256, 320)):
        ctx = _lib.Ctx(0, 3, 3, 3, B, H, W)
        out = torch.empty((B, 3, H, W), dtype=torch.uint8, device=dev)
        new = lambda: _lib.check(lib.yf_preprocess_frames(ctx.handle, uni.data_ptr(), B, off.ctypes.data, Hs.ctypes.data, Ws.ctypes.data,  # noqa: E731
                                                          out.data_ptr(), stream()), ctx.handle)
        ab("-> 3x%dx%d" % (H, W), [("yf_preprocess_frames", new)], args.reps, B * fb + out.numel())
        ctx.close()
    del uni

    sizes = [(512, 640), (480, 640), (333, 517), (1080, 1920), (128, 160)]
    say("(c) ragged batch of %d frames cycling %s" % (B, ", ".join("%dx%d" % s for s in sizes)))
    order = [sizes[b % len(sizes)] for b in range(B)]
    # the old kernel takes one size per call: its arm sees the same frames grouped by size, one call per group
    groups = {s: [b for b in range(B) if order[b] == s] for s in sizes}
    perm = [b for s in sizes for b in groups[s]]
    frames = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in order]
    off_r, Ho_r, Wo_r, nb = yf.detector.frame_layout(frames)
    buf = np.zeros(nb, np.uint8)
    yf.detector.pack_frames(frames, buf, off_r)
    ragged = torch.from_numpy(buf).to(dev)
    grouped = torch.from_numpy(np.concatenate([frames[b].reshape(-1) for b in perm])).to(dev)
    gstart, pos = {}, 0
    for s in sizes:
        gstart[s] = pos
        pos += len(groups[s]) * s[0] * s[1] * 3
    src_bytes = sum(h * w * 3 for h, w in order)
    say("    %.1f MB of frames" % (src_bytes / 1e6))
    for chans in (1, 3):
        for (H, W) in ((512, 640), (256, 320)):
            ctx = _lib.Ctx(0, chans, 3, 3, B, H, W)
            shape = (B, H, W) if chans == 1 else (B, 3, H, W)
            out_new = torch.empty(shape, dtype=torch.uint8, device=dev)
            new = lambda: _lib.check(lib.yf_preprocess_frames(ctx.handle, ragged.data_ptr(), B, off_r.ctypes.data, Ho_r.ctypes.data,  # noqa: E731
                                                              Wo_r.ctypes.data, out_new.data_ptr(), stream()), ctx.handle)
            arms = [("yf_preprocess_frames (1 call)", new)]
            if chans == 1:
                out_old = torch.empty(shape, dtype=torch.uint8, device=dev)

                def old():
                    o = 0
                    for s in sizes:
                        n = len(groups[s])
                        _lib.check(lib.yf_preprocess_bgr(ctx.handle, grouped.data_ptr() + gstart[s], n, s[0], s[1],
                                                         out_old.data_ptr() + o * H * W, stream()), ctx.handle)
                        o += n
                arms = [("yf_preprocess_bgr (1 call per size)", old)] + arms
            ab("in_ch=%d -> %dx%d" % (chans, H, W), arms, args.reps, src_bytes + out_new.numel())
            if chans == 1:
                torch.cuda.synchronize()
                say("    outputs equal: %s" % bool(torch.equal(out_old, out_new[perm])))
            ctx.close()
    del ragged, grouped

    say("(d) end to end from host frames, %d x %dx%d (host clock, the call synchronises)" % (B, Ho, Wo))
    host = [rng.integers(0, 256, (Ho, Wo, 3), dtype=np.uint8) for _ in range(B)]
    for res in ("512x640", "256x320"):
        det = yf.Detect_YOLO(dev, os.path.join(ROOT, "tests", "golden", "weights", "yolo_fastest_%s.pth" % res), yf.config_for(res), None)
        arms = [("detect_bgr_batch(np.stack(frames))", lambda: det.detect_bgr_batch(np.stack(host))),
                ("detect_frames(frames)", lambda: det.detect_frames(host))]
        for _, fn in arms:
            fn()
            fn()
        t = {label: [] for label, _ in arms}
        for _ in range(max(args.reps // 3, 5)):
            for label, fn in arms:
                t0 = time.perf_counter()
                fn()
                t[label].append((time.perf_counter() - t0) * 1e3)
        base = float(np.median(t[arms[0][0]]))
        for label, _ in arms:
            med = float(np.median(t[label]))
            say("  %-44s median %8.2f ms  min %8.2f ms  %7.0f img/s  x%.3f" % (res + " " + label, med, min(t[label]), B / med * 1e3, med / base))
        a, b = det.detect_bgr_batch(np.stack(host)), det.detect_frames(host)
        say("    detections equal: %s (%d rows)" % (a == b, sum(len(r) for r in a)))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
