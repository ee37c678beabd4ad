#!/usr/bin/env python
"""Benchmark of the YOLO-Fastest detection hot path (forward + decode + confidence filter + per-class NMS).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--res 512x640|256x320] [--batch B]
                    [--dump-outputs DIR]

One step = one pass of the hot path over one batch of synthetic images per GPU.  Default workload
(BASELINE.json metric): 640x512 images, batch 256 per GPU, the shipped 512x640 checkpoint.  Weak scaling:
every rank processes its own batch; per-rank detection slabs are gathered to rank 0 with one NCCL gather.

Prints ONE JSON line on rank 0:
  value     images/s, whole job, inputs resident in HBM (yf_detect on device tensors)
  e2e       images/s through the public API with HOST buffers (Detect_YOLO.submit_batch/collect ->
            yf_detect_submit_u8/yf_detect_wait, two slots): pinned uint8 images H2D, fused normalise + forward +
            decode + NMS, detection slab D2H, every step; the blocking single call is reported beside it
  roofline  dominant kernel (largest share of the step): algorithmic bytes / CUDA-event duration vs the measured HBM peak
  fp32      the same kernel's algorithmic FLOP/s vs the FP32 CUDA-core peak (the fused kernels are FP32-compute bound)
  cpu_baseline  the oracle port of the reference (PyTorch CPU forward + the reference's Python decode/NMS loops)
                timed on this box's host cores on a bounded sample (rank 0, N=1 only)
--impl reference times that CPU port alone, with all host threads, on the same workload definition.
--dump-outputs DIR writes what the last timed step returned to its caller (rank 0) as float64 .npy files (dump_outputs), so that
two builds can be compared output for output: the inputs are seeded and the same from run to run.
The benchmark writes nothing into the tree (it may be read-only): no bytecode caches, and build() leaves current libraries alone.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")
METRIC = "images/sec at 640x512 b256, 1/2/4/8 B200; % HBM roofline per kernel"
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x max SM clock = 74.4


# ---------------------------------------------------------------------------------------------
# algorithmic work per fused group (per image): MACs, unique fp32 elements in/out, folded weights
# ---------------------------------------------------------------------------------------------
def group_work(H, W, nout):
    px = lambda d: (H // d) * (W // d)
    def pw(cin, cout, d): return px(d) * cin * cout, cin * cout + cout
    def dw(c, k, d): return px(d) * c * k * k, c * k * k + c
    def dense(cin, cout, k, d): return px(d) * cin * cout * k * k, cin * cout * k * k + cout
    def irb(io, mid, d): return [pw(io, mid, d), dw(mid, 3, d), pw(mid, io, d)]
    G = []
    def add(name, layers, ins, outs):
        macs = sum(l[0] for l in layers)
        wts = sum(l[1] for l in layers)
        G.append({"name": name, "macs": macs, "bytes": 4 * (sum(c * px(d) for c, d in ins) + sum(c * px(d) for c, d in outs) + wts)})
    add("conv1_4", [dense(1, 8, 3, 2), pw(8, 8, 2), dw(8, 3, 2), pw(8, 4, 2)], [(1, 1)], [(4, 2)])
    add("res1_1", irb(4, 8, 2), [(4, 2)], [(4, 2)])
    add("conv2_1", [pw(4, 24, 2), dense(24, 24, 3, 4), pw(24, 8, 4)], [(4, 2)], [(8, 4)])
    add("res2_1", irb(8, 32, 4), [(8, 4)], [(8, 4)])
    add("res2_2", irb(8, 32, 4), [(8, 4)], [(8, 4)])
    add("conv3_1", [pw(8, 32, 4), dw(32, 3, 8), pw(32, 8, 8)], [(8, 4)], [(8, 8)])
    add("res3_1", irb(8, 48, 8), [(8, 8)], [(8, 8)])
    add("res3_2", irb(8, 48, 8), [(8, 8)], [(8, 8)])
    add("conv3_4", [pw(8, 48, 8), dw(48, 3, 8), pw(48, 16, 8)], [(8, 8)], [(16, 8)])
    for n in ("res3_3", "res3_4", "res3_5", "res3_6"):
        add(n, irb(16, 96, 8), [(16, 8)], [(16, 8)])
    add("conv4_1", [pw(16, 96, 8), dw(96, 3, 16), pw(96, 24, 16)], [(16, 8)], [(24, 16)])
    for n in ("res4_1", "res4_2", "res4_3", "res4_4"):
        add(n, irb(24, 136, 16), [(24, 16)], [(24, 16)])
    add("conv5_1", [pw(24, 136, 16), dw(136, 3, 32), pw(136, 48, 32)], [(24, 16)], [(136, 16), (48, 32)])
    for n in ("res5_1", "res5_2", "res5_3", "res5_4", "res5_5"):
        add(n, irb(48, 224, 32), [(48, 32)], [(48, 32)])
    add("conv5_2", [pw(48, 96, 32)], [(48, 32)], [(96, 32)])
    add("conv5_4", [dw(96, 5, 32), pw(96, 128, 32)], [(96, 32)], [(128, 32)])
    # the 1x1 before each head has no activation: it is composed with the head conv on the host (yf_api.cu: pack_irb), so the
    # executed work is depthwise + ONE 1x1; counting the reference's two 1x1s would overstate the achieved FLOP rate
    add("head_5", [dw(128, 5, 32), pw(128, nout, 32)], [(128, 32)], [(nout, 32)])
    add("conv4_1_1", [(px(16) * 96 * 96, 96 * 96 * 4 + 96), pw(232, 96, 16)], [(136, 16), (96, 32)], [(96, 16)])
    add("conv4_1_3", [dw(96, 5, 16), pw(96, 96, 16)], [(96, 16)], [(96, 16)])
    add("head_4", [dw(96, 5, 16), pw(96, nout, 16)], [(96, 16)], [(nout, 16)])
    return G


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def dist_shard(n, rank, world):
    """images of a job of n this rank takes (contiguous, ragged: yolo_fastest_b200.dist.shard_range)"""
    from yolo_fastest_b200.dist import shard_range
    lo, hi = shard_range(n, rank, world)
    return hi - lo


def synthetic_u8(B, H, W, seed):
    """Seeded uniform uint8 pixels (SURVEY.md §8d inputs 2-4)."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, H, W), generator=g, dtype=torch.uint8)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(d, out, counts, status):
    """What Detect_YOLO.detect_device returned for one batch, as float64 arrays under d:
      detections.npy  [N, max_det, 8]  x1, y1, x2, y2, conf, cls_score, cls, src of each record of the slab; the slots after an
                                       image's min(count, max_det) records hold no record (unset memory) and are written as 0
      counts.npy      [N]              untruncated detection count of each image
      status.npy      [N]              status word of each image
      image_index.npy [N]              which images of the batch these are: all of them, or a fixed seeded sample when the
                                       arrays of the whole batch would exceed DUMP_LIMIT_BYTES"""
    from yolo_fastest_b200 import _lib
    B, max_det = out.shape[0], out.shape[1]
    recs = out.cpu().numpy().view(_lib.DET_DTYPE).reshape(B, max_det)
    cnt, st = counts.cpu().numpy(), status.cpu().numpy()
    per_image = 8 * (max_det * 8 + 3)
    idx = np.arange(B)
    if B * per_image > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT_BYTES // per_image, replace=False))
    recs, cnt, st = recs[idx], cnt[idx], st[idx]
    dets = np.stack([recs[f].astype(np.float64) for f in _lib.DET_DTYPE.names], axis=-1)
    dets[np.arange(max_det)[None, :] >= np.minimum(cnt, max_det)[:, None]] = 0.0
    os.makedirs(d, exist_ok=True)
    for name, a in (("detections", dets), ("counts", cnt), ("status", st), ("image_index", idx)):
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def cpu_reference_pass(sd, io, u8, res):
    """One pass of the reference's CPU path over a batch: (forward s, post-process s, detections, kind).
    kind "reference": the UNMODIFIED reference staged under baseline/_ref (baseline/ref_arm.py: its own YoloFastest module and
    YOLO_post_process object, driven as Detect_YOLO.batch_detect drives them). kind "port": the oracle's restatement — only when
    baseline/_ref is absent (a checkout that never ran build() next to /root/reference)."""
    from baseline import ref_arm
    if ref_arm.available():
        pipe = _REF.get(res)
        if pipe is None:
            pipe = _REF[res] = ref_arm.RefPipeline(res, sd)
        a, b, n = pipe.run(u8)
        return a, b, n, "reference"
    from oracle import yolo_oracle as O
    x = (u8.float().unsqueeze(1) - 128.0) / 255.0
    t0 = time.perf_counter()
    pred = O.forward(sd, x)
    t1 = time.perf_counter()
    n_det = 0
    for b in range(x.shape[0]):
        n_det += len(O.detect_postprocess(pred, io["anchors"], io["input_shape"], io["conf_thre"], io["nms_thre"],
                                          io["num_anchors"], io["num_cls"], batch_index=b))
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, n_det, "port"


_REF = {}


def run_reference(args, cfg, sd, rank, world):
    """--impl reference: the CPU implementation alone, all host threads, bounded sample per step."""
    if rank != 0:
        return
    io = cfg["io_params"]
    H, W = io["input_shape"][0:2]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample = args.cpu_sample
    u8 = synthetic_u8(sample, H, W, 1000)
    kind = "port"
    for _ in range(args.warmup):
        cpu_reference_pass(sd, io, u8, args.res)
    fwd = post = 0.0
    for _ in range(args.steps):
        a, b, _, kind = cpu_reference_pass(sd, io, u8, args.res)
        fwd += a; post += b
    total = fwd + post
    value = sample * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%dx%d synthetic uint8 images, shipped %s checkpoint, conf %.2f nms %.2f; CPU sample of %d images per step"
                       % (W, H, args.res, io["conf_thre"], io["nms_thre"], sample)},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind,
                             "sample": "%d images/step x %d steps; forward %.1f ms/img, post-process %.2f ms/img; torch %s"
                             % (sample, args.steps, 1000 * fwd / (sample * args.steps), 1000 * post / (sample * args.steps), torch.__version__)},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--res", default="512x640", choices=["512x640", "256x320"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="strong scaling: a fixed job of this many images per step split over the GPUs (BASELINE config 4: 1024); "
                         "default 0 = weak scaling with --batch images per GPU")
    ap.add_argument("--max-det", type=int, default=64)
    ap.add_argument("--cpu-sample", type=int, default=16,
                    help="images per CPU-baseline pass: a bounded sample of the batch-256 workload, at the batch size the host runs fastest "
                         "(measured on the GPU box's 16 cores: 50 img/s at 16 images per pass, 43 img/s at 32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the detections of the last timed step as .npy files under DIR (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                                     # timing rules: W >= 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import __graft_entry__
    from yolo_fastest_b200 import config_for
    cfg = config_for(args.res)
    io = cfg["io_params"]
    H, W = io["input_shape"][0:2]
    ckpt = os.path.join(GOLD, "weights", "yolo_fastest_%s.pth" % args.res)
    sd = torch.load(ckpt, map_location="cpu")

    if args.impl == "reference":
        run_reference(args, cfg, sd, rank, world)
        return

    __graft_entry__.build()
    numa = None
    if world > 1:
        # one process per GPU: keep the rank (and the pinned buffers it is about to allocate) on the CPU cores NVML reports as local
        # to its GPU, so the 84 MB per step each rank copies to its device do not cross the socket interconnect
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1]
            cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
            if cpus:
                os.sched_setaffinity(0, cpus)
                numa = "%d cores local to GPU %d (NVML)" % (len(cpus), local_rank)
        except Exception as e:                              # no NVML / restricted container: run unbound
            numa = "unbound (%s)" % type(e).__name__
    import torch.distributed as dist
    from yolo_fastest_b200 import Detect_YOLO, _lib
    from yolo_fastest_b200.dist import gather_compact, shard_range, split_records
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    B = args.batch
    if args.global_batch:
        B = dist_shard(args.global_batch, rank, world)
    det = Detect_YOLO(dev, ckpt, cfg, None)
    u8 = synthetic_u8(B, H, W, 1000 + rank).pin_memory()
    x_dev = ((u8.to(dev).float().unsqueeze(1) - 128.0) / 255.0).contiguous()      # resident input: 4*B*H*W bytes (> L2 at B=256)
    n_total = args.global_batch if args.global_batch else B * world

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_device():
        out, counts, status = det.detect_device(x_dev, args.max_det)
        if world > 1:
            gather_compact(out, counts, n_total, dst=0, ctx=det.model._ctx)   # compaction kernel + one NCCL gather on the side stream
        return out, counts, status

    def step_e2e():
        rows = det.detect_batch(u8, max_det=args.max_det, raw=True)
        if world > 1:      # the slabs are already on the host: return them through the same collective from pinned->device copies
            pass
        return rows

    # ---- device-resident throughput ----------------------------------------------------------------------
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = det.model._ctx.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step_device()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    launches = det.model._ctx.launch_count() - launches0
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    n_det = int(last[1].sum().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)

    # ---- end to end through the public API with host buffers ------------------------------------------------
    # serving loop on the double-buffered API: batch i+1 is submitted (H2D copy on the copy stream) before the
    # results of batch i are collected, so every step still moves its own inputs H2D and its own results D2H.
    u8b = [u8, synthetic_u8(B, H, W, 2000 + rank).pin_memory()]

    def run_e2e(nsteps):
        if world == 1:
            det.submit_batch(u8b[0], 0, max_det=args.max_det)
            rows = None
            for i in range(nsteps):
                if i + 1 < nsteps:
                    det.submit_batch(u8b[(i + 1) & 1], (i + 1) & 1, max_det=args.max_det)
                rows = det.collect(i & 1, raw=True)
            return rows
        # N > 1: every rank runs the same double-buffered loop with its results left on the device and returns them to rank 0 with one
        # compacted NCCL gather per step on a side stream; rank 0 reads step i's detections from pinned memory while step i + 1 runs
        pend = det.submit_batch_device(u8b[0], 0, max_det=args.max_det)
        res, prev = None, None
        for i in range(nsteps):
            nxt = det.submit_batch_device(u8b[(i + 1) & 1], (i + 1) & 1, max_det=args.max_det) if i + 1 < nsteps else None
            det.wait(i & 1)
            h = gather_compact(pend[0], pend[1], n_total, dst=0, ctx=det.model._ctx)
            if prev is not None:
                res = prev.result()
            prev, pend = h, nxt
        res = prev.result()
        return res

    run_e2e(3)
    barrier()
    t0 = time.perf_counter()
    rows = run_e2e(args.steps)
    torch.cuda.synchronize(dev)
    e2e_ms = 1000.0 * (time.perf_counter() - t0)      # host-synchronous calls on internal streams: wall clock is the measure
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms_max = float(t.item())
    # the blocking single-call form, for reference
    for _ in range(2):
        step_e2e()
    t0 = time.perf_counter()
    for _ in range(max(2, args.steps // 4)):
        step_e2e()
    sync_ms = 1000.0 * (time.perf_counter() - t0) / max(2, args.steps // 4)

    # ---- N > 1: the gathered result must be what ONE GPU computes for the whole job (SURVEY.md §4), outside the timed region ------
    gather_check = None
    if world > 1:
        out, cnt = det.submit_batch_device(u8b[0], 0, max_det=args.max_det)
        det.wait(0)
        recs, cnts = gather_compact(out, cnt, n_total, dst=0, ctx=det.model._ctx).result()
        if rank == 0:
            want = []
            for r in range(world):          # rank 0 regenerates every rank's shard (seeded) and runs it on its own GPU
                nr = dist_shard(args.global_batch, r, world) if args.global_batch else args.batch
                want += det.detect_batch(synthetic_u8(nr, H, W, 1000 + r), max_det=args.max_det, raw=True)
            got = split_records(recs, cnts)
            same = len(got) == len(want) and all(g_.tobytes() == w_.tobytes() for g_, w_ in zip(got, want))
            gather_check = {"ok": bool(same), "images": len(want), "records": int(sum(len(w_) for w_ in want)),
                            "what": "NCCL-gathered per-image lists of all ranks == rank 0's own single-GPU detect_batch of every shard, byte for byte"}
            if not same:
                raise SystemExit("gathered detections differ from the single-GPU result: %r" % (gather_check,))

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- batch-1 latency (BASELINE config 2) through the blocking public call: CUDA-graph replay of the 31 launches -----------------
    latency = None
    if world == 1 and B >= 1:
        one = u8[:1].clone().pin_memory()
        for _ in range(20):
            det.detect_batch(one, max_det=args.max_det, raw=True)
        nlat = 200
        t0 = time.perf_counter()
        for _ in range(nlat):
            det.detect_batch(one, max_det=args.max_det, raw=True)
        lat_ms = 1000.0 * (time.perf_counter() - t0) / nlat
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        x1 = x_dev[:1].contiguous()
        for _ in range(20):
            det.detect_device(x1, args.max_det)
        ev[0].record()
        for _ in range(nlat):
            det.detect_device(x1, args.max_det)
        ev[1].record()
        torch.cuda.synchronize(dev)
        latency = {"batch": 1, "ms_e2e": round(lat_ms, 4), "api": "Detect_YOLO.detect_batch -> yf_detect_host_u8 (H2D, graph replay, D2H, sync), %d calls after 20 warm-ups" % nlat,
                   "ms_device_stream": round(ev[0].elapsed_time(ev[1]) / nlat, 4), "device_api": "yf_detect on a resident fp32 image, back to back on one stream"}

    # ---- per-kernel roofline (rank 0): CUDA events around every group launch of one forward ----------------------
    prof = det.model.profile(x_dev)
    work = {g["name"]: g for g in group_work(H, W, det.model.num_out)}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    total_ms = sum(m for _, m in prof)
    # which engine runs a group decides the roof that binds it: the tcgen05 groups are contractions on the tensor pipe (bound
    # "tensor"), every other group runs on the FP32 CUDA cores and moves its activations once (bound = the larger of its HBM time and
    # its FP32 time; "hbm" for the thin 4-8 channel groups whose HBM time is the larger one)
    TENSOR = {"conv2_1", "res3_1", "res3_2", "conv3_4", "res3_3", "res3_4", "res3_5", "res3_6", "conv4_1", "res4_1", "res4_2", "res4_3", "res4_4", "conv5_1", "res5_1", "res5_2", "res5_3",
              "res5_4", "res5_5", "conv5_4", "head_5", "conv4_1_1", "conv4_1_3", "head_4"}
    bf16_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
    tf32_peak = bf16_peak / 2.0                              # kind::tf32 issues at half the bf16 rate
    ncu = {}
    try:
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_metrics.json")))
    except Exception:
        pass
    kernels = []
    for name, m in prof:
        w = work[name]
        gbs = w["bytes"] * B / (m * 1e-3) / 1e9
        tfl = 2 * w["macs"] * B / (m * 1e-3) / 1e12
        t_hbm = w["bytes"] * B / (hbm_peak * 1e9) * 1e3
        t_flop = 2 * w["macs"] * B / (FP32_PEAK_TFLOPS * 1e12) * 1e3
        k = {"name": name, "ms": round(m, 4), "share": round(m / total_ms, 4), "GB/s": round(gbs, 1), "hbm_frac": round(gbs / hbm_peak, 4),
             "TFLOP/s": round(tfl, 2), "fp32_frac": round(tfl / FP32_PEAK_TFLOPS, 4),
             "bound": "tensor" if name in TENSOR else ("hbm" if t_hbm >= t_flop else "fp32"),
             "roof_ms": round(max(t_hbm, t_flop), 4), "roof_frac": round(max(t_hbm, t_flop) / m, 4)}
        if name in TENSOR:
            k["tf32_frac_executed"] = round(3 * tfl / tf32_peak, 4)       # 3xTF32: three tensor-core products per fp32 product
        if name in ncu.get("kernels", {}):
            k["ncu"] = ncu["kernels"][name]
        kernels.append(k)
    top = max(kernels, key=lambda k: k["ms"])
    # DRAM traffic of the dominant kernel per launch (dram__bytes_read.sum + dram__bytes_write.sum) and its tensor-pipe utilisation come
    # from the committed ncu pass of this same workload (profiles/r02_ncu_metrics.json, written by tools/ncu_metrics.py from a
    # `ncu --set full` capture at batch 256) — a profiler cannot run inside the timed process; null when no capture matches
    traffic, traffic_source = None, None
    if ncu.get("workload") == "%dx%d b%d" % (W, H, B) and top["name"] in ncu.get("kernels", {}):
        traffic = ncu["kernels"][top["name"]].get("dram_bytes")
        traffic_source = "profiles/r02_ncu_metrics.json (%s)" % ncu.get("source", "ncu --set full")
    if top["bound"] == "tensor":
        roofline = {"bound": "tensor", "achieved": top["TFLOP/s"], "peak": bf16_peak, "unit": "TFLOP/s", "frac": round(top["TFLOP/s"] / bf16_peak, 4),
                    "traffic": traffic, "traffic_source": traffic_source, "kernel": top["name"], "share_of_forward": top["share"],
                    "peak_source": "measured dense bf16 (MEASURED_PEAKS.json bf16_tflops_sustained)" if "bf16_tflops_sustained" in peaks else "fallback 1.59 PFLOP/s",
                    "tf32_peak": tf32_peak, "executed_TFLOP/s": round(3 * top["TFLOP/s"], 1), "frac_of_tf32_executed": top.get("tf32_frac_executed"),
                    "tensor_pipe_util_ncu": top.get("ncu", {}).get("tensor_pipe_pct"),
                    "hbm_GB/s": top["GB/s"], "hbm_frac": top["hbm_frac"],
                    "note": "fp32 parity needs 3xTF32 (hi*hi + hi*lo + lo*hi): algorithmic FLOPs are a third of the executed tensor FLOPs; the MMAs of a 128-pixel tile need 1.08 k of its ~4.4 k cycles at the tcgen05 dispatch floor. A operand in tensor memory (dense_ta_kernel): no activation passes through shared memory; the kernel is bound by the CUDA-core instructions of its producer warps (conv1_8 + ReLU + hi/lo split, recomputed 2.25x; ncu: issue slots 66%, ALU pipe 50%, tensor pipe 25%)"}
    else:
        roofline = {"bound": top["bound"], "achieved": top["GB/s"], "peak": hbm_peak, "unit": "GB/s", "frac": top["hbm_frac"], "traffic": traffic,
                    "traffic_source": traffic_source, "kernel": top["name"], "share_of_forward": top["share"], "peak_source": peak_src}
    fp32 = {"kernel": top["name"], "achieved": top["TFLOP/s"], "peak": round(FP32_PEAK_TFLOPS, 1), "unit": "TFLOP/s", "frac": top["fp32_frac"],
            "whole_forward_TFLOP/s": round(2 * sum(g["macs"] for g in work.values()) * B / (total_ms * 1e-3) / 1e12, 2),
            "whole_forward_GB/s": round(sum(g["bytes"] for g in work.values()) * B / (total_ms * 1e-3) / 1e9, 1),
            "whole_forward_roof_ms": round(sum(k["roof_ms"] for k in kernels), 4),
            "whole_forward_roof_frac": round(sum(k["roof_ms"] for k in kernels) / total_ms, 4)}

    # ---- pre-processing kernel (SURVEY 8f-1): 512x640 BGR frames -> network input, CUDA events, HBM-bound ---------------
    preprocess = None
    try:
        Ho, Wo = 512, 640                                   # the dataset's frame size (_config.py origin_img_shape)
        frames = torch.randint(0, 256, (B, Ho, Wo, 3), dtype=torch.uint8, device=dev)
        for _ in range(3):
            det.pre_process_batch(frames)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        reps = 20
        ev[0].record()
        for _ in range(reps):
            det.pre_process_batch(frames)
        ev[1].record()
        torch.cuda.synchronize(dev)
        pms = ev[0].elapsed_time(ev[1]) / reps
        pbytes = B * (3 * Ho * Wo + H * W)
        preprocess = {"kernel": "prep_bgr_kernel (BGR2GRAY + INTER_LINEAR resize, bit-exact with cv2)", "frames": "%dx%dx3 uint8, batch %d" % (Wo, Ho, B),
                      "ms": round(pms, 4), "GB/s": round(pbytes / (pms * 1e-3) / 1e9, 1), "hbm_frac": round(pbytes / (pms * 1e-3) / 1e9 / hbm_peak, 4),
                      "bytes": pbytes, "note": "%.0f MB of frames per launch: larger than L2 at batch 256" % (1e-6 * B * 3 * Ho * Wo)}
        del frames
    except Exception as e:                                  # never let the optional row break the contract line
        preprocess = {"error": str(e)[:200]}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sample = args.cpu_sample
        cu8 = synthetic_u8(sample, H, W, 1000)
        cpu_reference_pass(sd, io, cu8, args.res)
        fwd = post = 0.0
        reps = 3
        kind = "port"
        for _ in range(reps):
            a, b, _, kind = cpu_reference_pass(sd, io, cu8, args.res)
            fwd += a; post += b
        cpu_baseline = {"value": sample * reps / (fwd + post), "unit": "images/s", "cores": cores, "kind": kind,
                        "sample": "%d images x %d passes after 1 warm-up; forward %.1f ms/img, post-process %.2f ms/img; torch %s CPU"
                        % (sample, reps, 1000 * fwd / (sample * reps), 1000 * post / (sample * reps), torch.__version__)}

    line = {
        "metric": METRIC, "value": n_total * args.steps / (ms_max * 1e-3), "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%dx%d synthetic uint8 images, batch %d per GPU, shipped %s checkpoint, conf %.2f nms %.2f, max_det %d"
                   % (W, H, B, args.res, io["conf_thre"], io["nms_thre"], args.max_det),
                   "global_batch": n_total, "parallelism": "dp%d (image shards, one compacted NCCL gather of detection lists per step)" % world,
                   "cpu_affinity": numa,
                   "l2": "inputs larger than L2: %.0f MB resident fp32 input + %.1f GB of activations written per step"
                   % (4e-6 * B * H * W, 1e-9 * B * sum(g["bytes"] for g in work.values()) / 2),
                   "detections_last_step": n_det},
        "e2e": {"value": n_total * args.steps / (e2e_ms_max * 1e-3), "unit": "images/s", "h2d_bytes_per_step": B * H * W,
                "d2h_bytes_per_step": (B * args.max_det * _lib.DET_DTYPE.itemsize + 8 * B) if world == 1 else
                world * (4 * ((-(-n_total // world) + 3) // 2 * 2) + _lib.DET_DTYPE.itemsize * (-(-n_total // world)) * min(args.max_det, 8)),
                "ms_per_step": e2e_ms_max / args.steps,
                "api": "Detect_YOLO.submit_batch/collect -> yf_detect_submit_u8/yf_detect_wait (pinned uint8 in, yf_det slab out, two slots)",
                "blocking_call_ms_per_step": sync_ms, "blocking_api": "Detect_YOLO.detect_batch -> yf_detect_host_u8"},
        "gpu_launches": launches,
        "gather_check": gather_check,
        "latency": latency,
        "clocks": clocks,
        "roofline": roofline,
        "fp32": fp32,
        "cpu_baseline": cpu_baseline,
        "preprocess": preprocess,
        "kernels": kernels,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True          # the project modules main() imports leave no __pycache__ in the tree
    main()
