"""A/B of the depthwise 5x5 -> 1x1 groups (conv5_4, head_5, conv4_1_3, head_4): the TMA-fed kernel (dwpw_tma_kernel, the default
library) against the cp.async kernel it replaces (dwpw_tc_kernel, a -DYF_DWPW_TMA=0 build of the same sources). GPU box.

    python tools/dwpw_ab.py [--res 512x640] [--batch 256] [--rounds 5] [--old-lib PATH] [--out FILE]

The comparison library is compiled with __graft_entry__.NVCC_FLAGS into a temporary directory (never into the tree) unless --old-lib
names one. Each round runs both libraries in fresh processes (YF_B200_LIB), alternating, and each process reports the per-group
device times of yf_profile_forward (best of 3 calls) and sha256 digests of the conv5_4 / conv4_1_3 taps and both heads on the same
seeded input. Printed: per-round times, the medians of the four groups and of the step, and whether every digest is equal.
Exit status 1 when a digest differs."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUPS = ("conv5_4", "head_5", "conv4_1_3", "head_4")


def build_old(out_dir):
    """Compile the library with the cp.async kernel on every depthwise 5x5 -> 1x1 group into out_dir; returns its path."""
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    lib = os.path.join(out_dir, "libyf_b200_dwpw_cpasync.so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + ge.NVCC_FLAGS + ["-DYF_DWPW_TMA=0", "-o", lib, os.path.join(ge.CSRC, "yf_api.cu")]
    r = subprocess.run(cmd, cwd=ge.CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (r.stdout, r.stderr))
    return lib


def run_child(lib, res, batch, nc=3, profile=True, seed=11):
    """One process on library `lib`: digests of the taps and heads (and per-group times) as a dict."""
    cmd = [sys.executable, os.path.abspath(__file__), "--child", "--res", res, "--batch", str(batch), "--nc", str(nc), "--seed", str(seed)]
    if not profile:
        cmd.append("--no-profile")
    r = subprocess.run(cmd, env=dict(os.environ, YF_B200_LIB=lib), capture_output=True, text=True, timeout=1200)
    if r.returncode != 0:
        raise RuntimeError("child on %s failed:\n%s\n%s" % (lib, r.stdout[-3000:], r.stderr[-3000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def child(args):
    sys.path.insert(0, ROOT)
    import torch
    import yolo_fastest_b200 as yf
    H, W = (int(v) for v in args.res.split("x"))
    wname = "stress80_416" if args.nc == 80 else "yolo_fastest_512x640"
    sd = torch.load(os.path.join(ROOT, "tests", "golden", "weights", wname + ".pth"), map_location="cpu")
    m = yf.YoloFastest({"num_cls": args.nc, "input_channel": 1, "num_anchors": 3})
    m.load_state_dict(sd)
    m = m.cuda().eval()
    g = torch.Generator().manual_seed(args.seed)
    x = ((torch.randint(0, 256, (args.batch, 1, H, W), generator=g).float() - 128.0) / 255.0).cuda()
    out = {"lib": os.environ.get("YF_B200_LIB", "default")}
    if not args.no_profile:
        best = None
        for _ in range(3):
            p = m.profile(x)
            best = p if best is None else [(n, min(a, b)) for (n, a), (_, b) in zip(best, p)]
        out["step_ms"] = sum(t for _, t in best)
        out["groups"] = {n: t for n, t in best if n in GROUPS}
    hl, hs = m(x)
    torch.cuda.synchronize()
    digest = lambda t: hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()
    out["sha"] = {"head_large": digest(hl), "head_small": digest(hs)}
    for name in ("conv5_4", "conv4_1_3"):
        out["sha"][name] = digest(m.tap(name, args.batch))
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", default="512x640")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--nc", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--old-lib")
    ap.add_argument("--out")
    ap.add_argument("--child", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args()
    if args.child:
        return child(args)
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    ge.build()
    with tempfile.TemporaryDirectory() as tmp:
        libs = {"tma": ge.LIB, "cpasync": args.old_lib or build_old(tmp)}
        runs = {k: [] for k in libs}
        for rnd in range(args.rounds):
            for k in (("cpasync", "tma") if rnd % 2 == 0 else ("tma", "cpasync")):
                runs[k].append(run_child(libs[k], args.res, args.batch, args.nc, seed=args.seed))
    lines = ["dwpw A/B at %s, batch %d, %d classes, %d rounds (alternating; per-group device ms of yf_profile_forward, best of 3 calls per process)"
             % (args.res, args.batch, args.nc, args.rounds)]
    for k in ("cpasync", "tma"):
        for i, r in enumerate(runs[k]):
            lines.append("  %-8s round %d: step %.4f  %s  sum4 %.4f" % (k, i, r["step_ms"], "  ".join("%s %.4f" % (n, r["groups"][n]) for n in GROUPS),
                                                                         sum(r["groups"][n] for n in GROUPS)))
    med = {}
    for k in ("cpasync", "tma"):
        med[k] = {n: statistics.median(r["groups"][n] for r in runs[k]) for n in GROUPS}
        med[k]["sum4"] = statistics.median(sum(r["groups"][n] for n in GROUPS) for r in runs[k])
        med[k]["step"] = statistics.median(r["step_ms"] for r in runs[k])
        spread = max(r["step_ms"] for r in runs[k]) - min(r["step_ms"] for r in runs[k])
        lines.append("median %-8s: %s  sum4 %.4f  step %.4f (step spread %.4f)" % (k, "  ".join("%s %.4f" % (n, med[k][n]) for n in GROUPS),
                                                                                  med[k]["sum4"], med[k]["step"], spread))
    same = all(r["sha"] == runs["cpasync"][0]["sha"] for k in runs for r in runs[k])
    lines.append("sum of the four groups %.4f -> %.4f ms (%.2fx), step %.4f -> %.4f ms" % (
        med["cpasync"]["sum4"], med["tma"]["sum4"], med["cpasync"]["sum4"] / med["tma"]["sum4"], med["cpasync"]["step"], med["tma"]["step"]))
    lines.append("taps conv5_4, conv4_1_3 and both heads byte-equal between the libraries: %s" % same)
    text = "\n".join(lines)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
