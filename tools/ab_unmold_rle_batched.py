"""A/B of the evaluation tail, alternated in one process: B x (unmold_detections(..., return_device_planes=True) +
rle.encode) against one unmold_detections_batched call.

    python tools/ab_unmold_rle_batched.py [--reps 15] [--json out.json]

D = 100 detections per image.  Boxes are drawn like bench.py's unmold_metric (sides log-uniform in [24, 600] pixels,
placed uniformly inside a 1024^2 image); the 28x28 masks are Gaussian blobs with a little noise, the shape a trained
head's sigmoid masks have (bench.py's uniform-noise masks would overflow the default run capacity and go through the
full-plane retry).  One more batch mixes image sizes.  For each batch it reports the median wall time per batch (host
clock around a device synchronise), images/s, CUDA kernels per call (torch.profiler, in a separate pass), host syncs
and device-to-host bytes (counted on Tensor.cpu), device bytes touched by the paste and RLE stages (computed from the
shapes and boxes), and whether both arms returned identical results.  Reads the card name and power limit in the
same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from sln_amodal_b200 import rle, unmold, unmold_detections_batched  # noqa: E402

D, MH, K = 100, 28, 2


def make_batch(shapes, windows, seed):
    rng = np.random.default_rng(seed)
    B = len(shapes)
    det = np.zeros((B, D, 6), np.float32)
    mm = np.zeros((B, D, MH, MH, K), np.float32)
    yy, xx = np.mgrid[0:MH, 0:MH].astype(np.float32)
    for b, (shape, win) in enumerate(zip(shapes, windows)):
        wh, ww = win[2] - win[0], win[3] - win[1]
        hw = np.minimum(np.exp(rng.uniform(np.log(24), np.log(600), (D, 2))), [wh - 1, ww - 1])
        y1x1 = rng.uniform(0, 1, (D, 2)) * ([wh, ww] - hw) + [win[0], win[1]]
        det[b, :, :4] = np.concatenate([y1x1, y1x1 + hw], 1)
        det[b, :, 4] = rng.integers(1, 81, D)
        det[b, :, 5] = rng.random(D)
        for d in range(D):
            cy, cx = rng.uniform(6, MH - 6, 2)
            s = rng.uniform(20, 90)
            mm[b, d, :, :, 1] = np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / s) + 0.02 * rng.random((MH, MH))
    return torch.from_numpy(det).cuda(), torch.from_numpy(mm).cuda()


def single_arm(det, mm, shapes, windows):
    out = []
    for b in range(det.shape[0]):
        boxes, cls, scores, planes = unmold.unmold_detections(det[b], mm[b], shapes[b], np.asarray(windows[b]),
                                                              return_device_planes=True)
        out.append((boxes, cls, scores, rle.encode(planes) if boxes.shape[0] else []))
    return out


def batched_arm(det, mm, shapes, windows):
    return unmold_detections_batched(det, mm, shapes, windows)


def same(a, b):
    return len(a) == len(b) and all(
        all(x.dtype == y.dtype and np.array_equal(x, y) for x, y in zip(p[:3], q[:3])) and p[3] == q[3]
        for p, q in zip(a, b))


class D2HCounter:
    """Counts Tensor.cpu() calls on CUDA tensors (each one a host wait plus a device-to-host copy) and their bytes."""

    def __enter__(self):
        self.calls, self.bytes, self._orig = 0, 0, torch.Tensor.cpu
        counter = self

        def cpu(t, *a, **kw):
            if t.is_cuda:
                counter.calls += 1
                counter.bytes += t.numel() * t.element_size()
            return counter._orig(t, *a, **kw)
        torch.Tensor.cpu = cpu
        return self

    def __exit__(self, *exc):
        torch.Tensor.cpu = self._orig


def kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())


def touched_bytes(res, shapes):
    """Paste + RLE device bytes.  Full-plane path: the paste writes n*H*W, the transpose reads and writes them, the
    RLE reads them (4 n H W).  Box path: the paste writes each box's area and the RLE reads it (2 sum of areas)."""
    full = sum(4 * len(r[0]) * s[0] * s[1] for r, s in zip(res, shapes))
    box = sum(2 * int(((r[0][:, 2] - r[0][:, 0]) * (r[0][:, 3] - r[0][:, 1])).sum()) for r in res)
    return full, box


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = card()
    sq = ((1024, 1024, 3), (0, 0, 1024, 1024))
    mixed = [((1024, 1024, 3), (0, 0, 1024, 1024)), ((480, 640, 3), (128, 0, 896, 1024)),
             ((1440, 1920, 3), (128, 0, 896, 1024)), ((130, 131, 3), (2, 0, 1022, 1024))] * 2
    configs = [(f"B={B} 1024^2", [sq] * B) for B in (1, 4, 8, 16)] + [("B=8 mixed sizes", mixed)]
    rows = []
    for i, (label, imgs) in enumerate(configs):
        shapes, windows = [s for s, _ in imgs], [w for _, w in imgs]
        det, mm = make_batch(shapes, windows, seed=100 + i)
        arms = {"single": lambda: single_arm(det, mm, shapes, windows),
                "batched": lambda: batched_arm(det, mm, shapes, windows)}
        outs = {k: f() for k, f in arms.items()}                 # warm-up, and the results compared
        identical = same(outs["single"], outs["batched"])
        times = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, f in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                torch.cuda.synchronize()
                times[k].append(time.perf_counter() - t0)
        row = {"batch": label, "B": len(imgs), "identical": identical}
        for k, f in arms.items():
            with D2HCounter() as c:
                f()
            ms = float(np.median(times[k])) * 1e3
            row[k] = {"ms": round(ms, 3), "images_per_s": round(len(imgs) / ms * 1e3, 1), "kernels": kernels(f),
                      "host_syncs": c.calls, "d2h_bytes": c.bytes}
        full, box = touched_bytes(outs["single"], shapes)
        row["device_bytes"] = {"full_plane": full, "box_local": box}
        row["speedup"] = round(row["single"]["ms"] / row["batched"]["ms"], 2)
        rows.append(row)
        print(json.dumps(row), flush=True)
    res = {"card": name, "power_limit": power, "reps": args.reps, "rows": rows}
    print(json.dumps({"card": name, "power_limit": power}))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
