"""A/B of the detection targets, alternated in one process: B x detection_target_layer against one
detection_target_layer_batched call.

    python tools/ab_batched_targets.py [--reps 20] [--json out.json]

Each image comes from bench.py's detection_targets_metric generator with its own seed (1000 proposals, 240 of them
jittered GT boxes, 12 GT instances, L = 1, 1024^2 u8 masks, 100 sampled ROIs with 32x32 mask targets).  Both arms are
seeded the same before every call, so they sample the same rows.  For B in {1, 4, 8, 16} it reports the median wall
time per batch (host clock around a device synchronise), images/s, CUDA kernels per call (torch.profiler, in a
separate pass), host syncs and device-to-host bytes (counted on Tensor.cpu), and whether the two arms returned
identical results image by image.  Reads the card name and power limit in the same run.
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

from sln_amodal_b200 import detection_target_layer, detection_target_layer_batched, synth  # noqa: E402


class Cfg:
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    TRAIN_ROIS_PER_IMAGE = 100
    ROI_POSITIVE_RATIO = 0.7
    MASK_SHAPE = [32, 32]
    USE_MINI_MASK = False


def make_image(seed, G=12, N=1000, S=1024):
    """bench.py detection_targets_metric's inputs under another seed."""
    rng = np.random.default_rng(seed)
    gt = np.zeros((G, 4), np.float32)
    masks = np.zeros((1, G, S, S), np.uint8)
    for i in range(G):
        h, w = rng.uniform(0.1, 0.4, 2)
        y1, x1 = rng.uniform(0, 1 - h), rng.uniform(0, 1 - w)
        gt[i] = (y1, x1, y1 + h, x1 + w)
        masks[0, i, int(y1 * S):int((y1 + h) * S), int(x1 * S):int((x1 + w) * S)] = 1
    jit = gt[rng.integers(0, G, 240)] + rng.normal(0, 0.02, (240, 4)).astype(np.float32)
    props = np.clip(np.concatenate([jit, synth.roi_boxes(N - 240, seed=9 + seed)], 0), 0, 1).astype(np.float32)
    return props, np.ones(G, np.int32), gt, masks


def make_batch(B, seed):
    imgs = [make_image(seed + b) for b in range(B)]
    return [torch.from_numpy(np.stack([im[j] for im in imgs])).cuda() for j in range(4)]


def single_arm(props, ids, gt, masks):
    torch.manual_seed(5)
    return [detection_target_layer(props[b:b + 1], ids[b:b + 1], gt[b:b + 1], masks[b:b + 1], Cfg())
            for b in range(props.shape[0])]


def batched_arm(props, ids, gt, masks):
    torch.manual_seed(5)
    return detection_target_layer_batched(props, ids, gt, masks, Cfg())


def same(single, batched):
    rois, cls, deltas, tm, _, n_rois = batched
    for b, (r, c, d, m) in enumerate(single):
        k = int(n_rois[b])
        if k != (r.shape[0] if r.numel() else 0):
            return False
        if k and not (torch.equal(rois[b, :k], r) and torch.equal(cls[b, :k], c) and torch.equal(deltas[b, :k], d)
                      and torch.equal(tm[b, :k], m)):
            return False
    return True


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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = card()
    rows = []
    for B in (1, 4, 8, 16):
        data = make_batch(B, seed=303 + 100 * B)
        arms = {"single": lambda: single_arm(*data), "batched": lambda: batched_arm(*data)}
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
        row = {"B": B, "identical": identical, "rois": [int(v) for v in outs["batched"][5].tolist()]}
        for k, f in arms.items():
            with D2HCounter() as c:
                f()
            ms = float(np.median(times[k])) * 1e3
            row[k] = {"ms": round(ms, 3), "images_per_s": round(B / ms * 1e3, 1), "kernels": kernels(f),
                      "host_syncs": c.calls, "d2h_bytes": c.bytes}
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
