"""Batched against per-image proposals and detection heads, config-1 shapes, all arms alternated in one process.

    python tools/ab_batched_head.py [--reps 30] [--out results.json]

Inputs: 261 888 anchors per image, P2..P5 at C = 256 (256^2 .. 32^2), pools 7 and 14, 1000 proposals, top-100
detections, a static classifier output of 81 classes.
  proposals   B sequential ops.proposal_device calls  vs  one ops.proposal_batched_device call, B = 1, 4, 8, 16
  head graph  pipeline.MultiHeadGraph (B parallel single-image branches)  vs  pipeline.BatchedHeadGraph, B = 4, 8, 16
Times are CUDA events around each arm, median over --reps alternated rounds.  Kernel counts come from one
torch.profiler pass per arm, run before the timing.  The GPU's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from sln_amodal_b200 import ops, pipeline, synth  # noqa: E402

A, C, NCLS, R = 261888, 256, 81, 1000
SIDES = (256, 128, 64, 32)
STD = np.array([0.1, 0.1, 0.2, 0.2])
HW = (1024, 1024)


class Cfg:
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    RPN_BBOX_STD_DEV = STD
    RPN_NMS_THRESHOLD = 0.7
    POOL_SIZE = 7
    MASK_POOL_SIZE = 14


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
               and "memset" not in e.name.lower() and "memcpy" not in e.name.lower())


def timed(fn):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    e.synchronize()
    return s.elapsed_time(e)


def image_inputs(rng, dev):
    fg = rng.permutation(np.linspace(0, 1, A)).astype(np.float32)
    return (torch.from_numpy(np.stack([1 - fg, fg], 1).astype(np.float32)).to(dev),
            torch.from_numpy((rng.standard_normal((A, 4)) * 0.5).astype(np.float32)).to(dev))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "reps": args.reps, "proposals": [], "head_graph": []}
    print(json.dumps(res["gpu"]), flush=True)
    rng = np.random.default_rng(0)
    anchors = torch.from_numpy(synth.nms_boxes(A, seed=4, kind="rpn")).to(dev)
    imgs = [image_inputs(rng, dev) for _ in range(16)]

    # ---- proposals
    for B in (1, 4, 8, 16):
        P = torch.stack([p for p, _ in imgs[:B]])
        D = torch.stack([d for _, d in imgs[:B]])
        seq = lambda: [ops.proposal_device(P[b], D[b], anchors, R, 0.7, STD, HW) for b in range(B)]
        bat = lambda: ops.proposal_batched_device(P, D, anchors, R, 0.7, STD, HW)
        for _ in range(3):
            seq(), bat()
        got, num = bat()
        for b in range(B):                                 # the arms compute the same thing
            w, wn = ops.proposal_device(P[b], D[b], anchors, R, 0.7, STD, HW)
            assert int(num[b]) == int(wn[0]) and torch.equal(got[b], w), b
        ks, kb = kernels(seq), kernels(bat)
        ts, tb = [], []
        for _ in range(args.reps):
            ts.append(timed(seq))
            tb.append(timed(bat))
        r = {"B": B, "sequential_ms": float(np.median(ts)), "batched_ms": float(np.median(tb)),
             "sequential_kernels": ks, "batched_kernels": kb}
        r["speedup"] = r["sequential_ms"] / r["batched_ms"]
        res["proposals"].append(r)
        print(json.dumps(r), flush=True)

    # ---- head graphs
    cfg = Cfg()
    cls_p = torch.softmax(torch.randn(16 * R, NCLS, device=dev) * 3.0, 1)
    cls_d = torch.randn(16 * R, NCLS, 4, device=dev) * 0.3
    maps_all = [torch.randn(16, C, s, s, device=dev).contiguous(memory_format=torch.channels_last) for s in SIDES]
    with torch.no_grad():
        for B in (4, 8, 16):
            heads = [pipeline.HeadGraph(anchors, cfg, [m[b:b + 1].contiguous(memory_format=torch.channels_last) for m in maps_all],
                                        imgs[b][0], imgs[b][1], (cls_p[b * R:(b + 1) * R], cls_d[b * R:(b + 1) * R]),
                                        capture=False) for b in range(B)]
            multi = pipeline.MultiHeadGraph(heads)
            bat = pipeline.BatchedHeadGraph(anchors, cfg, [m[:B] for m in maps_all],
                                            torch.stack([p for p, _ in imgs[:B]]), torch.stack([d for _, d in imgs[:B]]),
                                            (cls_p[:B * R], cls_d[:B * R]))
            for _ in range(3):
                multi.replay(), bat.replay()
            torch.cuda.synchronize()
            for b, o in enumerate(multi.out):                  # same detections per image
                nd = int(o["num_detections"].item())
                assert int(bat.out["num_detections"][b]) == nd and torch.equal(bat.out["detections"][b], o["detections"]), b
            km, kb = kernels(multi.replay), kernels(bat.replay)
            tm, tb = [], []
            for _ in range(args.reps):
                tm.append(timed(multi.replay))
                tb.append(timed(bat.replay))
            r = {"B": B, "multi_ms": float(np.median(tm)), "batched_ms": float(np.median(tb)),
                 "multi_images_per_s": B / float(np.median(tm)) * 1e3, "batched_images_per_s": B / float(np.median(tb)) * 1e3,
                 "multi_kernels": km, "batched_kernels": kb}
            res["head_graph"].append(r)
            print(json.dumps(r), flush=True)
            del heads, multi, bat
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
