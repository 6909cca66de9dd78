"""Batched against per-image NMS and per-class-NMS detection heads, all arms alternated in one process.

    python tools/ab_batched_nms.py [--reps 30] [--out results.json]

  per-class NMS   the refine step's problem: n = 1000 rounded detections, 81 classes, thresh 0.3.
                  B sequential ops.nms_device calls  vs  one ops.nms_batched_device call, B = 1, 4, 8, 16
  agnostic NMS    n = 6000 RPN-like boxes, thresh 0.7, the same two arms
  head graph      USE_NMS = True (per-class NMS 0.3, 81 classes): pipeline.MultiHeadGraph (B parallel single-image
                  branches)  vs  pipeline.BatchedHeadGraph, B = 4, 8, 16; 261 888 anchors, P2..P5 at C = 256
Times are CUDA events around each arm, median over --reps alternated rounds; both arms' outputs are compared before the
timing.  Kernel counts come from one torch.profiler pass per arm, run before the timing.  The GPU's name and power limit
are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from ab_batched_head import A, C, NCLS, R, SIDES, gpu_info, image_inputs, kernels, timed  # noqa: E402
from sln_amodal_b200 import ops, pipeline, synth  # noqa: E402


class Cfg:
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    RPN_NMS_THRESHOLD = 0.7
    POOL_SIZE = 7
    MASK_POOL_SIZE = 14
    USE_NMS = True
    DETECTION_MIN_CONFIDENCE = 0.0
    DETECTION_NMS_THRESHOLD = 0.3


def nms_problems(B, n, K, dev, seed):
    rng = np.random.default_rng(seed)
    dets, cls = [], []
    for b in range(B):
        boxes = synth.nms_boxes(n, seed=seed + 7 * b, kind="rpn", rounded=K is not None)
        dets.append(np.concatenate([boxes, synth.nms_scores(n, seed=seed + 7 * b + 1)[:, None]], 1))
        cls.append(rng.integers(1, K, n).astype(np.int32) if K else None)
    D = torch.from_numpy(np.stack(dets).astype(np.float32)).to(dev)
    Cl = torch.from_numpy(np.stack(cls)).to(dev) if K else None
    return D, Cl


def nms_arms(name, n, K, thresh, dev, reps):
    out = []
    for B in (1, 4, 8, 16):
        D, Cl = nms_problems(B, n, K, dev, seed=10 * B + n)
        seq = lambda: [ops.nms_device(D[b], thresh, class_ids=None if Cl is None else Cl[b]) for b in range(B)]
        bat = lambda: ops.nms_batched_device(D, thresh, class_ids=Cl)
        for _ in range(3):
            seq(), bat()
        keep, num = bat()
        for b, (wk, wn) in enumerate(seq()):               # the arms compute the same thing
            k = int(wn.item())
            assert int(num[b]) == k and torch.equal(keep[b, :k], wk[:k]), (name, B, b)
        ks, kb = kernels(seq), kernels(bat)
        ts, tb = [], []
        for _ in range(reps):
            ts.append(timed(seq))
            tb.append(timed(bat))
        r = {"arm": name, "n": n, "classes": K, "thresh": thresh, "B": B, "sequential_ms": float(np.median(ts)),
             "batched_ms": float(np.median(tb)), "sequential_kernels": ks, "batched_kernels": kb}
        r["speedup"] = r["sequential_ms"] / r["batched_ms"]
        out.append(r)
        print(json.dumps(r), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "reps": args.reps}
    print(json.dumps(res["gpu"]), flush=True)
    res["per_class_nms"] = nms_arms("per_class_nms", 1000, NCLS, 0.3, dev, args.reps)
    res["agnostic_nms"] = nms_arms("agnostic_nms", 6000, None, 0.7, dev, args.reps)

    # ---- head graphs with the per-class NMS branch
    res["head_graph"] = []
    rng = np.random.default_rng(0)
    anchors = torch.from_numpy(synth.nms_boxes(A, seed=4, kind="rpn")).to(dev)
    imgs = [image_inputs(rng, dev) for _ in range(16)]
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
                assert nd > 0 and int(bat.out["num_detections"][b]) == nd, b
                assert torch.equal(bat.out["detections"][b], o["detections"]) and torch.equal(bat.out["keep"][b], o["keep"]), b
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
