"""A/B of the config-2 RoIAlign step on bf16 maps (DESIGN 4.6): three arms alternated in one process.

    (a) f32     f32 maps and grads: bench.py's headline step
    (b) today   bf16 maps through the f32 path, what an autocast user got before the 2-byte kernels: every map is widened
                to an f32 channels_last copy per call, crops come out f32; bf16 grads are widened, f32 gradient maps
                written and then cast to bf16 (autograd's cast)
    (c) native  bf16 maps, crops, grads and gradient maps through the 2-byte kernels

A step is bench.py's: for 7x7 and 14x14, plan the backward on the side stream, one pyramid forward, one pyramid
backward (8 x 1000 ROIs, C = 256, P2-P5 256^2 .. 32^2).  Reports ms per step (CUDA events), per-call times of the
forward and the planned backward, algorithmic bytes (DESIGN 4.1 / 4.3 with the element size of the arm) over the HBM
copy bandwidth measured in the same run, the card name and power limit, and a bitwise check of (c) against (a) run on
the widened maps and grads, rounded.

    python tools/ab_lowp.py [--rounds 5] [--steps 10] [--dtype bf16|f16]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from sln_amodal_b200 import ops  # noqa: E402


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in r.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:          # no nvidia-smi: the name from the driver, the limit unknown
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({type(e).__name__})"}


def copy_peak_gbs(dev, nbytes=2 << 30, reps=10):
    """HBM bandwidth of a device-to-device copy of nbytes (read + write), GB/s: the yardstick of the fractions."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device=dev).normal_()
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e6)


def fwd_bytes(boxes, level, pool, esz):
    total_r = 0
    for l, side in enumerate(bench.LEVEL_SIDES):
        sel = level == l
        if sel.any():
            b = boxes[sel]
            u = bench._distinct_taps(b[:, 0], b[:, 2], side, pool) * bench._distinct_taps(b[:, 1], b[:, 3], side, pool)
            total_r += esz * bench.CHANNELS * min(int(u.sum()), bench.IMAGES_PER_GPU * side * side)
    n = boxes.shape[0]
    return esz * n * bench.CHANNELS * pool * pool + total_r + 20 * n


def bwd_bytes(level, pool, esz):
    C, B = bench.CHANNELS, bench.IMAGES_PER_GPU
    return sum(esz * int((level == l).sum()) * C * pool * pool + 20 * int((level == l).sum()) + esz * B * C * side * side
               for l, side in enumerate(bench.LEVEL_SIDES))


def bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    na, nb = torch.isnan(a), torch.isnan(b)
    if not torch.equal(na, nb):
        return False
    iv = torch.int16 if a.element_size() == 2 else torch.int32
    return bool(torch.equal(a.view(iv)[~na], b.view(iv)[~nb]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--dtype", choices=["bf16", "f16"], default="bf16")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ab_lowp.py measures on a CUDA device; there is nothing to measure without one"
    D = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    dev = torch.device("cuda", 0)
    boxes_np, ind_np, level_np = bench.make_workload()
    n = boxes_np.shape[0]
    boxes, ind, level = (torch.from_numpy(a).to(dev) for a in (boxes_np, ind_np, level_np))
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    cl = torch.channels_last
    maps32 = [torch.randn((bench.IMAGES_PER_GPU, bench.CHANNELS, s, s), device=dev, generator=g).contiguous(memory_format=cl)
              for s in bench.LEVEL_SIDES]
    mapsD = [m.to(D) for m in maps32]
    sizes = [tuple(m.shape) for m in maps32]
    grads32 = {p: torch.randn((n, bench.CHANNELS, p, p), device=dev, generator=g).contiguous(memory_format=cl) for p in bench.POOLS}
    gradsD = {p: t.to(D) for p, t in grads32.items()}

    def fwd(arm, p):
        if arm == "f32":
            return ops.pyramid_crop_forward(maps32, boxes, ind, level, p, p)
        return ops.pyramid_crop_forward(mapsD, boxes, ind, level, p, p, keep_dtype=(arm == "native"))

    def bwd(arm, p, plan):
        if arm == "f32":
            return ops.pyramid_crop_backward(grads32[p], boxes, ind, level, sizes, plan=plan)
        if arm == "today":
            return [o.to(D) for o in ops.pyramid_crop_backward(gradsD[p], boxes, ind, level, sizes, plan=plan)]
        return ops.pyramid_crop_backward(gradsD[p], boxes, ind, level, sizes, plan=plan, out_dtype=D)

    def step(arm):
        outs = {}
        for p in bench.POOLS:
            plan = ops.pyramid_crop_backward_plan(boxes, ind, level, sizes, bench.CHANNELS, p, p)
            outs[p] = (fwd(arm, p), bwd(arm, p, plan))
        return outs

    arms = ["f32", "today", "native"]
    for arm in arms:
        for _ in range(3):
            step(arm)
    torch.cuda.synchronize()

    # ---- ms per step, arms alternated round by round
    per_step = {a: [] for a in arms}
    for _ in range(args.rounds):
        for arm in arms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                last = None
                last = step(arm)
            e1.record()
            torch.cuda.synchronize()
            per_step[arm].append(e0.elapsed_time(e1) / args.steps)
            del last

    # ---- per-call times (same buffers; the working set is far larger than L2)
    def time_op(fn, reps=10):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    peak = copy_peak_gbs(dev)
    calls = []
    for p in bench.POOLS:
        plan = ops.pyramid_crop_backward_plan(boxes, ind, level, sizes, bench.CHANNELS, p, p)
        for arm in arms:
            esz = 4 if arm == "f32" else 2
            tf = time_op(lambda: fwd(arm, p))
            tb = time_op(lambda: bwd(arm, p, plan))
            bf, bb = fwd_bytes(boxes_np, level_np, p, esz), bwd_bytes(level_np, p, esz)
            calls.append({"arm": arm, "pool": p, "fwd_ms": round(tf, 4), "bwd_planned_ms": round(tb, 4),
                          "fwd_bytes": bf, "bwd_bytes": bb,
                          "fwd_frac": round(bf / tf / 1e6 / peak, 4), "bwd_frac": round(bb / tb / 1e6 / peak, 4)})

    # ---- bitwise: (c) against (a) on the widened maps and grads, rounded
    wide = [m.float() for m in mapsD]
    checks = {}
    for p in bench.POOLS:
        plan = ops.pyramid_crop_backward_plan(boxes, ind, level, sizes, bench.CHANNELS, p, p)
        got_c = ops.pyramid_crop_forward(mapsD, boxes, ind, level, p, p, keep_dtype=True)
        want_c = ops.pyramid_crop_forward(wide, boxes, ind, level, p, p).to(D)
        got_g = ops.pyramid_crop_backward(gradsD[p], boxes, ind, level, sizes, plan=plan, out_dtype=D)
        want_g = ops.pyramid_crop_backward(gradsD[p].float(), boxes, ind, level, sizes, plan=plan)
        checks[f"{p}x{p}"] = {"crops": bits_equal(got_c, want_c),
                              "grad_maps": all(bits_equal(a, b.to(D)) for a, b in zip(got_g, want_g))}

    step_bytes = {a: sum(c["fwd_bytes"] + c["bwd_bytes"] for c in calls if c["arm"] == a) for a in arms}
    med = {a: float(np.median(v)) for a, v in per_step.items()}
    res = {"what": "config-2 step (8 x 1000 ROIs, C=256, P2-P5, 7x7 + 14x14, backward planned), arms alternated",
           "dtype": args.dtype, "card": card(), "copy_peak_gbs": round(peak, 1),
           "ms_per_step_median": {a: round(v, 4) for a, v in med.items()},
           "ms_per_step_all": {a: [round(x, 4) for x in v] for a, v in per_step.items()},
           "step_bytes": step_bytes,
           "step_frac_of_copy_peak": {a: round(step_bytes[a] / med[a] / 1e6 / peak, 4) for a in arms},
           "calls": calls, "bitwise_native_vs_widened_f32": checks}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
