#!/usr/bin/env python
"""bench.py -- throughput of the SLN-Amodal detection-head hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (our arm)
    python bench.py --impl reference --gpus N --steps K --warmup W   (reference CPU arm)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs bench_outputs  (also the last step's outputs)

Headline metric (BASELINE.json configs[1]): RoIAlign crop_and_resize fwd+bwd ROIs/s on
256-channel FPN P2-P5, batch 8 per GPU, 1000 ROIs/img, 7x7 and 14x14, fp32.  A "step" is one
pass of that path over one batch: for each pool size, one pyramid forward launch plus one
deterministic backward call covering every level.  `value` counts ROI crops (fwd+bwd) per second with
inputs resident in HBM; `e2e` is the same work through the reference-facing operator
(CropAndResizeFunction) with HOST buffers, H2D/D2H copies inside the timed region.
The line also carries `roofline` (dominant kernel vs the measured HBM copy peak),
`cpu_baseline` (the reference's own C ops on this host) and `extra` (NMS us @12k, proposal
layer, layer decode, EDT) so every number of BASELINE.json's metric appears in one run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True    # the tree may be read-only: the benchmark writes nothing into it
if "reference" in sys.argv:
    # the reference arm uses every host core; torchrun exports OMP_NUM_THREADS=1 to its workers, and the OpenMP runtime
    # reads the variable when it is first loaded (with torch, below), so it has to be overridden here
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)

from sln_amodal_b200 import synth  # noqa: E402

IMAGES_PER_GPU = 8
ROIS_PER_IMAGE = 1000
CHANNELS = 256
POOLS = (7, 14)
LEVEL_SIDES = (256, 128, 64, 32)
CPU_SAMPLE_ROIS = 500             # bounded CPU sample: the first 500 ROIs of image 0, both pools
WORKLOAD = ("config2: RoIAlign crop_and_resize fwd+bwd, %d imgs/GPU, C=%d, FPN P2-P5 (256^2..32^2), "
            "%d ROIs/img, pools 7x7+14x14, fp32" % (IMAGES_PER_GPU, CHANNELS, ROIS_PER_IMAGE))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            # the driver's file names the copy bandwidth `hbm_gbs`; tolerate nesting / near-synonyms of that key
            flat = dict(d)
            for v in d.values():
                if isinstance(v, dict):
                    flat.update(v)
            for key in ("hbm_gbs", "hbm_gb_s", "hbm_copy_gbs", "hbm_bandwidth_gbs", "hbm"):
                if key in flat and float(flat[key]) > 0:
                    v = float(flat[key])
                    return (v * 1000.0 if v < 100.0 else v), "measured (MEASURED_PEAKS.json %s)" % key     # TB/s -> GB/s
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _ncu_traffic(k):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/)."""
    try:
        name = "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else "r01_traffic.json"
        t = json.load(open(os.path.join(ROOT, "profiles", name)))["bytes"]
        pool = "14x14" if "14x14" in k["what"] else "7x7"
        return t.get("%s %s" % (k["kernel"], pool))
    except Exception:
        return None


def make_workload(seed_shift=0):
    n = IMAGES_PER_GPU * ROIS_PER_IMAGE
    boxes = synth.roi_boxes(n, seed=4321 + seed_shift)
    level = synth.fpn_level(boxes) - 2
    box_ind = np.repeat(np.arange(IMAGES_PER_GPU, dtype=np.int32), ROIS_PER_IMAGE)
    return boxes, box_ind, level.astype(np.int32)


DUMP_SEED = 20241020
DUMP_CROP_SAMPLES = 1 << 21       # per pool: 8 MB of the 100 MB (7x7) / 401 MB (14x14) of crops
DUMP_GRAD_SAMPLES = 1 << 20       # per pool and level: 4 MB; 48 MB in all


def dump_outputs(out_dir, outs):
    """Writes what one step returned to its caller -- per pool the crops [N, C, p, p] and the four gradient maps
    [B, C, H_l, W_l] -- as float32 .npy files.  Each array is a fixed, seeded sample of its elements (flat indices in
    NCHW order, ascending), so two builds run with the same arguments can be compared element for element."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = []
    for p in POOLS:
        crops, gmaps = outs[p]
        arrays.append(("crops_%dx%d" % (p, p), crops, DUMP_CROP_SAMPLES))
        arrays += [("grad_p%d_%dx%d" % (l + 2, p, p), gm, DUMP_GRAD_SAMPLES) for l, gm in enumerate(gmaps)]
    for k, (name, t, n) in enumerate(arrays):
        rng = np.random.default_rng([DUMP_SEED, k])
        idx = np.sort(rng.choice(t.numel(), min(n, t.numel()), replace=False))
        sample = torch.take(t, torch.from_numpy(idx).to(t.device))    # logical (NCHW) order whatever the strides
        np.save(os.path.join(out_dir, name + ".npy"), sample.cpu().numpy().astype(np.float32))


# --------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY.md section 8(d))
# --------------------------------------------------------------------------------------
def _distinct_taps(a1, a2, extent, crop):
    """Per ROI: number of distinct source rows (or columns) its valid samples touch."""
    f = np.float32
    a1, a2 = a1.astype(f), a2.astype(f)
    em1 = f(extent - 1)
    scale = (a2 - a1) * em1 / f(crop - 1)
    k = np.arange(crop, dtype=f)[None, :]
    pos = (a1 * em1)[:, None] + k * scale[:, None]
    valid = (pos >= 0) & (pos <= em1)
    lo = np.floor(pos).astype(np.int64)
    hi = np.ceil(pos).astype(np.int64)
    vals = np.concatenate([np.where(valid, lo, -1), np.where(valid, hi, -1)], 1)
    vals.sort(axis=1)
    distinct = (np.diff(vals, axis=1) != 0).sum(1) + 1
    distinct -= (vals[:, 0] == -1)          # the -1 placeholder is not a tap
    return np.maximum(distinct, 0)


def fwd_bytes(boxes, box_ind, level, pool):
    total_r = 0
    for l, side in enumerate(LEVEL_SIDES):
        sel = level == l
        if not sel.any():
            continue
        b = boxes[sel]
        u = _distinct_taps(b[:, 0], b[:, 2], side, pool) * _distinct_taps(b[:, 1], b[:, 3], side, pool)
        total_r += 4 * CHANNELS * min(int(u.sum()), IMAGES_PER_GPU * side * side)
    n = boxes.shape[0]
    return 4 * n * CHANNELS * pool * pool + total_r + 20 * n


def bwd_bytes(n_level, side, pool):
    return 4 * n_level * CHANNELS * pool * pool + 20 * n_level + 4 * IMAGES_PER_GPU * CHANNELS * side * side


# --------------------------------------------------------------------------------------
# clocks sampling during the timed region
# --------------------------------------------------------------------------------------
class ClockSampler:
    """One `nvidia-smi -lms 20` child process; samples are time-stamped on arrival so that the ones taken
    inside the timed window can be selected afterwards."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []          # (host time, fields)
        self.proc = None
        self.t = None

    def _run(self):
        try:
            for line in self.proc.stdout:
                self.samples.append((time.perf_counter(), [x.strip() for x in line.strip().split(",")]))
        except Exception:
            pass

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.t.join(timeout=5)

    def summary(self, t0=None, t1=None):
        sel = [f for (t, f) in self.samples if t0 is None or (t0 <= t <= t1)]
        window = "timed region"
        if len(sel) < 3:
            sel = [f for (_, f) in self.samples]
            window = "timed region + load extension"
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in sel:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
                for nm, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# --------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    from sln_amodal_b200 import _lib, ops, dist as sdist
    from sln_amodal_b200.crop_and_resize import CropAndResizeFunction

    # keep stdout clean for the single JSON line: libraries (NCCL's version banner, ...) write to fd 1
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world = sdist.init()
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback exists)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.lib()

    boxes_np, ind_np, level_np = make_workload(seed_shift=rank)
    n_rois = boxes_np.shape[0]
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    maps = [torch.randn((IMAGES_PER_GPU, CHANNELS, s, s), device=dev, generator=g).contiguous(memory_format=torch.channels_last)
            for s in LEVEL_SIDES]
    boxes = torch.from_numpy(boxes_np).to(dev)
    box_ind = torch.from_numpy(ind_np).to(dev)
    level = torch.from_numpy(level_np).to(dev)
    grads = {p: torch.randn((n_rois, CHANNELS, p, p), device=dev, generator=g).contiguous(memory_format=torch.channels_last)
             for p in POOLS}
    sizes = [tuple(m.shape) for m in maps]

    plan_ahead = os.environ.get("SLN_BENCH_NO_PLAN", "0") != "1"

    def step():
        # what the autograd operator does (pyramid._PyramidCrop): the backward's ROI lists are planned on a side stream
        # beside the forward kernel (they depend on the boxes only); the plan launches are inside the timed region
        outs = {}
        for p in POOLS:
            plan = ops.pyramid_crop_backward_plan(boxes, box_ind, level, sizes, CHANNELS, p, p) if plan_ahead else None
            crops = ops.pyramid_crop_forward(maps, boxes, box_ind, level, p, p, 0.0)
            outs[p] = (crops, ops.pyramid_crop_backward(grads[p], boxes, box_ind, level, sizes, plan=plan))
        return outs

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launches()
    with ClockSampler(local_rank) as clocks:
        barrier()
        t_start = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            # the previous step's outputs go back to the allocator first: every timed step then allocates exactly like the
            # warmup steps, from blocks the allocator already holds (no cudaMalloc inside the timed region)
            last = None
            last = step()
        e1.record()
        barrier()
        t_end = time.perf_counter()
        launches_timed = _lib.launches() - l0
        # the timed region can be shorter than nvidia-smi's sampling period: keep the same load running
        # (untimed) until a few clock samples exist, so throttling during this workload is visible
        t_ext = time.perf_counter()
        while time.perf_counter() - t_ext < 0.6:
            step()
        torch.cuda.synchronize()
    clocks_summary = clocks.summary(t_start, t_end)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    del last
    launches = launches_timed
    ms_total = sdist.max_over_ranks(e0.elapsed_time(e1))
    ms_per_step = ms_total / args.steps
    crops_per_step = n_rois * len(POOLS) * world
    value = crops_per_step / (ms_per_step * 1e-3)

    # ---- per-kernel timings for the roofline (separate pass, same buffers; working set >> L2)
    def time_op(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    peak, peak_src = measured_peak_gbs()
    kernels = []
    for p in POOLS:
        ms = time_op(lambda: ops.pyramid_crop_forward(maps, boxes, box_ind, level, p, p, 0.0))
        by = fwd_bytes(boxes_np, ind_np, level_np, p)
        kernels.append({"kernel": "crop_fwd_nhwc_kernel", "what": "pyramid fwd %dx%d" % (p, p), "ms": ms,
                        "algorithmic_bytes": by, "achieved_gbs": by / ms / 1e6})
        ms = time_op(lambda: ops.pyramid_crop_backward(grads[p], boxes, box_ind, level, sizes))
        by = sum(bwd_bytes(int((level_np == l).sum()), side, p) for l, side in enumerate(LEVEL_SIDES))
        pl = ops.pyramid_crop_backward_plan(boxes, box_ind, level, sizes, CHANNELS, p, p)
        ms_pl = time_op(lambda: ops.pyramid_crop_backward(grads[p], boxes, box_ind, level, sizes, plan=pl))
        if plan_ahead:       # what the step runs: the ROI lists come from the plan (built beside the forward)
            kernels.append({"kernel": "crop_bwd_tma_kernel",
                            "what": "pyramid bwd %dx%d, all levels (ROI lists planned ahead; republish + main kernel)" % (p, p),
                            "ms": ms_pl, "algorithmic_bytes": by, "achieved_gbs": by / ms_pl / 1e6,
                            "ms_incl_prep_launches": ms, "frac_incl_prep_launches": by / ms / 1e6})
        else:
            kernels.append({"kernel": "crop_bwd_tma_kernel",
                            "what": "pyramid bwd %dx%d, all levels (incl. 3 prep launches)" % (p, p),
                            "ms": ms, "algorithmic_bytes": by, "achieved_gbs": by / ms / 1e6,
                            "ms_planned_ahead": ms_pl, "frac_planned_ahead": by / ms_pl / 1e6})
    for k in kernels:
        k["frac"] = k["achieved_gbs"] / peak
        for kk in ("frac_planned_ahead", "frac_incl_prep_launches"):
            if kk in k:
                k[kk] = k[kk] / peak
    dom = max(kernels, key=lambda k: k["ms"])
    step_bytes = sum(k["algorithmic_bytes"] for k in kernels)
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "what": dom["what"], "achieved": round(dom["achieved_gbs"], 1),
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": round(dom["frac"], 4),
                "traffic": _ncu_traffic(dom),
                "step": {"algorithmic_bytes": step_bytes, "achieved": round(step_bytes / ms_per_step / 1e6, 1),
                         "frac": round(step_bytes / ms_per_step / 1e6 / peak, 4),
                         "frac_of_8TBs_nominal": round(step_bytes / ms_per_step / 1e6 / 8000.0, 4)}}

    # ---- e2e: reference-facing operator with HOST buffers (pinned), copies inside the timed region
    def pinned_like(t):
        return torch.empty(t.shape, dtype=torch.float32, memory_format=torch.channels_last).pin_memory()

    lvl_sel = [np.nonzero(level_np == l)[0] for l in range(4)]
    h_maps = [pinned_like(m) for m in maps]
    for hm, m in zip(h_maps, maps):
        hm.copy_(m)
    h_boxes = [boxes[torch.from_numpy(ix).to(dev)].cpu().pin_memory() for ix in lvl_sel]
    h_ind = [box_ind[torch.from_numpy(ix).to(dev)].cpu().pin_memory() for ix in lvl_sel]
    h_grads = {p: [pinned_like(grads[p][: len(ix)]) for ix in lvl_sel] for p in POOLS}
    for p in POOLS:
        for l, ix in enumerate(lvl_sel):
            h_grads[p][l].copy_(grads[p][: len(ix)])
    # results land in one of two sets of host buffers (steps alternate), so a step's results stay readable while the next
    # step's copies are already under way
    h_out_sets = [{p: [pinned_like(grads[p][: len(ix)]) for ix in lvl_sel] for p in POOLS} for _ in range(2)]
    h_gmaps_sets = [[pinned_like(m) for m in maps] for _ in range(2)]
    h_out, h_gmaps = h_out_sets[0], h_gmaps_sets[0]
    step_no = [0]
    # SLN_BENCH_E2E_SERIAL=1: every step drains its device->host copies before the next step's host->device copies start
    pipelined = os.environ.get("SLN_BENCH_E2E_SERIAL", "0") != "1"
    h2d = (sum(hm.numel() for hm in h_maps) + sum(t.numel() for t in h_boxes) + sum(t.numel() for t in h_ind)
           + sum(t.numel() for p in POOLS for t in h_grads[p])) * 4
    d2h = (sum(t.numel() for p in POOLS for t in h_out[p]) + sum(hm.numel() for hm in h_gmaps)) * 4

    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def e2e_step():
        # the call a reference user makes (modals.py:96): CropAndResizeFunction(ph,pw,0)(P_l, boxes_l, ind_l), then
        # backward.  Host->device copies run on their own stream, device->host copies on another, so the two PCIe
        # directions and the kernels overlap; every byte still moves inside the timed region.
        cur = torch.cuda.current_stream()
        if not pipelined:
            s_in.wait_stream(cur)
        h_out, h_gmaps = h_out_sets[step_no[0] % 2], h_gmaps_sets[step_no[0] % 2]
        step_no[0] += 1
        order = [(p, l) for p in POOLS for l in (3, 2, 1, 0)]      # small maps first: kernels and D2H start at once
        d_maps, d_boxes, d_ind, ev_lvl, d_g, ev_g = {}, {}, {}, {}, {}, {}
        with torch.cuda.stream(s_in):
            for p, l in order:
                if l not in d_maps:                                 # a level's map / boxes travel right before first use
                    d_maps[l] = h_maps[l].to(dev, non_blocking=True)
                    d_boxes[l] = h_boxes[l].to(dev, non_blocking=True)
                    d_ind[l] = h_ind[l].to(dev, non_blocking=True)
                    ev_lvl[l] = torch.cuda.Event()
                    ev_lvl[l].record(s_in)
                d_g[p, l] = h_grads[p][l].to(dev, non_blocking=True)
                ev_g[p, l] = torch.cuda.Event()
                ev_g[p, l].record(s_in)
        seen = set()
        for p, l in order:
            if l not in seen:
                seen.add(l)
                cur.wait_event(ev_lvl[l])
                for t in (d_maps[l], d_boxes[l], d_ind[l]):
                    t.record_stream(cur)
                d_maps[l].requires_grad_(True)
            cur.wait_event(ev_g[p, l])
            d_g[p, l].record_stream(cur)
            out = CropAndResizeFunction(p, p, 0)(d_maps[l], d_boxes[l], d_ind[l])
            out.backward(d_g[p, l])                                 # autograd sums both pools' gradients into .grad
            last = p == POOLS[-1]
            gm = d_maps[l].grad if last else None
            s_out.wait_stream(cur)
            with torch.cuda.stream(s_out):
                h_out[p][l].copy_(out.detach(), non_blocking=True)
                if last:                                            # one copy per map, as a training step would do
                    h_gmaps[l].copy_(gm, non_blocking=True)
            out.record_stream(s_out)
            if last:
                gm.record_stream(s_out)
                d_maps[l].grad = None
        if not pipelined:
            cur.wait_stream(s_out)

    e2e_steps = max(2, min(args.steps, 5))
    e2e_step()
    barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.current_stream().wait_stream(s_out)           # the last step's results are on the host before the clock stops
    b.record()
    barrier()
    e2e_ms = sdist.max_over_ranks(a.elapsed_time(b)) / e2e_steps
    e2e = {"value": round(crops_per_step / (e2e_ms * 1e-3), 1), "unit": "roi_crops/s", "ms_per_step": round(e2e_ms, 3),
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
           "api": "CropAndResizeFunction(ph,pw,0)(image,boxes,box_ind) + .backward per FPN level; pinned host buffers in and out; "
                  "H2D, kernels and D2H on three streams (both PCIe directions overlap); the gradient maps of the two pools are summed "
                  "on the device by autograd and copied once; " +
                  ("steps pipelined: step k+1's H2D runs while step k's D2H drains into the other of two host result sets, the "
                   "clock stops after the last D2H" if pipelined else "every step drains its D2H before the next H2D starts")}
    del h_maps, h_grads, h_out, h_gmaps, h_out_sets, h_gmaps_sets

    # ---- config 1 on every rank: images/s of the detection-head path over rank-sharded images (BASELINE metric 3)
    images = head_throughput(dev, rank, world, barrier, sdist)

    # ---- config 5 on every rank: the full training step, data-parallel with DDP all-reduce (tools/train_step.py)
    train = None
    if os.environ.get("SLN_BENCH_TRAIN", "1") != "0":
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import train_step
            torch.cuda.empty_cache()
            train = train_step.run(dev, rank, world, steps=2, warmup=1)
        except Exception as e:                               # the harness is outside the hot path: never lose the headline to it
            train = {"error": "%s: %s" % (type(e).__name__, e)}
        torch.cuda.empty_cache()

    # ---- the rest of the config-2 sweep (rank 0): 16x16, and 4000 ROIs per image, same maps
    sweep = []
    if rank == 0:
        del grads
        torch.cuda.empty_cache()
        for per in (ROIS_PER_IMAGE, 4000):
            n = IMAGES_PER_GPU * per
            b_np = synth.roi_boxes(n, seed=4321)
            l_np = (synth.fpn_level(b_np) - 2).astype(np.int32)
            i_np = np.repeat(np.arange(IMAGES_PER_GPU, dtype=np.int32), per)
            tb, ti, tl = (torch.from_numpy(a).to(dev) for a in (b_np, i_np, l_np))
            for p in (7, 14, 16):
                if per == ROIS_PER_IMAGE and p in POOLS:
                    continue                                        # already in `kernels`
                gp = torch.randn((n, CHANNELS, p, p), device=dev, generator=g).contiguous(memory_format=torch.channels_last)
                tf = time_op(lambda: ops.pyramid_crop_forward(maps, tb, ti, tl, p, p, 0.0))
                tbw = time_op(lambda: ops.pyramid_crop_backward(gp, tb, ti, tl, sizes))
                bf = fwd_bytes(b_np, i_np, l_np, p)
                bb = sum(bwd_bytes(int((l_np == l).sum()), side, p) for l, side in enumerate(LEVEL_SIDES))
                sweep.append({"rois_per_img": per, "pool": p, "fwd_ms": round(tf, 4), "fwd_frac": round(bf / tf / 1e6 / peak, 4),
                              "bwd_ms": round(tbw, 4), "bwd_frac": round(bb / tbw / 1e6 / peak, 4),
                              "fwd_bwd_rois_per_s": round(n / ((tf + tbw) * 1e-3), 1)})
                del gp
        torch.cuda.empty_cache()

    extra = {}
    cpu_baseline = None
    if rank == 0:
        extra = side_metrics(dev, peak)
        extra["head_pipeline"] = head_pipeline(dev, cpu=(world == 1))
        extra["detection_targets"] = detection_targets_metric(dev, cpu=(world == 1))
        extra["rpn_targets"] = rpn_targets_metric(dev, cpu=(world == 1))
        extra["rle"] = rle_metric(dev, peak, cpu=(world == 1))
        extra["unmold"] = unmold_metric(dev, peak, cpu=(world == 1))
        extra["rpn_pack"] = rpn_pack_metric(dev, peak, cpu=(world == 1))
        extra["resize_image"] = resize_image_metric(dev, cpu=(world == 1))
        try:
            extra["nchw_dropin"] = nchw_dropin_metric(dev, maps, boxes, box_ind, level, peak)
        except Exception as e:
            extra["nchw_dropin"] = {"error": "%s: %s" % (type(e).__name__, e)}
        if world == 1:
            try:
                extra["ref_cuda"] = ref_cuda_metric(dev, maps, boxes_np, ind_np, level_np)
            except Exception as e:
                extra["ref_cuda"] = {"error": "%s: %s" % (type(e).__name__, e)}
        if world == 1:
            cpu_baseline = cpu_reference_sample(boxes_np, ind_np, level_np, maps)

    if rank == 0:
        # the other numbers BASELINE.json's metric names, where the driver's record keeps them (it drops `extra`)
        nms12k = [r for r in extra.get("nms", []) if r.get("n") == 12000]
        by_kernel = {k["what"].split(",")[0]: round(k["frac"], 4) for k in kernels}
        also = {"frac_by_kernel_of_measured_hbm": by_kernel,
                "config2_sweep": sweep,
                "nms_us_12k": {r["boxes"]: r["us_median"] for r in nms12k},
                "nms_us_12k_sync_free_call": {r["boxes"]: r["us_with_fallback"] for r in nms12k},
                "nms_us_12k_dense_fallback": {r["boxes"]: r["us_dense_pipeline"] for r in nms12k if "us_dense_pipeline" in r},
                "nms_us_1k": {r["boxes"]: r["us_median"] for r in extra.get("nms", []) if r.get("n") == 1000},
                "proposal_layer_us": extra.get("proposal_layer", {}).get("us_median"),
                "edt_frac": extra.get("edt", {}).get("frac"), "edt_us_320_maps": extra.get("edt", {}).get("us_median"),
                "layer_decode_frac": extra.get("layer_decode", {}).get("frac"),
                "images_per_s": images["images_per_s"], "images_per_s_e2e": images["e2e"]["images_per_s"],
                "images_per_s_graph_replay": images["graph"]["images_per_s"],
                "images_per_s_graph_4_images_per_launch": images["graph"].get("images_per_s_4_images_per_launch"),
                "images_per_s_graph_8_images_per_launch": images["graph"].get("images_per_s_8_images_per_launch"),
                "ref_cuda_sm100a": extra.get("ref_cuda"), "nchw_dropin": extra.get("nchw_dropin"),
                "train_step_images_per_s": (train or {}).get("images_per_s"),
                "train_step_allreduce_share": (train or {}).get("allreduce_share")}
        roofline["also_measured"] = also
        line = {
            "metric": "roialign_fwd_bwd_roi_crops_per_s", "value": round(value, 1), "unit": "roi_crops/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "layout": "channels_last (NHWC kernels)", "rois_per_step_per_gpu": n_rois,
                       "l2_policy": "working set 4.7 GB per step >> 126 MB L2 (no flush needed)",
                       "sharding": "images (box_ind) across ranks; no data-path collective",
                       "backward_planning": ("ROI lists planned on a side stream beside the forward (inside the timed region)"
                                             if plan_ahead else "ROI lists planned inside the backward call"),
                       "images_per_s": images["images_per_s"], "images_per_s_e2e": images["e2e"]["images_per_s"],
                       "images_per_s_graph_replay": images["graph"]["images_per_s"],
                       "images_per_s_graph_4_images_per_launch": images["graph"].get("images_per_s_4_images_per_launch"),
                       "images_per_s_what": images["what"]},
            "clocks": clocks_summary, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "cpu_baseline": cpu_baseline,
            "kernels": [{k2: (round(v, 4) if isinstance(v, float) else v) for k2, v in k.items()} for k in kernels],
            "images": images,
            "train_step": train,
            "extra": extra,
        }
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def head_throughput(dev, rank, world, barrier, sdist, n_img=32):
    """BASELINE.json's third metric: images/s of the detection-head path (configs[0] without the out-of-scope convolutions)
    on EVERY rank over its own shard of images.  Per image: 261 888 anchors -> proposal_layer (top 6000, NMS 0.7, 1000 ROIs)
    -> pyramid_roi_align 7x7 -> refine_detections with the reference's shipped default config (USE_NMS = False: top-100,
    config.py:78) -> pyramid_roi_align 14x14 on the detections, every call through the reference's own signatures.
    Two timed regions (barrier + CUDA events, max over ranks): inputs resident in HBM, and end to end with the RPN /
    classifier outputs and the FPN maps copied from pinned host memory and the detections copied back, per image."""
    import torch
    from sln_amodal_b200 import proposal_layer, pyramid_roi_align, refine_detections
    A, K, n_sets = 261888, 81, 4
    anchors = torch.from_numpy(synth.nms_boxes(A, seed=4, kind="rpn")).to(dev)
    cfg = _HeadCfg()
    cfg.USE_NMS = False
    window = (0.0, 0.0, 1024.0, 1024.0)
    host, devs = [], []
    for k in range(n_sets):
        rng = np.random.default_rng(1000 * rank + 101 + k)
        fg = rng.permutation(np.linspace(0, 1, A)).astype(np.float32)
        cls_logits = rng.standard_normal((1000, K)).astype(np.float32) * 3.0
        arrs = {"probs": np.stack([1 - fg, fg], 1).astype(np.float32)[None],
                "deltas": (rng.standard_normal((A, 4)) * 0.5).astype(np.float32)[None],
                "cls_probs": (np.exp(cls_logits) / np.exp(cls_logits).sum(1, keepdims=True)).astype(np.float32),
                "cls_deltas": (rng.standard_normal((1000, K, 4)) * 0.3).astype(np.float32)}
        h = {k2: torch.from_numpy(v).pin_memory() for k2, v in arrs.items()}
        h["maps"] = [torch.randn((1, CHANNELS, s_, s_)).contiguous(memory_format=torch.channels_last).pin_memory() for s_ in LEVEL_SIDES]
        host.append(h)
        devs.append({k2: ([m.to(dev) for m in v] if k2 == "maps" else v.to(dev)) for k2, v in h.items()})
    h_det = torch.empty((100, 6), dtype=torch.float32).pin_memory()
    h2d = sum(v.numel() for k2, v in host[0].items() if k2 != "maps") * 4 + sum(m.numel() for m in host[0]["maps"]) * 4

    def one_image(d):
        rois = proposal_layer([d["probs"], d["deltas"]], 1000, 0.7, anchors, cfg)           # [1,k,4]
        k = rois.shape[1]
        pooled = pyramid_roi_align([rois] + d["maps"], 7, cfg.IMAGE_SHAPE)                  # classifier input
        det, keep = refine_detections(rois[0], d["cls_probs"][:k], d["cls_deltas"][:k], window, cfg)
        masks_in = pyramid_roi_align([(det[:, :4] / 1024.0).unsqueeze(0)] + d["maps"], 14, cfg.IMAGE_SHAPE)
        return det, pooled, masks_in

    def one_image_e2e(h):
        d = {k2: ([m.to(dev, non_blocking=True) for m in v] if k2 == "maps" else v.to(dev, non_blocking=True)) for k2, v in h.items()}
        det, _, _ = one_image(d)
        h_det[: det.shape[0]].copy_(det, non_blocking=True)
        return det

    def timed(fn, sets):
        for i in range(3):
            fn(sets[i % n_sets])
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n_img):
            fn(sets[i % n_sets])
        b.record()
        barrier()
        return sdist.max_over_ranks(a.elapsed_time(b))

    ms_dev = timed(one_image, devs)
    ms_e2e = timed(one_image_e2e, host)
    det = one_image(devs[0])[0]
    # the same kernels driven the B200 way: every step padded and sync-free, captured once per resident input set into a
    # CUDA graph, one launch per image (sln_amodal_b200/pipeline.py); detections checked against the eager call above
    from sln_amodal_b200 import pipeline
    gcfg = _HeadCfg()
    gcfg.USE_NMS = False
    gcfg.RPN_NMS_THRESHOLD, gcfg.POOL_SIZE, gcfg.MASK_POOL_SIZE = 0.7, 7, 14
    graphs = [pipeline.HeadGraph(anchors, gcfg, d["maps"], d["probs"][0], d["deltas"][0], (d["cls_probs"], d["cls_deltas"]))
              for d in devs]
    ms_graph = timed(lambda g: g.replay(), graphs)
    # and several independent images per launch: the chains of the resident input sets as parallel branches of one graph
    multi_res = {}
    for per_launch in (n_sets, 2 * n_sets):
        srcs = [devs[i % n_sets] for i in range(per_launch)]
        multi = pipeline.MultiHeadGraph([pipeline.HeadGraph(anchors, gcfg, d["maps"], d["probs"][0], d["deltas"][0],
                                                            (d["cls_probs"], d["cls_deltas"]), capture=False) for d in srcs])
        for _ in range(3):
            multi.replay()
        barrier()
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev_a.record()
        for _ in range(n_img // n_sets):
            multi.replay()
        ev_b.record()
        barrier()
        ms_multi = sdist.max_over_ranks(ev_a.elapsed_time(ev_b))
        m_out = multi.out[0]
        torch.cuda.synchronize()
        same = bool(int(m_out["num_detections"].item()) == det.shape[0] and torch.equal(m_out["detections"][: det.shape[0]], det))
        multi_res[per_launch] = (round(world * (n_img // n_sets) * per_launch / (ms_multi * 1e-3), 1), same)
        del multi, m_out
    g_out = graphs[0].replay()
    torch.cuda.synchronize()
    nd = int(g_out["num_detections"].item())
    graph_same = bool(nd == det.shape[0] and torch.equal(g_out["detections"][:nd], det))
    res = {"what": "proposal_layer -> pyramid_roi_align 7x7 -> refine_detections (USE_NMS=False, top-100) -> pyramid_roi_align "
                   "14x14, one 1024^2 image = 261888 anchors, C=256 FPN maps, K=81; synthetic RPN / classifier outputs "
                   "(convolutions out of scope); %d images per rank per timed region, images sharded over ranks" % n_img,
           "n_gpus": world, "images_per_rank": n_img, "detections_per_image": int(det.shape[0]),
           "ms_per_image_per_rank": round(ms_dev / n_img, 4), "images_per_s": round(world * n_img / (ms_dev * 1e-3), 1),
           "graph": {"images_per_s": round(world * n_img / (ms_graph * 1e-3), 1), "ms_per_image_per_rank": round(ms_graph / n_img, 4),
                     "detections_identical_to_eager": graph_same,
                     "images_per_s_%d_images_per_launch" % n_sets: multi_res[n_sets][0],
                     "images_per_s_%d_images_per_launch" % (2 * n_sets): multi_res[2 * n_sets][0],
                     "multi_detections_identical_to_eager": bool(multi_res[n_sets][1] and multi_res[2 * n_sets][1]),
                     "what": "pipeline.HeadGraph: the same steps padded and sync-free, captured once, one cudaGraphLaunch per image"},
           "e2e": {"images_per_s": round(world * n_img / (ms_e2e * 1e-3), 1), "ms_per_image_per_rank": round(ms_e2e / n_img, 4),
                   "h2d_bytes_per_image": int(h2d), "d2h_bytes_per_image": int(det.numel() * 4),
                   "note": "inputs from pinned host memory (RPN + classifier outputs 8 MB, FPN maps 89 MB per image: PCIe-bound), "
                           "detections copied back"},
           "timing": "CUDA events on the launching stream, barrier on both sides, max over ranks"}
    del host, devs, graphs, g_out
    torch.cuda.empty_cache()
    return res


def nchw_dropin_metric(dev, maps, boxes, box_ind, level, peak):
    """What the UNMODIFIED reference pays: its tensors are NCHW (cuDNN's default), so every map is transposed to
    channels_last once per forward pass (remembered across the crop calls that share it), crops come back channels_last,
    and the backward converts the incoming NCHW gradient and returns NCHW gradient maps (two more transposes).  Same
    config-2 inputs as the headline; `first` = with the map transposes, `cached` = later calls on the same maps."""
    import torch
    from sln_amodal_b200 import ops

    def ev_ms(fn, reps=5):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    sizes = [tuple(m.shape) for m in maps]
    rows = []
    for p in POOLS:
        def fresh():
            return [m.contiguous(memory_format=torch.contiguous_format).clone() for m in maps]
        # first call on new NCHW tensors: includes the four map transposes
        ts = []
        for _ in range(3):
            nchw = fresh()
            ts.append(ev_ms(lambda: ops.pyramid_crop_forward(nchw, boxes, box_ind, level, p, p, 0.0), reps=1))
        nchw = fresh()
        ops.pyramid_crop_forward(nchw, boxes, box_ind, level, p, p, 0.0)
        cached = ev_ms(lambda: ops.pyramid_crop_forward(nchw, boxes, box_ind, level, p, p, 0.0))
        nhwc = ev_ms(lambda: ops.pyramid_crop_forward(maps, boxes, box_ind, level, p, p, 0.0))
        g_nchw = torch.randn((boxes.shape[0], CHANNELS, p, p), device=dev)
        g_nhwc = g_nchw.contiguous(memory_format=torch.channels_last)
        b_nchw = ev_ms(lambda: ops.pyramid_crop_backward(g_nchw, boxes, box_ind, level, sizes, channels_last_out=[False] * 4))
        b_nhwc = ev_ms(lambda: ops.pyramid_crop_backward(g_nhwc, boxes, box_ind, level, sizes))
        rows.append({"pool": p, "fwd_ms_nhwc": round(nhwc, 4), "fwd_ms_nchw_first": round(float(np.median(ts)), 4),
                     "fwd_ms_nchw_cached": round(cached, 4), "bwd_ms_nhwc": round(b_nhwc, 4), "bwd_ms_nchw": round(b_nchw, 4),
                     "fwd_bwd_ratio_nchw_over_nhwc": round((float(np.median(ts)) + b_nchw) / (nhwc + b_nhwc), 3)})
        del g_nchw, g_nhwc, nchw
    return {"what": "config 2 with NCHW tensors in and out (the unmodified reference's layout)", "rows": rows,
            "note": "model.to(memory_format=torch.channels_last) -- install(channels_last_model=...) -- removes the transposes"}


def ref_cuda_metric(dev, maps, boxes_np, ind_np, level_np):
    """Speed-only comparator (BASELINE.md section 4): the reference's own CUDA kernels, unmodified, recompiled for sm_100a
    (oracle/_ref/libref_cuda.so), on the same config-2 inputs -- per FPN level like modals.py:70-97 drives them, NCHW maps,
    with the memsets the reference's host code issues (crop_and_resize_gpu.c:25, :57) -- and the reference's GPU NMS
    (nms_kernel.cu bit matrix + the blocking D2H copy + the host scan of nms_cuda.c:33-58) at 12k boxes.  torchvision's
    roi_align / nms ride along as a second, stock point.  None of this is a parity check."""
    import torch
    from oracle import oracle
    if not oracle.ref_cuda_available():
        return {"unavailable": "oracle/_ref/libref_cuda.so was not built (needs nvcc and the reference checkout at build time)"}

    def ev_ms(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    st = torch.cuda.current_stream().cuda_stream
    res = {"what": "reference CUDA kernels (unmodified, sm_100a) on the config-2 inputs, per FPN level, NCHW", "crop": []}
    nchw = [m.contiguous(memory_format=torch.contiguous_format) for m in maps]
    lv = [np.nonzero(level_np == l)[0] for l in range(4)]
    bx = [torch.from_numpy(boxes_np[ix]).to(dev) for ix in lv]
    bi = [torch.from_numpy(ind_np[ix]).to(dev) for ix in lv]
    for p in (7, 14):
        outs = [torch.empty((len(ix), CHANNELS, p, p), device=dev) for ix in lv]
        gin = [torch.randn((len(ix), CHANNELS, p, p), device=dev) for ix in lv]
        gout = [torch.empty_like(m) for m in nchw]

        def fwd():
            for l in range(4):
                outs[l].zero_()
                oracle.ref_cuda_crop_fwd(nchw[l].data_ptr(), bx[l].data_ptr(), bi[l].data_ptr(), len(lv[l]), IMAGES_PER_GPU,
                                         LEVEL_SIDES[l], LEVEL_SIDES[l], p, p, CHANNELS, 0.0, outs[l].data_ptr(), st)

        def bwd():
            for l in range(4):
                gout[l].zero_()
                oracle.ref_cuda_crop_bwd(gin[l].data_ptr(), bx[l].data_ptr(), bi[l].data_ptr(), len(lv[l]), IMAGES_PER_GPU,
                                         LEVEL_SIDES[l], LEVEL_SIDES[l], p, p, CHANNELS, gout[l].data_ptr(), st)
        row = {"pool": p, "fwd_ms": round(ev_ms(fwd), 4), "bwd_ms": round(ev_ms(bwd), 4)}
        try:
            from torchvision.ops import roi_align
            rois = [torch.cat([bi[l].float().unsqueeze(1), bx[l][:, [1, 0, 3, 2]] * (LEVEL_SIDES[l] - 1)], 1) for l in range(4)]
            row["torchvision_roi_align_fwd_ms"] = round(ev_ms(lambda: [roi_align(nchw[l], rois[l], (p, p), 1.0, 1, True) for l in range(4)]), 4)
        except Exception as e:
            row["torchvision_roi_align_fwd_ms"] = "unavailable: %s" % type(e).__name__
        res["crop"].append(row)
        del outs, gin, gout
    # NMS at 12k RPN-like boxes, thresh 0.7: the reference GPU path wants boxes sorted by score (nms_kernel.cu:16-24 reads
    # x1,y1,x2,y2,score rows)
    n = 12000
    d_np = np.concatenate([synth.nms_boxes(n, seed=7, kind="rpn"), synth.nms_scores(n, seed=8)[:, None]], 1).astype(np.float32)
    d_np = d_np[np.argsort(-d_np[:, 4], kind="stable")]
    dets = torch.from_numpy(d_np).to(dev)
    col = (n + 63) // 64
    mask = torch.empty((n, col), dtype=torch.int64, device=dev)
    h_mask = torch.empty((n, col), dtype=torch.int64).pin_memory()
    torch.cuda.synchronize()

    def ref_nms():
        oracle.ref_cuda_nms_mask(n, dets.data_ptr(), mask.data_ptr(), 0.7)       # default stream, like nms_kernel.cu:79
        h_mask.copy_(mask)                                                      # blocking D2H (nms_cuda.c:30-33)
        torch.cuda.synchronize()
        return oracle.nms_mask_scan(h_mask.numpy().view(np.uint64))
    ref_nms()
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        keep = ref_nms()
        ts.append(time.perf_counter() - t0)
    res["nms_12k_rpn"] = {"us_wall_incl_d2h_and_host_scan": round(float(np.median(ts)) * 1e6, 1), "kept": int(keep.size),
                          "mask_bytes": int(n * col * 8)}
    try:
        from torchvision.ops import nms as tv_nms
        b_xyxy = dets[:, [1, 0, 3, 2]].contiguous()
        sc = dets[:, 4].contiguous()
        tv_nms(b_xyxy, sc, 0.7)
        torch.cuda.synchronize()
        ts = []
        for _ in range(10):
            t0 = time.perf_counter()
            k2 = tv_nms(b_xyxy, sc, 0.7)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        res["nms_12k_rpn"]["torchvision_nms_us_wall"] = round(float(np.median(ts)) * 1e6, 1)
    except Exception as e:
        res["nms_12k_rpn"]["torchvision_nms_us_wall"] = "unavailable: %s" % type(e).__name__
    return res


def side_metrics(dev, peak):
    """The other numbers BASELINE.json's metric names: NMS us @ n boxes, proposal layer, layer decode, EDT."""
    import torch
    from sln_amodal_b200 import ops

    def time_us(fn, reps=20, flush=None):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            if flush is not None:
                flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) * 1e3)
        return float(np.median(ts)), float(np.min(ts))

    def graphed(fn):
        """One call captured in a CUDA graph (the whole C-ABI path is stream-ordered: cluster and cooperative launches
        included); replays measure device time without per-launch host latency."""
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        g = torch.cuda.CUDAGraph()
        # thread_local: other threads of the process (e.g. the NCCL watchdog under torchrun) may keep making CUDA calls
        with torch.cuda.graph(g, capture_error_mode="thread_local"):
            keepalive = fn()
        g.keepalive = keepalive
        return g

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    out = {"nms": [], "note": "median / min over 20 runs, CUDA events; L2 flushed between runs; us_graph = the same call "
                              "captured once in a CUDA graph and replayed"}
    for n in (1000, 2000, 4000, 6000, 8000, 12000):
        for kind, thr in (("rpn", 0.7), ("uniform", 0.7)):
            dets = torch.from_numpy(np.concatenate([synth.nms_boxes(n, seed=7, kind=kind), synth.nms_scores(n, seed=8)[:, None]], 1)).to(dev)
            keep, num, path = ops.nms_device(dets, thr, return_path=True)
            sparse = int(path.item()) == 1
            # what nms(dets, thresh) launches: the sparse pipeline alone when it takes the input (a bail-out would show as
            # num_keep < 0 and be retried dense); us_with_fallback = the sync-free call that also enqueues the dense kernels
            med, mn = time_us(lambda: ops.nms_device(dets, thr, sparse_only=sparse), flush=flush)
            med_fb, _ = time_us(lambda: ops.nms_device(dets, thr), flush=flush)
            g = graphed(lambda: ops.nms_device(dets, thr, sparse_only=sparse))
            med_g, _ = time_us(g.replay, flush=flush)
            del g
            row = {"n": n, "boxes": kind, "thresh": thr, "kept": int(num.item()), "us_median": round(med, 1),
                   "us_min": round(mn, 1), "us_with_fallback": round(med_fb, 1), "us_graph": round(med_g, 1),
                   "pairs_per_s": round(n * (n - 1) / 2 / (med * 1e-6), 0),
                   "pipeline": "sparse" if sparse else "dense"}
            if n == 12000:      # what an input outside the sparse contract pays: the dense bit-matrix pipeline alone
                row["us_dense_pipeline"] = round(time_us(lambda: ops.nms_device(dets, thr, dense_only=True), flush=flush)[0], 1)
            out["nms"].append(row)
    for K in (81, 61):
        n = 12000
        rng = np.random.default_rng(K)
        dets = torch.from_numpy(np.concatenate([synth.nms_boxes(n, seed=9, rounded=True), synth.nms_scores(n, seed=8)[:, None]], 1)).to(dev)
        cls = torch.from_numpy(rng.integers(1, K, n).astype(np.int32)).to(dev)
        path = ops.nms_device(dets, 0.3, class_ids=cls, return_path=True)[2]
        sparse = int(path.item()) == 1
        med, mn = time_us(lambda: ops.nms_device(dets, 0.3, class_ids=cls, sparse_only=sparse), flush=flush)
        med_fb, _ = time_us(lambda: ops.nms_device(dets, 0.3, class_ids=cls), flush=flush)
        out["nms"].append({"n": n, "boxes": "per-class K=%d rounded" % K, "thresh": 0.3, "us_median": round(med, 1), "us_min": round(mn, 1),
                           "us_with_fallback": round(med_fb, 1), "pipeline": "sparse" if sparse else "dense"})
    # proposal layer, 261 888 anchors
    A = 261888
    rng = np.random.default_rng(31)
    an = torch.from_numpy(synth.nms_boxes(A, seed=4, kind="rpn")).to(dev)
    fg = rng.permutation(np.linspace(0, 1, A)).astype(np.float32)
    probs = torch.from_numpy(np.stack([1 - fg, fg], 1).astype(np.float32)).to(dev)
    dl = torch.from_numpy((rng.standard_normal((A, 4)) * 0.5).astype(np.float32)).to(dev)
    prop = lambda: ops.proposal_device(probs, dl, an, 1000, 0.7, (0.1, 0.1, 0.2, 0.2), (1024, 1024))
    med, mn = time_us(prop, flush=flush)
    g = graphed(prop)
    med_g, _ = time_us(g.replay, flush=flush)
    del g
    out["proposal_layer"] = {"anchors": A, "pre_nms": 6000, "post_nms": 1000, "us_median": round(med, 1), "us_min": round(mn, 1),
                             "us_graph": round(med_g, 1)}
    # sem-dist encode: config 4 = 16 images x 20 instances x L planes of 1024^2
    Bn, n_inst, L = 16, 20, 1
    labels = np.stack([synth.label_map(1024, 1024, n=n_inst, seed=2024 + (i % 4)) for i in range(4)])
    labels = torch.from_numpy(np.tile(labels, (Bn // 4, 1, 1)).view(np.int64)).to(dev)
    planes, n_obj = ops.layer_decode_device(labels, L, n_inst)
    med, mn = time_us(lambda: ops.layer_decode_device(labels, L, n_inst), reps=5)
    g = graphed(lambda: ops.layer_decode_device(labels, L, n_inst))
    med_g, _ = time_us(g.replay, reps=5)
    del g
    by = Bn * 1024 * 1024 * (8 + n_inst * L)
    out["layer_decode"] = {"images": Bn, "n_max": n_inst, "L": L, "us_median": round(med, 1), "us_graph": round(med_g, 1),
                           "algorithmic_bytes": by, "achieved_gbs": round(by / med / 1e3, 1), "frac": round(by / med / 1e3 / peak, 4),
                           "frac_graph": round(by / med_g / 1e3 / peak, 4)}
    med, mn = time_us(lambda: ops.edt_sq_device(planes), reps=5)
    g = graphed(lambda: ops.edt_sq_device(planes))
    med_g, _ = time_us(g.replay, reps=5)
    del g
    M = Bn * n_inst * L
    by = M * 1024 * 1024 * 5
    out["edt"] = {"maps": M, "us_median": round(med, 1), "us_graph": round(med_g, 1), "maps_per_s": round(M / (med * 1e-6), 1),
                  "mpx_per_s": round(M * 1.048576 / (med * 1e-6), 1), "algorithmic_bytes": by,
                  "achieved_gbs": round(by / med / 1e3, 1), "frac": round(by / med / 1e3 / peak, 4),
                  "frac_graph": round(by / med_g / 1e3 / peak, 4)}
    del flush
    return out


# --------------------------------------------------------------------------------------
# config 1: the detection-head hot path of one image through the drop-in operator API
# --------------------------------------------------------------------------------------
class _HeadCfg:
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    IMAGE_SHAPE = np.array([1024, 1024, 3])
    USE_NMS = True
    DETECTION_MIN_CONFIDENCE = 0          # inference setting (amodal_train.py:571)
    DETECTION_NMS_THRESHOLD = 0.3


def head_pipeline(dev, cpu=True):
    """BASELINE.json configs[0] without the (out-of-scope) convolutions: 261 888 anchors -> proposal_layer (top 6000,
    NMS 0.7, 1000 ROIs) -> pyramid_roi_align 7x7 -> refine_detections (per-class NMS 0.3, K=81) -> pyramid_roi_align
    14x14 on the detections, every call through the reference's own function signatures.  RPN / classifier outputs and
    the FPN maps are synthetic.  Returns images/s on one GPU (images are independent: ranks shard them) and, on the host,
    the same sequence through the oracle (numpy + the reference's C crop / NMS)."""
    import torch
    from sln_amodal_b200 import proposal_layer, pyramid_roi_align, refine_detections
    A, K = 261888, 81
    rng = np.random.default_rng(101)
    anchors_np = synth.nms_boxes(A, seed=4, kind="rpn")
    fg = rng.permutation(np.linspace(0, 1, A)).astype(np.float32)
    probs_np = np.stack([1 - fg, fg], 1).astype(np.float32)
    deltas_np = (rng.standard_normal((A, 4)) * 0.5).astype(np.float32)
    maps_np = [rng.standard_normal((1, CHANNELS, s_, s_), dtype=np.float32) for s_ in LEVEL_SIDES]
    cls_logits = rng.standard_normal((1000, K)).astype(np.float32) * 3.0
    cls_probs_np = (np.exp(cls_logits) / np.exp(cls_logits).sum(1, keepdims=True)).astype(np.float32)
    cls_deltas_np = (rng.standard_normal((1000, K, 4)) * 0.3).astype(np.float32)
    window = (0.0, 0.0, 1024.0, 1024.0)
    cfg = _HeadCfg()
    t = lambda a: torch.from_numpy(a).to(dev)
    anchors, probs, deltas = t(anchors_np), t(probs_np).unsqueeze(0), t(deltas_np).unsqueeze(0)
    maps = [t(m).contiguous(memory_format=torch.channels_last) for m in maps_np]
    cls_probs, cls_deltas = t(cls_probs_np), t(cls_deltas_np)

    def one_image():
        rois = proposal_layer([probs, deltas], 1000, 0.7, anchors, cfg)                     # [1,k,4]
        k = rois.shape[1]
        pooled = pyramid_roi_align([rois] + maps, 7, cfg.IMAGE_SHAPE)                       # classifier input
        det, keep = refine_detections(rois[0], cls_probs[:k], cls_deltas[:k], window, cfg)
        boxes = det[:, :4] / 1024.0
        masks_in = pyramid_roi_align([boxes.unsqueeze(0)] + maps, 14, cfg.IMAGE_SHAPE)      # mask / sem-dist head input
        return rois, pooled, det, masks_in

    out = one_image()
    torch.cuda.synchronize()
    ts = []
    for _ in range(20):
        t0 = time.perf_counter()
        one_image()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    ms = float(np.median(ts)) * 1e3
    res = {"what": "proposal_layer -> pyramid_roi_align 7x7 -> refine_detections (per-class NMS) -> pyramid_roi_align 14x14, "
                   "one 1024^2 image, 261888 anchors, K=81, synthetic RPN / classifier outputs (convolutions out of scope)",
           "rois": int(out[0].shape[1]), "detections": int(out[2].shape[0]), "ms_per_image": round(ms, 3),
           "images_per_s_per_gpu": round(1e3 / ms, 1), "timing": "host wall clock incl. the API's own host reads, median of 20"}
    if cpu:
        from oracle import oracle
        t0 = time.perf_counter()
        rois_c = oracle.proposal_layer(probs_np, deltas_np, anchors_np, 1000, 0.7)
        pooled_c = oracle.pyramid_roi_align(rois_c, maps_np, 7)
        kc = rois_c.shape[0]
        det_c, _ = oracle.refine_detections(rois_c, cls_probs_np[:kc], cls_deltas_np[:kc], window, min_confidence=0, nms_threshold=0.3)
        masks_c = oracle.pyramid_roi_align(det_c[:, :4] / np.float32(1024.0), maps_np, 14)
        cpu_s = time.perf_counter() - t0
        rois_g, det_g = out[0][0].cpu().numpy(), out[2].cpu().numpy()
        checks = {"rois_max_abs_diff": float(np.abs(rois_c - rois_g).max()) if rois_c.shape == rois_g.shape else None,
                  # (proposal boxes agree to 1 ulp -- exp through double vs torch's CPU exp -- so the crops are compared
                  # by value, not bit for bit)
                  "crops7_max_abs_diff": float(np.abs(pooled_c - out[1].contiguous().cpu().numpy()).max())
                  if pooled_c.shape == tuple(out[1].shape) else None,
                  "detections_identical": bool(det_c.shape == det_g.shape and np.array_equal(det_c, det_g)),
                  "detections": [int(det_c.shape[0]), int(det_g.shape[0])]}
        res["cpu_oracle"] = {"ms_per_image": round(cpu_s * 1e3, 1), "images_per_s": round(1.0 / cpu_s, 3), "cores": os.cpu_count(),
                             "kind": "port (numpy) + the reference's C crop / NMS", "parity": checks}
    return res


def detection_targets_metric(dev, cpu=True):
    """SURVEY 8(f)-1: detection_target_layer for one training image (1000 proposals, 12 GT instances, L = 1, 1024^2
    GT masks, 100 sampled ROIs -> 32x32 mask targets) through the reference's signature, next to the oracle on the host."""
    import torch
    from sln_amodal_b200 import detection_target_layer
    rng = np.random.default_rng(303)
    G_, N_ = 12, 1000
    gt = np.zeros((G_, 4), np.float32)
    masks = np.zeros((1, G_, 1024, 1024), np.uint8)
    for i in range(G_):
        h, w = rng.uniform(0.1, 0.4, 2)
        y1, x1 = rng.uniform(0, 1 - h), rng.uniform(0, 1 - w)
        gt[i] = (y1, x1, y1 + h, x1 + w)
        masks[0, i, int(y1 * 1024):int((y1 + h) * 1024), int(x1 * 1024):int((x1 + w) * 1024)] = 1
    jit = gt[rng.integers(0, G_, 240)] + rng.normal(0, 0.02, (240, 4)).astype(np.float32)       # 20 per GT, like config 5
    props = np.clip(np.concatenate([jit, synth.roi_boxes(N_ - 240, seed=9)], 0), 0, 1).astype(np.float32)
    ids = np.ones(G_, np.int32)

    class Cfg:
        BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
        TRAIN_ROIS_PER_IMAGE = 100
        ROI_POSITIVE_RATIO = 0.7
        MASK_SHAPE = [32, 32]
        USE_MINI_MASK = False

    t = lambda a: torch.from_numpy(a).to(dev)
    args = (t(props).unsqueeze(0), t(ids).unsqueeze(0), t(gt).unsqueeze(0), t(masks).unsqueeze(0))
    torch.manual_seed(5)
    out = detection_target_layer(*args, Cfg())
    torch.cuda.synchronize()
    ts = []
    for _ in range(20):
        t0 = time.perf_counter()
        detection_target_layer(*args, Cfg())
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    ms = float(np.median(ts)) * 1e3
    res = {"what": "detection_target_layer, 1000 proposals, 12 GT, L=1, 1024^2 masks -> 100 ROIs with 32x32 mask targets",
           "ms_per_image": round(ms, 3), "images_per_s_per_gpu": round(1e3 / ms, 1), "sampled_rois": int(out[0].shape[0])}
    if cpu:
        from oracle import oracle
        torch.manual_seed(5)
        t0 = time.perf_counter()
        ro, co, do, mo = oracle.detection_target_layer(props, ids, gt, masks)
        cpu_s = time.perf_counter() - t0
        res["cpu_oracle"] = {"ms_per_image": round(cpu_s * 1e3, 1), "cores": os.cpu_count(),
                             "parity": {"rois_identical": bool(np.array_equal(ro, out[0].cpu().numpy())),
                                        "class_ids_identical": bool(np.array_equal(co, out[1].cpu().numpy())),
                                        "masks_identical": bool(np.array_equal(mo, out[3].cpu().numpy())),
                                        "deltas_max_abs_diff": float(np.abs(do - out[2].cpu().numpy()).max()) if do.size else 0.0}}
    return res


def rpn_targets_metric(dev, cpu=True):
    """SURVEY 8(f)-2: build_rpn_targets for one training image, 261 888 anchors x 12 GT boxes, numpy in / numpy out like
    the reference (the float64 IoU reductions on the device, matching rules and sampling in numpy)."""
    import torch
    from sln_amodal_b200 import build_rpn_targets
    anchors = synth.pyramid_anchors()
    rng = np.random.default_rng(404)
    c = rng.uniform(100, 924, (12, 2))
    s_ = rng.uniform(40, 400, (12, 2))
    gt = np.clip(np.concatenate([c - s_ / 2, c + s_ / 2], 1), 0, 1024).astype(np.int32)
    ids = np.ones(12, np.int32)

    class Cfg:
        RPN_TRAIN_ANCHORS_PER_IMAGE = 256
        RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])

    np.random.seed(1)
    out = build_rpn_targets((1024, 1024, 3), anchors, ids, gt, Cfg(), device=dev)
    ts = []
    for _ in range(10):
        t0 = time.perf_counter()
        build_rpn_targets((1024, 1024, 3), anchors, ids, gt, Cfg(), device=dev)
        ts.append(time.perf_counter() - t0)
    ms = float(np.median(ts)) * 1e3
    res = {"what": "build_rpn_targets, %d anchors x 12 GT boxes, float64" % anchors.shape[0], "ms_per_image": round(ms, 3),
           "positives": int((out[0] == 1).sum()), "negatives": int((out[0] == -1).sum())}
    if cpu:
        from oracle import oracle
        np.random.seed(1)
        t0 = time.perf_counter()
        m, b = oracle.build_rpn_targets(anchors, ids, gt)
        cpu_s = time.perf_counter() - t0
        res["cpu_oracle"] = {"ms_per_image": round(cpu_s * 1e3, 1), "cores": os.cpu_count(),
                             "identical": bool(np.array_equal(m, out[0]) and np.array_equal(b, out[1]))}
    return res


def rle_metric(dev, peak, cpu=True):
    """SURVEY 8(f)-3: COCO RLE of 100 full-resolution (1024^2) detection masks (blobs), device run-length kernel + host
    string coder, next to the reference's own maskApi.c (oracle/_ref) on the host."""
    import torch
    from sln_amodal_b200 import rle
    n, h, w = 100, 1024, 1024
    rng = np.random.default_rng(505)
    yy, xx = np.mgrid[0:h, 0:w]
    masks = np.zeros((n, h, w), np.uint8)
    for i in range(n):
        cy, cx = rng.uniform(0.2, 0.8, 2) * h
        ry, rx = rng.uniform(0.05, 0.2, 2) * h
        masks[i] = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
    d = torch.from_numpy(masks).to(dev)
    cols = d.transpose(1, 2).contiguous().view(n, h * w)
    out = rle.encode(d)
    torch.cuda.synchronize()
    ev = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rle.rle_counts_device(cols)
        b.record()
        torch.cuda.synchronize()
        ev.append(a.elapsed_time(b) * 1e3)
    t0 = time.perf_counter()
    rle.encode(d)
    wall = time.perf_counter() - t0
    us = float(np.median(ev))
    res = {"what": "COCO RLE of 100 masks of 1024^2", "kernel_us": round(us, 1), "algorithmic_bytes": n * h * w,
           "achieved_gbs": round(n * h * w / us / 1e3, 1), "frac": round(n * h * w / us / 1e3 / peak, 4),
           "encode_ms_incl_transpose_d2h_and_strings": round(wall * 1e3, 2)}
    if cpu:
        from oracle import oracle
        colh = np.ascontiguousarray(masks.transpose(0, 2, 1)).reshape(n, h * w)
        t0 = time.perf_counter()
        ref = oracle.ref_rle_encode(colh, h, w) if oracle.ref_mask_available() else [(oracle.rle_encode(c), None) for c in colh]
        cpu_s = time.perf_counter() - t0
        res["cpu_baseline"] = {"ms": round(cpu_s * 1e3, 1), "kind": "reference" if oracle.ref_mask_available() else "port", "cores": 1,
                               "identical": bool(all(o["counts"] == (r[1] if r[1] is not None else oracle.rle_to_string(r[0]))
                                                     for o, r in zip(out, ref)))}
    return res


def _event_us(fn, reps=10, flush=None):
    import torch
    fn()
    torch.cuda.synchronize()
    ev = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ev.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ev))


def unmold_metric(dev, peak, cpu=True):
    """SURVEY 8(f)-3: utils.unmold_mask for the 100 detections of one 1024^2 image (28x28 masks -> resize to the box,
    threshold, paste) as one launch, then the device RLE; next to the oracle (scipy bytescale restated + Pillow-exact
    resample) on the host for a bounded sample of the same detections.  Algorithmic bytes: the N*H*W planes written."""
    import torch
    from sln_amodal_b200 import rle, unmold
    rng = np.random.default_rng(3)
    N, H, W = 100, 1024, 1024
    masks_np = rng.random((N, 28, 28)).astype(np.float32)
    hw = np.exp(rng.uniform(np.log(24), np.log(600), (N, 2)))
    y1x1 = rng.uniform(0, 1, (N, 2)) * (1024 - hw)
    boxes_np = np.concatenate([y1x1, y1x1 + hw], 1).astype(np.int32)
    masks, boxes = torch.from_numpy(masks_np).to(dev), torch.from_numpy(boxes_np).to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    us = _event_us(lambda: unmold.unmold_masks(masks, boxes, (H, W)), flush=flush)
    planes = unmold.unmold_masks(masks, boxes, (H, W))
    t0 = time.perf_counter()
    enc = rle.encode(unmold.unmold_masks(masks, boxes, (H, W)))
    wall = time.perf_counter() - t0
    res = {"what": "unmold_mask of 100 detections (28x28 -> box, threshold, paste) into 1024^2 planes, one launch",
           "kernel_us": round(us, 1), "algorithmic_bytes": N * H * W, "achieved_gbs": round(N * H * W / us / 1e3, 1),
           "frac": round(N * H * W / us / 1e3 / peak, 4), "l2": "flushed between iterations",
           "unmold_plus_rle_encode_ms": round(wall * 1e3, 2)}
    if cpu:
        from oracle import oracle
        k = 20
        t0 = time.perf_counter()
        want = [oracle.unmold_mask(masks_np[i], boxes_np[i], (H, W)) for i in range(k)]
        cpu_s = time.perf_counter() - t0
        got = planes[:k].cpu().numpy()
        res["cpu_baseline"] = {"ms_per_100_detections": round(cpu_s * 1e3 * N / k, 1), "kind": "port", "cores": 1,
                               "sample": "first %d of the 100 detections" % k,
                               "identical": bool(all(np.array_equal(got[i], want[i]) for i in range(k)))}
        del enc
    return res


def rpn_pack_metric(dev, peak, cpu=True):
    """SURVEY 8(f)-4: RPN output re-layout for one 1024^2 image (five levels, 261 888 anchors): one launch against the
    reference's expression (10 permute copies + 5 softmax + 3 cat) in torch on the same device and on the host."""
    import torch
    from sln_amodal_b200 import rpn
    torch.manual_seed(5)
    sizes = (256, 128, 64, 32, 16)
    cls_maps = [torch.randn(1, 6, s, s, device=dev) * 4 for s in sizes]
    box_maps = [torch.randn(1, 12, s, s, device=dev) for s in sizes]

    def ref_expr(cm, bm):
        lg = [c.permute(0, 2, 3, 1).contiguous().view(c.size(0), -1, 2) for c in cm]
        pr = [torch.softmax(x, dim=2) for x in lg]
        bx = [b.permute(0, 2, 3, 1).contiguous().view(b.size(0), -1, 4) for b in bm]
        return torch.cat(lg, 1), torch.cat(pr, 1), torch.cat(bx, 1)

    us = _event_us(lambda: rpn.rpn_pack(cls_maps, box_maps), reps=20)
    us_t = _event_us(lambda: ref_expr(cls_maps, box_maps), reps=20)
    ours, ref = rpn.rpn_pack(cls_maps, box_maps), ref_expr(cls_maps, box_maps)
    A = ours[0].shape[1]
    nbytes = A * (2 + 4) * 4 * 2 + A * 2 * 4                                  # read 6 floats, write 8 per anchor
    res = {"what": "RPN re-layout + softmax + concat, 5 levels, %d anchors, one launch" % A, "us": round(us, 1),
           "torch_expression_same_device_us": round(us_t, 1), "algorithmic_bytes": nbytes,
           "achieved_gbs": round(nbytes / us / 1e3, 1), "bound": "launch latency (6.3 MB per image)",
           "copies_identical": bool(torch.equal(ours[0], ref[0]) and torch.equal(ours[2], ref[2])),
           "softmax_bit_identical_to_torch_cuda": bool(torch.equal(ours[1], ref[1])),
           "softmax_max_rel_err_vs_torch_cuda": float(((ours[1] - ref[1]).abs() / ref[1].abs().clamp_min(1e-30)).max().item())}
    if cpu:
        cm, bm = [c.cpu() for c in cls_maps], [b.cpu() for b in box_maps]
        ref_expr(cm, bm)
        t0 = time.perf_counter()
        for _ in range(5):
            ref_expr(cm, bm)
        res["cpu_baseline"] = {"ms": round((time.perf_counter() - t0) / 5 * 1e3, 2), "kind": "port",
                               "cores": torch.get_num_threads(), "sample": "the same image, torch-CPU expression of modals.py:394-410 + model.py:553-563"}
    return res


def resize_image_metric(dev, cpu=True):
    """SURVEY 8(f)-2: utils.resize_image of one D2SA-sized RGB image (1440 x 1920 -> 1024^2, Pillow-exact bilinear) in
    three launches, image already on the device; next to Pillow itself on one host core (what the reference calls)."""
    import torch
    from sln_amodal_b200 import targets
    rng = np.random.default_rng(12)
    img_np = rng.integers(0, 256, (1440, 1920, 3)).astype(np.uint8)
    img = torch.from_numpy(img_np).to(dev)
    us = _event_us(lambda: targets.resize_image_device(img, (1024, 1024)), reps=20)
    nbytes = img_np.size + 1024 * 1024 * 3
    res = {"what": "resize_image 1440x1920x3 u8 -> 1024x1024x3 (Pillow-exact bilinear), 3 launches", "us": round(us, 1),
           "algorithmic_bytes": nbytes, "achieved_gbs": round(nbytes / us / 1e3, 1), "bound": "launch latency (11.4 MB per image)"}
    if cpu:
        from oracle import oracle
        got = targets.resize_image_device(img, (1024, 1024)).cpu().numpy()
        try:
            oracle.resize_image_pil(img_np, (1024, 1024))
            t0 = time.perf_counter()
            want = oracle.resize_image_pil(img_np, (1024, 1024))
            kind, cpu_s = "reference library (Pillow)", time.perf_counter() - t0
        except ImportError:
            t0 = time.perf_counter()
            want = oracle.resize_image(img_np, (1024, 1024))
            kind, cpu_s = "port", time.perf_counter() - t0
        res["cpu_baseline"] = {"ms": round(cpu_s * 1e3, 2), "kind": kind, "cores": 1, "sample": "the same image",
                               "identical": bool(np.array_equal(got, want))}
    return res


# --------------------------------------------------------------------------------------
# CPU reference (oracle/_ref when present: the reference's own C, unmodified)
# --------------------------------------------------------------------------------------
def _cpu_sample(boxes_np, ind_np, level_np):
    sel = np.nonzero(ind_np == 0)[0][:CPU_SAMPLE_ROIS]
    return boxes_np[sel], level_np[sel]


def _cpu_pass(oracle, use_ref, maps_np, boxes, level, grads):
    fwd = oracle.ref_crop_and_resize_fwd if use_ref else oracle.crop_and_resize_fwd
    bwd = oracle.ref_crop_and_resize_bwd if use_ref else oracle.crop_and_resize_bwd
    for p in POOLS:
        for l in range(4):
            ix = np.nonzero(level == l)[0]
            if ix.size == 0:
                continue
            z = np.zeros(ix.size, np.int32)
            fwd(maps_np[l], boxes[ix], z, p, p, 0.0)
            bwd(grads[p][ix], boxes[ix], z, maps_np[l].shape)


def cpu_reference_sample(boxes_np, ind_np, level_np, maps=None, steps=1, warmup=1):
    from oracle import oracle
    use_ref = oracle.ref_available()
    cores = os.cpu_count() or 1
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the reference arm is meant to use every host core it can
    os.environ["OMP_NUM_THREADS"] = str(cores)
    try:                                                     # an OpenMP runtime that is already loaded ignores the variable
        import ctypes
        ctypes.CDLL("libgomp.so.1").omp_set_num_threads(cores)
    except Exception:
        pass
    boxes, level = _cpu_sample(boxes_np, ind_np, level_np)
    rng = np.random.default_rng(99)
    if maps is not None:
        maps_np = [m[:1].contiguous().cpu().numpy() for m in maps]
    else:
        maps_np = [rng.standard_normal((1, CHANNELS, s, s), dtype=np.float32) for s in LEVEL_SIDES]
    grads = {p: rng.standard_normal((boxes.shape[0], CHANNELS, p, p), dtype=np.float32) for p in POOLS}
    for _ in range(warmup):
        _cpu_pass(oracle, use_ref, maps_np, boxes[:64], level[:64], {p: grads[p][:64] for p in POOLS})
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        _cpu_pass(oracle, use_ref, maps_np, boxes, level, grads)
        ts.append(time.perf_counter() - t0)
    t = float(np.mean(ts))
    crops = boxes.shape[0] * len(POOLS)
    return {"value": round(crops / t, 1), "unit": "roi_crops/s", "cores": cores,
            "kind": "reference" if use_ref else "port", "seconds_per_sample": round(t, 3),
            "sample": "first %d ROIs of image 0 over P2-P5, pools 7x7+14x14, fwd+bwd through the reference's "
                      "crop_and_resize.c (fwd OpenMP over boxes, bwd single-threaded by construction)" % boxes.shape[0],
            "all_step_times_s": [round(x, 3) for x in ts]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    boxes_np, ind_np, level_np = make_workload()
    warm = max(args.warmup, 1)
    res = cpu_reference_sample(boxes_np, ind_np, level_np, None, steps=args.steps, warmup=min(warm, 2))
    t = res["seconds_per_sample"]
    line = {"impl": "reference", "metric": "roialign_fwd_bwd_roi_crops_per_s", "value": res["value"], "unit": "roi_crops/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": res["sample"],
                       "note": "one CPU process on rank 0 with all host cores, whatever --gpus says: the CPU arm does not scale "
                               "with N, so only the N=1 ratio against it is meaningful"},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": res["value"], "unit": "roi_crops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of what the last timed step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
