"""A/B of the bulk-async backward's stage configurations (crop_bwd_tma.cuh) in one process (SLN_BWD_CFG is read per
   call): "auto" = by crop size, c0 = 32 x 3, c1 = 16 x 6.  Checks every arm against auto on the config-2 workload (exact
   mode: bit-equal; default mode: max rel error against auto's exact result) and times each with CUDA events
   (working set >> L2).   python tools/ab_bwd_impl.py [rois_per_img ...]"""
import json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from sln_amodal_b200 import ops, synth

dev = torch.device("cuda", 0)
peak, src = bench.measured_peak_gbs()
pers = [int(a) for a in sys.argv[1:]] or [1000]
maps_shape = [(8, 256, s, s) for s in bench.LEVEL_SIDES]


def timed(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


rows = []
for per in pers:
    n = 8 * per
    boxes_np = synth.roi_boxes(n, seed=4321)
    level_np = (synth.fpn_level(boxes_np) - 2).astype(np.int32)
    ind_np = np.repeat(np.arange(8, dtype=np.int32), per)
    boxes, ind, level = (torch.from_numpy(a).to(dev) for a in (boxes_np, ind_np, level_np))
    for p in (7, 14, 16):
        g = torch.randn((n, 256, p, p), device=dev).contiguous(memory_format=torch.channels_last)
        bb = sum(bench.bwd_bytes(int((level_np == l).sum()), side, p) for l, side in enumerate(bench.LEVEL_SIDES))
        row = {"rois_per_img": per, "pool": p}
        outs = {}
        for impl in ("auto", "c0", "c1"):
            os.environ.pop("SLN_BWD_CFG", None)
            if impl != "auto":
                os.environ["SLN_BWD_CFG"] = impl[1]
            for exact in (False, True):
                outs[(impl, exact)] = ops.pyramid_crop_backward(g, boxes, ind, level, maps_shape, exact=exact)
            ms = timed(lambda: ops.pyramid_crop_backward(g, boxes, ind, level, maps_shape))
            row["ms_impl%s" % impl] = round(ms, 4)
            row["frac_impl%s" % impl] = round(bb / ms / 1e6 / peak, 3)
        row["exact_bit_equal"] = all(all(torch.equal(a, b) for a, b in zip(outs[("auto", True)], outs[(k, True)]))
                                     for k in ("c0", "c1"))
        err = 0.0
        for k in ("auto", "c0", "c1"):
            for b, e in zip(outs[(k, False)], outs[("auto", True)]):
                err = max(err, float((b - e).abs().max() / e.abs().max()))
        row["default_max_rel_err"] = err
        rows.append(row)
        print(row, flush=True)
        del g, outs
print(json.dumps({"peak_gbs": peak, "peak_source": src, "rows": rows}))
