"""ncu driver: the config-2 backward (8 images, C=256, P2-P5, 8 x per ROIs), pools 7 and 14, two calls each.
   python tools/prof_bwd.py [rois_per_img]"""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from sln_amodal_b200 import ops, synth
per = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
dev = torch.device("cuda", 0)
n = 8 * per
boxes_np = synth.roi_boxes(n, seed=4321)
level_np = (synth.fpn_level(boxes_np) - 2).astype(np.int32)
ind_np = np.repeat(np.arange(8, dtype=np.int32), per)
boxes, ind, level = (torch.from_numpy(a).to(dev) for a in (boxes_np, ind_np, level_np))
sizes = [(8, 256, s, s) for s in bench.LEVEL_SIDES]
for p in (7, 14):
    g = torch.randn((n, 256, p, p), device=dev).contiguous(memory_format=torch.channels_last)
    for _ in range(2):
        ops.pyramid_crop_backward(g, boxes, ind, level, sizes)
    torch.cuda.synchronize()
