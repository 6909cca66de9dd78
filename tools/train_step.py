"""BASELINE config 5 harness: a full SLN-style Mask R-CNN training step on synthetic D2SA-shaped data, data-parallel over
the GPUs of one box.  Test / measurement infrastructure -- NOT part of the product (sln_amodal_b200/ holds the hot path only).

What the reference does per optimizer step (model.py:370-461, train_epoch): 16 x { one image through MaskRCNN.predict(
mode='training'), losses (model.py:423-436), backward }, gradient clipping, SGD step.  Here:

  * backbone / heads: a ResNet-101-FPN Mask R-CNN in STOCK PyTorch (cuDNN convolutions, random init; the architecture of
    the reference's model.py:44-160 + modals.py RPN / Classifier / Mask, written from the published Mask R-CNN layout --
    out of the graft's scope, it only has to produce realistic tensors and gradient traffic), wrapped by
    sln_amodal_b200.dist.wrap_ddp (bucketed NCCL all-reduce overlapped with backward);
  * the hot path goes through this repo's drop-ins: rpn_pack (RPN re-layout + softmax, one launch each way),
    proposal_layer, detection_target_layer (IoU matching, box refinement, mask targets), pyramid_roi_align 7x7 and 16x16
    with the bulk-async backward kernel;
  * GT-jittered proposals are injected (20 per GT box, SURVEY 7) so that random weights still give ~70 positives;
  * "batch 16" = 16 images per optimizer step: strong scaling splits them over the ranks (16 / N images per rank, gradient
    accumulation under DDP.no_sync() until the rank's last image), weak scaling gives every rank 16.

    python tools/train_step.py                 (one GPU)
    python tools/train_step.py --images-per-forward 16   (16 images per forward: batched proposals, targets, crops)
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/train_step.py --gpus N
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

IMAGE = 1024


# ----------------------------------------------------------------------------- stock-PyTorch model (out of scope)
class Bottleneck(nn.Module):
    def __init__(self, cin, planes, stride=1):
        super().__init__()
        self.c1 = nn.Conv2d(cin, planes, 1, stride=stride, bias=False)
        self.b1 = nn.BatchNorm2d(planes)
        self.c2 = nn.Conv2d(planes, planes, 3, padding=1, bias=False)
        self.b2 = nn.BatchNorm2d(planes)
        self.c3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.b3 = nn.BatchNorm2d(planes * 4)
        self.down = None
        if stride != 1 or cin != planes * 4:
            self.down = nn.Sequential(nn.Conv2d(cin, planes * 4, 1, stride=stride, bias=False), nn.BatchNorm2d(planes * 4))

    def forward(self, x):
        y = F.relu(self.b1(self.c1(x)))
        y = F.relu(self.b2(self.c2(y)))
        y = self.b3(self.c3(y))
        return F.relu(y + (x if self.down is None else self.down(x)))


class ResNetFPN(nn.Module):
    def __init__(self, blocks=(3, 4, 23, 3)):
        super().__init__()
        self.stem = nn.Sequential(nn.Conv2d(3, 64, 7, stride=2, padding=3, bias=False), nn.BatchNorm2d(64), nn.ReLU(),
                                  nn.MaxPool2d(3, stride=2, padding=1))
        cin, stages = 64, []
        for i, n in enumerate(blocks):
            planes = 64 << i
            layers = [Bottleneck(cin, planes, stride=1 if i == 0 else 2)]
            cin = planes * 4
            layers += [Bottleneck(cin, planes) for _ in range(n - 1)]
            stages.append(nn.Sequential(*layers))
        self.stages = nn.ModuleList(stages)
        self.lat = nn.ModuleList([nn.Conv2d(256 << i, 256, 1) for i in range(4)])
        self.smooth = nn.ModuleList([nn.Conv2d(256, 256, 3, padding=1) for _ in range(4)])

    def forward(self, x):
        x = self.stem(x)
        cs = []
        for st in self.stages:
            x = st(x)
            cs.append(x)
        p = self.lat[3](cs[3])
        outs = [p]
        for i in (2, 1, 0):
            p = self.lat[i](cs[i]) + F.interpolate(p, scale_factor=2.0, mode="nearest")
            outs.append(p)
        outs = outs[::-1]                                               # P2..P5
        outs = [s(o) for s, o in zip(self.smooth, outs)]
        return outs + [F.max_pool2d(outs[3], 1, stride=2)]              # + P6


class RPNHead(nn.Module):
    def __init__(self, a=3):
        super().__init__()
        self.shared = nn.Conv2d(256, 512, 3, padding=1)
        self.cls = nn.Conv2d(512, 2 * a, 1)
        self.box = nn.Conv2d(512, 4 * a, 1)

    def forward(self, x):
        h = F.relu(self.shared(x))
        return self.cls(h), self.box(h)


class ClassifierHead(nn.Module):
    def __init__(self, pool=7, classes=2):
        super().__init__()
        self.c1 = nn.Conv2d(256, 1024, pool)
        self.b1 = nn.BatchNorm2d(1024)
        self.c2 = nn.Conv2d(1024, 1024, 1)
        self.b2 = nn.BatchNorm2d(1024)
        self.cls = nn.Linear(1024, classes)
        self.box = nn.Linear(1024, classes * 4)

    def forward(self, pooled):
        x = F.relu(self.b1(self.c1(pooled)))
        x = F.relu(self.b2(self.c2(x))).flatten(1)
        return self.cls(x), self.box(x).view(x.shape[0], -1, 4)


class MaskHead(nn.Module):
    def __init__(self, classes=2):
        super().__init__()
        self.convs = nn.ModuleList([nn.Conv2d(256, 256, 3, padding=1) for _ in range(4)])
        self.bns = nn.ModuleList([nn.BatchNorm2d(256) for _ in range(4)])
        self.deconv = nn.ConvTranspose2d(256, 256, 2, stride=2)
        self.out = nn.Conv2d(256, classes, 1)

    def forward(self, pooled):
        x = pooled
        for c, b in zip(self.convs, self.bns):
            x = F.relu(b(c(x)))
        return self.out(F.relu(self.deconv(x)))                         # logits [n, classes, 2*pool, 2*pool]


class Cfg:
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])
    IMAGE_SHAPE = np.array([IMAGE, IMAGE, 3])
    TRAIN_ROIS_PER_IMAGE = 100
    ROI_POSITIVE_RATIO = 0.7
    MASK_SHAPE = [32, 32]
    MASK_POOL_SIZE = 16
    POOL_SIZE = 7
    USE_MINI_MASK = False
    GPU_COUNT = 1
    POST_NMS_ROIS_TRAINING = 1000
    RPN_NMS_THRESHOLD = 0.7


class SLNTrainNet(nn.Module):
    """forward(image, targets) -> total loss of one image (the reference is batch 1, Functions.py:128)."""

    def __init__(self, anchors):
        super().__init__()
        self.fpn = ResNetFPN()
        self.rpn = RPNHead()
        self.classifier = ClassifierHead()
        self.mask = MaskHead()
        self.register_buffer("anchors", anchors, persistent=False)
        self.cfg = Cfg()

    def forward(self, image, rpn_match=None, rpn_bbox_t=None, gt_ids=None, gt_boxes=None, gt_masks=None, injected=None):
        if isinstance(image, dict):                                   # B images at once (batch_inputs)
            return self.forward_batch(**image)
        from sln_amodal_b200 import detection_target_layer, proposal_layer, pyramid_roi_align, rpn as srpn
        cfg = self.cfg
        feats = self.fpn(image)
        cls_maps, box_maps = zip(*[self.rpn(p) for p in feats])
        logits, probs, deltas = srpn.rpn_pack(list(cls_maps), list(box_maps))        # [1,A,2], [1,A,2], [1,A,4]
        with torch.no_grad():
            rois = proposal_layer([probs, deltas], cfg.POST_NMS_ROIS_TRAINING, cfg.RPN_NMS_THRESHOLD, self.anchors, cfg)
            rois = torch.cat([injected.unsqueeze(0), rois], 1)[:, : cfg.POST_NMS_ROIS_TRAINING]
            t_rois, t_ids, t_deltas, t_masks = detection_target_layer(rois, gt_ids, gt_boxes, gt_masks, cfg)
        # RPN losses (model.py:423-426)
        m = rpn_match.view(-1)
        sel = torch.nonzero(m != 0).view(-1)
        loss = F.cross_entropy(logits[0, sel], (m[sel] == 1).long())
        pos = torch.nonzero(m == 1).view(-1)
        if pos.numel():
            loss = loss + F.smooth_l1_loss(deltas[0, pos], rpn_bbox_t[: pos.numel()])
        n_pos = 0
        if t_rois.numel():
            maps = feats[:4]
            pooled = pyramid_roi_align([t_rois.unsqueeze(0)] + maps, cfg.POOL_SIZE, cfg.IMAGE_SHAPE)
            cls_logits, bbox = self.classifier(pooled)
            loss = loss + F.cross_entropy(cls_logits, t_ids.long())
            posr = torch.nonzero(t_ids > 0).view(-1)
            n_pos = int(posr.numel())
            if n_pos:
                cid = t_ids[posr].long()
                loss = loss + F.smooth_l1_loss(bbox[posr, cid], t_deltas[posr])
                pooled_m = pyramid_roi_align([t_rois[posr].unsqueeze(0)] + maps, cfg.MASK_POOL_SIZE, cfg.IMAGE_SHAPE)
                mlog = self.mask(pooled_m)
                tm = t_masks[posr]
                tm = tm[:, 0] if tm.dim() == 4 else tm
                loss = loss + F.binary_cross_entropy_with_logits(mlog[torch.arange(n_pos, device=mlog.device), cid], tm)
        return loss, n_pos

    def forward_batch(self, images, rpn_match, rpn_bbox_t, gt_ids, gt_boxes, gt_masks, num_gt, injected):
        """B images per forward: images [B,3,H,W] through the FPN as one batch (BatchNorms in eval mode, so every image
        sees what it sees alone), rpn_pack, proposal_layer_batched, the injected proposals in front of each image's
        proposals, detection_target_layer_batched, pyramid_roi_align_batched on the sampled rows.  gt_ids [B,G] /
        gt_boxes [B,G,4] are padded beyond num_gt (B host ints), gt_masks a list of B [L,G_b,H,W]; rpn_match, rpn_bbox_t
        and injected are lists of B.  Returns the sum over the images of forward()'s per-image loss, and the positives."""
        from sln_amodal_b200 import detection_target_layer_batched, proposal_layer_batched, pyramid_roi_align_batched
        from sln_amodal_b200 import rpn as srpn
        cfg = self.cfg
        B, dev = images.shape[0], images.device
        feats = self.fpn(images)
        cls_maps, box_maps = zip(*[self.rpn(p) for p in feats])
        logits, probs, deltas = srpn.rpn_pack(list(cls_maps), list(box_maps))        # [B,A,2], [B,A,2], [B,A,4]
        K = cfg.POST_NMS_ROIS_TRAINING
        with torch.no_grad():
            rois, num = proposal_layer_batched([probs, deltas], K, cfg.RPN_NMS_THRESHOLD, self.anchors, cfg)
            n_inj = [int(j.shape[0]) for j in injected]
            rois = torch.stack([torch.cat([injected[b], rois[b, : max(K - n_inj[b], 0)]])[:K] for b in range(B)])
            num = torch.clamp(num + torch.tensor(n_inj, dtype=torch.int32, device=dev), max=K).to(torch.int32)
            t_rois, t_ids, t_deltas, t_masks, _, t_num = detection_target_layer_batched(rois, gt_ids, gt_boxes, gt_masks, cfg,
                                                                                     num_proposals=num, num_gt=num_gt)
        loss = logits.new_zeros(())
        for b in range(B):                                            # RPN losses (model.py:423-426), per image
            m = rpn_match[b].view(-1)
            sel = torch.nonzero(m != 0).view(-1)
            loss = loss + F.cross_entropy(logits[b, sel], (m[sel] == 1).long())
            pos = torch.nonzero(m == 1).view(-1)
            if pos.numel():
                loss = loss + F.smooth_l1_loss(deltas[b, pos], rpn_bbox_t[b][: pos.numel()])
        T = t_rois.shape[1]
        k = t_num.cpu().tolist()
        rows = torch.from_numpy(np.concatenate([b * T + np.arange(k[b]) for b in range(B)]).astype(np.int64)).to(dev)
        if rows.numel() == 0:
            return loss, 0
        img = torch.div(rows, T, rounding_mode="floor")

        def per_image_mean(v, idx, n):                                # sum over the images of each image's mean
            return (torch.zeros(B, device=dev).index_add_(0, idx, v) / n).sum()

        ids = t_ids.view(-1)[rows].long()
        boxes = t_rois.view(-1, 4)[rows]
        maps = feats[:4]
        pooled = pyramid_roi_align_batched(boxes, img.to(torch.int32), maps, cfg.POOL_SIZE, cfg.IMAGE_SHAPE)
        cls_logits, bbox = self.classifier(pooled)
        loss = loss + per_image_mean(F.cross_entropy(cls_logits, ids, reduction="none"), img,
                                     torch.tensor(k, dtype=torch.float32, device=dev).clamp(min=1))
        posr = torch.nonzero(ids > 0).view(-1)
        n_pos = int(posr.numel())
        if n_pos:
            cid, pimg = ids[posr], img[posr]
            pcnt = torch.zeros(B, device=dev).index_add_(0, pimg, torch.ones(n_pos, device=dev)).clamp(min=1)
            dl = F.smooth_l1_loss(bbox[posr, cid], t_deltas.view(-1, 4)[rows][posr], reduction="none")
            loss = loss + per_image_mean(dl.sum(1), pimg, 4 * pcnt)
            pooled_m = pyramid_roi_align_batched(boxes[posr], pimg.to(torch.int32), maps, cfg.MASK_POOL_SIZE, cfg.IMAGE_SHAPE)
            mlog = self.mask(pooled_m)
            tm = t_masks.view(B * T, *t_masks.shape[2:])[rows][posr][:, 0]
            bce = F.binary_cross_entropy_with_logits(mlog[torch.arange(n_pos, device=dev), cid], tm, reduction="none")
            loss = loss + per_image_mean(bce.flatten(1).sum(1), pimg, pcnt * tm[0].numel())
        return loss, n_pos


# ----------------------------------------------------------------------------- synthetic D2SA-shaped data
def make_image(seed, dev, anchors_np):
    """One training example: image, 8-15 rectangular / elliptic instances (L = 1, one foreground class,
    amodal_train.py:122,606), their boxes and masks, RPN targets and 20 jittered proposals per GT box."""
    from sln_amodal_b200 import build_rpn_targets
    rng = np.random.default_rng(seed)
    n = int(rng.integers(8, 16))
    masks = np.zeros((1, n, IMAGE, IMAGE), np.uint8)
    boxes = np.zeros((n, 4), np.float32)
    yy, xx = np.mgrid[0:IMAGE, 0:IMAGE]
    for i in range(n):
        h, w = rng.uniform(0.08, 0.35, 2) * IMAGE
        y1, x1 = rng.uniform(0, IMAGE - h), rng.uniform(0, IMAGE - w)
        boxes[i] = (y1, x1, y1 + h, x1 + w)
        if rng.random() < 0.5:
            masks[0, i, int(y1):int(y1 + h), int(x1):int(x1 + w)] = 1
        else:
            masks[0, i] = ((yy - (y1 + h / 2)) / (h / 2)) ** 2 + ((xx - (x1 + w / 2)) / (w / 2)) ** 2 <= 1.0
    ids = np.ones(n, np.int32)
    np.random.seed(seed)
    rpn_match, rpn_bbox = build_rpn_targets((IMAGE, IMAGE, 3), anchors_np, ids, boxes.astype(np.int32), RCfg(), device=dev)
    nb = boxes / IMAGE
    jit = np.clip(np.repeat(nb, 20, 0) + rng.normal(0, 0.01, (20 * n, 4)), 0, 1).astype(np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return {"image": torch.randn(1, 3, IMAGE, IMAGE, generator=torch.Generator().manual_seed(seed)).to(dev).contiguous(memory_format=torch.channels_last),
            "rpn_match": t(rpn_match.astype(np.int32)), "rpn_bbox": t(rpn_bbox.astype(np.float32)),
            "gt_ids": t(ids).unsqueeze(0), "gt_boxes": t(nb).unsqueeze(0), "gt_masks": t(masks).unsqueeze(0), "injected": t(jit)}


def batch_inputs(items):
    """SLNTrainNet.forward_batch's inputs for a list of make_image examples: the images as one [B,3,H,W] batch, the GT
    ids / boxes padded to the largest instance count, the masks as a list (never stacked)."""
    B, dev = len(items), items[0]["image"].device
    num_gt = [int(d["gt_ids"].shape[1]) for d in items]
    gt_ids = torch.zeros((B, max(num_gt)), dtype=torch.int32, device=dev)
    gt_boxes = torch.zeros((B, max(num_gt), 4), dtype=torch.float32, device=dev)
    for b, d in enumerate(items):
        gt_ids[b, :num_gt[b]] = d["gt_ids"][0]
        gt_boxes[b, :num_gt[b]] = d["gt_boxes"][0]
    return {"images": torch.cat([d["image"] for d in items]).contiguous(memory_format=torch.channels_last),
            "rpn_match": [d["rpn_match"] for d in items], "rpn_bbox_t": [d["rpn_bbox"] for d in items],
            "gt_ids": gt_ids, "gt_boxes": gt_boxes, "gt_masks": [d["gt_masks"][0] for d in items], "num_gt": num_gt,
            "injected": [d["injected"] for d in items]}


class RCfg:
    RPN_TRAIN_ANCHORS_PER_IMAGE = 256
    RPN_BBOX_STD_DEV = np.array([0.1, 0.1, 0.2, 0.2])


# ----------------------------------------------------------------------------- the measurement
def run(dev, rank, world, steps=2, warmup=1, images_per_step=16, weak=False, log=None, images_per_forward=1):
    """Times `steps` optimizer steps (CUDA events, barrier on both sides, max over ranks).  strong scaling: the 16 images
    of a step are split over the ranks; weak: 16 per rank.  images_per_forward > 1 sends that many images through one
    forward (SLNTrainNet.forward_batch) instead of one at a time.  Returns a dict for bench.py."""
    import torch.distributed as dist
    from sln_amodal_b200 import dist as sdist, synth
    from contextlib import nullcontext
    torch.backends.cudnn.benchmark = True
    anchors_np = synth.pyramid_anchors()
    torch.manual_seed(0)                                              # identical initial weights on every rank
    net = SLNTrainNet(torch.from_numpy(anchors_np.astype(np.float32))).to(dev).to(memory_format=torch.channels_last)
    net.train()
    for m in net.modules():                                           # the reference keeps BatchNorm in eval mode (model.py:525-531)
        if isinstance(m, nn.BatchNorm2d):
            m.eval()
    n_params = sum(p.numel() for p in net.parameters())
    ddp = sdist.wrap_ddp(net, device_ids=[dev.index])
    opt = torch.optim.SGD(net.parameters(), lr=1e-3, momentum=0.9, weight_decay=1e-4)
    per_rank = images_per_step if weak else max(1, images_per_step // world)
    data = [make_image(1000 * rank + 7 + i, dev, anchors_np) for i in range(min(per_rank, 4))]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    B = max(1, min(int(images_per_forward), per_rank))
    groups = [batch_inputs([data[(g + j) % len(data)] for j in range(min(B, per_rank - g))])
              for g in range(0, per_rank, B)] if B > 1 else []

    def step_batched(sync=True):
        opt.zero_grad(set_to_none=True)
        pos = 0
        for i, grp in enumerate(groups):
            last = i == len(groups) - 1
            ctx = nullcontext() if (world == 1 or (last and sync)) else ddp.no_sync()
            with ctx:
                loss, n_pos = ddp(grp)
                (loss / per_rank).backward()
            pos += n_pos
        torch.nn.utils.clip_grad_norm_(net.parameters(), 5.0)
        opt.step()
        return float(loss.detach()) / len(groups[-1]["num_gt"]), pos      # per image, like the per-image step's

    def step(sync=True):
        if groups:
            return step_batched(sync)
        opt.zero_grad(set_to_none=True)
        pos = 0
        for i in range(per_rank):
            d = data[i % len(data)]
            last = i == per_rank - 1
            ctx = nullcontext() if (world == 1 or (last and sync)) else ddp.no_sync()
            with ctx:
                loss, n_pos = ddp(d["image"], d["rpn_match"], d["rpn_bbox"], d["gt_ids"], d["gt_boxes"], d["gt_masks"], d["injected"])
                (loss / per_rank).backward()
            pos += n_pos
        torch.nn.utils.clip_grad_norm_(net.parameters(), 5.0)        # model.py:443
        opt.step()
        return float(loss.detach()), pos

    def timed(sync):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            out = step(sync)
        b.record()
        barrier()
        return sdist.max_over_ranks(a.elapsed_time(b)) / steps, out

    for _ in range(warmup):
        step()
    ms, (loss, pos) = timed(True)
    res = {"what": "SLN-style training step, synthetic D2SA-shaped 1024^2 images (8-15 instances, L=1): ResNet-101-FPN + RPN + "
                   "classifier + mask head in stock PyTorch (fp32, TF32 convolutions), hot path through the drop-ins "
                   "(rpn_pack, proposal_layer, detection_target_layer, pyramid_roi_align 7x7 + 16x16 fwd/bwd), losses, "
                   "backward, clip, SGD; %d images per optimizer step per rank" % per_rank,
           "n_gpus": world, "scaling": "weak" if weak else "strong", "images_per_step_global": per_rank * world,
           "ms_per_step": round(ms, 2), "images_per_s": round(per_rank * world / (ms * 1e-3), 2),
           "parameters": n_params, "positives_last_step": pos, "loss_last_step": round(loss, 4), "steps": steps}
    if groups:
        res["images_per_forward"] = B
    if world > 1:
        ms_ns, _ = timed(False)                                       # the same step without the gradient all-reduce
        res["ms_per_step_without_allreduce"] = round(ms_ns, 2)
        res["allreduce_share"] = round(max(0.0, ms - ms_ns) / ms, 4)
        res["allreduce_bytes_per_step"] = n_params * 4
        res["collective"] = "DDP bucketed NCCL all-reduce (25 MB buckets), one per optimizer step (no_sync on the other images)"
        # evaluation-side collective: all-gather of per-image detections (dist.gather_detections) over NCCL
        dets = [torch.rand((50 + 10 * rank + i, 6), device=dev) for i in range(2)]
        barrier()
        t0 = time.perf_counter()
        allg = sdist.gather_detections(dets)
        torch.cuda.synchronize()
        res["gather_detections"] = {"images": len(allg), "ms": round((time.perf_counter() - t0) * 1e3, 2),
                                    "rows": int(sum(int(x.shape[0]) for x in allg))}
    if log:
        log(res)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--weak", action="store_true")
    ap.add_argument("--images-per-forward", type=int, default=1,
                    help="images per forward pass (B > 1: FPN on a [B,3,H,W] batch, batched proposals and targets)")
    args = ap.parse_args()
    from sln_amodal_b200 import dist as sdist
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world = sdist.init()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    res = run(torch.device("cuda", local), rank, world, steps=args.steps, warmup=args.warmup, weak=args.weak,
              images_per_forward=args.images_per_forward)
    if rank == 0:
        os.write(real_stdout, (json.dumps(res) + "\n").encode())
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
