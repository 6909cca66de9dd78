"""CUDA-graph replay of the detection-head path of one image (BASELINE.json configs[0], SURVEY section 3.1).

The reference walks the path with one Python call per step and a host read after most of them (proposal count, level
masks, detection count: model.py:570-646, modal/modals.py:70-108, modal/Functions.py:526-546).  The drop-ins keep those
signatures and therefore the host reads that define their return shapes.  This module is the other way to drive the SAME
kernels: every step in its padded, sync-free form (`ops.*_device`), captured ONCE into a CUDA graph on static buffers and
replayed with a single launch per image -- no Python between the kernels, no host read inside the image:

    proposal_layer (top-6000 select, decode, clip, NMS, top-k; `num` stays on the device)
      -> FPN level of every ROI + one crop launch for all levels            (pyramid_roi_align, pool 7)
      -> [classifier callback: the model's own head, out of scope here]
      -> refine_detections, the branch config.USE_NMS names (rows beyond `num` masked out):
           USE_NMS = False: decode + top-100 in two launches
           USE_NMS = True:  decode + batched class-aware NMS + one emit launch (refine_detections_batched)
      -> FPN level + crop of the detections                                 (pyramid_roi_align, pool 14 / 16)

With USE_NMS = True the graph keeps the first `max_detections` survivors; the reference keeps all of them.  Pass
max_detections = proposal_count for its untruncated output.

Padding contract: `rois` has `proposal_count` rows, zeros beyond `num`; `detections` has 100 rows, zeros beyond `num_det`;
the crops of padded rows are crops of the zero box (harmless, never read by a caller that honours the counts).  Rows
below the counts are bit-identical to what the eager drop-ins return (tests/test_gpu_parity.py::test_head_graph_*).
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .detection import refine_detections_batched
from .proposal import PRE_NMS_LIMIT


class HeadGraph:
    """graph = HeadGraph(anchors, config, feature_maps, rpn_probs, rpn_bbox, classifier);  out = graph.replay()

    anchors [A,4] pixels; config: IMAGE_SHAPE, RPN_BBOX_STD_DEV, RPN_NMS_THRESHOLD, POOL_SIZE, MASK_POOL_SIZE (the
    reference's config.py names).  feature_maps / rpn_probs [A,2] / rpn_bbox [A,4] are the STATIC input tensors: the graph
    reads these addresses on every replay, so the caller refreshes their contents in place (copy_) between replays.
    classifier(pooled [R,C,p,p], rois [R,4]) -> (probs [R,K], deltas [R,K,4]) runs inside the capture (any capturable
    torch code: the model's classifier head); it may also be a pair of static tensors (probs, deltas).
    With config.USE_NMS true (also reading DETECTION_MIN_CONFIDENCE and DETECTION_NMS_THRESHOLD) refine_detections takes
    its per-class NMS branch and keeps the first max_detections survivors; the reference keeps all of them, so pass
    max_detections = proposal_count for its untruncated output.  Without the attribute, or with it false, the top-k
    branch runs."""

    def __init__(self, anchors, config, feature_maps, rpn_probs, rpn_bbox, classifier, proposal_count=1000,
                 max_detections=100, window=None, capture=True):
        self.dev = rpn_probs.device
        self.cfg = config
        self.anchors = anchors
        self.maps = list(feature_maps)
        self.rpn_probs, self.rpn_bbox = rpn_probs, rpn_bbox
        self.classifier = classifier
        self.R, self.D = int(proposal_count), int(max_detections)
        h, w = config.IMAGE_SHAPE[:2]
        self.image_hw = (int(h), int(w))
        self.window = tuple(float(v) for v in (window if window is not None else (0, 0, h, w)))
        self.std_rpn = np.reshape(config.RPN_BBOX_STD_DEV, [4])
        self.out = None
        self._bg = None
        self.graph = None
        if capture:
            self.graph = torch.cuda.CUDAGraph()
            self._capture()

    # the image's steps on the current stream, sync-free; called once eagerly (warm-up: workspaces, lazy module loads) and
    # once under capture
    def _steps(self):
        cfg, R, D = self.cfg, self.R, self.D
        rois, num = ops.proposal_device(self.rpn_probs, self.rpn_bbox, self.anchors, R, float(cfg.RPN_NMS_THRESHOLD),
                                        self.std_rpn, self.image_hw, pre_nms_limit=PRE_NMS_LIMIT)
        box_ind = self._box_ind if self._bg is not None else torch.zeros(R, dtype=torch.int32, device=self.dev)
        level = ops.roi_levels_device(rois, self.image_hw)
        pooled = ops.pyramid_crop_forward(self.maps, rois, box_ind, level, int(cfg.POOL_SIZE), int(cfg.POOL_SIZE), 0.0)
        if callable(self.classifier):
            probs, deltas = self.classifier(pooled, rois)
        else:
            probs, deltas = self.classifier
        # rows beyond the proposal count must not become detections: give them the background class (Functions.py:486-489
        # keeps only class_ids > 0)
        if self._bg is None:                       # constants: made in the eager warm-up pass (host -> device copies cannot be captured)
            self._bg = torch.zeros_like(probs[:1])
            self._bg[0, 0] = 1.0
            h, w = self.image_hw
            self._norm = torch.tensor([h, w, h, w], dtype=torch.float32, device=self.dev)
            self._ar_r = torch.arange(R, device=self.dev, dtype=torch.int32)
            self._ar_d = torch.arange(D, device=self.dev, dtype=torch.int32)
            self._box_ind = torch.zeros(R, dtype=torch.int32, device=self.dev)
        valid = self._ar_r < num
        probs = torch.where(valid[:, None], probs[:R], self._bg)
        if getattr(cfg, "USE_NMS", False):
            # per-class NMS branch, the B = 1 case of the batched form: rows zero beyond num_det, keep too
            det, keep, num_det = refine_detections_batched(rois[None], probs[None], deltas[:R][None], self.window, cfg, D)
            det, keep = det[0], keep[0]
        else:
            dets, _, class_ids, n_excl = ops.refine_decode_device(rois, probs, deltas[:R], self.std_rpn, self.image_hw, self.window, 0.0)
            det, keep = ops.refine_topk_device(dets, class_ids, D)
            num_det = torch.clamp(R - n_excl, max=D)
            rows = self._ar_d < num_det
            det = torch.where(rows[:, None], det, torch.zeros_like(det))     # rows beyond num_det were never written
        boxes = det[:, :4] / self._norm
        lvl_d = ops.roi_levels_device(boxes, self.image_hw)
        mp = int(cfg.MASK_POOL_SIZE)
        mask_in = ops.pyramid_crop_forward(self.maps, boxes, box_ind[:D], lvl_d, mp, mp, 0.0)
        return {"rois": rois, "num_rois": num, "pooled": pooled, "detections": det, "keep": keep, "num_detections": num_det,
                "mask_pooled": mask_in}

    def _warm_up(self):
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        with torch.cuda.stream(side):                     # outside the capture: workspaces, constants, lazy module loads
            self._steps()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        torch.cuda.synchronize(self.dev)

    def _capture(self):
        self._warm_up()
        with torch.cuda.graph(self.graph):
            self.out = self._steps()

    def replay(self):
        """One graph launch on the current stream; returns the static output tensors (valid until the next replay)."""
        self.graph.replay()
        return self.out


class MultiHeadGraph:
    """Several images per launch: the step chains of `heads` (HeadGraph objects built with capture=False, one per image,
    each on its own static inputs) are captured into ONE graph as parallel branches (fork / join on side streams).  The
    path's kernels are short and narrow -- the NMS stages are single clusters, the selects a few hundred CTAs -- so a lone
    image leaves most of the GPU idle between dependent launches; independent images fill it.  Images never interact:
    every branch has its own workspaces and outputs, and each image's results are those of its own HeadGraph."""

    def __init__(self, heads):
        self.heads = list(heads)
        self.dev = self.heads[0].dev
        for h in self.heads:
            h._warm_up()
        self.graph = torch.cuda.CUDAGraph()
        streams = [torch.cuda.Stream(device=self.dev) for _ in self.heads]
        with torch.cuda.graph(self.graph):
            main = torch.cuda.current_stream(self.dev)
            for h, st in zip(self.heads, streams):
                st.wait_stream(main)                       # fork
                with torch.cuda.stream(st):
                    h.out = h._steps()
            for st in streams:
                main.wait_stream(st)                       # join
        self.out = [h.out for h in self.heads]

    def replay(self):
        self.graph.replay()
        return self.out


class BatchedHeadGraph(HeadGraph):
    """HeadGraph's steps for B images at once, one launch per stage for all of them (the per-image dense NMS fallback of
    sln_proposal_layer_batched aside), captured into one graph.

    feature_maps: per level [B,C,H_l,W_l]; rpn_probs [B,A,2]; rpn_bbox [B,A,4]; anchors [A,4] shared.  classifier(pooled
    [B*R,C,p,p], rois [B*R,4]) -> (probs [B*R,K], deltas [B*R,K,4]), or a pair of static tensors of those shapes (or
    [B,R,K] / [B,R,K,4]).  Outputs are [B, ...]: rois [B,R,4] and detections [B,D,6] zero beyond num_rois[b] /
    num_detections[b] (keep too), pooled [B,R,C,p,p], mask_pooled [B,D,C,mp,mp].  Below the counts every image's outputs
    are bit-identical to its own HeadGraph's: the crops, the level rule and the refine front are per row, and the
    proposals, the top-k and the per-class NMS (config.USE_NMS, as in HeadGraph, with the same max_detections cap) run
    within the image."""

    def __init__(self, anchors, config, feature_maps, rpn_probs, rpn_bbox, classifier, proposal_count=1000,
                 max_detections=100, window=None, capture=True):
        self.B = int(rpn_probs.shape[0])
        super().__init__(anchors, config, feature_maps, rpn_probs, rpn_bbox, classifier, proposal_count=proposal_count,
                         max_detections=max_detections, window=window, capture=capture)

    def _steps(self):
        cfg, B, R, D = self.cfg, self.B, self.R, self.D
        rois, num = ops.proposal_batched_device(self.rpn_probs, self.rpn_bbox, self.anchors, R, float(cfg.RPN_NMS_THRESHOLD),
                                                self.std_rpn, self.image_hw, pre_nms_limit=PRE_NMS_LIMIT)
        if self._bg is None:                       # constants: made in the eager warm-up pass (host -> device copies cannot be captured)
            h, w = self.image_hw
            self._norm = torch.tensor([h, w, h, w], dtype=torch.float32, device=self.dev)
            self._ar_r = torch.arange(R, device=self.dev, dtype=torch.int32)
            self._ar_d = torch.arange(D, device=self.dev, dtype=torch.int32)
            img = torch.arange(B, device=self.dev, dtype=torch.int32)
            self._box_ind_r = img.repeat_interleave(R)
            self._box_ind_d = img.repeat_interleave(D)
        flat = rois.reshape(B * R, 4)
        level = ops.roi_levels_device(flat, self.image_hw)
        pooled = ops.pyramid_crop_forward(self.maps, flat, self._box_ind_r, level, int(cfg.POOL_SIZE), int(cfg.POOL_SIZE), 0.0)
        if callable(self.classifier):
            probs, deltas = self.classifier(pooled, flat)
        else:
            probs, deltas = self.classifier
        probs = probs.reshape(B * R, probs.shape[-1])
        deltas = deltas.reshape(B * R, deltas.shape[-2], 4)
        if self._bg is None:
            self._bg = torch.zeros_like(probs[:1])
            self._bg[0, 0] = 1.0
        # rows beyond each image's proposal count get the background class, as in HeadGraph
        valid = (self._ar_r[None, :] < num[:, None]).reshape(B * R)
        probs = torch.where(valid[:, None], probs, self._bg)
        if getattr(cfg, "USE_NMS", False):
            det, keep, num_det = refine_detections_batched(rois, probs.view(B, R, -1), deltas.view(B, R, -1, 4), self.window,
                                                           cfg, D)
        else:
            dets, _, class_ids, _ = ops.refine_decode_device(flat, probs, deltas, self.std_rpn, self.image_hw, self.window, 0.0)
            det, keep, num_det = ops.refine_topk_batched_device(dets.view(B, R, 5), class_ids.view(B, R), D)
            rows = self._ar_d[None, :] < num_det[:, None]
            det = torch.where(rows[..., None], det, torch.zeros_like(det))   # rows beyond num_det were never written
            keep = torch.where(rows, keep, torch.zeros_like(keep))
        boxes = (det[..., :4] / self._norm).reshape(B * D, 4)
        lvl_d = ops.roi_levels_device(boxes, self.image_hw)
        mp = int(cfg.MASK_POOL_SIZE)
        mask_in = ops.pyramid_crop_forward(self.maps, boxes, self._box_ind_d, lvl_d, mp, mp, 0.0)
        return {"rois": rois, "num_rois": num, "pooled": pooled.unflatten(0, (B, R)), "detections": det, "keep": keep,
                "num_detections": num_det, "mask_pooled": mask_in.unflatten(0, (B, D))}
