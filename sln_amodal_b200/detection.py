"""Detection refinement (reference modal/Functions.py:453-575), both branches of config.USE_NMS.

refine_detections keeps the reference's signature and return convention.  USE_NMS = True: the python loop
over class ids (:506-525 -- one nonzero + sort + nms + unique1d per class, each with host syncs) is one
class-aware NMS call.  USE_NMS = False (the shipped default, config.py:78): top-100 by score in one launch.
refine_detections_batched runs either branch for B images with no host read (padded outputs, device counts).
"""
from __future__ import annotations

import numpy as np
import torch


def _refine_detections_fused(rois, probs, deltas, window, config):
    """CUDA path with USE_NMS: one decode launch (argmax, delta decode, clip, round, keep filter), one class-aware
    NMS call, one host read.  Filtered-out boxes ride through the NMS with score -inf and a private class and are
    dropped from the tail of its score-ordered output."""
    from . import ops
    height, width = config.IMAGE_SHAPE[:2]
    std_dev = np.reshape(config.RPN_BBOX_STD_DEV, [4])
    min_conf = float(config.DETECTION_MIN_CONFIDENCE or 0.0)
    dets, cls_nms, class_ids, n_excl = ops.refine_decode_device(rois, probs, deltas, std_dev, (height, width), window, min_conf)
    thr = config.DETECTION_NMS_THRESHOLD
    keep, num = ops.nms_device(dets, thr, class_ids=cls_nms, sparse_only=True)
    k, n_ex = (int(v) for v in torch.cat((num, n_excl)).tolist())          # the one host read
    if k < 0:                                                               # outside the sparse NMS contract
        keep, num = ops.nms_device(dets, thr, class_ids=cls_nms, dense_only=True)
        k = int(num.item())
    k -= n_ex
    if k <= 0:
        return [], []
    keep = keep[:k]                                                         # score-descending (:538-546)
    sel = dets[keep]
    result = torch.cat((sel[:, :4], class_ids[keep].unsqueeze(1).float(), sel[:, 4:5]), dim=1)
    return result, keep


def _refine_detections_topk(rois, probs, deltas, window, config):
    """CUDA path without NMS -- the reference's shipped default (config.py:78 USE_NMS = False; Functions.py:526-546):
    the decode launch, then one launch that ranks the non-background ROIs by score and writes the best 100 (the
    reference hard-codes 100, :530-532) as finished [M,6] rows; one host read for M.  DETECTION_MIN_CONFIDENCE does not
    apply on this branch (it sits inside `if config.USE_NMS`, :492-495)."""
    from . import ops
    height, width = config.IMAGE_SHAPE[:2]
    std_dev = np.reshape(config.RPN_BBOX_STD_DEV, [4])
    dets, _, class_ids, n_excl = ops.refine_decode_device(rois, probs, deltas, std_dev, (height, width), window, 0.0)
    result, keep = ops.refine_topk_device(dets, class_ids, 100)
    m = min(100, rois.shape[0] - int(n_excl.item()))                          # the one host read
    if m <= 0:
        return [], []
    return result[:m], keep[:m]


def refine_detections_batched(rois, probs, deltas, window, config, max_detections=100):
    """refine_detections for B images of N rows each, sync-free: rois [B,N,4] normalised, probs [B,N,K], deltas
    [B,N,K,4], window (y1,x1,y2,x2) pixels shared by the batch -> (detections f32 [B,D,6] (y1,x1,y2,x2,class_id,score),
    keep int64 [B,D] row indices within the image, num_detections int32 [B]), all on the device, zero beyond the counts.

    USE_NMS = False: decode + the top-D non-background rows (refine_topk_batched_device); with D = 100 every image's
    rows equal refine_detections'.  USE_NMS = True: decode with DETECTION_MIN_CONFIDENCE, one class-aware NMS for all
    images at DETECTION_NMS_THRESHOLD (nms_batched_device, max_keep = D), and one launch that writes the rows.  Image b's
    rows are the first D of refine_detections' for that image: the reference does not cap the survivors, so pass
    max_detections = N for its untruncated output."""
    from . import ops
    from ._lib import SlnError
    for t, nm in ((rois, "rois"), (probs, "probs"), (deltas, "deltas")):
        ops._require_cuda(t, nm)
    if rois.dim() != 3 or rois.shape[2] != 4:
        raise SlnError(f"rois must be [B,N,4], got {tuple(rois.shape)}")
    B, N = int(rois.shape[0]), int(rois.shape[1])
    if probs.dim() != 3 or tuple(probs.shape[:2]) != (B, N):
        raise SlnError(f"probs {tuple(probs.shape)} disagrees with rois {tuple(rois.shape)}")
    K = int(probs.shape[2])
    if tuple(deltas.shape) != (B, N, K, 4):
        raise SlnError(f"deltas {tuple(deltas.shape)} disagrees with probs {tuple(probs.shape)}")
    D = int(max_detections)
    if D < 0:
        raise SlnError(f"max_detections must be >= 0, got {max_detections}")
    height, width = config.IMAGE_SHAPE[:2]
    std_dev = np.reshape(config.RPN_BBOX_STD_DEV, [4])
    use_nms = bool(getattr(config, "USE_NMS", False))
    min_conf = float(config.DETECTION_MIN_CONFIDENCE or 0.0) if use_nms else 0.0
    dets, cls_nms, class_ids, _ = ops.refine_decode_device(rois.reshape(B * N, 4), probs.reshape(B * N, K),
                                                          deltas.reshape(B * N, K, 4), std_dev, (height, width), window,
                                                          min_conf)
    dets, cls_nms, class_ids = dets.view(B, N, 5), cls_nms.view(B, N), class_ids.view(B, N)
    if use_nms:
        if D == 0:                                  # max_keep = 0 would mean "all" to the NMS
            keep, num = torch.empty((B, 0), dtype=torch.int64, device=dets.device), torch.zeros(B, dtype=torch.int32, device=dets.device)
        else:
            keep, num = ops.nms_batched_device(dets, config.DETECTION_NMS_THRESHOLD, class_ids=cls_nms, max_keep=D)
        return ops.refine_nms_emit_batched_device(dets, class_ids, keep, num, D)
    det, keep, num_det = ops.refine_topk_batched_device(dets, class_ids, D)
    rows = torch.arange(D, device=dets.device, dtype=torch.int32)[None, :] < num_det[:, None]
    det = torch.where(rows[..., None], det, torch.zeros_like(det))             # rows beyond num_det were never written
    keep = torch.where(rows, keep, torch.zeros_like(keep))
    return det, keep, num_det


def refine_detections(rois, probs, deltas, window, config):
    """rois [N,4] normalised, probs [N,K], deltas [N,K,4], window (y1,x1,y2,x2) pixels
    -> (detections [M,6] (y1,x1,y2,x2,class_id,score), keep indices) or ([], []).
    Device tensors only: the product has no CPU / eager-PyTorch path (DESIGN.md section 1)."""
    if not rois.is_cuda:
        raise RuntimeError("refine_detections: CUDA tensors required (no CPU fallback in sln_amodal_b200)")
    if rois.shape[0] == 0:
        return [], []
    if config.USE_NMS:
        return _refine_detections_fused(rois, probs, deltas, window, config)
    return _refine_detections_topk(rois, probs, deltas, window, config)
