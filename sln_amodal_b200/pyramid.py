"""Drop-in for pyramid_roi_align / pyramid_roi_align_image (reference modal/modals.py:20-157).

The reference loops over FPN levels with nonzero / gather / crop / cat / sort and >= 8 host
syncs (modals.py:70-108).  Here the level of every ROI is computed on the device with the
reference's own formula and torch ops (modals.py:53-64), and ONE kernel launch crops all
ROIs from their level and writes them in the original order.
"""
from __future__ import annotations

import torch

from . import ops
from .crop_and_resize import CropAndResizeFunction, keeps_dtype


# Training: plan the backward (its three ROI-list launches) beside the forward kernel; False restores plan-in-backward.
PLAN_BACKWARD_IN_FORWARD = True


def log2(x):
    """modals.py:8-13: log2 as log(x)/log(2)."""
    ln2 = torch.log(torch.tensor([2.0], dtype=torch.float32, device=x.device))
    return torch.log(x) / ln2


def roi_level(boxes, image_shape):
    """modals.py:53-64.  boxes [N,4] normalised -> int32 [N] in {2,3,4,5}.  CUDA tensors take one kernel launch
    (ops.roi_levels_device: the same fp32 operation sequence); CPU tensors the reference's torch expression."""
    if boxes.is_cuda and boxes.dtype == torch.float32:
        return ops.roi_levels_device(boxes, image_shape) + 2
    y1, x1, y2, x2 = boxes.chunk(4, dim=1)
    h = y2 - y1
    w = x2 - x1
    image_area = torch.tensor([float(image_shape[0] * image_shape[1])], dtype=torch.float32, device=boxes.device)
    lvl = 4 + log2(torch.sqrt(h * w) / (224.0 / torch.sqrt(image_area)))
    return lvl.round().int().clamp(2, 5).view(-1)


class _PyramidCrop(torch.autograd.Function):
    @staticmethod
    def forward(ctx, boxes, box_ind, level, pool, *maps):
        ctx.sizes = [tuple(m.shape) for m in maps]
        ctx.cl = [ops.is_channels_last(m) for m in maps]
        ctx.needs = [m.requires_grad for m in maps]
        ctx.plan = None
        lowp = keeps_dtype(*maps)
        ctx.grad_dtype = maps[0].dtype if lowp else torch.float32
        if PLAN_BACKWARD_IN_FORWARD and any(ctx.needs) and boxes.shape[0] and not torch.cuda.is_current_stream_capturing():
            # the backward's ROI lists only depend on the boxes: build them on a side stream while the forward kernel runs
            ctx.plan = ops.pyramid_crop_backward_plan(boxes, box_ind, level, ctx.sizes, maps[0].shape[1], pool, pool)
        out = ops.pyramid_crop_forward(list(maps), boxes, box_ind, level, pool, pool, 0.0, keep_dtype=lowp)
        ctx.save_for_backward(boxes, box_ind, level)
        return out

    @staticmethod
    def backward(ctx, grad):
        boxes, box_ind, level = ctx.saved_tensors
        outs = ops.pyramid_crop_backward(grad, boxes, box_ind, level, ctx.sizes, channels_last_out=ctx.cl, plan=ctx.plan,
                                         out_dtype=ctx.grad_dtype)
        grads = [o if need else None for o, need in zip(outs, ctx.needs)]
        return (None, None, None, None) + tuple(grads)


def pyramid_roi_align(inputs, pool_size, image_shape):
    """inputs = [boxes [1,N,4] normalised, P2, P3, P4, P5 each [1,C,H_l,W_l]]
    -> pooled [N,C,pool,pool] in the order of the boxes (modals.py:20-110)."""
    boxes = inputs[0].reshape(-1, 4)
    feature_maps = [m if m.dim() == 4 else m.unsqueeze(0) for m in inputs[1:]]
    level = roi_level(boxes.detach(), image_shape) - 2           # 0..3 -> P2..P5
    box_ind = torch.zeros(boxes.shape[0], dtype=torch.int32, device=boxes.device)
    return _PyramidCrop.apply(boxes.detach(), box_ind, level, pool_size, *feature_maps)


def pyramid_roi_align_batched(boxes, box_ind, feature_maps, pool_size, image_shape):
    """Batch > 1 extension (the reference is batch-1 only, modals.py:39): boxes [N,4], box_ind [N]
    names the image of each box, feature_maps [B,C,H_l,W_l]."""
    level = roi_level(boxes.detach(), image_shape) - 2
    return _PyramidCrop.apply(boxes.detach(), box_ind, level, pool_size, *feature_maps)


def pyramid_roi_align_image(inputs, pool_size, image_shape, istrain=False):
    """Single-map crop (modals.py:112-157): inputs = [boxes, feature_map]."""
    boxes = inputs[0].reshape(-1, 4)
    fm = inputs[1]
    if fm.dim() == 3:
        fm = fm.unsqueeze(0)
    elif fm.dim() == 5:
        fm = fm.squeeze(0)
    ind = torch.zeros(boxes.shape[0], dtype=torch.int32, device=boxes.device)
    return CropAndResizeFunction(pool_size, pool_size, 0)(fm, boxes, ind)
