"""Drop-in for proposal_layer (reference modal/Functions.py:114-178).

    proposal_layer(inputs, proposal_count, nms_threshold, anchors, config=None)
        inputs  = [rpn_probs [1,A,2], rpn_bbox [1,A,4]]
        anchors = [A,4] pixels (y1,x1,y2,x2)
        -> [1, k, 4] normalised proposals, k <= proposal_count, NOT zero padded

The whole layer (top-6000 select, delta decode, clip, NMS, top-k, normalise) is one C-ABI
call with no host synchronisation; the only host read is the survivor count needed to
return an unpadded tensor like the reference does.
"""
from __future__ import annotations

import numpy as np

from . import ops

PRE_NMS_LIMIT = 6000          # Functions.py:144


def proposal_layer(inputs, proposal_count, nms_threshold, anchors, config=None):
    # Currently only supports batchsize 1 (Functions.py:128-130; the reference mutates `inputs`)
    inputs[0] = inputs[0].squeeze(0)
    inputs[1] = inputs[1].squeeze(0)
    std_dev = np.reshape(config.RPN_BBOX_STD_DEV, [4]) if config is not None else (0.1, 0.1, 0.2, 0.2)
    height, width = (config.IMAGE_SHAPE[:2] if config is not None else (1024, 1024))
    boxes, num = ops.proposal_device(inputs[0], inputs[1], anchors, proposal_count, nms_threshold,
                                     std_dev, (height, width), pre_nms_limit=PRE_NMS_LIMIT)
    k = int(num.item())
    return boxes[:k].unsqueeze(0)


def proposal_layer_batched(inputs, proposal_count, nms_threshold, anchors, config=None):
    """proposal_layer for B images in one call: inputs = [rpn_probs [B,A,2], rpn_bbox [B,A,4]] (not modified), anchors
    [A,4] pixels shared by the images.  Returns (rois [B,proposal_count,4] normalised, zero padded beyond num[b]; num
    int32 [B]) as device tensors, no host sync; rois[b, :num[b]] is proposal_layer's result for image b alone."""
    std_dev = np.reshape(config.RPN_BBOX_STD_DEV, [4]) if config is not None else (0.1, 0.1, 0.2, 0.2)
    height, width = (config.IMAGE_SHAPE[:2] if config is not None else (1024, 1024))
    return ops.proposal_batched_device(inputs[0], inputs[1], anchors, proposal_count, nms_threshold, std_dev,
                                       (height, width), pre_nms_limit=PRE_NMS_LIMIT)


def proposal_layer_padded(rpn_probs, rpn_bbox, anchors, proposal_count, nms_threshold,
                          std_dev=(0.1, 0.1, 0.2, 0.2), image_hw=(1024, 1024)):
    """Sync-free variant for batched / graph-captured use: returns (boxes [proposal_count,4]
    zero padded, num int32[1]) as device tensors."""
    return ops.proposal_device(rpn_probs, rpn_bbox, anchors, proposal_count, nms_threshold, std_dev,
                               image_hw, pre_nms_limit=PRE_NMS_LIMIT)
