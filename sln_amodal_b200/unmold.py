"""Mask paste after the path -- utils.unmold_mask (utils.py:447-465) and MaskRCNN.unmold_detections
(model.py:747-806) with the per-detection python loop replaced by one launch (SURVEY.md section 8(f), row 3).

    unmold_mask(mask, bbox, image_shape)                               -> u8 [H, W]   (the reference's signature)
    unmold_masks(masks [N,h,w], boxes [N,4], image_shape)              -> u8 [N, H, W] on the device
    unmold_detections(detections, mrcnn_mask, image_shape, window)     -> boxes, class_ids, scores, masks [H, W, N]
    unmold_detections_batched(detections [B,D,6], mrcnn_mask [B,D,h,w,K], image_shapes, windows)
                                                                       -> per image: boxes, class_ids, scores, COCO RLEs

The reference resizes with scipy.misc.imresize(interp='bilinear') = scipy's bytescale + Pillow's 8-bit resampler;
sln_unmold_masks reproduces both bit for bit (csrc/unmold.cu).  The planes stay on the device so that
rle.encode() -- the next step of the reference's evaluation (amodal_train.py:371-400) -- takes them without a copy.
The batched form goes from B images' detections to COCO RLE strings on the device without any H x W plane
(ops.unmold_rle_batched_device); its results are those of unmold_detections followed by rle.encode, image by image.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops, rle
from ._lib import check, lib, ptr, stream_ptr


def unmold_masks(masks, boxes, image_shape):
    """masks f32 [N, h, w] and boxes int [N, 4] (numpy or tensors; moved to the current CUDA device when they are not
    there yet) -> u8 [N, H, W] CUDA tensor."""
    H, W = int(image_shape[0]), int(image_shape[1])
    if not torch.cuda.is_available():
        raise _lib.SlnError("unmold_masks needs a CUDA device (there is no CPU fallback)")
    dev = masks.device if isinstance(masks, torch.Tensor) and masks.is_cuda else torch.device("cuda", torch.cuda.current_device())
    m = torch.as_tensor(masks, dtype=torch.float32).to(dev).contiguous()
    b = torch.as_tensor(np.asarray(boxes) if not isinstance(boxes, torch.Tensor) else boxes).to(dev).to(torch.int32).contiguous()
    if m.dim() != 3 or b.dim() != 2 or b.shape[1] != 4 or b.shape[0] != m.shape[0]:
        raise _lib.SlnError("unmold_masks: masks [N, h, w] and boxes [N, 4] expected")
    n, mh, mw = m.shape
    out = torch.empty((n, H, W), dtype=torch.uint8, device=dev)
    if n:
        with torch.cuda.device(dev):
            check(lib().sln_unmold_masks(ptr(m), n, mh, mw, ptr(b), H, W, ptr(out), stream_ptr()), "sln_unmold_masks")
        _lib.count_launches(1)
    return out


def unmold_mask(mask, bbox, image_shape, device=False):
    """utils.py:447-465: one small float mask -> binary full-image mask, numpy u8 [H, W] like the reference's (callers
    np.stack the results, model.py:794-800); device=True keeps the CUDA tensor.  Like the reference, the box must lie
    inside the image with positive height and width (there the paste raises a shape mismatch; here it is an error too)."""
    m = torch.as_tensor(mask, dtype=torch.float32)
    m = m.reshape([s for s in m.shape if s != 1] or [1, 1])               # mask.squeeze()
    if m.dim() != 2:
        raise _lib.SlnError("unmold_mask: a [height, width] mask expected")
    y1, x1, y2, x2 = (int(v) for v in bbox)
    if not (0 <= y1 < y2 <= int(image_shape[0]) and 0 <= x1 < x2 <= int(image_shape[1])):
        raise ValueError("unmold_mask: box %s is not inside the %dx%d image" % ((y1, x1, y2, x2), image_shape[0], image_shape[1]))
    out = unmold_masks(m[None], np.asarray([[y1, x1, y2, x2]], np.int32), image_shape)[0]
    return out if device else out.cpu().numpy()


def unmold_detections(detections, mrcnn_mask, image_shape, window, return_device_planes=False):
    """model.py:747-806.  detections [N, 6] and mrcnn_mask [N, h, w, num_classes] as numpy (the reference's calling
    convention) or tensors.  The box arithmetic is the reference's numpy (float64 scale / shift, astype(int32),
    zero-area filter); the resize / threshold / paste loop is one launch.  Returns boxes, class_ids, scores and
    masks [H, W, N] (numpy, like the reference) or, with return_device_planes, the u8 [N, H, W] CUDA planes."""
    det = detections.detach().cpu().numpy() if isinstance(detections, torch.Tensor) else np.asarray(detections)
    zero_ix = np.where(det[:, 4] == 0)[0]
    N = zero_ix[0] if zero_ix.shape[0] > 0 else det.shape[0]
    boxes = det[:N, :4]
    class_ids = det[:N, 4].astype(np.int32)
    class_ids[class_ids > 0] = 1                                           # model.py:769 (classes collapsed)
    scores = det[:N, 5]
    idx = np.arange(N)
    if isinstance(mrcnn_mask, torch.Tensor):
        masks = mrcnn_mask[torch.as_tensor(idx, device=mrcnn_mask.device), :, :,
                           torch.as_tensor(class_ids.astype(np.int64), device=mrcnn_mask.device)]
    else:
        masks = np.asarray(mrcnn_mask)[idx, :, :, class_ids]
    h_scale = image_shape[0] / (window[2] - window[0])
    w_scale = image_shape[1] / (window[3] - window[1])
    shift = window[:2]
    scales = np.array([h_scale, w_scale, h_scale, w_scale])
    shifts = np.array([shift[0], shift[1], shift[0], shift[1]])
    boxes = np.multiply(boxes - shifts, scales).astype(np.int32)
    # model.py:789-793 drops zero-area boxes (the product test also passes boxes with NEGATIVE height and width); a box
    # that rounding pushed past the image border or turned inside out makes the reference's paste raise -- here such a
    # detection is dropped together with its score and class, so boxes, scores and masks stay consistent
    H_, W_ = int(image_shape[0]), int(image_shape[1])
    keep = np.where(((boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1]) > 0) & (boxes[:, 2] > boxes[:, 0]) &
                    (boxes[:, 0] >= 0) & (boxes[:, 1] >= 0) & (boxes[:, 2] <= H_) & (boxes[:, 3] <= W_))[0]
    if keep.shape[0] != N:
        boxes, class_ids, scores = boxes[keep], class_ids[keep], scores[keep]
        masks = masks[torch.as_tensor(keep, device=masks.device)] if isinstance(masks, torch.Tensor) else masks[keep]
        N = class_ids.shape[0]
    if N == 0:
        empty = np.empty((0,) + tuple(np.shape(mrcnn_mask)[1:3]))          # model.py:804 (the reference's quirk)
        return boxes, class_ids, scores, empty
    planes = unmold_masks(masks, boxes, image_shape)
    if return_device_planes:
        return boxes, class_ids, scores, planes
    return boxes, class_ids, scores, np.ascontiguousarray(planes.permute(1, 2, 0).cpu().numpy())


def unmold_detections_batched(detections, mrcnn_mask, image_shapes, windows, cap=None):
    """unmold_detections + rle.encode for B images at once.  detections f32 [B,D,6] (BatchedHeadGraph's output, or a
    stack of per-image [D,6]) and mrcnn_mask f32 [B,D,h,w,K] (any strides: a permuted view of [B,D,K,h,w] works) on
    the device; image_shapes and windows: B host values each (images may differ in size).  Returns, per image,
    (boxes int32 [n,4], class_ids int32 [n], scores f32 [n], rles) with rles a list of {"size": [H, W], "counts": bytes}:
    what unmold_detections(..., return_device_planes=True) followed by rle.encode(planes) returns for that image (for an
    image with no kept detection, rles is [] where the single-image path returns the reference's placeholder array).
    The device work runs sync-free (ops.unmold_rle_batched_device); the host waits once, then copies the metadata and
    the packed strings.  Masks with more than `cap` runs (see the ops function) are re-encoded through unmold_masks +
    rle.encode."""
    B = int(detections.shape[0]) if isinstance(detections, torch.Tensor) else len(detections)
    out = ops.unmold_rle_batched_device(detections, mrcnn_mask, image_shapes, windows, cap=cap)
    if B == 0:
        return []
    D = int(detections.shape[1])
    meta = out.meta.cpu().numpy()                                       # the one wait for the device
    boxes, cls, scores, src, m, off, slen, num_kept, total = ops.unmold_meta_views(meta, B, D)
    strings = out.strings[: int(total[0])].cpu().numpy().tobytes() if int(total[0]) else b""
    results = []
    for b in range(B):
        n = int(num_kept[b])
        if n < 0:
            raise IndexError(f"image {b}: a detection's class indexes outside the {int(mrcnn_mask.shape[4])} mask channels")
        H, W = int(image_shapes[b][0]), int(image_shapes[b][1])
        rles = [{"size": [H, W], "counts": strings[int(off[b, k]): int(off[b, k]) + int(slen[b, k])]} if m[b, k] > 0
                else None for k in range(n)]
        retry = [k for k in range(n) if m[b, k] <= 0]
        if retry:                                                       # more runs than cap: the full-plane path
            dev = mrcnn_mask.device
            masks = mrcnn_mask[b][torch.as_tensor(src[b, retry].astype(np.int64), device=dev), :, :,
                                  torch.as_tensor(cls[b, retry].astype(np.int64), device=dev)]
            for k, r in zip(retry, rle.encode(unmold_masks(masks, boxes[b, retry], image_shapes[b]))):
                rles[k] = r
        results.append((boxes[b, :n].copy(), cls[b, :n].copy(), scores[b, :n].copy(), rles))
    return results
