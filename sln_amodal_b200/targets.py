"""Drop-in for bbox_overlaps / detection_target_layer (reference modal/Functions.py:184-416) and
utils.box_refinement (utils.py:96-117) -- SURVEY.md section 8(f), row 1.

Same signatures and return conventions as the reference.  The IoU matching (two [N*G,4] repeat tensors and ~20
elementwise kernels in the reference) and the box refinement are one launch each; the mask targets go through this
repo's CropAndResizeFunction (A12).  Subsampling draws `torch.randperm` from the CPU generator at the same two places
as the reference (:288, :361), so with the same seed the sampled ROIs are the same ones.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, ops
from .crop_and_resize import CropAndResizeFunction


def bbox_overlaps(boxes1, boxes2):
    """IoU overlaps [N1,N2] between two sets of (y1,x1,y2,x2) boxes (Functions.py:184-218)."""
    return ops.bbox_overlaps_device(boxes1, boxes2)


def box_refinement(box, gt_box):
    """Refinement (dy, dx, log dh, log dw) that maps box onto gt_box (utils.py:96-117)."""
    return ops.box_refinement_device(box, gt_box)


def _sample_rois(positive_h, negative_h, config):
    """The reference's subsampling (:281-291, :353-366) of one image on the host: bool [n] positive / negative rows ->
    (positive rows, negative rows) as int64 index arrays, drawn with `torch.randperm` from the CPU generator under the
    reference's conditions and in its order (the negative draw only after at least one positive).  Both
    detection_target_layer and detection_target_layer_batched sample through here."""
    pos_sel = neg_sel = np.zeros(0, np.int64)
    if positive_h.any():
        positive_indices = np.nonzero(positive_h)[0]
        want = int(config.TRAIN_ROIS_PER_IMAGE * config.ROI_POSITIVE_RATIO)
        rand_idx = torch.randperm(positive_indices.shape[0])[:want].numpy()   # CPU generator, like the reference
        pos_sel = positive_indices[rand_idx]
    if pos_sel.shape[0] > 0 and negative_h.any():
        negative_indices = np.nonzero(negative_h)[0]
        r = 1.0 / config.ROI_POSITIVE_RATIO
        negative_count = int(r * pos_sel.shape[0] - pos_sel.shape[0])
        rand_idx = torch.randperm(negative_indices.shape[0])[:negative_count].numpy()
        neg_sel = negative_indices[rand_idx]
    return pos_sel, neg_sel


def rois_per_image(config):
    """Most rows detection_target_layer can return for one image: max over p = 1..want of p + int(r*p - p), with the
    reference's own float expressions (want positives at most, r = 1 / ROI_POSITIVE_RATIO)."""
    want = int(config.TRAIN_ROIS_PER_IMAGE * config.ROI_POSITIVE_RATIO)
    r = 1.0 / config.ROI_POSITIVE_RATIO
    return max((p + int(r * p - p) for p in range(1, want + 1)), default=0)


def detection_target_layer(proposals, gt_class_ids, gt_boxes, gt_masks, config):
    """proposals [1,N,4] normalised, gt_class_ids [1,G], gt_boxes [1,G,4] normalised, gt_masks [1,L,G,H,W]
    -> (rois [R,4], roi_gt_class_ids [R], deltas [R,4], masks [R,L,mh,mw]); empty tensors when nothing is sampled
    (Functions.py:223-416, batch 1 like the reference).

    Host round trips: the reference pays one per `if tensor.size()` / `nonzero` (about ten per image).  Here the
    per-proposal decisions (positive / negative, one byte each) come back in ONE copy together with the class ids; the
    index selection and the reference's `torch.randperm` draws (CPU generator, same sizes in the same order, so a seeded
    run samples the same ROIs) happen on the host, and the chosen indices go back in one copy."""
    dev = proposals.device
    proposals = proposals.squeeze(0).float().contiguous()
    gt_class_ids = gt_class_ids.squeeze(0)
    gt_boxes = gt_boxes.squeeze(0).float().to(dev)
    gt_masks = gt_masks.squeeze(0)
    n = proposals.shape[0]
    G = gt_class_ids.shape[0]

    # overlaps [proposals, gt_boxes] reduced on the fly: row maximum and its (first) index, :274-277, :297 -- launched for
    # the common case of no crowd boxes before the class ids are known on the host
    _, roi_iou_max, roi_argmax = ops.bbox_overlaps_device(proposals, gt_boxes, matrix=False, reduce=True)
    codes = (roi_iou_max >= 0.5).to(torch.uint8)
    if gt_class_ids.is_cuda:
        packed = torch.cat([codes, gt_class_ids.to(torch.int32).view(torch.uint8)]).cpu().numpy()      # the one sync
        codes_h, cls_h = packed[:n], packed[n:].view(np.int32)
    else:
        cls_h = gt_class_ids.to(torch.int32).numpy()
        codes_h = None
    gt_class_ids = gt_class_ids.to(dev)
    no_crowd_h = np.ones(n, dtype=bool)
    if (cls_h < 0).any():                                                     # COCO crowds, :253-267 (rare: redo without them)
        crowd_ix = torch.from_numpy(np.nonzero(cls_h < 0)[0]).to(dev)
        non_crowd_ix = torch.from_numpy(np.nonzero(cls_h > 0)[0]).to(dev)
        crowd_boxes = gt_boxes[crowd_ix]
        gt_class_ids = gt_class_ids[non_crowd_ix]
        gt_boxes = gt_boxes[non_crowd_ix]
        gt_masks = gt_masks[:, non_crowd_ix.to(gt_masks.device)]
        _, crowd_iou_max, _ = ops.bbox_overlaps_device(proposals, crowd_boxes, matrix=False, reduce=True)
        _, roi_iou_max, roi_argmax = ops.bbox_overlaps_device(proposals, gt_boxes, matrix=False, reduce=True)
        both = torch.stack([(roi_iou_max >= 0.5), (crowd_iou_max < 0.001)]).to(torch.uint8).cpu().numpy()
        codes_h, no_crowd_h = both[0], both[1].astype(bool)
    elif codes_h is None:
        codes_h = codes.cpu().numpy()
    positive_h = codes_h.astype(bool)
    negative_h = ~positive_h & no_crowd_h                                     # :351-352

    L = gt_masks.shape[0]
    mh, mw = int(config.MASK_SHAPE[0]), int(config.MASK_SHAPE[1])
    pos_sel, neg_sel = _sample_rois(positive_h, negative_h, config)
    positive_count, negative_count = pos_sel.shape[0], neg_sel.shape[0]
    if positive_count > 0:
        sel = torch.from_numpy(np.concatenate([pos_sel, neg_sel]) if negative_count > 0 else pos_sel).to(dev)
        positive_indices = sel[:positive_count]
        positive_rois = proposals[positive_indices]
        assignment = roi_argmax[positive_indices].long()
        roi_gt_boxes = gt_boxes[assignment]
        roi_gt_class_ids = gt_class_ids[assignment]
        deltas = ops.box_refinement_device(positive_rois, roi_gt_boxes, np.reshape(config.BBOX_STD_DEV, [4]))
        boxes = positive_rois
        if config.USE_MINI_MASK:                                              # :316-325
            y1, x1, y2, x2 = positive_rois.chunk(4, dim=1)
            gt_y1, gt_x1, gt_y2, gt_x2 = roi_gt_boxes.chunk(4, dim=1)
            gt_h, gt_w = gt_y2 - gt_y1, gt_x2 - gt_x1
            boxes = torch.cat([(y1 - gt_y1) / gt_h, (x1 - gt_x1) / gt_w, (y2 - gt_y1) / gt_h, (x2 - gt_x1) / gt_w], dim=1)
        if gt_masks.is_cuda and gt_masks.dtype in (torch.uint8, torch.bool):
            # gather by assignment + crop + round in one launch, sampling the u8 planes directly (:327-346)
            masks = ops.mask_targets_device(gt_masks, assignment, boxes, mh, mw)
        else:
            roi_masks = gt_masks[:, assignment.to(gt_masks.device)].to(dev)   # [L,P,H,W]
            box_ids = torch.arange(positive_count, dtype=torch.int32, device=dev)
            crop = CropAndResizeFunction(mh, mw, 0)
            masks = torch.stack([crop(roi_masks[i].unsqueeze(1).float(), boxes, box_ids).detach() for i in range(L)], dim=1)
            masks = torch.round(masks.squeeze(2))                             # :346
        if negative_count > 0:
            negative_rois = proposals[sel[positive_count:]]

    if positive_count > 0 and negative_count > 0:                             # :370-384
        rois = torch.cat((positive_rois, negative_rois), dim=0)
        roi_gt_class_ids = torch.cat([roi_gt_class_ids.int(), torch.zeros(negative_count, dtype=torch.int32, device=dev)], dim=0)
        deltas = torch.cat([deltas, torch.zeros(negative_count, 4, device=dev)], dim=0)
        masks = torch.cat([masks, torch.zeros(negative_count, L, mh, mw, device=dev)], dim=0)
    elif positive_count > 0:
        rois = positive_rois
        roi_gt_class_ids = roi_gt_class_ids.int()
    else:                                                                     # nothing sampled: empty tensors, :400-409
        rois = torch.empty(0, device=dev)
        roi_gt_class_ids = torch.empty(0, dtype=torch.int32, device=dev)
        deltas = torch.empty(0, device=dev)
        masks = torch.empty(0, device=dev)
    return rois, roi_gt_class_ids, deltas, masks


def detection_target_layer_batched(proposals, gt_class_ids, gt_boxes, gt_masks, config, num_proposals=None, num_gt=None):
    """detection_target_layer for B images: one match launch, one host round trip, one emit launch.

    proposals f32 [B,R,4] normalised (e.g. proposal_layer_batched's zero-padded rois), gt_class_ids int [B,G], gt_boxes
    f32 [B,G,4] normalised, gt_masks u8 / bool on the device: one tensor [B,L,G,H,W] or a list of B tensors [L,G_b,H,W]
    with G_b = num_gt[b] (never stacked or copied); num_proposals int32 device [B] (None: all R rows are proposals),
    num_gt B host ints (None: all G rows are GT boxes).  Every image has the same L, H, W.
    Returns (rois f32 [B,T,4], class_ids int32 [B,T], deltas f32 [B,T,4], masks f32 [B,T,L,mh,mw], num_positive int32
    [B], num_rois int32 [B]) on the device, T = rois_per_image(config): image b's rows [0, num_positive[b]) are its
    positives, then its negatives up to num_rois[b], then zeros.  Rows below num_rois[b] equal what
    detection_target_layer returns for proposals[b, :num_proposals[b]] and gt_*[b, :num_gt[b]] alone (num_rois[b] = 0
    where it returns empty tensors), and a seeded call draws the same `torch.randperm`s from the CPU generator in the same
    order as the B single-image calls in image order.
    One difference: a proposal whose IoU maximum is NaN (a zero-area proposal against a zero-area GT box) is neither
    positive nor negative here, as in the reference (Functions.py:351, NaN < 0.5 is false); detection_target_layer counts
    it as a negative.
    The sampling runs on the host between the two launches (one wait, one device-to-host copy of a byte per proposal, one
    host-to-device copy of the sampled rows), so the call cannot be captured in a CUDA graph."""
    B, R, G, num_gt, gt_class_ids, num_proposals = ops.target_inputs(proposals, gt_class_ids, gt_boxes, num_gt, num_proposals)
    dev = proposals.device
    planes, mask_g, LHW = ops.target_mask_planes(gt_masks, B, G, num_gt, dev)
    proposals, gt_boxes = proposals.contiguous(), gt_boxes.contiguous()
    T = rois_per_image(config)
    codes, argmax = ops.target_match_batched_device(proposals, gt_class_ids, gt_boxes, num_gt, num_proposals)
    codes_h = codes.cpu().numpy()                                             # the one wait
    lay = ops.target_stage_layout(B, T)
    stage_h = torch.empty(lay["total"], dtype=torch.int32, pin_memory=True)
    h = stage_h.numpy()
    h[lay["planes"]:lay["mask_g"]].view(np.int64)[:] = [m.data_ptr() for m in planes]
    h[lay["mask_g"]:lay["num_positive"]] = mask_g
    sel = h[lay["sel"]:].reshape(B, T)
    sel[:] = -1
    for b in range(B):
        pos_sel, neg_sel = _sample_rois((codes_h[b] & 1) != 0, (codes_h[b] & 2) != 0, config)
        n_pos, n_rois = pos_sel.shape[0], pos_sel.shape[0] + neg_sel.shape[0]
        sel[b, :n_pos] = pos_sel
        sel[b, n_pos:n_rois] = neg_sel
        h[lay["num_positive"] + b] = n_pos
        h[lay["num_rois"] + b] = n_rois
    stage = torch.empty(lay["total"], dtype=torch.int32, device=dev)
    stage.copy_(stage_h, non_blocking=True)
    rois, class_ids, deltas, masks = ops.detection_targets_emit_batched_device(
        proposals, argmax, gt_boxes, gt_class_ids, stage, T, LHW, config.MASK_SHAPE, np.reshape(config.BBOX_STD_DEV, [4]),
        config.USE_MINI_MASK)
    return (rois, class_ids, deltas, masks, stage[lay["num_positive"]:lay["num_rois"]],
            stage[lay["num_rois"]:lay["sel"]])


_ANCHOR_CACHE = {}


def _device_anchors(anchors, dev):
    """The anchor pyramid is a constant of the configuration: keep its float64 device copy between calls."""
    key = (anchors.__array_interface__["data"][0], anchors.shape, str(anchors.dtype), str(dev))
    hit = _ANCHOR_CACHE.get(key)
    if hit is None or hit[0] is not anchors:
        _ANCHOR_CACHE.clear()
        hit = (anchors, torch.from_numpy(np.ascontiguousarray(anchors, dtype=np.float64)).to(dev))
        _ANCHOR_CACHE[key] = hit
    return hit[1]


def build_rpn_targets(image_shape, anchors, gt_class_ids, gt_boxes, config, device=None):
    """Drop-in for build_rpn_targets (modal/Functions.py:739-847): numpy in, numpy out --
    (rpn_match int32 [A], rpn_bbox float64 [RPN_TRAIN_ANCHORS_PER_IMAGE, 4]).
    The [A,G] float64 IoU matrix of the reference (utils.compute_overlaps) is never built: its three reductions come
    from the device (ops.rpn_overlap_reductions_device); the matching rules, the two `np.random.choice` subsampling
    draws (:806, :814 -- same global numpy generator, same order) and the <= 128 positive deltas stay in numpy exactly
    as the reference has them."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    anchors = np.asarray(anchors)
    gt_class_ids = np.asarray(gt_class_ids)
    gt_boxes = np.asarray(gt_boxes)
    A = anchors.shape[0]
    rpn_match = np.zeros([A], dtype=np.int32)
    rpn_bbox = np.zeros((config.RPN_TRAIN_ANCHORS_PER_IMAGE, 4))
    d_anchors = _device_anchors(anchors, dev)
    crowd_ix = np.where(gt_class_ids < 0)[0]
    if crowd_ix.shape[0] > 0:                                                 # :759-770
        non_crowd_ix = np.where(gt_class_ids > 0)[0]
        crowd_boxes = gt_boxes[crowd_ix]
        gt_class_ids = gt_class_ids[non_crowd_ix]
        gt_boxes = gt_boxes[non_crowd_ix]
        crowd_iou_max = ops.rpn_overlap_reductions_device(
            d_anchors, torch.from_numpy(np.ascontiguousarray(crowd_boxes, dtype=np.float64)), want_argmax=False)[0].cpu().numpy()
        no_crowd_bool = crowd_iou_max < 0.001
    else:
        no_crowd_bool = np.ones([A], dtype=bool)
    if gt_boxes.shape[0] == 0:
        # the reference fails here too: np.argmax over the empty axis of the [A, 0] overlap matrix (Functions.py:786)
        raise ValueError("build_rpn_targets: no non-crowd GT box left (attempt to get argmax of an empty sequence)")
    if anchors.dtype != np.float64:
        # the reference computes the IoU in the anchors' dtype; the device reductions are float64 (what the reference's
        # generate_pyramid_anchors produces), so narrower anchors would no longer be bit-identical
        raise TypeError("build_rpn_targets: float64 anchors expected (utils.generate_pyramid_anchors), got %s" % anchors.dtype)
    mx, am, ga = ops.rpn_overlap_reductions_device(d_anchors, torch.from_numpy(np.ascontiguousarray(gt_boxes, dtype=np.float64)))
    anchor_iou_max, anchor_iou_argmax, gt_iou_argmax = mx.cpu().numpy(), am.cpu().numpy(), ga.cpu().numpy()
    # matching rules (:789-795): negatives first, then one anchor per GT box whatever its IoU, then every anchor >= 0.7
    rpn_match[(anchor_iou_max < 0.3) & no_crowd_bool] = -1
    rpn_match[gt_iou_argmax] = 1
    rpn_match[anchor_iou_max >= 0.7] = 1
    # balance (:799-816): at most half positives, the rest negatives; the surplus of either kind goes back to neutral.
    # Same two draws from numpy's global generator, in the same order and with the same arguments, as the reference.
    budget = config.RPN_TRAIN_ANCHORS_PER_IMAGE
    for label, allowed in ((1, lambda: budget // 2), (-1, lambda: budget - np.sum(rpn_match == 1))):
        members = np.where(rpn_match == label)[0]
        surplus = len(members) - allowed()
        if surplus > 0:
            rpn_match[np.random.choice(members, surplus, replace=False)] = 0
    # refinement targets of the surviving positives (:820-845), all at once: the same float64 operations element by
    # element (GT boxes keep their integer dtype until the first float operand, as in the reference's scalar code)
    pos = np.where(rpn_match == 1)[0]
    if pos.size:
        a = anchors[pos]
        g = gt_boxes[anchor_iou_argmax[pos]]
        g_h, g_w = g[:, 2] - g[:, 0], g[:, 3] - g[:, 1]
        g_cy, g_cx = g[:, 0] + 0.5 * g_h, g[:, 1] + 0.5 * g_w
        a_h, a_w = a[:, 2] - a[:, 0], a[:, 3] - a[:, 1]
        a_cy, a_cx = a[:, 0] + 0.5 * a_h, a[:, 1] + 0.5 * a_w
        t = np.stack([(g_cy - a_cy) / a_h, (g_cx - a_cx) / a_w, np.log(g_h / a_h), np.log(g_w / a_w)], axis=1)
        rpn_bbox[: pos.size] = t / config.RPN_BBOX_STD_DEV
    return rpn_match, rpn_bbox


def _jitter_boxes(tight):
    """utils.extract_bboxes :51-53 on tight boxes [N,4]: jitter each by +-1/15 of its side with `np.random.rand(4)` drawn per
    instance from the global numpy generator in the reference's order, negatives clipped to 0, truncated to int32."""
    boxes = np.zeros([tight.shape[0], 4], dtype=np.int32)
    for i in range(tight.shape[0]):
        y1, x1, y2, x2 = (int(v) for v in tight[i])
        box = np.array([y1, x1, y2, x2]) + (np.random.rand(4) * 2 - 1) * (y2 - y1, x2 - x1, y2 - y1, x2 - x1) / 15
        box[box < 0] = 0
        boxes[i] = box
    return boxes.astype(np.int32)


def extract_bboxes(mask):
    """Drop-in for utils.extract_bboxes (utils.py:28-54).  mask [H,W,N] (numpy, like the reference) or a CUDA tensor of
    planes [N,H,W] (what sem_dist_targets / decode_layers leave on the device: no trip of the masks through the host).
    Returns int32 [N,4] = the tight box of every instance jittered by +-1/15 of its side with `np.random.rand(4)` drawn
    per instance from the global numpy generator in the reference's order (:51), negatives clipped to 0 (:52)."""
    if isinstance(mask, np.ndarray):
        planes = torch.from_numpy(np.ascontiguousarray(np.moveaxis(mask, -1, 0)).astype(np.uint8)).cuda()
    else:
        planes = mask
    tight = ops.plane_bboxes_device(planes).cpu().numpy().reshape(-1, 4)
    return _jitter_boxes(tight)


def compose_image_meta(image_id, image_shape, window, active_class_ids):
    """modal/Functions.py:612-630: [image_id] + shape (3) + window (4) + active_class_ids as one 1-D array."""
    return np.array([image_id] + list(image_shape) + list(window) + list(active_class_ids))


def load_image_gt(dataset, config, image_id, augment=False, use_mini_mask=False, device=False):
    """Drop-in for load_image_gt (modal/Functions.py:675-736), the per-image ground-truth loader of the training set
    (model.py:80), with the geometry on the device:
      * the label map `<path>.npz['layer']` is inflated into pinned memory and copied asynchronously (npz.py), decoded into
        the [n, L, H, W] visibility planes by sln_layer_decode -- what AmodalDataset.load_layer2 (amodal_train.py:236-271)
        builds with one full-image compare per (object, label piece);
      * utils.resize_image (Pillow-exact 8-bit bilinear, sln_resize_image_u8), utils.resize_layer + the horizontal flip
        (one gather launch reproducing scipy.ndimage.zoom(order=0), sln_gather_planes);
      * the amodal box of an instance = the union of its layers' tight boxes (sln_plane_bboxes; np.sum(mask_layers, 2)
        + np.any in the reference, :718-720), jittered by utils.extract_bboxes' np.random.rand draws in the same order.
    Same draws from the same generators as the reference (`random.randint(0, 1)` only when augment, then 4 numbers of
    `np.random.rand` per instance), so a seeded run returns the reference's values: (image u8 [D,D,3], image_meta,
    class_ids int32 [n], bbox int32 [n,4], mask_layers u8 [D,D,n,L]).  device=True keeps the planes as a CUDA tensor
    [n, L, D, D] (what detection_target_layer's mask-target crop reads) instead of the reference's numpy layout.
    use_mini_mask: the reference's shipped configuration is False (config.py:90) and utils.minimize_mask cannot take the
    4-D layer array it is handed (:726-727), so True raises here instead of failing inside imresize."""
    import random
    from . import npz, semdist
    if use_mini_mask:
        raise ValueError("use_mini_mask=True is not supported: the reference's own minimize_mask cannot process the layer masks "
                         "(modal/Functions.py:726-727, config.py:90 ships False)")
    image = dataset.load_image(image_id)
    info = dataset.image_info[image_id]
    label = npz.load_layer_label(info['path'][:-4] + '.npz')
    planes, n_obj = semdist.decode_layers(label, config.NUM_CLASSES, n_max=32)
    n = int(n_obj[0].item())
    if n == 0:
        # no object decodes: the reference's load_layer2 returns utils.Dataset's empty mask here and load_image_gt then
        # fails inside scipy.ndimage.zoom (a 4-element zoom on a 3-D array)
        raise RuntimeError("image %r has no decodable instance: the reference's load_image_gt cannot process it either "
                           "(utils.resize_layer expects [H,W,L,n])" % (image_id,))
    class_ids = np.ones(n, dtype=np.int32)                               # amodal_train.py:262
    shape = image.shape
    image, window, scale, padding = resize_image(image, min_dim=config.IMAGE_MIN_DIM, max_dim=config.IMAGE_MAX_DIM,
                                                 padding=config.IMAGE_PADDING)
    flip = bool(random.randint(0, 1)) if augment else False              # :712-715
    if flip:
        image = np.fliplr(image)
    planes = resize_layer_device(planes[0, :n], scale, flip=flip)        # [n, L, D, D]
    per_layer = ops.plane_bboxes_device(planes).cpu().numpy()            # [n, L, 4], zeros for an empty plane
    tight = np.zeros((n, 4), np.int64)
    for i in range(n):
        live = per_layer[i][per_layer[i][:, 2] > 0]
        if live.shape[0]:
            tight[i] = (live[:, 0].min(), live[:, 1].min(), live[:, 2].max(), live[:, 3].max())
    bbox = _jitter_boxes(tight)
    active_class_ids = np.zeros([128], dtype=np.int32)
    active_class_ids[range(128)] = 1
    image_meta = compose_image_meta(image_id, shape, window, active_class_ids)
    if device:
        return image, image_meta, class_ids, bbox, planes
    mask_layers = planes.permute(2, 3, 0, 1).contiguous().cpu().numpy()   # np.swapaxes(mask_layers, 2, 3) > 0 as uint8
    return image, image_meta, class_ids, bbox, mask_layers


def zoom_index_map(n_in, n_out):
    """Source index of every output line of scipy.ndimage.zoom(order=0, mode='constant') along one axis, in scipy's own
    float64 arithmetic: position = o * (n_in-1)/(n_out-1), index = floor(position + 0.5); a position outside
    [0, n_in-1] -- the last line overshoots by one rounding error for some size pairs -- reads the constant 0 (index -1)."""
    if n_out <= 1:
        return np.zeros(max(n_out, 0), np.int32)
    z = (n_in - 1) / (n_out - 1)
    cc = np.arange(n_out, dtype=np.float64) * z
    idx = np.floor(cc + 0.5).astype(np.int64)
    idx[(cc < 0) | (cc > n_in - 1)] = -1
    return idx.astype(np.int32)


def resize_layer_device(planes, scale, flip=False):
    """utils.resize_layer (utils.py:358-362: scipy.ndimage.zoom(mask, [sy, sx, 1, 1], order=0)) and the optional
    np.fliplr of load_image_gt (Functions.py:712-715) for device-resident planes [..., H, W] in one gather launch."""
    H, W = planes.shape[-2:]
    H2, W2 = int(round(H * scale[0])), int(round(W * scale[1]))
    iy, ix = zoom_index_map(H, H2), zoom_index_map(W, W2)
    if flip:
        ix = ix[::-1].copy()
    return ops.gather_planes_device(planes, iy, ix)


def resize_layer(mask, scale, padding=None):
    """Drop-in for utils.resize_layer: numpy mask [H, W, ...] in, numpy out (the planes take one trip through the
    device; use resize_layer_device on the output of decode_layers / sem_dist_targets to stay there)."""
    m = np.asarray(mask)
    planes = torch.from_numpy(np.ascontiguousarray(np.moveaxis(m, (0, 1), (-2, -1))).astype(np.uint8)).cuda()
    out = resize_layer_device(planes, scale).cpu().numpy()
    return np.moveaxis(out, (-2, -1), (0, 1)).astype(m.dtype)


def resize_image_device(image, out_hw):
    """scipy.misc.imresize(image, out_hw) (interp='bilinear') of a uint8 image [h, w] or [h, w, C] on the device:
    Pillow's 8-bit bilinear resample per band, bit for bit (sln_resize_image_u8).  numpy or tensor in, CUDA u8 out."""
    if not torch.cuda.is_available():
        raise _lib.SlnError("resize_image_device needs a CUDA device (there is no CPU fallback)")
    t = torch.as_tensor(image)
    if t.dtype != torch.uint8 or t.dim() not in (2, 3):
        raise _lib.SlnError("resize_image_device: uint8 [h, w] or [h, w, C] expected")
    if not t.is_cuda:
        t = t.cuda()
    t = t.contiguous()
    h, w = int(t.shape[0]), int(t.shape[1])
    C = int(t.shape[2]) if t.dim() == 3 else 1
    H2, W2 = int(out_hw[0]), int(out_hw[1])
    out = torch.empty((H2, W2, C) if t.dim() == 3 else (H2, W2), dtype=torch.uint8, device=t.device)
    need = int(_lib.lib().sln_resize_image_workspace_bytes(h, w, C, H2, W2))
    ws = torch.empty(max(need, 1), dtype=torch.uint8, device=t.device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.lib().sln_resize_image_u8(_lib.ptr(t), h, w, C, H2, W2, _lib.ptr(out), _lib.ptr(ws), need, _lib.stream_ptr()),
                   "sln_resize_image_u8")
    _lib.count_launches(3)
    return out


def resize_image(image, min_dim=None, max_dim=None, padding=False, device=False):
    """Drop-in for utils.resize_image (utils.py:301-356): the reference squashes every image to (max_dim, max_dim) with
    scipy.misc.imresize -- min_dim and padding are ignored by its body too -- and returns (image, window, scale, padding).
    The image comes back as a numpy uint8 array like the reference's (callers do image.astype(np.float32), model.py
    mold_inputs); device=True keeps it a CUDA u8 tensor.  uint8 input only (imresize would bytescale anything else)."""
    h, w = image.shape[:2]
    out = resize_image_device(image, (max_dim, max_dim))
    if not device:
        out = out.cpu().numpy()
    window = (0, 0, max_dim, max_dim)
    scale = (max_dim / h, max_dim / w)
    return out, window, scale, [(0, 0), (0, 0), (0, 0)]
