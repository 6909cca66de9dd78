"""Drop-in for the reference's roialign/roi_align/crop_and_resize.py and roi_align.py.

Same names, argument meaning and return conventions as the reference
(crop_and_resize.py:10-67, roi_align.py:9-48):

    CropAndResizeFunction(crop_height, crop_width, extrapolation_value=0)(image, boxes, box_ind)
    CropAndResize(crop_height, crop_width, extrapolation_value=0)(image, boxes, box_ind)
    RoIAlign(crop_height, crop_width, extrapolation_value=0, transform_fpcoor=True)(featuremap, boxes, box_ind)

The reference's CropAndResizeFunction is a legacy (instance) autograd.Function, which
torch >= 1.3 refuses to run; here it is a plain callable class around a static
autograd.Function.  Gradient flows to `image` only (crop_and_resize.py:50).
"""
from __future__ import annotations

import torch
from torch import nn

from . import ops


def keeps_dtype(*maps):
    """Inside an enabled CUDA autocast region, bf16 / fp16 maps (all of one dtype) are cropped in their own dtype, like
    torchvision's roi_align, and their gradient is written in it; the values are today's f32 results rounded once, which
    is what autocast's cast hands a low-precision consumer anyway.  Outside autocast, crops are f32."""
    dt = maps[0].dtype
    return torch.is_autocast_enabled("cuda") and dt in ops.LOWP_DTYPES and all(m.dtype == dt for m in maps)


class _CropAndResize(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image, boxes, box_ind, crop_height, crop_width, extrapolation_value):
        lowp = keeps_dtype(image)
        crops = ops.crop_and_resize_forward(image, boxes, box_ind, crop_height, crop_width, extrapolation_value,
                                            keep_dtype=lowp)
        ctx.im_size = tuple(image.shape)                       # crop_and_resize.py:30-31
        ctx.im_channels_last = ops.is_channels_last(image)
        ctx.grad_dtype = image.dtype if lowp else torch.float32
        ctx.save_for_backward(boxes, box_ind)
        return crops

    @staticmethod
    def backward(ctx, grad_outputs):
        boxes, box_ind = ctx.saved_tensors
        grad_image = ops.crop_and_resize_backward(grad_outputs, boxes, box_ind, ctx.im_size,
                                                  channels_last_out=ctx.im_channels_last, out_dtype=ctx.grad_dtype)
        return grad_image, None, None, None, None, None       # crop_and_resize.py:50


class CropAndResizeFunction(object):
    """CropAndResizeFunction(ch, cw, ext)(image, boxes, box_ind) -> crops [N,C,ch,cw].

    image   f32 [B,C,H,W] (CUDA); NCHW or channels_last memory, the result follows it.  bf16 / fp16 images
            give crops of their dtype inside torch.autocast (see keeps_dtype), f32 crops outside it
    boxes   f32 [N,4] (y1,x1,y2,x2) normalised to [0,1] over (H-1, W-1)
    box_ind i32 [N] image index of each box"""

    def __init__(self, crop_height, crop_width, extrapolation_value=0):
        self.crop_height = crop_height
        self.crop_width = crop_width
        self.extrapolation_value = extrapolation_value

    def __call__(self, image, boxes, box_ind):
        return _CropAndResize.apply(image, boxes, box_ind, self.crop_height, self.crop_width,
                                    self.extrapolation_value)

    # the reference's legacy Function is sometimes driven through .forward()
    forward = __call__


class CropAndResize(nn.Module):
    """Crop and resize ported from tensorflow (reference crop_and_resize.py:53-67)."""

    def __init__(self, crop_height, crop_width, extrapolation_value=0):
        super(CropAndResize, self).__init__()
        self.crop_height = crop_height
        self.crop_width = crop_width
        self.extrapolation_value = extrapolation_value

    def forward(self, image, boxes, box_ind):
        return CropAndResizeFunction(self.crop_height, self.crop_width, self.extrapolation_value)(image, boxes, box_ind)


class RoIAlign(nn.Module):
    """RoIAlign on top of crop_and_resize (reference roi_align.py:9-48): boxes are
    (x1,y1,x2,y2) in pixels of the feature map, without normalisation."""

    def __init__(self, crop_height, crop_width, extrapolation_value=0, transform_fpcoor=True):
        super(RoIAlign, self).__init__()
        self.crop_height = crop_height
        self.crop_width = crop_width
        self.extrapolation_value = extrapolation_value
        self.transform_fpcoor = transform_fpcoor

    def forward(self, featuremap, boxes, box_ind):
        x1, y1, x2, y2 = torch.split(boxes, 1, dim=1)
        image_height, image_width = featuremap.size()[2:4]
        if self.transform_fpcoor:                              # roi_align.py:29-37
            spacing_w = (x2 - x1) / float(self.crop_width)
            spacing_h = (y2 - y1) / float(self.crop_height)
            nx0 = (x1 + spacing_w / 2 - 0.5) / float(image_width - 1)
            ny0 = (y1 + spacing_h / 2 - 0.5) / float(image_height - 1)
            nw = spacing_w * float(self.crop_width - 1) / float(image_width - 1)
            nh = spacing_h * float(self.crop_height - 1) / float(image_height - 1)
            boxes = torch.cat((ny0, nx0, ny0 + nh, nx0 + nw), 1)
        else:                                                  # roi_align.py:38-43
            x1 = x1 / float(image_width - 1)
            x2 = x2 / float(image_width - 1)
            y1 = y1 / float(image_height - 1)
            y2 = y2 / float(image_height - 1)
            boxes = torch.cat((y1, x1, y2, x2), 1)
        boxes = boxes.detach().contiguous()
        box_ind = box_ind.detach()
        return CropAndResizeFunction(self.crop_height, self.crop_width, self.extrapolation_value)(featuremap, boxes, box_ind)
