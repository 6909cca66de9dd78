"""Functional host layer over the C ABI: torch CUDA tensors in, torch CUDA tensors out.

Every function here enqueues hand-written sm_100a kernels from libsln_b200.so on the
current torch stream.  Nothing falls back to PyTorch or the CPU: non-CUDA inputs raise.
PyTorch only provides device memory (outputs and workspaces are torch tensors owned by
the caller side, as the ABI requires) and the stream.
"""
from __future__ import annotations

import collections
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import LAYOUT_NCHW, LAYOUT_NHWC, check, lib, ptr, stream_ptr


# Default rounding mode of the RoIAlign backward: False = fma per term (fast, <= 1e-6 relative of
# the reference, deterministic); True = the reference's exact rounding sequence (bit-identical).
EXACT_BACKWARD = False


def _require_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.SlnError(f"{name} must be a CUDA tensor: this path has no CPU implementation "
                            "(the CPU oracle lives under oracle/ and is test infrastructure only)")


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _i32c(t):
    return t.detach().to(torch.int32).contiguous()


def is_channels_last(t) -> bool:
    """True when the 4-D tensor's memory is [B,H,W,C]-contiguous."""
    return t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _check_rois(N, box_ind, level=None):
    """The kernels read box_ind[i] (and level[i]) for every one of the N boxes: a shorter array is read out of bounds."""
    if box_ind.shape[0] != N:
        raise _lib.SlnError(f"box_ind has {box_ind.shape[0]} entries for {N} boxes")
    if level is not None and level.shape[0] != N:
        raise _lib.SlnError(f"level has {level.shape[0]} entries for {N} boxes")


def _check_map_sizes(map_sizes, channels):
    """map_sizes of the pyramid backward: (B, C, H, W) per level, one B for all, C == channels.  Returns B."""
    B = int(map_sizes[0][0])
    for sz in map_sizes:
        if int(sz[0]) != B or int(sz[1]) != int(channels):
            raise _lib.SlnError(f"map size {tuple(sz)} disagrees with batch {B} / channels {int(channels)}")
    return B


_AUX_STREAMS = {}


def _aux_stream(device):
    """One side stream per device for work that runs beside the caller's stream (the backward's planning launches)."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    s = _AUX_STREAMS.get(idx)
    if s is None:
        s = _AUX_STREAMS[idx] = torch.cuda.Stream(device=idx)
    return s


# ---------------------------------------------------------------------------
# layout converters
# ---------------------------------------------------------------------------
def to_channels_last(x):
    """Any 4-D tensor -> the same logical tensor as f32 in channels_last memory (our transpose kernel)."""
    _require_cuda(x, "x")
    if x.dtype != torch.float32:
        x = x.detach().float()                # keeps the memory format: a channels_last input stays channels_last
    if is_channels_last(x):
        return x
    x = x.detach().contiguous()
    B, Cc, H, W = x.shape
    out = torch.empty((B, Cc, H, W), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    if out.numel():
        with torch.cuda.device(x.device):
            check(lib().sln_nchw_to_nhwc(ptr(x), ptr(out), B, Cc, H, W, stream_ptr()), "sln_nchw_to_nhwc")
        _lib.count_launches(1)
    return out


def to_contiguous_nchw(x):
    """Any 4-D tensor -> the same logical tensor as f32, NCHW-contiguous (channels_last input: our transpose kernel)."""
    _require_cuda(x, "x")
    if x.dtype != torch.float32:
        x = x.detach().float()
    if x.is_contiguous():
        return x
    if not is_channels_last(x):
        return x.contiguous()
    B, Cc, H, W = x.shape
    out = torch.empty((B, Cc, H, W), dtype=torch.float32, device=x.device)
    if out.numel():
        with torch.cuda.device(x.device):
            check(lib().sln_nhwc_to_nchw(ptr(x), ptr(out), B, Cc, H, W, stream_ptr()), "sln_nhwc_to_nchw")
        _lib.count_launches(1)
    return out


# 2-byte element types the crop kernels run natively (SLN_DTYPE_* codes of the *_ex entry points).  The caller asks for
# it (keep_dtype= / out_dtype=); the autograd functions do so inside an enabled CUDA autocast region only.
LOWP_DTYPES = {torch.bfloat16: _lib.DTYPE_BF16, torch.float16: _lib.DTYPE_F16}


def _b16_transpose(x, to_nhwc):
    """A 2-byte [B,C,H,W] tensor -> the same tensor, same dtype, in channels_last (to_nhwc) or NCHW-contiguous memory
    (sln_nchw_to_nhwc_b16 / sln_nhwc_to_nchw_b16: the bits move, nothing is converted)."""
    x = x.detach()
    if to_nhwc and is_channels_last(x):
        return x
    if not to_nhwc and x.is_contiguous():
        return x
    src = x.contiguous() if to_nhwc else x
    if not to_nhwc and not is_channels_last(src):
        return src.contiguous()
    B, Cc, H, W = x.shape
    out = torch.empty((B, Cc, H, W), dtype=x.dtype, device=x.device,
                      memory_format=torch.channels_last if to_nhwc else torch.contiguous_format)
    if out.numel():
        fn = lib().sln_nchw_to_nhwc_b16 if to_nhwc else lib().sln_nhwc_to_nchw_b16
        with torch.cuda.device(x.device):
            check(fn(ptr(src), ptr(out), B, Cc, H, W, stream_ptr()), "sln_nchw_to_nhwc_b16" if to_nhwc else "sln_nhwc_to_nchw_b16")
        _lib.count_launches(1)
    return out


def _aligned16(t):
    return t.data_ptr() % 16 == 0


def _bwd_native_lowp(grads, out_dtype, Cc, ph, pw):
    """True when the 2-byte backward runs natively (bulk-async kernel): grads already in out_dtype, C % 8 == 0, crops of
    at most 32 per side, and channels_last grads 16-byte aligned (other layouts are transposed into a fresh buffer)."""
    if grads.dtype != out_dtype or Cc % 8 or ph > 32 or pw > 32:
        return False
    return not is_channels_last(grads) or _aligned16(grads)


# NCHW callers (the unmodified reference: cuDNN hands out NCHW tensors unless the model was converted) on the fast path:
# the NHWC gather kernel is ~3x faster than the NCHW one at C = 256, and the same FPN map is cropped several times per
# step (classifier 7x7, mask head 14x14 / 16x16, every level call of the reference's pyramid_roi_align).  So a wide NCHW
# map is transposed ONCE (sln_nchw_to_nhwc) and the channels_last copy is remembered for as long as the source tensor is
# alive and unmodified.  The key is the identity of the tensor that owns the memory (its autograd base for views such as
# the reference's squeeze(0) / unsqueeze(0), modals.py:39-41) plus its version counter, view offset, shape and strides; the
# weak reference guarantees the memory has not been freed and handed to another tensor in between.
NHWC_CACHE_MIN_CHANNELS = 32
_nhwc_cache = {}          # key -> (weakref to the owning tensor, channels_last copy)
_NHWC_CACHE_MAX = 16


def _nhwc_cached(image, keep_dtype=False):
    """keep_dtype: a 2-byte map is remembered in its own dtype (sln_nchw_to_nhwc_b16) instead of as an f32 copy."""
    import weakref
    owner = image._base if image._base is not None else image
    key = (id(owner), owner._version, image.storage_offset(), tuple(image.shape), tuple(image.stride()), image.device.index,
           bool(keep_dtype))
    hit = _nhwc_cache.get(key)
    if hit is not None and hit[0]() is owner:
        return hit[1]
    for k in [k for k, v in _nhwc_cache.items() if v[0]() is None]:
        del _nhwc_cache[k]
    while len(_nhwc_cache) >= _NHWC_CACHE_MAX:
        del _nhwc_cache[next(iter(_nhwc_cache))]
    cl = _b16_transpose(image, True) if keep_dtype else to_channels_last(image)
    _nhwc_cache[key] = (weakref.ref(owner), cl)
    return cl


# ---------------------------------------------------------------------------
# crop_and_resize
# ---------------------------------------------------------------------------
def crop_and_resize_forward(image, boxes, box_ind, crop_height, crop_width, extrapolation_value=0.0, keep_dtype=False):
    """crops[N,C,ph,pw] = crop_and_resize(image[B,C,H,W], boxes[N,4], box_ind[N]).

    channels_last images go through the NHWC gather kernel and give channels_last crops.  NCHW images with at least
    NHWC_CACHE_MIN_CHANNELS channels (a multiple of 4) do too, through a remembered channels_last copy (see above); narrow
    NCHW images (mask targets C = 1, image crops C = 3) take the NCHW kernel and give NCHW crops.  Values are identical
    either way.  Crops are f32 whatever the image dtype, unless keep_dtype is set and the image is bf16 / fp16: then the
    crops come in the image's dtype, bit-identical to the f32 crops of image.float() rounded to it (_crop_forward_lowp)."""
    _require_cuda(image, "image")
    _require_cuda(boxes, "boxes")
    _require_cuda(box_ind, "box_ind")
    if image.dim() != 4:
        raise _lib.SlnError("image must be [B,C,H,W]")
    boxes = _f32c(boxes).view(-1, 4)
    box_ind = _i32c(box_ind).view(-1)
    N = boxes.shape[0]
    if box_ind.shape[0] != N:
        raise _lib.SlnError("box_ind and boxes disagree on N")
    B, Cc, H, W = image.shape
    if keep_dtype and image.dtype in LOWP_DTYPES:
        return _crop_forward_lowp(image, boxes, box_ind, crop_height, crop_width, extrapolation_value)
    nhwc = is_channels_last(image) and image.dtype == torch.float32
    if (not nhwc and image.dtype == torch.float32 and Cc >= NHWC_CACHE_MIN_CHANNELS and Cc % 4 == 0 and N and H * W > 1):
        image = _nhwc_cached(image)
        nhwc = True
    if nhwc:
        img = image.detach()
        out = torch.empty((N, Cc, crop_height, crop_width), dtype=torch.float32, device=image.device,
                          memory_format=torch.channels_last)
        if N and Cc and not is_channels_last(out):        # degenerate shapes: fall to NCHW kernel
            nhwc = False
    if not nhwc:
        img = _f32c(image)
        out = torch.empty((N, Cc, crop_height, crop_width), dtype=torch.float32, device=image.device)
    with torch.cuda.device(image.device):
        check(lib().sln_crop_and_resize_fwd(ptr(img), B, Cc, H, W, LAYOUT_NHWC if nhwc else LAYOUT_NCHW,
                                            ptr(boxes), ptr(box_ind), N, int(crop_height), int(crop_width),
                                            float(extrapolation_value), ptr(out), stream_ptr()),
              "sln_crop_and_resize_fwd")
    if N and Cc:
        _lib.count_launches(1)
    return out


def _crop_forward_lowp(image, boxes, box_ind, crop_height, crop_width, extrapolation_value):
    """bf16 / fp16 image -> crops of its dtype.  channels_last images and wide NCHW ones (through a remembered 2-byte
    channels_last copy) take the 2-byte NHWC gather kernel; narrow NCHW images take the f32 NCHW kernel on the widened
    image and are rounded once, which gives the same bits."""
    B, Cc, H, W = image.shape
    N = boxes.shape[0]
    img = None
    if is_channels_last(image):
        img = image.detach()
    elif Cc >= NHWC_CACHE_MIN_CHANNELS and Cc % 4 == 0 and N and H * W > 1:
        img = _nhwc_cached(image, keep_dtype=True)
    out = torch.empty((N, Cc, crop_height, crop_width), dtype=image.dtype, device=image.device,
                      memory_format=torch.channels_last)
    if img is None or (N and Cc and not is_channels_last(out)):
        return crop_and_resize_forward(image, boxes, box_ind, crop_height, crop_width, extrapolation_value).to(image.dtype)
    with torch.cuda.device(image.device):
        check(lib().sln_crop_and_resize_fwd_ex(LOWP_DTYPES[image.dtype], ptr(img), B, Cc, H, W, LAYOUT_NHWC, ptr(boxes),
                                               ptr(box_ind), N, int(crop_height), int(crop_width), float(extrapolation_value),
                                               ptr(out), stream_ptr()), "sln_crop_and_resize_fwd_ex")
    if N and Cc:
        _lib.count_launches(1)
    return out


def _prep_grads(grads):
    g = grads.detach()
    if g.dtype != torch.float32:
        g = g.float()
    cl = is_channels_last(g)
    if not cl:
        g = to_channels_last(g)
    return g, cl


def crop_and_resize_backward(grads, boxes, box_ind, image_size, channels_last_out=None, exact=None, out_dtype=torch.float32):
    """grad_image[B,C,H,W] of crop_and_resize w.r.t. the image (deterministic gather kernel).

    channels_last_out: memory format of the returned gradient (default: follow `grads`).
    exact: True -> round every term like crop_and_resize.c (bit-identical to the reference CPU
    backward); False -> fused multiply-add per term (default; see EXACT_BACKWARD).
    out_dtype: f32 (default), or bf16 / fp16: the gradient in that dtype, bit-identical to the f32 gradient of
    grads.float() rounded to it.  bf16 / fp16 grads of that dtype are read natively (C % 8 == 0, crops of at most 32
    per side, 16-byte aligned); other shapes run the f32 kernels and round."""
    _require_cuda(grads, "grads")
    if exact is None:
        exact = EXACT_BACKWARD
    flags = _lib.BWD_EXACT if exact else 0
    boxes = _f32c(boxes).view(-1, 4)
    box_ind = _i32c(box_ind).view(-1)
    B, Cc, H, W = [int(v) for v in image_size]
    N, Cg, ph, pw = grads.shape
    if Cg != Cc or boxes.shape[0] != N:
        raise _lib.SlnError("grads / boxes / image_size disagree")
    _check_rois(N, box_ind)
    lowp = out_dtype in LOWP_DTYPES
    if lowp and not _bwd_native_lowp(grads, out_dtype, Cc, ph, pw):
        return crop_and_resize_backward(grads, boxes, box_ind, image_size, channels_last_out, exact).to(out_dtype)
    if lowp:
        g_cl = is_channels_last(grads)
        g = _b16_transpose(grads, True)
    else:
        g, g_cl = _prep_grads(grads)
    if channels_last_out is None:
        channels_last_out = g_cl
    out = torch.empty((B, Cc, H, W), dtype=out_dtype if lowp else torch.float32, device=grads.device,
                      memory_format=torch.channels_last)
    with torch.cuda.device(grads.device):
        ws = _workspace(lib().sln_crop_and_resize_bwd_workspace_bytes(N, B, ph, pw), grads.device)
        if lowp:
            check(lib().sln_crop_and_resize_bwd_ex(LOWP_DTYPES[out_dtype], ptr(g), ptr(boxes), ptr(box_ind), N, Cc, ph, pw,
                                                   ptr(out), B, H, W, LAYOUT_NHWC, flags, ptr(ws), ws.numel(), stream_ptr()),
                  "sln_crop_and_resize_bwd_ex")
        else:
            check(lib().sln_crop_and_resize_bwd(ptr(g), ptr(boxes), ptr(box_ind), N, Cc, ph, pw, ptr(out), B, H, W,
                                                LAYOUT_NHWC, flags, ptr(ws), ws.numel(), stream_ptr()),
                  "sln_crop_and_resize_bwd")
    if out.numel():
        _lib.count_launches(4 if N else 1)
    if not channels_last_out:
        out = _b16_transpose(out, False) if lowp else to_contiguous_nchw(out)
    return out


class BackwardPlan:
    """The backward's ROI lists for one (boxes, box_ind, level, map sizes, channels, pool) -- they do not depend on the
    gradients, so they can be built while the forward of the same ROIs runs.  Holds the workspace and the event that marks
    the lists ready; valid while boxes / box_ind / level are unchanged."""

    def __init__(self, ws, event, key):
        self.ws, self.event, self.key = ws, event, key


def _plan_key(boxes, box_ind, level, map_sizes, Cc, ph, pw):
    return (boxes.data_ptr(), boxes._version, boxes.dtype, box_ind.data_ptr(), box_ind._version, box_ind.dtype,
            level.data_ptr(), level._version, level.dtype, int(boxes.numel()),
            tuple(tuple(int(v) for v in sz) for sz in map_sizes), int(Cc), int(ph), int(pw))


def pyramid_crop_backward_plan(boxes, box_ind, level, map_sizes, channels, crop_height, crop_width, stream=None):
    """Build the lists of pyramid_crop_backward ahead of time (sln_pyramid_crop_bwd with SLN_BWD_PLAN_ONLY) on `stream`
    (default: this module's side stream, forked from the current stream) and return a BackwardPlan to pass as `plan=`.
    Three small latency-bound launches that then run BESIDE the bandwidth-bound forward instead of in front of the
    backward's main kernel."""
    _require_cuda(boxes, "boxes")
    ph, pw = int(crop_height), int(crop_width)
    # keyed on the CALLER's tensors (storage + version counter): an in-place change of any of them invalidates the plan
    key = _plan_key(boxes, box_ind, level, map_sizes, channels, ph, pw)
    boxes = _f32c(boxes).view(-1, 4)
    box_ind = _i32c(box_ind).view(-1)
    level = _i32c(level).view(-1)
    N = boxes.shape[0]
    _check_rois(N, box_ind, level)
    nl = len(map_sizes)
    B = _check_map_sizes(map_sizes, channels)
    dev = boxes.device
    cur = torch.cuda.current_stream(dev)
    side = stream if stream is not None else _aux_stream(dev)
    with torch.cuda.device(dev):
        ws = _workspace(lib().sln_pyramid_crop_bwd_workspace_bytes(N, B, nl, ph, pw), dev)     # allocated on the current stream
        mp = (C.c_void_p * nl)(*[ws.data_ptr()] * nl)             # plausible (non-null) addresses: nothing is accessed through them
        hs = (C.c_int * nl)(*[int(sz[2]) for sz in map_sizes])
        ws_ = (C.c_int * nl)(*[int(sz[3]) for sz in map_sizes])
        for t in (ws, boxes, box_ind, level):       # read / written on the side stream: a tensor dropped right after this
            t.record_stream(side)                   # call must not hand its block back before the plan launches are done
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            check(lib().sln_pyramid_crop_bwd(None, ptr(boxes), ptr(box_ind), ptr(level), N, int(channels), ph, pw, mp, hs, ws_, nl,
                                             B, _lib.BWD_PLAN_ONLY, ptr(ws), ws.numel(), C.c_void_p(side.cuda_stream)),
                  "sln_pyramid_crop_bwd(plan)")
            ev = torch.cuda.Event()
            ev.record(side)
    if N:
        _lib.count_launches(3)
    return BackwardPlan(ws, ev, key)


def pyramid_crop_backward(grads, boxes, box_ind, level, map_sizes, channels_last_out=None, exact=None, plan=None,
                          out_dtype=torch.float32):
    """Backward of pyramid_crop_forward for all levels in one call.  map_sizes: list of (B,C,H_l,W_l).
    Returns the list of grad maps (channels_last unless channels_last_out[l] is False).
    plan: a BackwardPlan from pyramid_crop_backward_plan for the same ROIs (ignored when it does not match); a plan does
    not depend on the dtype.  out_dtype: as in crop_and_resize_backward."""
    _require_cuda(grads, "grads")
    if exact is None:
        exact = EXACT_BACKWARD
    flags = _lib.BWD_EXACT if exact else 0
    key_src = (boxes, box_ind, level)                    # the caller's tensors (the conversions below may copy)
    boxes = _f32c(boxes).view(-1, 4)
    box_ind = _i32c(box_ind).view(-1)
    level = _i32c(level).view(-1)
    N, Cc, ph, pw = grads.shape
    if boxes.shape[0] != N:
        raise _lib.SlnError(f"grads hold {N} crops for {boxes.shape[0]} boxes")
    _check_rois(N, box_ind, level)
    nl = len(map_sizes)
    B = _check_map_sizes(map_sizes, Cc)
    lowp = out_dtype in LOWP_DTYPES
    if lowp and not _bwd_native_lowp(grads, out_dtype, Cc, ph, pw):
        return [o.to(out_dtype) for o in pyramid_crop_backward(grads, *key_src, map_sizes, channels_last_out, exact, plan)]
    g = _b16_transpose(grads, True) if lowp else _prep_grads(grads)[0]
    outs = [torch.empty(tuple(int(v) for v in sz), dtype=out_dtype if lowp else torch.float32, device=grads.device,
                        memory_format=torch.channels_last) for sz in map_sizes]
    mp = (C.c_void_p * nl)(*[o.data_ptr() for o in outs])
    hs = (C.c_int * nl)(*[int(sz[2]) for sz in map_sizes])
    ws_ = (C.c_int * nl)(*[int(sz[3]) for sz in map_sizes])
    planned = plan is not None and plan.key == _plan_key(*key_src, map_sizes, Cc, ph, pw)
    with torch.cuda.device(grads.device):
        if planned:
            torch.cuda.current_stream(grads.device).wait_event(plan.event)
            ws = plan.ws
            flags |= _lib.BWD_PLANNED
        else:
            ws = _workspace(lib().sln_pyramid_crop_bwd_workspace_bytes(N, B, nl, ph, pw), grads.device)
        if lowp:
            check(lib().sln_pyramid_crop_bwd_ex(LOWP_DTYPES[out_dtype], ptr(g), ptr(boxes), ptr(box_ind), ptr(level), N, Cc,
                                                ph, pw, mp, hs, ws_, nl, B, flags, ptr(ws), ws.numel(), stream_ptr()),
                  "sln_pyramid_crop_bwd_ex")
        else:
            check(lib().sln_pyramid_crop_bwd(ptr(g), ptr(boxes), ptr(box_ind), ptr(level), N, Cc, ph, pw, mp, hs, ws_, nl, B,
                                             flags, ptr(ws), ws.numel(), stream_ptr()), "sln_pyramid_crop_bwd")
    _lib.count_launches((2 if planned else 4) if N else 1)
    if channels_last_out is not None:
        outs = [o if cl else (_b16_transpose(o, False) if lowp else to_contiguous_nchw(o))
                for o, cl in zip(outs, channels_last_out)]
    return outs


def pyramid_crop_forward(feature_maps, boxes, box_ind, level, crop_height, crop_width, extrapolation_value=0.0,
                         keep_dtype=False):
    """One launch for all FPN levels: feature_maps = list of channels_last [B,C,H_l,W_l] tensors,
    level[i] in [0, len(feature_maps)) names the source map of ROI i.  Output channels_last
    [N,C,ph,pw] in the original ROI order.  Maps of another dtype are cropped from their f32 values, into f32 crops --
    unless keep_dtype is set and every map is bf16, or every map fp16: then the 2-byte kernel writes crops of that dtype,
    bit-identical to the f32 crops rounded to it (NCHW maps are transposed once and remembered, in their dtype)."""
    for m in feature_maps:
        _require_cuda(m, "feature map")
        if m.dim() != 4:
            raise _lib.SlnError("feature maps must be [B,C,H_l,W_l]")
    boxes = _f32c(boxes).view(-1, 4)
    box_ind = _i32c(box_ind).view(-1)
    level = _i32c(level).view(-1)
    N = boxes.shape[0]
    _check_rois(N, box_ind, level)
    B, Cc = feature_maps[0].shape[0], feature_maps[0].shape[1]
    for m in feature_maps:
        if m.shape[0] != B or m.shape[1] != Cc:
            raise _lib.SlnError("feature maps disagree on batch / channels")
    dt = feature_maps[0].dtype
    lowp = keep_dtype and dt in LOWP_DTYPES and all(m.dtype == dt for m in feature_maps)
    maps = []
    for m in feature_maps:
        if lowp:
            maps.append(m.detach() if is_channels_last(m) else _nhwc_cached(m, keep_dtype=True))
        elif is_channels_last(m) and m.dtype == torch.float32:
            maps.append(m.detach())
        elif m.dtype == torch.float32:
            maps.append(_nhwc_cached(m))                 # NCHW map: transposed once, remembered while the tensor lives
        else:
            maps.append(to_channels_last(m))
    nl = len(maps)
    out = torch.empty((N, Cc, crop_height, crop_width), dtype=dt if lowp else torch.float32, device=boxes.device,
                      memory_format=torch.channels_last)
    mp = (C.c_void_p * nl)(*[m.data_ptr() for m in maps])
    hs = (C.c_int * nl)(*[m.shape[2] for m in maps])
    ws_ = (C.c_int * nl)(*[m.shape[3] for m in maps])
    with torch.cuda.device(boxes.device):
        if lowp:
            check(lib().sln_pyramid_crop_fwd_ex(LOWP_DTYPES[dt], mp, hs, ws_, nl, B, Cc, ptr(boxes), ptr(box_ind), ptr(level),
                                                N, int(crop_height), int(crop_width), float(extrapolation_value), ptr(out),
                                                stream_ptr()), "sln_pyramid_crop_fwd_ex")
        else:
            check(lib().sln_pyramid_crop_fwd(mp, hs, ws_, nl, B, Cc, ptr(boxes), ptr(box_ind), ptr(level), N,
                                             int(crop_height), int(crop_width), float(extrapolation_value), ptr(out),
                                             stream_ptr()), "sln_pyramid_crop_fwd")
    if N and Cc:
        _lib.count_launches(1)
    return out


def roi_levels_device(boxes, image_hw):
    """FPN level index (0..3 for P2..P5) of each ROI, modals.py:53-64, in one launch.  boxes [N,4] normalised (CUDA)."""
    _require_cuda(boxes, "boxes")
    boxes = _f32c(boxes).view(-1, 4)
    N = boxes.shape[0]
    out = torch.empty(N, dtype=torch.int32, device=boxes.device)
    if N:
        with torch.cuda.device(boxes.device):
            check(lib().sln_roi_levels(ptr(boxes), N, int(image_hw[0]), int(image_hw[1]), ptr(out), stream_ptr()),
                  "sln_roi_levels")
        _lib.count_launches(1)
    return out


# ---------------------------------------------------------------------------
# NMS
# ---------------------------------------------------------------------------
def nms_device(dets, thresh, class_ids=None, max_keep=0, dense_only=False, return_path=False, sparse_only=False):
    """Greedy NMS fully on the device.  Returns (keep int64[n] padded, num_keep int32[1]) -- both
    device tensors, no host sync.  keep[:num_keep] are indices into dets, score-descending.
    dense_only forces the dense bit-matrix pipeline; return_path appends a device int32[1] that is 1 when
    the sparse (binned) pipeline produced the result (include/sln_b200.h, sln_nms_ex).
    sparse_only launches the sparse pipeline alone: num_keep < 0 then means "outside its contract, call again with
    dense_only=True" (what `nms()` does, which reads num_keep on the host anyway)."""
    _require_cuda(dets, "dets")
    dets = _f32c(dets)
    if dets.dim() != 2 or dets.shape[1] != 5:
        raise _lib.SlnError("dets must be [n,5] (y1,x1,y2,x2,score)")
    n = dets.shape[0]
    cls = None
    if class_ids is not None:
        cls = _i32c(class_ids).view(-1)
        if cls.shape[0] != n:
            raise _lib.SlnError("class_ids and dets disagree on n")
    keep = torch.empty(max(n, 1), dtype=torch.int64, device=dets.device)
    num = torch.empty(1, dtype=torch.int32, device=dets.device)
    with torch.cuda.device(dets.device):
        ws = _workspace(lib().sln_nms_workspace_bytes(n), dets.device)
        path = torch.zeros(1, dtype=torch.int32, device=dets.device) if return_path else None
        check(lib().sln_nms_ex(ptr(dets), ptr(cls), n, float(thresh), int(max_keep), (1 if dense_only else 0) | (2 if sparse_only else 0),
                               ptr(keep), ptr(num), ptr(path), ptr(ws), ws.numel(), stream_ptr()), "sln_nms_ex")
    if n:
        _lib.count_launches(4)
    if return_path:
        return keep, num, path
    return keep, num


def _dense_nms_launches(n):
    """Kernels of nms.cu's dense pipeline for n > 0 boxes: mask + scan, the fixed-point resolve from 160 words, and from
    16384 boxes two stages (stage A's mask + scan, suppress, compact, emit, then stage B)."""
    if n < 16384:
        return 2 + (((n + 63) // 64) >= 160)
    return 2 + 3 + 2 + (((n - 1024 + 63) // 64) >= 160)


def nms_batched_device(dets, thresh, class_ids=None, max_keep=0, dense_only=False, return_path=False):
    """B independent greedy NMS problems in one call (sln_nms_batched).  dets [B,n,5], class_ids integer [B,n] or None.
    Returns (keep int64 [B,mk], num_keep int32 [B]) on the device, mk = max_keep if 0 < max_keep <= n else n, plus a
    device int32 [B] path report with return_path.  keep[b, :num_keep[b]] and num_keep[b] are nms_device's for problem b
    alone; entries beyond num_keep[b] are undefined.  No host sync; graph capturable."""
    _require_cuda(dets, "dets")
    if dets.dim() != 3 or dets.shape[2] != 5:
        raise _lib.SlnError(f"dets must be [B,n,5] (y1,x1,y2,x2,score), got {tuple(dets.shape)}")
    if not dets.dtype.is_floating_point:
        raise _lib.SlnError(f"dets must be floating point, got {dets.dtype}")
    B, n = int(dets.shape[0]), int(dets.shape[1])
    if B > 65535:
        raise _lib.SlnError(f"B={B} problems in one call (at most 65535)")
    if int(max_keep) < 0:
        raise _lib.SlnError(f"max_keep must be >= 0 (0: all), got {max_keep}")
    if class_ids is not None:
        _require_cuda(class_ids, "class_ids")
        if tuple(class_ids.shape) != (B, n):
            raise _lib.SlnError(f"class_ids {tuple(class_ids.shape)} disagrees with dets {tuple(dets.shape)}")
        if class_ids.dtype.is_floating_point or class_ids.dtype == torch.bool:
            raise _lib.SlnError(f"class_ids must be an integer tensor, got {class_ids.dtype}")
    dets = _f32c(dets)
    cls = _i32c(class_ids) if class_ids is not None else None
    mk = n if int(max_keep) == 0 or int(max_keep) > n else int(max_keep)
    keep = torch.empty((B, mk), dtype=torch.int64, device=dets.device)
    num = torch.empty(B, dtype=torch.int32, device=dets.device)
    path = torch.empty(B, dtype=torch.int32, device=dets.device) if return_path else None
    with torch.cuda.device(dets.device):
        ws = _workspace(lib().sln_nms_batched_workspace_bytes(B, n), dets.device)
        check(lib().sln_nms_batched(ptr(dets), ptr(cls), B, n, float(thresh), int(max_keep), 1 if dense_only else 0,
                                    ptr(keep), ptr(num), ptr(path), ptr(ws), ws.numel(), stream_ptr()), "sln_nms_batched")
    if B:
        sparse = n > 0 and not dense_only and 65 <= n <= 65535 and float(thresh) >= 0.05
        launches = 2 + 3 * sparse + B * _dense_nms_launches(n) if n else 1      # rank memset + rank; bin, pairs, resolve
        if return_path:
            launches += 1 + sparse                                              # path memset (+ the status copy)
        _lib.count_launches(launches)
    if return_path:
        return keep, num, path
    return keep, num


def refine_decode_device(rois, probs, deltas, std_dev, image_hw, window, min_confidence=0.0):
    """Elementwise front of refine_detections in one launch (include/sln_b200.h, sln_refine_decode).
    Returns (dets [N,5], cls_nms int32[N], class_ids int32[N], n_excluded int32[1]) on the device."""
    _require_cuda(rois, "rois")
    rois = _f32c(rois).view(-1, 4)
    probs = _f32c(probs)
    deltas = _f32c(deltas)
    N, K = probs.shape
    if rois.shape[0] != N or deltas.shape[0] != N or deltas.shape[1] != K:
        raise _lib.SlnError("rois / probs / deltas disagree")
    dev = rois.device
    dets = torch.empty((N, 5), dtype=torch.float32, device=dev)
    cls_nms = torch.empty(N, dtype=torch.int32, device=dev)
    class_ids = torch.empty(N, dtype=torch.int32, device=dev)
    n_excl = torch.empty(1, dtype=torch.int32, device=dev)
    sd = (C.c_float * 4)(*[float(v) for v in std_dev])
    win = (C.c_float * 4)(*[float(v) for v in window])
    with torch.cuda.device(dev):
        check(lib().sln_refine_decode(ptr(rois), ptr(probs), ptr(deltas), N, K, sd, float(image_hw[0]), float(image_hw[1]),
                                      win, float(min_confidence), ptr(dets), ptr(cls_nms), ptr(class_ids), ptr(n_excl),
                                      stream_ptr()), "sln_refine_decode")
    if N:
        _lib.count_launches(1)
    return dets, cls_nms, class_ids, n_excl


def refine_topk_device(dets, class_ids, max_keep=100):
    """Top `max_keep` non-background ROIs by score, in descending score order (include/sln_b200.h, sln_refine_topk).
    Returns (result f32 [max_keep,6], keep int64 [max_keep]); only the first min(max_keep, #kept) rows are written."""
    _require_cuda(dets, "dets")
    N = dets.shape[0]
    result = torch.empty((int(max_keep), 6), dtype=torch.float32, device=dets.device)
    keep = torch.empty(int(max_keep), dtype=torch.int64, device=dets.device)
    if N and max_keep:
        with torch.cuda.device(dets.device):
            check(lib().sln_refine_topk(ptr(dets), ptr(class_ids), N, int(max_keep), ptr(result), ptr(keep), stream_ptr()),
                  "sln_refine_topk")
        _lib.count_launches(1)
    return result, keep


def refine_topk_batched_device(dets, class_ids, max_keep=100):
    """refine_topk_device for B images in one launch (sln_refine_topk_batched).  dets [B,N,5], class_ids int32 [B,N]
    (sln_refine_decode's outputs of the flattened [B*N] rows, viewed per image).  Returns (result f32 [B,max_keep,6],
    keep int64 [B,max_keep] row indices within the image, num_det int32 [B] = min(max_keep, kept rows of the image));
    only the first num_det[b] rows of image b are written."""
    _require_cuda(dets, "dets")
    _require_cuda(class_ids, "class_ids")
    if dets.dim() != 3 or dets.shape[2] != 5:
        raise _lib.SlnError(f"dets must be [B,N,5], got {tuple(dets.shape)}")
    B, N = int(dets.shape[0]), int(dets.shape[1])
    if tuple(class_ids.shape) != (B, N):
        raise _lib.SlnError(f"class_ids {tuple(class_ids.shape)} disagrees with dets {tuple(dets.shape)}")
    if int(max_keep) < 0:
        raise _lib.SlnError(f"max_keep must be >= 0, got {max_keep}")
    dets, class_ids = _f32c(dets), _i32c(class_ids)
    result = torch.empty((B, int(max_keep), 6), dtype=torch.float32, device=dets.device)
    keep = torch.empty((B, int(max_keep)), dtype=torch.int64, device=dets.device)
    num_det = torch.empty(B, dtype=torch.int32, device=dets.device)
    if B:
        with torch.cuda.device(dets.device):
            check(lib().sln_refine_topk_batched(ptr(dets), ptr(class_ids), B, N, int(max_keep), ptr(result), ptr(keep),
                                                ptr(num_det), stream_ptr()), "sln_refine_topk_batched")
        _lib.count_launches(2 if N and max_keep else 1)
    return result, keep, num_det


def refine_nms_emit_batched_device(dets, class_ids, nms_keep, nms_num, max_detections):
    """The per-class NMS branch's last step for B images (sln_refine_nms_emit_batched).  dets [B,N,5] and class_ids int32
    [B,N] are sln_refine_decode's outputs viewed per image; nms_keep [B,mk] / nms_num [B] are nms_batched_device's on
    (dets, cls_nms) with max_keep = max_detections.  Returns (result f32 [B,D,6], keep int64 [B,D], num_det int32 [B]),
    zero beyond num_det[b] = min(D, survivors with a finite score)."""
    _require_cuda(dets, "dets")
    if dets.dim() != 3 or dets.shape[2] != 5:
        raise _lib.SlnError(f"dets must be [B,N,5], got {tuple(dets.shape)}")
    B, N, D = int(dets.shape[0]), int(dets.shape[1]), int(max_detections)
    if D < 0:
        raise _lib.SlnError(f"max_detections must be >= 0, got {max_detections}")
    if tuple(class_ids.shape) != (B, N):
        raise _lib.SlnError(f"class_ids {tuple(class_ids.shape)} disagrees with dets {tuple(dets.shape)}")
    if nms_keep.dim() != 2 or int(nms_keep.shape[0]) != B or int(nms_keep.shape[1]) > N or tuple(nms_num.shape) != (B,):
        raise _lib.SlnError(f"nms keep {tuple(nms_keep.shape)} / num {tuple(nms_num.shape)} disagree with dets {tuple(dets.shape)}")
    if nms_keep.dtype != torch.int64 or nms_num.dtype != torch.int32:
        raise _lib.SlnError("nms keep must be int64 and num int32 (nms_batched_device's outputs)")
    dets, class_ids = _f32c(dets), _i32c(class_ids)
    nms_keep, nms_num = nms_keep.contiguous(), nms_num.contiguous()
    result = torch.empty((B, D, 6), dtype=torch.float32, device=dets.device)
    keep = torch.empty((B, D), dtype=torch.int64, device=dets.device)
    num_det = torch.empty(B, dtype=torch.int32, device=dets.device)
    if B:
        with torch.cuda.device(dets.device):
            check(lib().sln_refine_nms_emit_batched(ptr(dets), ptr(class_ids), B, N, ptr(nms_keep), ptr(nms_num),
                                                    int(nms_keep.shape[1]), D, ptr(result), ptr(keep), ptr(num_det),
                                                    stream_ptr()), "sln_refine_nms_emit_batched")
        _lib.count_launches(1)
    return result, keep, num_det


UNMOLD_BATCH_MAX = 512          # images per sln_unmold_rle_batched call (their sizes and windows travel as kernel parameters)


def unmold_scale_shift(image_shape, window):
    """model.py:774-779 for one image: (h_scale, w_scale, window[0], window[1]) as Python floats, computed with the
    reference's own expressions.  The device runs the box arithmetic in float64, which is what numpy does for integer
    and float64 windows; a float32 / float16 window would make numpy round in that type, and is refused."""
    if isinstance(window, torch.Tensor):
        window = window.detach().cpu().numpy()
    h_scale = image_shape[0] / (window[2] - window[0])
    w_scale = image_shape[1] / (window[3] - window[1])
    shift = window[:2]
    scales = np.array([h_scale, w_scale, h_scale, w_scale])
    shifts = np.array([shift[0], shift[1], shift[0], shift[1]])
    if np.result_type(np.float32, shifts.dtype, scales.dtype) != np.float64:
        raise _lib.SlnError(f"window {window!r}: the box arithmetic would run in "
                            f"{np.result_type(np.float32, shifts.dtype, scales.dtype)}, not float64 (pass integer or float64 windows)")
    return float(scales[0]), float(scales[1]), float(shifts[0]), float(shifts[1])


# Outputs of unmold_rle_batched_device, all on the device.  boxes int32 [B,D,4], class_ids int32 [B,D], scores f32 [B,D],
# src_row int32 [B,D], m int32 [B,D], str_off int32 [B,D], str_len int32 [B,D], num_kept int32 [B] and str_total int32
# [1] are views of one int32 buffer `meta` (one copy brings them all to the host); strings u8 holds the packed strings.
UnmoldRle = collections.namedtuple("UnmoldRle", "boxes class_ids scores src_row m str_off str_len num_kept str_total "
                                                "strings meta")


def unmold_meta_views(meta, B, D):
    """Split the int32 metadata buffer of unmold_rle_batched_device (device tensor or its host copy) into its fields:
    boxes [B,D,4], class_ids, scores (f32), src_row, m, str_off, str_len [B,D], num_kept [B], str_total [1]."""
    n, o, out = B * D, 0, []
    for size, shape in ((4 * n, (B, D, 4)), (n, (B, D)), (n, (B, D)), (n, (B, D)), (n, (B, D)), (n, (B, D)), (n, (B, D)),
                        (B, (B,)), (1, (1,))):
        out.append(meta[o:o + size].reshape(shape))
        o += size
    out[2] = out[2].view(torch.float32) if isinstance(out[2], torch.Tensor) else out[2].view(np.float32)
    return out


def unmold_rle_batched_device(detections, mrcnn_mask, image_shapes, windows, cap=None, workspace=None):
    """unmold_detections + COCO RLE for B images in one sync-free device pass (sln_unmold_rle_batched, five launches).
    detections f32 [B,D,6] and mrcnn_mask f32 [B,D,h,w,K] (any strides) on the device; image_shapes and windows: B host
    values each.  cap: most runs per mask (default 2 * max W + 1: a mask whose every column holds one stretch of ones has
    at most two changes per column); a mask with more gets m = -runs and no string.  workspace: a u8 CUDA tensor of at
    least sln_unmold_rle_batched_workspace_bytes (allocated when None).  Returns an UnmoldRle of device tensors."""
    _require_cuda(detections, "detections")
    _require_cuda(mrcnn_mask, "mrcnn_mask")
    if detections.dim() != 3 or detections.shape[2] != 6 or detections.dtype != torch.float32:
        raise _lib.SlnError(f"detections must be f32 [B,D,6], got {detections.dtype} {tuple(detections.shape)}")
    if mrcnn_mask.dim() != 5 or mrcnn_mask.dtype != torch.float32:
        raise _lib.SlnError(f"mrcnn_mask must be f32 [B,D,h,w,K], got {mrcnn_mask.dtype} {tuple(mrcnn_mask.shape)}")
    B, D = int(detections.shape[0]), int(detections.shape[1])
    if tuple(mrcnn_mask.shape[:2]) != (B, D):
        raise _lib.SlnError(f"mrcnn_mask {tuple(mrcnn_mask.shape)} disagrees with detections {tuple(detections.shape)}")
    if len(image_shapes) != B or len(windows) != B:
        raise _lib.SlnError(f"{len(image_shapes)} image shapes and {len(windows)} windows for B = {B} images")
    if B > UNMOLD_BATCH_MAX:
        raise _lib.SlnError(f"B = {B} images in one call (at most {UNMOLD_BATCH_MAX})")
    mh, mw, K = (int(v) for v in mrcnn_mask.shape[2:])
    if not (1 <= mh <= 256 and 1 <= mw <= 256 and K >= 1):
        raise _lib.SlnError(f"mask [h, w, K] = {(mh, mw, K)}: h, w in [1, 256] and K >= 1")
    Hs = [int(s[0]) for s in image_shapes]
    Ws = [int(s[1]) for s in image_shapes]
    if any(not (1 <= v <= 65535) for v in Hs + Ws):
        raise _lib.SlnError(f"image sides must be in [1, 65535], got {list(zip(Hs, Ws))}")
    ss = [unmold_scale_shift(image_shapes[b], windows[b]) for b in range(B)]
    cap = 2 * max(Ws, default=1) + 1 if cap is None else int(cap)
    n = B * D
    if cap < 1 or 7 * cap * n >= 1 << 31:
        raise _lib.SlnError(f"cap = {cap} for {n} masks: need cap >= 1 and 7 * cap * B * D < 2^31")
    dev = detections.device
    det = detections.detach().contiguous()
    mask = mrcnn_mask.detach()
    meta = torch.empty(10 * n + B + 1, dtype=torch.int32, device=dev)
    strings = torch.empty(max(7 * cap * n, 1), dtype=torch.uint8, device=dev)
    views = unmold_meta_views(meta, B, D)
    boxes, cls, scores, src, m, off, slen, num_kept, total = views
    Ha, Wa = (C.c_int * max(B, 1))(*Hs), (C.c_int * max(B, 1))(*Ws)
    sa = (C.c_double * max(4 * B, 1))(*[v for t in ss for v in t])
    st = (C.c_longlong * 5)(*[int(v) for v in mask.stride()])
    with torch.cuda.device(dev):
        need = lib().sln_unmold_rle_batched_workspace_bytes(B, D, Ha, Wa, cap)
        if workspace is None:
            workspace = _workspace(need, dev)
        elif workspace.numel() < need or not workspace.is_cuda:
            raise _lib.SlnError(f"workspace: need {need} bytes on the device, got {workspace.numel()}")
        check(lib().sln_unmold_rle_batched(ptr(det), B, D, ptr(mask), mh, mw, K, st, Ha, Wa, sa, cap, ptr(boxes), ptr(cls),
                                           ptr(scores), ptr(src), ptr(num_kept), ptr(m), ptr(off), ptr(slen), ptr(total),
                                           ptr(strings), strings.numel(), ptr(workspace), workspace.numel(), stream_ptr()),
              "sln_unmold_rle_batched")
    if B and D:
        _lib.count_launches(5)      # box prep, box-local paste, runs, string scan, string write
    return UnmoldRle(*views, strings, meta)


def rle_strings_device(counts, m):
    """The device string coder (sln_rle_strings): counts u32-as-int32 [n, cap] and m int32 [n] (the outputs of
    rle.rle_counts_device) -> (strings u8, str_off int32 [n], str_len int32 [n], str_total int32 [1]).  List i's
    rleToString string is strings[str_off[i] : str_off[i] + str_len[i]]; lists with m[i] <= 0 or > cap get none."""
    _require_cuda(counts, "counts")
    _require_cuda(m, "m")
    if counts.dim() != 2 or counts.dtype not in (torch.int32, torch.uint32) or m.dtype != torch.int32 or \
            tuple(m.shape) != (counts.shape[0],):
        raise _lib.SlnError(f"counts must be 32-bit [n, cap] and m int32 [n], got {tuple(counts.shape)} / {tuple(m.shape)}")
    n, cap = int(counts.shape[0]), int(counts.shape[1])
    if cap < 1 or 7 * cap * n >= 1 << 31:
        raise _lib.SlnError(f"counts [{n}, {cap}]: need cap >= 1 and 7 * cap * n < 2^31")
    counts, m = counts.contiguous(), m.contiguous()
    dev = counts.device
    strings = torch.empty(max(7 * cap * n, 1), dtype=torch.uint8, device=dev)
    off = torch.empty(n, dtype=torch.int32, device=dev)
    slen = torch.empty(n, dtype=torch.int32, device=dev)
    total = torch.empty(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        check(lib().sln_rle_strings(ptr(counts), n, cap, ptr(m), ptr(off), ptr(slen), ptr(total), ptr(strings),
                                    strings.numel(), stream_ptr()), "sln_rle_strings")
    if n:
        _lib.count_launches(3)
    return strings, off, slen, total


def bbox_overlaps_device(boxes1, boxes2, matrix=True, reduce=False):
    """IoU of boxes1 [N,4] against boxes2 [G,4] (include/sln_b200.h, sln_bbox_overlaps).
    Returns the [N,G] matrix, or (matrix | None, iou_max [N], argmax int32 [N]) with reduce=True."""
    _require_cuda(boxes1, "boxes1")
    b1 = _f32c(boxes1).view(-1, 4)
    b2 = _f32c(boxes2).view(-1, 4).to(b1.device)
    N, G = b1.shape[0], b2.shape[0]
    ov = torch.empty((N, G), dtype=torch.float32, device=b1.device) if matrix else None
    mx = torch.empty(N, dtype=torch.float32, device=b1.device) if reduce else None
    am = torch.empty(N, dtype=torch.int32, device=b1.device) if reduce else None
    if N:
        with torch.cuda.device(b1.device):
            check(lib().sln_bbox_overlaps(ptr(b1), N, ptr(b2), G, ptr(ov), ptr(mx), ptr(am), stream_ptr()), "sln_bbox_overlaps")
        _lib.count_launches(1)
    return (ov, mx, am) if reduce else ov


def box_refinement_device(box, gt_box, std_dev=None):
    """utils.box_refinement for M box pairs, optionally divided by std_dev (sln_box_refinement)."""
    _require_cuda(box, "box")
    b = _f32c(box).view(-1, 4)
    g = _f32c(gt_box).view(-1, 4)
    if g.shape != b.shape:
        raise _lib.SlnError("box and gt_box disagree")
    out = torch.empty_like(b)
    sd = (C.c_float * 4)(*[float(v) for v in std_dev]) if std_dev is not None else None
    if b.shape[0]:
        with torch.cuda.device(b.device):
            check(lib().sln_box_refinement(ptr(b), ptr(g), b.shape[0], sd, ptr(out), stream_ptr()), "sln_box_refinement")
        _lib.count_launches(1)
    return out


def mask_targets_device(gt_masks, assignment, boxes, mh, mw):
    """round(crop_and_resize(gt_masks[l, assignment[p]], boxes[p])) for every layer l and positive ROI p, straight from
    u8 / bool masks [L,G,H,W] (sln_mask_targets).  Returns f32 [P,L,mh,mw]."""
    _require_cuda(gt_masks, "gt_masks")
    if gt_masks.dtype == torch.bool:
        gt_masks = gt_masks.view(torch.uint8)
    if gt_masks.dtype != torch.uint8 or gt_masks.dim() != 4:
        raise _lib.SlnError("gt_masks must be uint8 / bool [L,G,H,W]")
    gt_masks = gt_masks.contiguous()
    L, G, H, W = gt_masks.shape
    boxes = _f32c(boxes).view(-1, 4)
    assignment = _i32c(assignment).view(-1)
    P = boxes.shape[0]
    if assignment.shape[0] != P:
        raise _lib.SlnError(f"assignment has {assignment.shape[0]} entries for {P} boxes")
    out = torch.empty((P, L, int(mh), int(mw)), dtype=torch.float32, device=gt_masks.device)
    if out.numel():
        with torch.cuda.device(gt_masks.device):
            check(lib().sln_mask_targets(ptr(gt_masks), L, G, H, W, ptr(assignment), ptr(boxes), P, int(mh), int(mw), ptr(out),
                                         stream_ptr()), "sln_mask_targets")
        _lib.count_launches(1)
    return out


TARGET_BATCH_MAX = 512          # images per batched detection-target call (their GT counts travel as kernel parameters)


def target_num_gt(num_gt, B, G):
    """num_gt of the batched detection targets as B host ints in [0, G] (None: G for every image)."""
    if num_gt is None:
        return [G] * B
    if isinstance(num_gt, torch.Tensor):
        if num_gt.is_cuda:
            raise _lib.SlnError("num_gt must be host ints (a device tensor would need a sync to read)")
        num_gt = num_gt.tolist()
    num_gt = [int(v) for v in num_gt]
    if len(num_gt) != B:
        raise _lib.SlnError(f"num_gt has {len(num_gt)} entries for B = {B} images")
    if any(not (0 <= v <= G) for v in num_gt):
        raise _lib.SlnError(f"num_gt {num_gt} outside [0, G = {G}]")
    return num_gt


def target_mask_planes(gt_masks, B, G, num_gt, device):
    """The GT masks of the batched detection targets: one u8 / bool tensor [B,L,G,H,W] or a list of B tensors
    [L,G_b,H,W] with G_b == num_gt[b], on `device`.  Returns (planes: B contiguous u8 tensors [L,G_b,H,W], their G_b,
    (L, H, W)).  Nothing is stacked or copied, except an entry that is not contiguous."""
    if isinstance(gt_masks, torch.Tensor):
        _require_cuda(gt_masks, "gt_masks")
        if gt_masks.dim() != 5 or int(gt_masks.shape[0]) != B or int(gt_masks.shape[2]) != G:
            raise _lib.SlnError(f"gt_masks must be [B={B},L,G={G},H,W] or a list of B tensors [L,G_b,H,W], "
                                f"got {tuple(gt_masks.shape)}")
        entries = [gt_masks[b] for b in range(B)]
        gs = [int(gt_masks.shape[2])] * B
    else:
        entries = list(gt_masks)
        if len(entries) != B:
            raise _lib.SlnError(f"gt_masks has {len(entries)} entries for B = {B} images")
        for b, m in enumerate(entries):
            if not isinstance(m, torch.Tensor) or m.dim() != 4:
                raise _lib.SlnError(f"gt_masks[{b}] must be a tensor [L,G_b,H,W]")
        gs = [int(m.shape[1]) for m in entries]
        if gs != list(num_gt):
            raise _lib.SlnError(f"gt_masks entries have G_b = {gs}, num_gt is {list(num_gt)}")
    planes = []
    for b, m in enumerate(entries):
        _require_cuda(m, f"gt_masks[{b}]")
        if m.dtype not in (torch.uint8, torch.bool):
            raise _lib.SlnError(f"gt_masks must be uint8 / bool, got {m.dtype}")
        if m.device != device:
            raise _lib.SlnError(f"gt_masks[{b}] is on {m.device}, the proposals on {device}")
        planes.append((m.view(torch.uint8) if m.dtype == torch.bool else m).contiguous())
    lhw = {(int(m.shape[0]), int(m.shape[2]), int(m.shape[3])) for m in planes}
    if len(lhw) > 1:
        raise _lib.SlnError(f"every image needs the same L, H, W of its masks, got {sorted(lhw)}")
    L, H, W = lhw.pop() if lhw else (0, 1, 1)
    if not (1 <= H <= 32767 and 1 <= W <= 32767):
        raise _lib.SlnError(f"mask side outside [1, 32767]: {H} x {W}")
    return planes, gs, (L, H, W)


def target_match_batched_device(proposals, gt_class_ids, gt_boxes, num_gt=None, num_proposals=None):
    """Match half of the batched detection targets (sln_target_match_batched, one launch): proposals f32 [B,R,4],
    gt_class_ids int [B,G], gt_boxes f32 [B,G,4] on the device, num_gt B host ints (None: all G rows), num_proposals
    int32 device [B] (None: all R rows).  Returns (codes u8 [B,R]: bit 0 positive, bit 1 negative-eligible; argmax
    int32 [B,R]: the matched row of gt_boxes[b])."""
    B, R, G, num_gt, cls, num_proposals = target_inputs(proposals, gt_class_ids, gt_boxes, num_gt, num_proposals)
    dev = proposals.device
    codes = torch.empty((B, R), dtype=torch.uint8, device=dev)
    argmax = torch.empty((B, R), dtype=torch.int32, device=dev)
    if B and R:
        ng = (C.c_int * B)(*num_gt)
        with torch.cuda.device(dev):
            check(lib().sln_target_match_batched(ptr(proposals.contiguous()), B, R, ptr(num_proposals), ptr(gt_boxes.contiguous()),
                                                 ptr(cls), G, ng, ptr(codes), ptr(argmax), stream_ptr()),
                  "sln_target_match_batched")
        _lib.count_launches(1)
    return codes, argmax


def target_inputs(proposals, gt_class_ids, gt_boxes, num_gt, num_proposals):
    """Checks the batched detection targets' inputs (SlnError on any mismatch, before anything is launched).  Returns
    (B, R, G, num_gt as B host ints, gt_class_ids as int32, num_proposals contiguous or None)."""
    for t, name in ((proposals, "proposals"), (gt_class_ids, "gt_class_ids"), (gt_boxes, "gt_boxes")):
        _require_cuda(t, name)
    if proposals.dim() != 3 or proposals.shape[2] != 4 or proposals.dtype != torch.float32:
        raise _lib.SlnError(f"proposals must be f32 [B,R,4], got {proposals.dtype} {tuple(proposals.shape)}")
    B, R = int(proposals.shape[0]), int(proposals.shape[1])
    if B > TARGET_BATCH_MAX:
        raise _lib.SlnError(f"B = {B} images in one call (at most {TARGET_BATCH_MAX})")
    if gt_boxes.dim() != 3 or int(gt_boxes.shape[0]) != B or gt_boxes.shape[2] != 4 or gt_boxes.dtype != torch.float32:
        raise _lib.SlnError(f"gt_boxes must be f32 [B={B},G,4], got {gt_boxes.dtype} {tuple(gt_boxes.shape)}")
    G = int(gt_boxes.shape[1])
    if tuple(gt_class_ids.shape) != (B, G) or gt_class_ids.dtype.is_floating_point or gt_class_ids.dtype == torch.bool:
        raise _lib.SlnError(f"gt_class_ids must be integer [B,G] = [{B},{G}], got {gt_class_ids.dtype} {tuple(gt_class_ids.shape)}")
    for t, name in ((gt_class_ids, "gt_class_ids"), (gt_boxes, "gt_boxes")):
        if t.device != proposals.device:
            raise _lib.SlnError(f"{name} is on {t.device}, the proposals on {proposals.device}")
    num_gt = target_num_gt(num_gt, B, G)
    if num_proposals is not None:
        _require_cuda(num_proposals, "num_proposals")
        if tuple(num_proposals.shape) != (B,) or num_proposals.dtype != torch.int32 or num_proposals.device != proposals.device:
            raise _lib.SlnError(f"num_proposals must be int32 [B={B}] beside the proposals, got {num_proposals.dtype} "
                                f"{tuple(num_proposals.shape)} on {num_proposals.device}")
        num_proposals = num_proposals.contiguous()
    return B, R, G, num_gt, _i32c(gt_class_ids), num_proposals


# Staging buffer of the batched detection targets (int32 slots): what the host's sampling sends to the emit kernel in
# one copy.  planes: B device addresses of the images' u8 masks (two slots each, int64); then mask_g, num_positive,
# num_rois [B] and sel [B,T].
def target_stage_layout(B, T):
    return {"planes": 0, "mask_g": 2 * B, "num_positive": 3 * B, "num_rois": 4 * B, "sel": 5 * B, "total": 5 * B + B * T}


def detection_targets_emit_batched_device(proposals, argmax, gt_boxes, gt_class_ids, stage, T, LHW, mask_shape,
                                          std_dev=None, use_mini_mask=False):
    """Emit half of the batched detection targets (sln_detection_targets_emit_batched, one launch).  proposals f32
    [B,R,4], argmax int32 [B,R] (target_match_batched_device's), gt_boxes f32 [B,G,4], gt_class_ids int32 [B,G]; stage:
    the int32 device buffer of target_stage_layout(B, T), filled by the host's sampling; LHW = (L, H, W) of the masks it
    points at.  Returns (rois f32 [B,T,4], class_ids int32 [B,T], deltas f32 [B,T,4], masks f32 [B,T,L,mh,mw]), every
    element written."""
    B, R, G = int(proposals.shape[0]), int(proposals.shape[1]), int(gt_boxes.shape[1])
    L, H, W = (int(v) for v in LHW)
    mh, mw = int(mask_shape[0]), int(mask_shape[1])
    lay = target_stage_layout(B, T)
    if stage.dtype != torch.int32 or stage.numel() != lay["total"]:
        raise _lib.SlnError(f"stage must be int32 [{lay['total']}], got {stage.dtype} [{stage.numel()}]")
    dev = proposals.device
    rois = torch.empty((B, T, 4), dtype=torch.float32, device=dev)
    class_ids = torch.empty((B, T), dtype=torch.int32, device=dev)
    deltas = torch.empty((B, T, 4), dtype=torch.float32, device=dev)
    masks = torch.empty((B, T, L, mh, mw), dtype=torch.float32, device=dev)
    if B and T:
        at = lambda k: C.c_void_p(stage.data_ptr() + 4 * lay[k])
        sd = (C.c_float * 4)(*[float(v) for v in std_dev]) if std_dev is not None else None
        with torch.cuda.device(dev):
            check(lib().sln_detection_targets_emit_batched(
                ptr(proposals.contiguous()), B, R, ptr(argmax), ptr(gt_boxes.contiguous()), ptr(gt_class_ids), G, at("sel"),
                at("num_positive"), at("num_rois"), at("planes"), at("mask_g"), T, L, H, W, mh, mw, sd, int(bool(use_mini_mask)),
                ptr(rois), ptr(class_ids), ptr(deltas), ptr(masks), stream_ptr()), "sln_detection_targets_emit_batched")
        _lib.count_launches(1)
    return rois, class_ids, deltas, masks


def rpn_overlap_reductions_device(anchors, gt_boxes, want_argmax=True):
    """float64 IoU reductions of build_rpn_targets (sln_rpn_overlap_reductions).  anchors f64 [A,4], gt_boxes f64 [G,4]
    on the device -> (anchor_iou_max f64 [A], anchor_argmax i32 [A] | None, gt_argmax i32 [G] | None)."""
    _require_cuda(anchors, "anchors")
    a = anchors.to(torch.float64).contiguous().view(-1, 4)
    g = gt_boxes.to(device=a.device, dtype=torch.float64).contiguous().view(-1, 4)
    A, G = a.shape[0], g.shape[0]
    mx = torch.zeros(A, dtype=torch.float64, device=a.device)
    am = torch.zeros(A, dtype=torch.int32, device=a.device) if want_argmax else None
    ga = torch.zeros(G, dtype=torch.int32, device=a.device) if want_argmax else None
    if A and G:
        with torch.cuda.device(a.device):
            ws = _workspace(lib().sln_rpn_overlap_workspace_bytes(G), a.device) if want_argmax else None
            check(lib().sln_rpn_overlap_reductions(ptr(a), A, ptr(g), G, ptr(mx), ptr(am), ptr(ga), ptr(ws),
                                                   ws.numel() if ws is not None else 0, stream_ptr()),
                  "sln_rpn_overlap_reductions")
        _lib.count_launches(3 if want_argmax else 1)
    return mx, am, ga


def plane_bboxes_device(planes):
    """Tight (y1, x1, y2, x2) of binary u8 / bool planes [..., H, W] on the device -> int32 [..., 4] (sln_plane_bboxes)."""
    _require_cuda(planes, "planes")
    if planes.dtype == torch.bool:
        planes = planes.view(torch.uint8)
    if planes.dtype != torch.uint8 or planes.dim() < 2:
        raise _lib.SlnError("planes must be uint8 / bool [..., H, W]")
    planes = planes.contiguous()
    H, W = planes.shape[-2:]
    M = planes.numel() // max(H * W, 1) if H * W else int(np.prod(planes.shape[:-2]))
    out = torch.empty(tuple(planes.shape[:-2]) + (4,), dtype=torch.int32, device=planes.device)
    if M:
        with torch.cuda.device(planes.device):
            check(lib().sln_plane_bboxes(ptr(planes), M, H, W, ptr(out), stream_ptr()), "sln_plane_bboxes")
        _lib.count_launches(1)
    return out


def gather_planes_device(planes, iy, ix):
    """dst[..., y, x] = planes[..., iy[y], ix[x]] (0 where an index is negative); planes u8 / bool [..., H, W] on the
    device, iy / ix int32 index maps (numpy or tensors) -> u8 [..., len(iy), len(ix)] (sln_gather_planes)."""
    _require_cuda(planes, "planes")
    was_bool = planes.dtype == torch.bool
    if was_bool:
        planes = planes.view(torch.uint8)
    if planes.dtype != torch.uint8 or planes.dim() < 2:
        raise _lib.SlnError("planes must be uint8 / bool [..., H, W]")
    planes = planes.contiguous()
    H, W = planes.shape[-2:]
    n = planes.numel() // max(H * W, 1)
    d_iy = torch.as_tensor(np.asarray(iy, dtype=np.int32)).to(planes.device) if not torch.is_tensor(iy) else _i32c(iy)
    d_ix = torch.as_tensor(np.asarray(ix, dtype=np.int32)).to(planes.device) if not torch.is_tensor(ix) else _i32c(ix)
    H2, W2 = d_iy.numel(), d_ix.numel()
    out = torch.empty(tuple(planes.shape[:-2]) + (H2, W2), dtype=torch.uint8, device=planes.device)
    if out.numel():
        with torch.cuda.device(planes.device):
            check(lib().sln_gather_planes(ptr(planes), n, H, W, ptr(d_iy), ptr(d_ix), H2, W2, ptr(out), stream_ptr()),
                  "sln_gather_planes")
        _lib.count_launches(1)
    return out.view(torch.bool) if was_bool else out


# ---------------------------------------------------------------------------
# proposal_layer
# ---------------------------------------------------------------------------
def proposal_device(probs, deltas, anchors, proposal_count, nms_threshold, std_dev, image_hw, pre_nms_limit=6000):
    """One image.  probs [A,2], deltas [A,4], anchors [A,4] (pixels).  Returns
    (boxes f32[proposal_count,4] normalised, zero padded; num int32[1]) on the device."""
    for t, nm in ((probs, "probs"), (deltas, "deltas"), (anchors, "anchors")):
        _require_cuda(t, nm)
    probs, deltas, anchors = _f32c(probs), _f32c(deltas), _f32c(anchors)
    A = anchors.shape[0]
    if probs.shape != (A, 2) or deltas.shape != (A, 4):
        raise _lib.SlnError("probs/deltas/anchors shapes disagree")
    out = torch.empty((max(int(proposal_count), 1), 4), dtype=torch.float32, device=probs.device)
    num = torch.empty(1, dtype=torch.int32, device=probs.device)
    sd = (C.c_float * 4)(*[float(v) for v in std_dev])
    with torch.cuda.device(probs.device):
        ws = _workspace(lib().sln_proposal_workspace_bytes(A, int(pre_nms_limit)), probs.device)
        check(lib().sln_proposal_layer(ptr(probs), ptr(deltas), ptr(anchors), A, int(pre_nms_limit),
                                       int(proposal_count), float(nms_threshold), sd, float(image_hw[0]),
                                       float(image_hw[1]), ptr(out), ptr(num), ptr(ws), ws.numel(), stream_ptr()),
              "sln_proposal_layer")
    if A and proposal_count:
        _lib.count_launches(14 if A > pre_nms_limit else 6)
    return out[:proposal_count], num


def _proposal_batched_launches(B, A, K, nms_threshold):
    """Launches of one sln_proposal_layer_batched call with K = min(A, pre_nms_limit) > 0: the shared stages once, the
    dense NMS fallback (nms.cu: mask + scan, the fixed-point resolve from 160 words, two stages from 16384 boxes) once
    per image."""
    shared = (6 if K < A else 1) + 3                     # histogram memset + 5 select kernels | select_all; rank memset, rank, decode
    shared += 3 if 65 <= K <= 65535 and nms_threshold >= 0.05 else 0     # bin, pairs, resolve
    shared += 1                                          # finalize
    if K < 16384:
        dense = 2 + (((K + 63) // 64) >= 160)
    else:
        dense = 2 + 3 + 2 + (((K - 1024 + 63) // 64) >= 160)
    return shared + B * dense


def proposal_batched_device(probs, deltas, anchors, proposal_count, nms_threshold, std_dev, image_hw, pre_nms_limit=6000):
    """B images in one call (sln_proposal_layer_batched).  probs [B,A,2], deltas [B,A,4], anchors [A,4] (pixels, shared).
    Returns (boxes f32 [B,proposal_count,4] normalised, zero padded; num int32 [B]) on the device; image b's rows are
    exactly proposal_device's for that image alone."""
    for t, nm in ((probs, "probs"), (deltas, "deltas"), (anchors, "anchors")):
        _require_cuda(t, nm)
    if probs.dim() != 3 or probs.shape[2] != 2:
        raise _lib.SlnError(f"probs must be [B,A,2], got {tuple(probs.shape)}")
    B, A = int(probs.shape[0]), int(probs.shape[1])
    if tuple(deltas.shape) != (B, A, 4):
        raise _lib.SlnError(f"deltas {tuple(deltas.shape)} disagrees with probs {tuple(probs.shape)}")
    if tuple(anchors.shape) != (A, 4):
        raise _lib.SlnError(f"anchors {tuple(anchors.shape)} disagree with A = {A}")
    if int(proposal_count) < 0 or int(pre_nms_limit) < 0:
        raise _lib.SlnError(f"proposal_count ({proposal_count}) and pre_nms_limit ({pre_nms_limit}) must be >= 0")
    probs, deltas, anchors = _f32c(probs), _f32c(deltas), _f32c(anchors)
    R = int(proposal_count)
    out = torch.empty((B, max(R, 1), 4), dtype=torch.float32, device=probs.device)
    num = torch.empty(B, dtype=torch.int32, device=probs.device)
    sd = (C.c_float * 4)(*[float(v) for v in std_dev])
    with torch.cuda.device(probs.device):
        ws = _workspace(lib().sln_proposal_batched_workspace_bytes(B, A, int(pre_nms_limit)), probs.device)
        check(lib().sln_proposal_layer_batched(ptr(probs), ptr(deltas), ptr(anchors), B, A, int(pre_nms_limit), R,
                                               float(nms_threshold), sd, float(image_hw[0]), float(image_hw[1]), ptr(out),
                                               ptr(num), ptr(ws), ws.numel(), stream_ptr()), "sln_proposal_layer_batched")
    K = min(A, int(pre_nms_limit))
    if B:
        _lib.count_launches(_proposal_batched_launches(B, A, K, float(nms_threshold)) if K and R else 1 + (R > 0))
    return out[:, :R], num


# ---------------------------------------------------------------------------
# sem-dist target encoding
# ---------------------------------------------------------------------------
def layer_decode_device(label, L, n_max):
    """label [B,H,W] (int64/uint64 bit patterns) -> (u8 [B,n_max,L,H,W], n_obj int32[B])."""
    _require_cuda(label, "label")
    if label.dtype not in (torch.int64, torch.uint64):
        raise _lib.SlnError("label must hold 64-bit patterns (int64 or uint64)")
    label = label.contiguous()
    if label.dim() == 2:
        label = label.unsqueeze(0)
    B, H, W = label.shape
    out = torch.empty((B, n_max, L, H, W), dtype=torch.uint8, device=label.device)
    n_obj = torch.empty(B, dtype=torch.int32, device=label.device)
    scratch = torch.empty(2 * max(B, 1), dtype=torch.int32, device=label.device)
    with torch.cuda.device(label.device):
        check(lib().sln_layer_decode(ptr(label), B, H, W, int(L), int(n_max), ptr(out), ptr(n_obj), ptr(scratch),
                                     stream_ptr()), "sln_layer_decode")
    if B and H * W:
        _lib.count_launches(2)
    return out, n_obj


def edt_sq_device(maps):
    """maps u8 [...,H,W] -> i32 same shape: squared distance to the nearest zero pixel of each map."""
    _require_cuda(maps, "maps")
    if maps.dtype == torch.bool:
        maps = maps.to(torch.uint8)
    if maps.dtype != torch.uint8:
        raise _lib.SlnError("maps must be uint8 or bool")
    maps = maps.contiguous()
    H, W = maps.shape[-2], maps.shape[-1]
    M = maps.numel() // max(H * W, 1) if H * W else 0
    out = torch.empty(maps.shape, dtype=torch.int32, device=maps.device)
    with torch.cuda.device(maps.device):
        nbytes = lib().sln_edt_workspace_bytes(M, H, W)
        ws = _workspace(nbytes, maps.device)
        check(lib().sln_edt_sq(ptr(maps), M, H, W, ptr(out), ptr(ws), ws.numel(), stream_ptr()), "sln_edt_sq")
    if M and H * W:
        per = 2 * H * W
        chunk = max(1, min(M, (2048 << 20) // per))
        _lib.count_launches(2 * ((M + chunk - 1) // chunk))
    return out
