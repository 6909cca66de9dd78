"""Functional host layer over the C ABI: torch CUDA tensors in, torch CUDA tensors out.

Every function here enqueues hand-written sm_100a kernels from libsln_b200.so on the
current torch stream.  Nothing falls back to PyTorch or the CPU: non-CUDA inputs raise.
PyTorch only provides device memory (outputs and workspaces are torch tensors owned by
the caller side, as the ABI requires) and the stream.
"""
from __future__ import annotations

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
