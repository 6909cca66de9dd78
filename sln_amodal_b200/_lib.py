"""ctypes binding of libsln_b200.so (C ABI declared in include/sln_b200.h).

There is no CPU fallback: if the library is missing or a call fails, the caller gets
an exception.  PyTorch is used only for device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsln_b200.so")

OK = 0
LAYOUT_NCHW = 0
LAYOUT_NHWC = 1
BWD_EXACT = 1
BWD_PLAN_ONLY = 2        # sln_pyramid_crop_bwd: build the ROI lists only
BWD_PLANNED = 4          # ... the workspace already holds them
DTYPE_F32 = 0            # element type of the *_ex crop entry points
DTYPE_BF16 = 1
DTYPE_F16 = 2

_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/sln_b200.h one to one
PROTOTYPES = {
    "sln_version": (_i, []),
    "sln_last_error_string": (C.c_char_p, []),
    "sln_device_info": (_i, [C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz), C.POINTER(_sz)]),
    "sln_crop_and_resize_fwd": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _f, _vp, _vp]),
    "sln_crop_and_resize_bwd_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "sln_crop_and_resize_bwd": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "sln_pyramid_crop_fwd": (_i, [C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _vp, _vp, _vp, _i,
                                  _i, _i, _f, _vp, _vp]),
    "sln_pyramid_crop_bwd_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "sln_pyramid_crop_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), _i, _i,
                                  _i, _vp, _sz, _vp]),
    "sln_crop_and_resize_fwd_ex": (_i, [_i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _f, _vp, _vp]),
    "sln_crop_and_resize_bwd_ex": (_i, [_i, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _sz, _vp]),
    "sln_pyramid_crop_fwd_ex": (_i, [_i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _vp, _vp, _vp, _i,
                                     _i, _i, _f, _vp, _vp]),
    "sln_pyramid_crop_bwd_ex": (_i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i),
                                     _i, _i, _i, _vp, _sz, _vp]),
    "sln_roi_levels": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "sln_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "sln_nhwc_to_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "sln_nchw_to_nhwc_b16": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "sln_nhwc_to_nchw_b16": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "sln_nms_workspace_bytes": (_sz, [_i]),
    "sln_nms": (_i, [_vp, _vp, _i, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "sln_nms_ex": (_i, [_vp, _vp, _i, _f, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sln_refine_decode": (_i, [_vp, _vp, _vp, _i, _i, C.POINTER(_f), _f, _f, C.POINTER(_f), _f, _vp, _vp, _vp, _vp, _vp]),
    "sln_refine_topk": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp]),
    "sln_bbox_overlaps": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "sln_box_refinement": (_i, [_vp, _vp, _i, C.POINTER(_f), _vp, _vp]),
    "sln_mask_targets": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "sln_rpn_overlap_workspace_bytes": (_sz, [_i]),
    "sln_rpn_overlap_reductions": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "sln_plane_bboxes": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "sln_rle_encode": (_i, [_vp, _i, C.c_longlong, _vp, _i, _vp, _vp]),
    "sln_rle_to_string": (C.c_longlong, [_vp, C.c_longlong, C.c_char_p, C.c_longlong]),
    "sln_unmold_masks": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "sln_resize_image_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "sln_resize_image_u8": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "sln_gather_planes": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "sln_rpn_pack": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "sln_rpn_unpack_grads": (_i, [_vp, _vp, C.POINTER(_i), C.POINTER(_i), _i, _i, _i, _i, C.POINTER(_vp), C.POINTER(_vp), _vp]),
    "sln_proposal_workspace_bytes": (_sz, [_i, _i]),
    "sln_proposal_layer": (_i, [_vp, _vp, _vp, _i, _i, _i, _f, C.POINTER(_f), _f, _f, _vp, _vp, _vp, _sz, _vp]),
    "sln_layer_decode": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "sln_edt_workspace_bytes": (_sz, [_i, _i, _i]),
    "sln_edt_sq": (_i, [_vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
}

_lib = None


class SlnError(RuntimeError):
    pass


def lib():
    """The loaded library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SlnError(
                f"{LIB_PATH} is missing: build it with `python -m sln_amodal_b200.build` "
                "(there is no CPU or PyTorch fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)       # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != OK:
        msg = lib().sln_last_error_string().decode("utf-8", "replace")
        raise SlnError(f"{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (or NULL for None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# Kernel-launch counter: every C-ABI call that enqueues our kernels reports how many it
# launched, so bench.py can state `gpu_launches` from a count rather than a guess.
_launches = 0


def count_launches(n: int) -> None:
    global _launches
    _launches += n


def launches() -> int:
    return _launches
