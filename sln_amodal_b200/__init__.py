"""sln_amodal_b200 -- B200-native (sm_100a) kernels for the SLN-Amodal detection-head hot path,
behind the reference's own operator API.

    from sln_amodal_b200 import CropAndResizeFunction, nms, proposal_layer, pyramid_roi_align

Importing the package does not load the CUDA library; the first operator call does, and it
fails loudly if sln_amodal_b200/libsln_b200.so has not been built
(`python -m sln_amodal_b200.build`).  There is no CPU or PyTorch fallback.
"""
from .crop_and_resize import CropAndResize, CropAndResizeFunction, RoIAlign  # noqa: F401
from .nms import batched_nms, nms, pth_nms  # noqa: F401
from .proposal import proposal_layer, proposal_layer_batched, proposal_layer_padded  # noqa: F401
from .pyramid import pyramid_roi_align, pyramid_roi_align_batched, pyramid_roi_align_image  # noqa: F401
from .semdist import decode_layers, load_layer2, sem_dist_targets  # noqa: F401
from .detection import refine_detections, refine_detections_batched  # noqa: F401
from .ops import nms_batched_device as nms_batched  # noqa: F401
from .targets import (bbox_overlaps, box_refinement, build_rpn_targets, detection_target_layer,  # noqa: F401
                      detection_target_layer_batched, extract_bboxes, resize_image, resize_image_device, resize_layer,
                      resize_layer_device, zoom_index_map)
from .rle import encode as rle_encode  # noqa: F401
from .rpn import rpn_forward_levels, rpn_pack  # noqa: F401
from .unmold import unmold_detections, unmold_detections_batched, unmold_mask, unmold_masks  # noqa: F401
from .install import install  # noqa: F401

__version__ = "0.1.0"
