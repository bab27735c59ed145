"""nuhtc_b200 -- B200 (sm_100a) native RoI stage + nucleus merge for NuHTC.

Host side mirrors of the reference's op surface (mmcv.ops RoIAlign / nms / batched_nms, mmdet's
SingleRoIExtractor and mask paste, tools/infer_wsi.py:mask_nms, tools/nuclei_merge.py:merge_overlap, mmdet's
test-time image pipeline behind inference_detector) over the C ABI of include/nuhtc_b200.h (libnuhtc_b200.so, hand-written CUDA).  GPU only: no CPU fallback.
"""
from . import _lib
from ._lib import NuhtcError, LIB_PATH
from .mmcv_ops import (RoIAlign, roi_align, nms, batched_nms, roi_align_levels, nms_groups, to_nhwc, to_cg32, clear_layout_cache,
                       layout_cache, StagedLevels, stage_levels)
from .mask_paste import _do_paste_mask, paste_masks, get_seg_masks, get_seg_masks_device
from .mask_nms import mask_nms, mask_nms_device, pack_masks
from .nuclei_merge import merge_arrays, merge_overlap
from .contours import mask_contours, mask2inst, rings_for_merge
from .preprocess import TilePipeline, inference_detector
from . import slide, synth, roi_stage, rpn, contours, watershed

__version__ = "0.1.0"
