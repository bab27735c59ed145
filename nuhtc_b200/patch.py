"""Rebind the reference's op surface to the B200 ops (see INTEGRATION.md).  Needs mmcv / mmdet / nuhtc importable,
i.e. it runs inside the reference's environment; nothing else in this package depends on them."""
from __future__ import annotations

import importlib


def patch_mmcv(verbose: bool = False):
    """``mmcv.ops.RoIAlign / roi_align / nms / batched_nms`` and the names the reference modules bound at import time
    (`batched_nms` in four modules, `_do_paste_mask` in fcn_mask_head) now point at nuhtc_b200.  Returns the list of
    rebound attributes."""
    from . import RoIAlign, _do_paste_mask, batched_nms, nms, roi_align
    import mmcv.ops
    # not `import mmcv.ops.nms as m`: mmcv/ops/__init__.py does `from .nms import nms`, so the attribute `mmcv.ops.nms` is
    # the function and that form would bind the function, not the submodule
    mmcv_nms = importlib.import_module("mmcv.ops.nms")

    done = []

    def bind(mod, name, obj):
        setattr(mod, name, obj)
        done.append(f"{mod.__name__}.{name}")

    bind(mmcv.ops, "RoIAlign", RoIAlign)
    bind(mmcv.ops, "roi_align", roi_align)
    bind(mmcv.ops, "nms", nms)
    bind(mmcv.ops, "batched_nms", batched_nms)
    bind(mmcv_nms, "nms", nms)
    bind(mmcv_nms, "batched_nms", batched_nms)
    for modname in ("nuhtc.models.bbox_head", "nuhtc.core.post_processing.bbox_nms", "mmdet.core.post_processing.bbox_nms",
                    "mmdet.models.dense_heads.rpn_head"):
        try:
            bind(importlib.import_module(modname), "batched_nms", batched_nms)
        except ImportError:
            pass
    try:
        bind(importlib.import_module("mmdet.models.roi_heads.mask_heads.fcn_mask_head"), "_do_paste_mask", _do_paste_mask)
    except ImportError:
        pass
    if verbose:
        print("nuhtc_b200.patch_mmcv:", ", ".join(done))
    return done


def patch_wsi_tools(infer_wsi_module=None, nuclei_merge_module=None):
    """Rebind the tile post-processing helpers of the reference's scripts: ``mask_nms`` and ``mask2inst`` of
    tools/infer_wsi.py (:51-84) and ``merge_overlap`` of tools/nuclei_merge.py (:62-174).  Pass the imported modules."""
    from . import mask2inst, mask_nms, merge_overlap
    done = []
    if infer_wsi_module is not None:
        infer_wsi_module.mask_nms = mask_nms
        infer_wsi_module.mask2inst = mask2inst
        done += ["infer_wsi.mask_nms", "infer_wsi.mask2inst"]
    if nuclei_merge_module is not None:
        nuclei_merge_module.merge_overlap = merge_overlap
        done.append("nuclei_merge.merge_overlap")
    return done


def patch_inference(infer_wsi_module):
    """Rebind ``inference_detector`` of tools/infer_wsi.py (called at :485) to :func:`nuhtc_b200.inference_detector`: the
    tiles' resize / normalise / pad run as one kernel on the GPU and cross PCIe as uint8.  Pass the imported module."""
    from . import inference_detector
    infer_wsi_module.inference_detector = inference_detector
    return ["infer_wsi.inference_detector"]
