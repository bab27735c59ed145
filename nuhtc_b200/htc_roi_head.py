"""HTC RoI head with the reference's call signature, on the device-resident RoI stage.

Drop-in for the test path of
  * ``HybridTaskCascadeRoIHead_Lite.simple_test(img, x, proposal_list, img_metas, rescale)``
        /root/reference/nuhtc/models/htc_roi_head_cus.py:2184-2376  (+ ``_bbox_forward`` :187-203)
  * stock ``HybridTaskCascadeRoIHead.simple_test(x, proposal_list, img_metas, rescale)``
        /root/reference/thirdparty/mmdetection/mmdet/models/roi_heads/htc_roi_head.py:330-503
Same arguments, same return value: ``list[(bbox_result, segm_result)]`` with ``bbox_result = list[num_classes] of float32
ndarray [k,5]`` (mmdet ``bbox2result``) and ``segm_result = list[num_classes] of list of bool ndarray [H,W]``
(``FCNMaskHead.get_seg_masks``), detections in the reference's order (score-descending per image, grouped by label).

What runs where: the RoI extractors (multi-level RoIAlign, cosine-attention pooling, semantic-feature fusion), box decode,
per-class NMS, detection truncation and mask paste are this package's kernels (``RoIStage``); the bbox / mask / semantic
heads are the caller's torch modules (stock cuDNN work, outside the target).  Nothing leaves the device between the
proposals and the final results; the only device->host copies are the returned arrays.

Head protocol (what the wrapper needs from the caller's modules -- mmdet's heads satisfy it through small adapters):
  bbox_head[i](roi_feats [K,C,7,7]) -> (cls_score [K,*], bbox_pred [K,4])      class-agnostic regression
  bbox_head[i].num_classes, .target_stds (4 floats), optional .score_activation(cls_score) -> [K, num_classes+1]
        (default softmax; ``seesaw_activation`` is the NuHTC configs' SeesawLoss.get_activation)
  mask_head(mask_feats [D,C,14,14]) -> logits [D,1,h,w]   (class-agnostic, as every NuHTC config sets)
  semantic_head(x) -> (semantic_pred, semantic_feat)       (optional)

Half precision: ``x`` and the semantic feature map may be fp16 or bf16 (mmcv's wrap_fp16_model, torch.autocast); the
heads then receive RoI features in that dtype and the result format is unchanged (fp32 boxes, bool masks).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from .roi_stage import RoIStage, RoIStageConfig, bbox2roi

__all__ = ["HybridTaskCascadeRoIHead_Lite", "HybridTaskCascadeRoIHead", "seesaw_activation", "bbox2result"]


def seesaw_activation(cls_score: torch.Tensor) -> torch.Tensor:
    """SeesawLoss.get_activation (mmdet/models/losses/seesaw_loss.py:157-175): [N, C+2] -> [N, C+1]."""
    cls, obj = cls_score[..., :-2], cls_score[..., -2:]
    sc = torch.softmax(cls, dim=-1)
    so = torch.softmax(obj, dim=-1)
    return torch.cat([sc * so[..., [0]], so[..., [1]]], dim=-1)


def bbox2result(bboxes: np.ndarray, labels: np.ndarray, num_classes: int) -> List[np.ndarray]:
    """mmdet/core/bbox/transforms.py:bbox2result on host arrays."""
    if bboxes.shape[0] == 0:
        return [np.zeros((0, 5), dtype=np.float32) for _ in range(num_classes)]
    return [bboxes[labels == i, :] for i in range(num_classes)]


class HybridTaskCascadeRoIHead_Lite:
    def __init__(self, num_stages: int, bbox_head: Sequence[Callable], mask_head: Callable, test_cfg: dict,
                 featmap_strides: Sequence[int] = (4, 8, 16, 32), extractor: str = "attention", start_level: int = 2,
                 thres: float = 0.0, finest_scale: float = 56.0, bbox_roi_layer: Optional[dict] = None,
                 mask_roi_layer: Optional[dict] = None, semantic_head: Optional[Callable] = None,
                 semantic_fusion: Sequence[str] = ("bbox", "mask"), semantic_roi_layer: Optional[dict] = None,
                 semantic_stride: int = 4, watershed_proposal=None, mask_classes: Optional[int] = None):
        """Config keys follow configs/nuhtc/htc_lite_swin_pytorch_fpn_PanNuke_seasaw_CAS.py:72-164.
        extractor: 'attention' (AttentionRoIExtractor, start_level / thres) or 'single' (SingleRoIExtractor, finest_scale).
        *_roi_layer: dict(type='RoIAlign', output_size=.., sampling_ratio=..).
        test_cfg: dict(score_thr, nms=dict(type='nms', iou_threshold=..), max_per_img, mask_thr_binary).
        watershed_proposal: True = prepend the watershed proposals of the semantic prediction to every image's proposals
        (`with_watershed_proposal`, htc_roi_head_cus.py:2217-2221; needs a semantic_head) with nuhtc_b200.watershed (device
        resident; the reference does this step on the host with scipy / skimage); a callable
        (semantic_pred, proposal_list, img_shape) -> proposal_list replaces it; None / False skips it."""
        assert len(bbox_head) == num_stages
        bl = dict(bbox_roi_layer or dict(type="RoIAlign", output_size=7, sampling_ratio=2))
        ml = dict(mask_roi_layer or dict(type="RoIAlign", output_size=14, sampling_ratio=0))
        sl = dict(semantic_roi_layer or dict(type="RoIAlign", output_size=14, sampling_ratio=0))
        for lay in (bl, ml, sl):
            if lay.get("type", "RoIAlign") != "RoIAlign":
                raise NotImplementedError("roi_layer type %r: NuHTC configures RoIAlign only" % lay.get("type"))
        if sl.get("sampling_ratio", 0) != 0:
            raise NotImplementedError("semantic_roi_extractor: sampling_ratio=0 (every shipped config)")
        self.num_stages = num_stages
        self.bbox_head = list(bbox_head)
        self.mask_head = mask_head
        self.semantic_head = semantic_head
        self.with_semantic = semantic_head is not None
        self.semantic_fusion = tuple(semantic_fusion) if self.with_semantic else ()
        if watershed_proposal is True:
            from .watershed import watershed_proposal as _ws

            def watershed_proposal(semantic_pred, proposal_list, img_shape):
                if semantic_pred.dtype != torch.float32:
                    raise NotImplementedError("watershed_proposal=True needs an fp32 semantic prediction: its blur and threshold "
                                              f"would otherwise run in {semantic_pred.dtype}, not as the fp32 reference does")
                return _ws(semantic_pred, proposal_list=proposal_list, img_shape=img_shape, min_area=10, thres=0)[0]
        self.watershed_proposal = watershed_proposal or None
        self.test_cfg = dict(test_cfg)
        self.num_classes = int(getattr(self.bbox_head[-1], "num_classes"))
        self.mask_classes = int(mask_classes if mask_classes is not None else self.num_classes)
        self._layers = (bl, ml, sl)
        self._strides = tuple(featmap_strides)
        self._extractor = extractor
        self._ext_args = dict(start_level=int(start_level), thres=float(thres), finest_scale=float(finest_scale),
                              semantic_stride=int(semantic_stride))
        self._stage_cache = {}

    # -- one RoIStage per (frame, scale_factor, rescale): the stage keeps per-device constants
    def _stage(self, img_shape, ori_shape, scale_factor: float, rescale: bool) -> RoIStage:
        key = (tuple(img_shape[:2]), tuple(ori_shape[:2]), float(scale_factor), bool(rescale))
        st = self._stage_cache.get(key)
        if st is None:
            bl, ml, sl = self._layers
            nms = self.test_cfg.get("nms", dict(type="nms", iou_threshold=0.5))
            if nms.get("type", "nms") != "nms":
                raise NotImplementedError("nms type %r" % nms.get("type"))
            cfg = RoIStageConfig(
                featmap_strides=self._strides, finest_scale=self._ext_args["finest_scale"],
                extractor=self._extractor, sum_levels=self._ext_args["start_level"], attention_thres=self._ext_args["thres"],
                semantic_fusion=self.semantic_fusion, semantic_stride=self._ext_args["semantic_stride"],
                semantic_out=int(sl["output_size"]),
                bbox_out=int(bl["output_size"]), bbox_sampling_ratio=int(bl.get("sampling_ratio", 0)),
                mask_out=int(ml["output_size"]), mask_sampling_ratio=int(ml.get("sampling_ratio", 0)),
                num_stages=self.num_stages, stage_stds=tuple(tuple(float(v) for v in h.target_stds) for h in self.bbox_head),
                num_classes=self.num_classes, score_thr=float(self.test_cfg["score_thr"]), nms_iou=float(nms["iou_threshold"]),
                max_per_img=int(self.test_cfg["max_per_img"]), mask_thr_binary=float(self.test_cfg.get("mask_thr_binary", 0.5)),
                img_shape=tuple(img_shape[:2]),
                # rescale=True: detections and masks live in the original frame; otherwise in the scaled frame
                # round(ori_shape * scale_factor) with unscaled boxes (fcn_mask_head.py:249-255)
                ori_shape=tuple(ori_shape[:2]) if rescale else tuple(int(np.round(v * scale_factor)) for v in ori_shape[:2]),
                scale_factor=float(scale_factor) if rescale else 1.0,
                dense_masks=True, fused_dense_bits=False, contour_max_pts=0, tile_postprocess=False)
            act = getattr(self.bbox_head[-1], "score_activation", None)
            st = RoIStage(cfg, [(lambda f, h=h: h(f)) for h in self.bbox_head], lambda f, cand: self.mask_head(f), score_fn=act)
            self._stage_cache[key] = st
        return st

    @torch.no_grad()
    def simple_test(self, img, x, proposal_list, img_metas, rescale=False):
        """htc_roi_head_cus.py:2184-2376.  `img` is only consulted by the reference's optional seg_head (not configured)."""
        semantic_feat = None
        if self.with_semantic:
            semantic_pred, semantic_feat = self.semantic_head(x)
            if self.watershed_proposal is not None:
                proposal_list = self.watershed_proposal(semantic_pred, proposal_list, img_metas[0]["img_shape"][:2])
        num_imgs = len(proposal_list)
        C = self.num_classes
        empty = [(bbox2result(np.zeros((0, 5), np.float32), np.zeros((0,), np.int64), C), [[] for _ in range(self.mask_classes)])
                 for _ in range(num_imgs)]
        rois = bbox2roi([p[:, :4] for p in proposal_list])
        if rois.shape[0] == 0:
            return empty
        img_shape, ori_shape = img_metas[0]["img_shape"], img_metas[0]["ori_shape"]
        sf = img_metas[0]["scale_factor"]
        sf0 = float(np.asarray(sf).reshape(-1)[0])
        for m in img_metas:   # one launch sequence serves the whole batch: the tiles of a batch share their geometry
            if tuple(m["img_shape"][:2]) != tuple(img_shape[:2]) or tuple(m["ori_shape"][:2]) != tuple(ori_shape[:2]) or \
                    not np.allclose(np.asarray(m["scale_factor"], dtype=np.float64).reshape(-1), sf0):
                raise NotImplementedError("simple_test: the images of a batch must share img_shape / ori_shape / a uniform scale_factor")
        stage = self._stage(img_shape, ori_shape, sf0, rescale)
        per_img = max(int(p.shape[0]) for p in proposal_list)
        res = stage.run(list(x[: len(self._strides)]), rois, max_rois_per_tile=per_img, semantic_feat=semantic_feat)
        res.check()
        # ---- reference result format
        valid = res.det_valid.cpu().numpy().astype(bool)
        boxes = res.det_boxes.cpu().numpy()
        scores = res.det_scores.cpu().numpy()
        labels = res.det_labels.cpu().numpy()
        tiles = res.det_tile.cpu().numpy()
        masks = res.masks.cpu().numpy().astype(bool)
        out = []
        for i in range(num_imgs):
            sel = np.nonzero(valid & (tiles == i))[0]      # slots are tile-major in score order
            det = np.concatenate([boxes[sel], scores[sel, None]], axis=1).astype(np.float32)
            lab = labels[sel]
            bbox_result = bbox2result(det, lab, C)
            segm = [[] for _ in range(self.mask_classes)]
            for j, l in zip(sel, lab):
                segm[int(l)].append(masks[j])
            out.append((bbox_result, segm))
        return out


class HybridTaskCascadeRoIHead(HybridTaskCascadeRoIHead_Lite):
    """Stock mmdet signature: simple_test(x, proposal_list, img_metas, rescale=False) (htc_roi_head.py:330)."""

    def simple_test(self, x, proposal_list, img_metas, rescale=False):  # type: ignore[override]
        return super().simple_test(None, x, proposal_list, img_metas, rescale=rescale)
