"""Device-resident HTC RoI stage for a batch of tiles.

Mirrors the control flow of the reference's RoI heads
  * stock ``HybridTaskCascadeRoIHead.simple_test``  thirdparty/mmdetection/mmdet/models/roi_heads/htc_roi_head.py:330-503
  * ``HybridTaskCascadeRoIHead_Lite.simple_test``   nuhtc/models/htc_roi_head_cus.py:2184-2376
followed by the per-tile post-processing of tools/infer_wsi.py:510-526 (margin / min_area filter, mask NMS),
but keeps every intermediate on the GPU: no per-image Python loop, no ``.cpu().numpy()`` between the mask head
and the paste, no per-instance D2H (SURVEY.md H7).  The ops are the ones in this package (one multi-level
RoIAlign launch per cascade stage, one grouped NMS launch for all tiles, fused paste, batched mask NMS); the
bbox / mask heads are callables supplied by the caller (stock PyTorch modules -- outside this package's target).

Precision: the FPN levels (and the semantic feature map) may be fp32, fp16 or bf16.  The RoI features reach the heads in
that dtype (see roi_align_levels), and the head outputs are upcast where mmdet's force_fp32 decorators upcast them:
cls_score / bbox_pred before the activation and the box decode, the mask probabilities before the paste.
"""
from __future__ import annotations

import contextlib
import math
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from . import det_ops
from .contours import mask_contours
from .mask_nms import mask_nms_device
from .mask_paste import paste_masks, paste_masks_dense_bits
from .mmcv_ops import StagedLevels, nms_groups, roi_align_levels, stage_levels

__all__ = ["RoIStageConfig", "RoIStage", "RoIStageResult", "delta2bbox", "bbox2roi"]


@dataclass
class RoIStageConfig:
    featmap_strides: Tuple[int, ...] = (4, 8, 16, 32)
    finest_scale: float = 56.0
    extractor: str = "single"          # 'single': SingleRoIExtractor routing; 'sum': levels [0, sum_levels) summed;
                                       # 'attention': AttentionRoIExtractor = 'sum' + cosine-attention pooling of the levels
                                       # from sum_levels on, added at the store (roi_extractors_cus.py:195-259)
    sum_levels: int = 2                # AttentionRoIExtractor pools levels 0,1 with RoIAlign (roi_extractors_cus.py:213-218)
    attention_thres: float = 0.0       # AttentionRoIExtractor(thres=...)
    semantic_fusion: Tuple[str, ...] = ()   # ('bbox', 'mask'): add the semantic RoI features (htc_roi_head_cus.py:193-199, 2332-2335)
    semantic_stride: int = 4           # semantic_roi_extractor featmap_strides=[4]
    semantic_out: int = 14             # its RoIAlign output size (sampling_ratio 0); pooled to bbox_out for the bbox branch
    bbox_out: int = 7
    bbox_sampling_ratio: int = 0       # stock HTC 0; NuHTC configs use 2
    mask_out: int = 14
    mask_sampling_ratio: int = 0
    num_stages: int = 3
    stage_stds: Tuple[Tuple[float, ...], ...] = ((0.1, 0.1, 0.2, 0.2), (0.05, 0.05, 0.1, 0.1), (0.033, 0.033, 0.067, 0.067))
    num_classes: int = 5
    score_thr: float = 0.05            # stock HTC 0.05; NuHTC 0.35
    nms_iou: float = 0.5
    max_per_img: int = 500             # NuHTC PanNuke 500; stock HTC 100
    mask_thr_binary: float = 0.5
    img_shape: Tuple[int, int] = (512, 512)   # network frame (tile x scale_factor)
    ori_shape: Tuple[int, int] = (256, 256)   # tile frame
    scale_factor: float = 2.0
    fused_dense_bits: bool = True      # dense frames + bit rows from one evaluation (needs W % 16 == 0)
    overlap_dense_paste: bool = True   # write the dense masks on a forked stream beside the mask NMS / contour kernels
    contour_max_pts: int = 0           # > 0: trace mask2inst contours of every detection slot (tools/infer_wsi.py:528)
    margin: int = 0                    # tools/infer_wsi.py --margin
    min_area: int = 10                 # tools/infer_wsi.py --min_area
    mask_nms_thr: float = 0.05         # tools/infer_wsi.py:526
    dense_masks: bool = True           # True: [D,H,W] uint8 masks as get_seg_masks builds them; False: bit rows only
    tile_postprocess: bool = True      # margin / min_area filter + per-tile mask NMS (+ contours) of tools/infer_wsi.py:510-534;
                                       # False stops where the RoI head's simple_test stops (detections + pasted masks)


@dataclass
class RoIStageResult:
    det_boxes: torch.Tensor      # [D,4] tile-frame boxes of the detections that entered the mask branch
    det_scores: torch.Tensor     # [D]
    det_labels: torch.Tensor     # [D] int64
    det_tile: torch.Tensor       # [D] int32 tile (image) index inside the batch
    masks: Optional[torch.Tensor]  # [D,H,W] bool (dense_masks) or None
    mask_bits: torch.Tensor      # [D,H,ceil(W/64)] int64 bit rows
    mask_area: torch.Tensor      # [D] int32
    keep: torch.Tensor           # [D] int32: per tile, kept detection indices (into D) in score order
    tile_start: torch.Tensor     # [B] int32
    tile_count: torch.Tensor     # [B] int32
    det_valid: Optional[torch.Tensor] = None   # [D] bool: D = B*max_per_img slots, tile-major; invalid slots are padding
    det_cand: Optional[torch.Tensor] = None    # [D] int64 candidate id (roi*num_classes + label) of each slot
    status: Optional[tuple] = None             # device status words of the NMS / mask-NMS (/ contour) launches
    contour_xy: Optional[torch.Tensor] = None  # [D,contour_max_pts,2] int32 contour points of the mask-NMS survivors (cfg.contour_max_pts > 0)
    contour_count: Optional[torch.Tensor] = None   # [D] int32

    def check(self) -> None:
        """Host-side check of the device status words (one small D2H)."""
        if self.status is not None:
            for name, st in zip(("nms", "mask_nms", "contours"), self.status):
                v = int(st.item())
                if v != 0:
                    raise RuntimeError(f"{name} status {v}: a tile exceeded its declared capacity" if name != "contours" else
                                       f"contours status {v}: a contour exceeded contour_max_pts (1) or a mask its window (2)")

    def kept_indices(self) -> List[torch.Tensor]:
        ts, tc = self.tile_start.cpu().tolist(), self.tile_count.cpu().tolist()
        return [self.keep[s:s + c].long() for s, c in zip(ts, tc)]

    def compact(self) -> "RoIStageResult":
        """Drop the padding slots (synchronises): detections tile-major in score order, `keep` re-indexed."""
        self.check()
        if self.det_valid is None or bool(self.det_valid.all()):
            return self
        v = self.det_valid
        new_index = torch.cumsum(v.to(torch.int64), 0) - 1
        # tile t's kept list sits at keep[tile_start[t] : tile_start[t]+tile_count[t]] and tile_start is the scan of the
        # ENTRANT counts, so the lists are not packed from 0: gather them tile by tile into a packed list
        ts, tc = self.tile_start.cpu().tolist(), self.tile_count.cpu().tolist()
        parts = [new_index[self.keep[s:s + c].long()].to(self.keep.dtype) for s, c in zip(ts, tc)]
        keep = torch.cat(parts) if parts else self.keep[:0]
        tcount = self.tile_count.clone()
        tstart = (torch.cumsum(tcount, 0) - tcount).to(self.tile_start.dtype)
        return RoIStageResult(self.det_boxes[v], self.det_scores[v], self.det_labels[v], self.det_tile[v],
                              None if self.masks is None else self.masks[v], self.mask_bits[v], self.mask_area[v], keep,
                              tstart, tcount, det_valid=None, det_cand=self.det_cand[v], status=None,
                              contour_xy=None if self.contour_xy is None else self.contour_xy[v],
                              contour_count=None if self.contour_count is None else self.contour_count[v])


def bbox2roi(bbox_list: Sequence[torch.Tensor]) -> torch.Tensor:
    """mmdet/core/bbox/transforms.py:59-78."""
    parts = []
    for img_id, b in enumerate(bbox_list):
        if b.size(0) > 0:
            parts.append(torch.cat([b.new_full((b.size(0), 1), img_id), b[:, :4]], dim=-1))
        else:
            parts.append(b.new_zeros((0, 5)))
    return torch.cat(parts, 0)


def delta2bbox(rois: torch.Tensor, deltas: torch.Tensor, stds, max_shape=None, means=(0., 0., 0., 0.),
               wh_ratio_clip: float = 16 / 1000) -> torch.Tensor:
    """Class-agnostic form of mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:163-260 (same op order)."""
    if deltas.size(0) == 0:
        return deltas
    stds_t = stds if isinstance(stds, torch.Tensor) else deltas.new_tensor(stds)
    means_t = means if isinstance(means, torch.Tensor) else deltas.new_tensor(means)
    d = deltas * stds_t.view(1, -1) + means_t.view(1, -1)
    pxy = (rois[:, :2] + rois[:, 2:]) * 0.5
    pwh = rois[:, 2:] - rois[:, :2]
    dxy_wh = pwh * d[:, :2]
    max_ratio = abs(math.log(wh_ratio_clip))
    dwh = d[:, 2:].clamp(min=-max_ratio, max=max_ratio)
    gxy = pxy + dxy_wh
    gwh = pwh * dwh.exp()
    out = torch.cat([gxy - gwh * 0.5, gxy + gwh * 0.5], dim=-1)
    if max_shape is not None:
        out[..., 0::2].clamp_(min=0, max=max_shape[1])
        out[..., 1::2].clamp_(min=0, max=max_shape[0])
    return out


class RoIStage:
    """``bbox_heads[i](roi_feats [K,C,7,7]) -> (cls_score [K,num_classes+1], bbox_pred [K,4])`` (class-agnostic
    regression, as every NuHTC config sets); ``mask_head(roi_feats [D,C,14,14], det_index [D]) -> logits [D,1,h,w]``;
    ``score_fn(cls_score) -> scores`` (softmax for stock HTC; the Seesaw activation for NuHTC)."""

    def __init__(self, cfg: RoIStageConfig, bbox_heads: Sequence[Callable], mask_head: Callable,
                 score_fn: Optional[Callable] = None):
        assert len(bbox_heads) == cfg.num_stages
        self.cfg = cfg
        self.bbox_heads = list(bbox_heads)
        self.mask_head = mask_head
        self.score_fn = score_fn or (lambda s: torch.softmax(s, dim=-1))
        self._consts = {}                       # per-device constant tensors (built once: nothing is copied H2D in run())
        self.timer: Optional[Callable] = None   # optional: timer(name) -> context manager (bench.py uses CUDA events)
        self.trace: Optional[dict] = None       # optional: filled with the tensors at every op boundary (parity tests)

    def _const(self, dev):
        c = self._consts.get(dev)
        if c is None:
            cfg = self.cfg
            c = dict(stds=[torch.tensor(s, dtype=torch.float32, device=dev) for s in cfg.stage_stds],
                     means=torch.zeros(4, dtype=torch.float32, device=dev),
                     far=torch.tensor([[-4096.0, -4096.0, -4095.0, -4095.0]], device=dev),
                     labels=torch.arange(cfg.num_classes, device=dev, dtype=torch.int64),
                     zero=torch.zeros((), device=dev), minus1=torch.full((), -1, dtype=torch.int32, device=dev))
            self._consts[dev] = c
        return c

    def _side_stream(self, dev):
        st = self._consts.get(("side", dev))
        if st is None:
            st = self._consts[("side", dev)] = torch.cuda.Stream(device=dev)
        return st

    def _t(self, name: str):
        return self.timer(name) if self.timer is not None else contextlib.nullcontext()

    def _rec(self, **kw):
        if self.trace is not None:
            for k, v in kw.items():
                self.trace.setdefault(k, []).append(v)

    # -- RoI extractors: one launch over all levels -------------------------------------------------------
    def extract(self, feats: StagedLevels, rois: torch.Tensor, out_size: int, sampling_ratio: int, semantic: Optional[StagedLevels] = None,
                branch: str = "bbox") -> torch.Tensor:
        """`semantic`: the staged semantic feature map; when cfg.semantic_fusion names this branch its RoI features are
        added INSIDE the same launch: as one more summed level (mask branch, same output size), or pooled at twice the
        output size and 2x2-averaged (bbox branch: adaptive_avg_pool2d of the 14x14 semantic RoIAlign, folded into the
        sampling grid -- see nuhtc_roi_align_cg32's pool2)."""
        cfg = self.cfg
        fuse = semantic is not None and branch in cfg.semantic_fusion
        if cfg.extractor == "attention":
            from .mmcv_ops import attention_pool
            L_all = min(len(feats), len(cfg.featmap_strides))
            bias = None
            for i in range(cfg.sum_levels, L_all):
                # the reference hard-codes the level stride as 4 * 2**i (roi_extractors_cus.py:222)
                bias = attention_pool(feats.nchw[i].float(), rois, 4 * 2 ** i, float(cfg.attention_thres), out=bias)
            lv = feats.sub(range(cfg.sum_levels))
            scales = [1.0 / s_ for s_ in cfg.featmap_strides[: cfg.sum_levels]]
            pool2 = [False] * cfg.sum_levels
            if fuse:
                assert cfg.semantic_out in (out_size, 2 * out_size), "semantic RoI size must equal the branch size or twice it"
                lv = lv.cat(semantic)
                scales = scales + [1.0 / cfg.semantic_stride]
                pool2 = pool2 + [cfg.semantic_out == 2 * out_size]
            return roi_align_levels(lv, rois, out_size, scales, sampling_ratio, True, mode="sum", bias=bias,
                                    pool2=pool2 if any(pool2) else None)
        if fuse:
            raise NotImplementedError("semantic fusion is wired for extractor='attention' (the shipped NuHTC configs)")
        if cfg.extractor == "single":
            n = min(len(feats), len(cfg.featmap_strides))
            lv = feats.sub(range(n))
            return roi_align_levels(lv, rois, out_size, [1.0 / s for s in cfg.featmap_strides[:n]], sampling_ratio,
                                    True, mode="route", finest_scale=cfg.finest_scale)
        if cfg.extractor == "sum":
            lv = feats.sub(range(cfg.sum_levels))
            return roi_align_levels(lv, rois, out_size, [1.0 / s for s in cfg.featmap_strides[: cfg.sum_levels]],
                                    sampling_ratio, True, mode="sum")
        raise ValueError(cfg.extractor)

    # -- the stage ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def run(self, feats, rois: torch.Tensor, max_rois_per_tile: Optional[int] = None,
            semantic_feat: Optional[torch.Tensor] = None) -> RoIStageResult:
        """feats: the FPN levels of the batch ([B,C,H_l,W_l] fp32, fp16 or bf16 CUDA tensors) or an already staged
        ``StagedLevels``.  The kernel layout is staged ONCE here and handed to the four RoIAlign calls explicitly (no cache
        involved).  semantic_feat [B,C,H/stride,W/stride]: the semantic head's feature map (cfg.semantic_fusion), in the
        levels' dtype."""
        cfg = self.cfg
        with self._t("stage_layout"):
            feats = stage_levels(feats)
            sem = stage_levels([semantic_feat]) if (semantic_feat is not None and cfg.semantic_fusion) else None
        B = feats.B
        dev = rois.device
        K = rois.shape[0]
        C = cfg.num_classes
        tile_of_roi = rois[:, 0].to(torch.int32)
        K0 = self._const(dev)
        ms_scores = []
        bbox_pred = None
        for i in range(cfg.num_stages):
            with self._t("roi_align_bbox"):
                bbox_feats = self.extract(feats, rois, cfg.bbox_out, cfg.bbox_sampling_ratio, sem, "bbox")
            self._rec(bbox_rois=rois, bbox_feats=bbox_feats)
            cls_score, bbox_pred = self.bbox_heads[i](bbox_feats)
            ms_scores.append(cls_score)
            if i < cfg.num_stages - 1:
                # regress_by_class with reg_class_agnostic=True (mmdet bbox_head.py:459-496), force_fp32 on bbox_pred
                rois = det_ops.delta2bbox(rois, bbox_pred.float(), stds=cfg.stage_stds[i], max_shape=cfg.img_shape)
        cls_score = sum(ms_scores) / float(len(ms_scores))   # in the heads' dtype, as simple_test averages them
        scores = self.score_fn(cls_score.float())           # get_bboxes is force_fp32 on cls_score / bbox_pred
        # rescale=True: detections live in the tile frame (bbox_head.py:373-376)
        bboxes = det_ops.delta2bbox(rois, bbox_pred.float(), stds=cfg.stage_stds[cfg.num_stages - 1], max_shape=cfg.img_shape,
                                    divide_by=cfg.scale_factor)[:, 1:]

        # multiclass_nms for every tile at once (nuhtc/models/bbox_head.py:12-102): class-agnostic boxes are
        # expanded per class, candidates at or below score_thr are parked in a negative group, the rest go
        # through one grouped NMS launch with the per-image class offsets.
        cand_boxes, cand_scores, cand_labels, cand_tile, groups = det_ops.multiclass_candidates(bboxes, scores, rois, C, cfg.score_thr)
        if max_rois_per_tile is None:
            max_rois_per_tile = int(torch.bincount(tile_of_roi.long(), minlength=B).max().item())
        with self._t("nms"):
            # decoded boxes are clamped to the frame (max_shape), so no coordinate is negative: class segments are exact
            # capacity is per (tile, class) segment: a RoI contributes one candidate per class
            keep, gstart, gcount, status = nms_groups(cand_boxes, cand_scores, cand_labels, groups, B, max_rois_per_tile,
                                                      cfg.nms_iou, 0, "offset", num_classes=C)
        self._rec(nms_boxes=bboxes, nms_scores=scores, nms_keep=keep, nms_start=gstart, nms_count=gcount)
        # max_per_img truncation WITHOUT a host round trip: every tile gets max_per_img detection slots; slot r of tile
        # b is its r-th kept candidate (score order) or invalid.  Invalid slots carry a box far outside the frame (RoIAlign
        # and paste see nothing there) and tile -1 (the mask NMS ignores them), so no kernel needs the counts on the host.
        if cfg.max_per_img > 0:
            det_boxes, det_scores, det_labels, det_tile, det_valid, det_cand, mask_rois = det_ops.detection_slots(
                keep, gstart, gcount, cfg.max_per_img, cand_boxes, cand_scores, cand_labels, cand_tile, cfg.scale_factor)
        else:  # unbounded detections per tile: sizes are data dependent, read them back
            host = torch.stack([gstart, gcount]).cpu()
            idx = torch.cat([torch.arange(s_, s_ + c_, device=dev) for s_, c_ in zip(host[0].tolist(), host[1].tolist())]) \
                if int(host[1].sum()) > 0 else torch.zeros(0, dtype=torch.int64, device=dev)
            det_cand = keep[idx]
            det_valid = torch.ones_like(det_cand, dtype=torch.bool)
        if cfg.max_per_img <= 0:
            det_boxes, det_scores, det_labels = cand_boxes[det_cand].contiguous(), cand_scores[det_cand].contiguous(), cand_labels[det_cand]
            det_tile = cand_tile[det_cand].contiguous()
            mask_rois = torch.cat([det_tile.to(torch.float32)[:, None], det_boxes * cfg.scale_factor], dim=1)
        D = det_boxes.shape[0]

        # mask branch: RoIAlign 14x14 on the detections (network frame), mask head, paste into the tile frame
        with self._t("roi_align_mask"):
            mask_feats = self.extract(feats, mask_rois, cfg.mask_out, cfg.mask_sampling_ratio, sem, "mask")
        self._rec(mask_rois=mask_rois, mask_feats=mask_feats)
        logits = self.mask_head(mask_feats, det_cand)
        probs = logits.sigmoid().float()   # the paste works in fp32 (mmdet's _do_paste_mask casts the probabilities)
        H, W = cfg.ori_shape
        # the bit rows (+ area / tight box) feed the mask NMS; the dense uint8 frames are what get_seg_masks returns.
        # Both come straight from the 28x28 maps: re-reading 64 KB per nucleus to pack it would cost more than
        # evaluating its ~1e3 reachable pixels twice.
        masks = None
        side = None
        if cfg.dense_masks and cfg.fused_dense_bits and W % 16 == 0:
            # one evaluation of every mask writes the dense frame (each byte once) and the bit rows
            with self._t("paste"):
                masks, bits, area, bbox = paste_masks_dense_bits(probs, det_boxes, H, W, cfg.mask_thr_binary)
        else:
            with self._t("paste_bits"):
                bits, area, bbox = paste_masks(probs, det_boxes, H, W, thr=cfg.mask_thr_binary, kind="bits", want_stats=True)
            # the dense frames are an output only (mask NMS and contours read the bit rows), and writing them is pure HBM
            # traffic while the mask NMS scan and the contour walk are latency bound: they run side by side on a forked stream
            if cfg.dense_masks:
                main = torch.cuda.current_stream(dev)
                if cfg.overlap_dense_paste and not (self.timer is not None and getattr(self.timer, 'enabled', True)):  # per-op timing keeps one stream
                    side = self._side_stream(dev)
                    side.wait_stream(main)
                with torch.cuda.stream(side) if side is not None else contextlib.nullcontext():
                    with self._t("paste"):
                        masks = paste_masks(probs, det_boxes, H, W, thr=cfg.mask_thr_binary, kind="bin")
                if side is not None:
                    masks.record_stream(main)
        self._rec(paste_probs=probs, paste_boxes=det_boxes)

        if not cfg.tile_postprocess:
            if side is not None:
                torch.cuda.current_stream(dev).wait_stream(side)
            return RoIStageResult(det_boxes, det_scores, det_labels, det_tile, masks, bits, area, None, None, None,
                                  det_valid=det_valid, det_cand=det_cand, status=(status,))
        # tools/infer_wsi.py:510-521 margin / min_area filter, then per-tile mask NMS (:526)
        tile_ids = det_ops.tile_filter(det_boxes, area, det_tile, cfg.margin, H, W, cfg.min_area)
        cap = cfg.max_per_img if cfg.max_per_img > 0 else max(D, 1)
        with self._t("mask_nms"):
            keep2, tstart, tcount, st2 = mask_nms_device(bits, area, bbox, det_scores, W, cfg.mask_nms_thr, tile=tile_ids,
                                                         num_tiles=B, max_tile_size=cap)
        self._rec(mnms_tile=tile_ids)
        cxy = ccnt = None
        stat = (status, st2)
        if cfg.contour_max_pts > 0:
            with self._t("contours"):   # only the survivors of the mask NMS are traced (infer_wsi.py:527-529)
                sel = det_ops.keep_flags(keep2, tstart, tcount, cap, D)
                cxy, ccnt, st3 = mask_contours(bits, W, cfg.contour_max_pts, check=False, bbox=bbox, select=sel)
            stat = (status, st2, st3)
        if side is not None:
            torch.cuda.current_stream(dev).wait_stream(side)
        return RoIStageResult(det_boxes, det_scores, det_labels, det_tile, masks, bits, area, keep2, tstart, tcount,
                              det_valid=det_valid, det_cand=det_cand, status=stat, contour_xy=cxy, contour_count=ccnt)
