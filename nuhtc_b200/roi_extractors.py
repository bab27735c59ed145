"""RoI extractors with the reference's call signature ``forward(feats, rois, roi_scale_factor=None)``, backed by ONE
multi-level RoIAlign launch (+ the fused attention pooling for AttentionRoIExtractor).

  * ``SingleRoIExtractor``     thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:10-115
  * ``AttentionRoIExtractor``  nuhtc/models/roi_extractors_cus.py:164-259 (aggregation='sum', no pre/post plugin modules:
                               what the four shipped configs use)
Both are plain ``nn.Module``s built from the same config dict (``roi_layer=dict(type='RoIAlign', output_size=..,
sampling_ratio=..)``, ``out_channels``, ``featmap_strides``); inference only, GPU only.

Precision: the reference's extractors are ``@force_fp32(apply_to=('feats',), out_fp16=True)``.  Here fp32, fp16 or bf16
feats are all accepted and the RoI features come back in the feats' dtype, computed in fp32 and rounded once -- what
force_fp32 does for fp16 once ``wrap_fp16_model`` has set ``fp16_enabled``, without its casts of the levels and results.
"""
from __future__ import annotations

from typing import Optional, Sequence

import torch
import torch.nn as nn

from .mmcv_ops import RoIAlign, attention_pool, roi_align_levels

__all__ = ["SingleRoIExtractor", "AttentionRoIExtractor"]


def _roi_rescale(rois: torch.Tensor, scale_factor: float) -> torch.Tensor:
    """BaseRoIExtractor.roi_rescale (base_roi_extractor.py:62-84)."""
    cx = (rois[:, 1] + rois[:, 3]) * 0.5
    cy = (rois[:, 2] + rois[:, 4]) * 0.5
    w = rois[:, 3] - rois[:, 1]
    h = rois[:, 4] - rois[:, 2]
    new_w = w * scale_factor
    new_h = h * scale_factor
    return torch.stack((rois[:, 0], cx - new_w * 0.5, cy - new_h * 0.5, cx + new_w * 0.5, cy + new_h * 0.5), dim=-1)


class _BaseRoIExtractor(nn.Module):
    def __init__(self, roi_layer: dict, out_channels: int, featmap_strides: Sequence[int], init_cfg=None):
        super().__init__()
        cfg = dict(roi_layer)
        layer_type = cfg.pop("type")
        if layer_type != "RoIAlign":
            raise NotImplementedError(f"roi_layer type {layer_type!r}: NuHTC configures RoIAlign only")
        self.roi_layers = nn.ModuleList([RoIAlign(spatial_scale=1 / s, **cfg) for s in featmap_strides])
        self.out_channels = out_channels
        self.featmap_strides = list(featmap_strides)
        self.fp16_enabled = False   # set by mmcv's wrap_fp16_model; the output dtype follows the feats either way

    @property
    def num_inputs(self) -> int:
        return len(self.featmap_strides)


class SingleRoIExtractor(_BaseRoIExtractor):
    """Each RoI is pooled on the one level ``map_roi_levels`` picks; the routing runs inside the kernel."""

    def __init__(self, roi_layer, out_channels, featmap_strides, finest_scale=56, init_cfg=None):
        super().__init__(roi_layer, out_channels, featmap_strides, init_cfg)
        self.finest_scale = finest_scale

    def map_roi_levels(self, rois: torch.Tensor, num_levels: int) -> torch.Tensor:
        scale = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
        target_lvls = torch.floor(torch.log2(scale / self.finest_scale + 1e-6))
        return target_lvls.clamp(min=0, max=num_levels - 1).long()

    @torch.no_grad()
    def forward(self, feats, rois, roi_scale_factor=None):
        l0 = self.roi_layers[0]
        num_levels = len(feats)
        if num_levels == 1:
            if len(rois) == 0:
                return feats[0].new_zeros(0, self.out_channels, *l0.output_size)
            return l0(feats[0], rois)
        # the level is chosen from the un-rescaled RoIs (single_level_roi_extractor.py:82-85): when a rescale is asked
        # for, route on the host side of the op and pool the rescaled boxes level by level
        if roi_scale_factor is not None:
            lv = self.map_roi_levels(rois, num_levels)
            rois = _roi_rescale(rois, roi_scale_factor)
            out = feats[0].new_zeros(rois.size(0), self.out_channels, *l0.output_size)
            for i in range(num_levels):
                inds = (lv == i).nonzero(as_tuple=False).squeeze(1)
                if inds.numel() > 0:
                    out[inds] = self.roi_layers[i](feats[i], rois[inds])
            return out
        return roi_align_levels(list(feats), rois, l0.output_size, [l.spatial_scale for l in self.roi_layers[:num_levels]],
                                l0.sampling_ratio, l0.aligned, mode="route", finest_scale=float(self.finest_scale))


class AttentionRoIExtractor(_BaseRoIExtractor):
    """Levels below ``start_level`` are pooled with RoIAlign on EVERY RoI and summed; levels from ``start_level`` on
    contribute one cosine-attention pooled vector per RoI, broadcast over the bins.  One attention launch per such level
    and one RoIAlign launch in all; the broadcast-add is fused into the RoIAlign store."""

    def __init__(self, aggregation="sum", pre_cfg=None, post_cfg=None, start_level=2, thres=0, **kwargs):
        super().__init__(**kwargs)
        if aggregation != "sum" or pre_cfg is not None or post_cfg is not None:
            raise NotImplementedError("AttentionRoIExtractor: aggregation='sum' without pre/post modules (the shipped configs)")
        self.aggregation = aggregation
        self.start_level = list(range(int(start_level), 10)) if not isinstance(start_level, list) else start_level
        self.thres = thres

    @torch.no_grad()
    def forward(self, feats, rois, roi_scale_factor=None):
        l0 = self.roi_layers[0]
        if len(feats) == 1:
            return l0(feats[0], rois)
        if rois.size(0) == 0:
            return feats[0].new_zeros(0, self.out_channels, *l0.output_size)
        if roi_scale_factor is not None:
            rois = _roi_rescale(rois, roi_scale_factor)
        num_levels = len(feats)
        pooled = [i for i in range(num_levels) if i not in self.start_level]
        attn = [i for i in range(num_levels) if i in self.start_level]
        bias: Optional[torch.Tensor] = None
        for i in attn:
            # the reference hard-codes the level stride as 4 * 2**i (roi_extractors_cus.py:222)
            bias = attention_pool(feats[i].float(), rois, 4 * 2 ** i, float(self.thres), out=bias)   # fp32 kernel, small levels
        if not pooled:
            return bias[:, :, None, None].expand(-1, -1, *l0.output_size).contiguous().to(feats[0].dtype)
        return roi_align_levels([feats[i] for i in pooled], rois, l0.output_size, [self.roi_layers[i].spatial_scale for i in pooled],
                                l0.sampling_ratio, l0.aligned, mode="sum", bias=bias)
