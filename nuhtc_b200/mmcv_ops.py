"""Drop-in mirrors of the mmcv.ops surface NuHTC's RoI stage uses, backed by libnuhtc_b200.so.

Signatures, argument meaning and error behaviour follow mmcv-full 1.7.2
(``mmcv.ops.RoIAlign`` / ``roi_align`` / ``nms`` / ``batched_nms``) as the reference calls them:
  * RoIAlign built by ``layer_cls(spatial_scale=1/s, **cfg)`` --
    /root/reference/thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/base_roi_extractor.py:54-60
  * ``roi_align(...)`` called positionally -- /root/reference/nuhtc/core/masks/structures.py:48-50
  * ``batched_nms(boxes, scores, idxs, nms_cfg, class_agnostic)`` --
    /root/reference/nuhtc/models/bbox_head.py:93,208
Forward (inference) only; GPU only.
"""
from __future__ import annotations

import ctypes
import os
from collections import OrderedDict
from typing import Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L

_RA_STATS = os.environ.get("NUHTC_RA_STATS") == "1"

__all__ = ["RoIAlign", "roi_align", "nms", "batched_nms", "roi_align_levels", "to_nhwc", "to_cg32", "clear_layout_cache",
           "layout_cache", "StagedLevels", "stage_levels",
           "nms_groups", "attention_pool"]


def _pair(x) -> Tuple[int, int]:
    if isinstance(x, (tuple, list)):
        assert len(x) == 2
        return int(x[0]), int(x[1])
    return int(x), int(x)


# ----------------------------------------------------------------------------- layout staging
# The RoIAlign kernels want the channel axis contiguous.  A level that arrives NCHW is re-laid out by our own kernels:
#   * CG32  [B][C/32][H][W][32]  -- the strip-shared kernels (7x7 / 14x14 outputs, C % 32 == 0): nuhtc_to_cg32
#   * NHWC  [B][H][W][C]         -- the attention pooling and the round-1 per-RoI kernels: nuhtc_nchw_to_nhwc
# Staging is done ONCE per batch by whoever owns the batch (RoIStage.run, the RoI extractors: `stage_levels`) and the
# staged buffers are passed down explicitly.  An optional cache keyed on (data_ptr, _version, shape) exists for callers
# that go through the per-level mmcv surface (RoIAlign.forward is called level by level, stage by stage); it is OFF by
# default and is never consulted while a CUDA graph is being captured, because `_version` does not see writes made by
# graph replays, by raw-pointer writers or by fresh tensor objects on recycled storage (a stale layout would be silent).
_LAYOUT_CACHE: "OrderedDict[tuple, tuple]" = OrderedDict()
_LAYOUT_CACHE_MAX = 16
_LAYOUT_CACHE_ON = [False]


def clear_layout_cache() -> None:
    _LAYOUT_CACHE.clear()


class layout_cache:
    """``with layout_cache():`` -- remember staged layouts of unmodified source tensors inside the block (e.g. around one
    forward pass that calls RoIAlign level by level).  The caller vouches that the features are only written through
    torch ops on tensors it holds (see the hazard note above); the cache is emptied on exit."""

    def __enter__(self):
        self.prev = _LAYOUT_CACHE_ON[0]
        _LAYOUT_CACHE_ON[0] = True
        return self

    def __exit__(self, *a):
        _LAYOUT_CACHE_ON[0] = self.prev
        if not self.prev:
            clear_layout_cache()


def _cached(x: torch.Tensor, kind: str, make):
    use = _LAYOUT_CACHE_ON[0] and not torch.cuda.is_current_stream_capturing()
    key = (kind, x.data_ptr(), x._version, tuple(x.shape), tuple(x.stride()), x.dtype, x.device.index)
    if use and key in _LAYOUT_CACHE:
        _LAYOUT_CACHE.move_to_end(key)
        return _LAYOUT_CACHE[key][1]
    out = make()
    if use:
        _LAYOUT_CACHE[key] = (x, out)  # holding `x` keeps its storage (and so the key) from being recycled
        while len(_LAYOUT_CACHE) > _LAYOUT_CACHE_MAX:
            _LAYOUT_CACHE.popitem(last=False)
    return out


def to_nhwc(x: torch.Tensor) -> torch.Tensor:
    """[B,C,H,W] fp32 CUDA (any strides) -> contiguous [B,H,W,C] buffer (returned as a [B,H,W,C] tensor)."""
    L.require_cuda(x, "input")
    assert x.dim() == 4 and x.dtype == torch.float32, "expected a 4-D fp32 feature map"
    B, C, H, W = x.shape
    if x.permute(0, 2, 3, 1).is_contiguous():  # already channels_last in memory
        return x.permute(0, 2, 3, 1)
    if not x.is_contiguous():
        x = x.contiguous()

    def make():
        out = torch.empty((B, H, W, C), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            L.check(L.lib().nuhtc_nchw_to_nhwc(x.data_ptr(), out.data_ptr(), B, C, H, W, L.stream_ptr(x.device)), "nchw_to_nhwc")
        L.count("nchw_to_nhwc")
        return out
    return _cached(x, "nhwc", make)


def _levels_dtype(levels: Sequence[torch.Tensor]) -> torch.dtype:
    """The one element type of a set of feature maps: fp32, fp16 or bf16 (ValueError otherwise)."""
    dts = {f.dtype for f in levels}
    if len(dts) != 1:
        raise ValueError(f"feature levels must share one dtype, got {sorted(str(d) for d in dts)}")
    dt = dts.pop()
    if dt not in L.DTYPE_CODES:
        raise ValueError(f"feature levels must be float32, float16 or bfloat16, got {dt}")
    return dt


def to_cg32(x: torch.Tensor) -> torch.Tensor:
    """[B,C,H,W] fp32, fp16 or bf16 CUDA, C % 32 == 0 (NCHW-contiguous or channels_last) -> [B, C/32, H, W, 32] fp32
    buffer.  A half-precision map is upcast exactly while it is staged: the buffer equals ``to_cg32(x.float())``."""
    L.require_cuda(x, "input")
    assert x.dim() == 4, "expected a 4-D feature map"
    code = L.DTYPE_CODES[_levels_dtype([x])]
    B, C, H, W = x.shape
    assert C % 32 == 0
    cl = x.permute(0, 2, 3, 1).is_contiguous() and not x.is_contiguous()
    if not cl and (not x.is_contiguous() or (H * W) % 4 != 0):
        x = x.contiguous(memory_format=torch.channels_last)   # odd map sizes: go through the line-permutation kernel
        cl = True

    def make():
        out = torch.empty((B, C // 32, H, W, 32), dtype=torch.float32, device=x.device)
        if B > 0:
            with torch.cuda.device(x.device):
                L.check(L.lib().nuhtc_to_cg32_dt(x.data_ptr(), code, out.data_ptr(), B, C, H, W, int(cl), L.stream_ptr(x.device)),
                        "to_cg32")
            L.count("to_cg32")
        return out
    return _cached(x, "cg32", make)


def _fast_path_ok(C: int, ph: int, pw: int) -> bool:
    return ph == pw and ph in (7, 14) and C % 32 == 0


class StagedLevels:
    """FPN levels of one batch, laid out for the RoIAlign kernels.  Build it once per batch with ``stage_levels`` and pass
    it wherever ``feats`` is accepted: the three cascade stages and the mask branch then share one re-layout.
    The levels are fp32, fp16 or bf16, all of one dtype (``self.dtype``, the dtype of the RoI features pooled from them);
    the staged CG32 buffers are fp32 either way."""

    def __init__(self, feats: Sequence[torch.Tensor]):
        f0 = feats[0]
        self.B, self.C = int(f0.shape[0]), int(f0.shape[1])
        self.shapes = [(int(f.shape[2]), int(f.shape[3])) for f in feats]
        self.device = f0.device
        for f in feats:
            L.require_cuda(f, "feats")
            assert f.shape[0] == self.B and f.shape[1] == self.C
        self.dtype = _levels_dtype(feats)
        self.nchw = list(feats)
        self.cg32 = [to_cg32(f) for f in feats] if self.C % 32 == 0 else None

    def __len__(self):
        return len(self.nchw)

    def cat(self, other: "StagedLevels") -> "StagedLevels":
        """these levels followed by `other`'s (same batch and channel count), e.g. FPN levels + the semantic feature map"""
        assert other.B == self.B and other.C == self.C
        if other.dtype != self.dtype:
            raise ValueError(f"feature levels must share one dtype, got {self.dtype} and {other.dtype}")
        o = object.__new__(StagedLevels)
        o.B, o.C, o.device, o.dtype = self.B, self.C, self.device, self.dtype
        o.shapes = self.shapes + other.shapes
        o.nchw = self.nchw + other.nchw
        o.cg32 = None if (self.cg32 is None or other.cg32 is None) else self.cg32 + other.cg32
        return o

    def sub(self, idx: Sequence[int]) -> "StagedLevels":
        o = object.__new__(StagedLevels)
        o.B, o.C, o.device, o.dtype = self.B, self.C, self.device, self.dtype
        o.shapes = [self.shapes[i] for i in idx]
        o.nchw = [self.nchw[i] for i in idx]
        o.cg32 = None if self.cg32 is None else [self.cg32[i] for i in idx]
        return o


def stage_levels(feats) -> StagedLevels:
    return feats if isinstance(feats, StagedLevels) else StagedLevels(list(feats))


def roi_align_levels(feats, rois: torch.Tensor, output_size, spatial_scales: Sequence[float],
                     sampling_ratio: int = 0, aligned: bool = True, mode: str = "route", finest_scale: float = 56.0,
                     impl: str = "auto", out: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                     pool2: Optional[Sequence[bool]] = None) -> torch.Tensor:
    """All FPN levels in ONE call.

    mode 'route': each RoI is pooled on the level SingleRoIExtractor.map_roi_levels picks
                  (single_level_roi_extractor.py:36-55); one level = plain roi_align.
    mode 'sum'  : every RoI is pooled on every level, results summed in level order
                  (AttentionRoIExtractor's RoIAlign branch, roi_extractors_cus.py:213-218,246).
    feats: NCHW CUDA tensors [B,C,H_l,W_l] (NCHW-contiguous or channels_last), or a ``StagedLevels``; fp32, fp16 or bf16,
           all levels of one dtype (ValueError otherwise).  The result has that dtype (a given ``out`` must have it too);
           ``bias`` stays fp32.  Everything is computed in fp32 and each output value is rounded once to the levels'
           dtype (mmcv's ``force_fp32(out_fp16=True)``).  On the channel-group path (impl 'auto', C % 32 == 0, 7x7 or
           14x14) half levels are staged and stored natively; every other shape and impl runs the fp32 kernels between
           ONE ``.float()`` of the levels and ONE rounding of the result (its copy into ``out``), both below.
    pool2: per level (mode 'sum'): the level enters as adaptive_avg_pool2d(RoIAlign(2P x 2P, sampling_ratio=0), P) -- the
           semantic branch of NuHTC's _bbox_forward -- pooled directly at P x P inside the same launch.
    impl : 'auto' (strip-shared kernels on the CG32 layout when the shape allows, else the literal kernel),
           'direct' (literal per-sample kernel, bit-exact with the reference's accumulation order),
           'nhwc' (round-1 per-RoI kernels on the NHWC layout; kept for A/B measurements)."""
    ph, pw = _pair(output_size)
    staged = feats if isinstance(feats, StagedLevels) else None
    nl = len(feats)
    assert 1 <= nl <= L.MAX_LEVELS and len(spatial_scales) == nl
    raw = staged.nchw if staged is not None else list(feats)
    dtype = staged.dtype if staged is not None else _levels_dtype(raw)
    L.require_cuda(rois, "rois")
    assert rois.dim() == 2 and rois.size(1) == 5, "rois must have shape [K,5]"
    B, C = raw[0].shape[0], raw[0].shape[1]
    K = rois.size(0)
    dev = raw[0].device
    rois = rois.to(torch.float32).contiguous()
    if out is None:
        out = torch.empty((K, C, ph, pw), dtype=dtype, device=dev)
    else:
        assert out.shape == (K, C, ph, pw) and out.is_contiguous() and out.dtype == dtype
    if K == 0:
        return out
    if bias is not None:
        assert bias.shape == (K, C) and bias.dtype == torch.float32 and bias.is_cuda
        bias = bias.contiguous()
    for f in raw:
        L.require_cuda(f, "feats")
        assert f.shape[0] == B and f.shape[1] == C
    native = impl == "auto" and _fast_path_ok(C, ph, pw)
    if dtype != torch.float32 and not native:
        # no half-precision kernel for this shape / impl: the fp32 result, rounded once
        res = roi_align_levels([f.float() for f in raw], rois, (ph, pw), spatial_scales, sampling_ratio, aligned, mode,
                               finest_scale, impl, None, bias, pool2)
        return out.copy_(res)
    Hs = (ctypes.c_int * nl)(*[int(f.shape[2]) for f in raw])
    Ws = (ctypes.c_int * nl)(*[int(f.shape[3]) for f in raw])
    sc = (ctypes.c_float * nl)(*[float(s) for s in spatial_scales])
    m = {"route": L.ROI_ROUTE, "sum": L.ROI_SUM}[mode]
    lib = L.lib()
    if native:
        bufs = staged.cg32 if staged is not None else [to_cg32(f) for f in raw]
        ptrs = (ctypes.c_void_p * nl)(*[b.data_ptr() for b in bufs])
        wsb = lib.nuhtc_roi_align_workspace_bytes(Hs, Ws, nl, B, K, ph, pw)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        p2 = None if pool2 is None else (ctypes.c_int * nl)(*[int(bool(v)) for v in pool2])
        with torch.cuda.device(dev):
            rc = lib.nuhtc_roi_align_cg32_dt(ptrs, Hs, Ws, sc, nl, B, C, rois.data_ptr(), K, ph, pw, int(sampling_ratio),
                                             int(bool(aligned)), m, float(finest_scale), p2, out.data_ptr(), L.DTYPE_CODES[dtype],
                                             L.ptr(bias), ws.data_ptr(), wsb, L.stream_ptr(dev))
        L.check(rc, "roi_align_cg32")
        L.count("roi_align_strip")
        if _RA_STATS:   # debugging aid (synchronises): how many RoIs missed the strip kernel
            print(f"RA_STATS P={ph} K={K} leftover={int(ws[8:12].view(torch.int32).item())}", flush=True)
        return out
    if pool2 is not None and any(pool2):
        raise NotImplementedError("pool2 levels need the channel-group path (C % 32 == 0, 7x7 or 14x14 output)")
    use_nhwc = impl == "nhwc" and ph == pw and ph in (7, 14) and C % 64 == 0
    bufs = [to_nhwc(f) for f in raw] if use_nhwc else [f if f.is_contiguous() else f.contiguous() for f in raw]
    layout = L.LAYOUT_NHWC if use_nhwc else L.LAYOUT_NCHW
    ptrs = (ctypes.c_void_p * nl)(*[b.data_ptr() for b in bufs])
    with torch.cuda.device(dev):
        rc = lib.nuhtc_roi_align_fwd(ptrs, Hs, Ws, sc, nl, B, C, layout, rois.data_ptr(), K, ph, pw, int(sampling_ratio),
                                     int(bool(aligned)), m, float(finest_scale),
                                     L.IMPL_AUTO if use_nhwc else L.IMPL_DIRECT, out.data_ptr(), L.ptr(bias),
                                     L.stream_ptr(dev))
    L.check(rc, "roi_align_fwd")
    L.count("roi_align")
    return out


def attention_pool(feat: torch.Tensor, rois: torch.Tensor, stride: float, thres: float = 0.0,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Cosine-attention global pooling of one level (AttentionRoIExtractor, roi_extractors_cus.py:220-238):
    feat [B,C,H,W] fp32 CUDA (C <= 64), rois [K,5] -> [K,C]; with ``out`` given the result is ADDED to it."""
    L.require_cuda(feat, "feat")
    L.require_cuda(rois, "rois")
    B, C, H, W = feat.shape
    K = rois.shape[0]
    dev = feat.device
    nhwc = to_nhwc(feat)
    rois = rois.to(torch.float32).contiguous()
    acc = out is not None
    if out is None:
        out = torch.empty((K, C), dtype=torch.float32, device=dev)
    if K == 0:
        return out
    lib = L.lib()
    wsb = lib.nuhtc_attention_pool_workspace_bytes(K, B)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        rc = lib.nuhtc_attention_pool(nhwc.data_ptr(), B, H, W, C, rois.data_ptr(), K, float(stride), float(thres), int(acc),
                                      out.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb, L.stream_ptr(dev))
    L.check(rc, "attention_pool")
    L.count("attention_pool")
    return out


def roi_align(input, rois, output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode="avg", aligned=True):
    """mmcv.ops.roi_align(input, rois, output_size, spatial_scale, sampling_ratio, pool_mode, aligned)."""
    if pool_mode != "avg":
        raise NotImplementedError("nuhtc_b200.roi_align implements pool_mode='avg' (the only mode NuHTC configures)")
    assert rois.size(1) == 5, "RoI must be (idx, x1, y1, x2, y2)!"
    return roi_align_levels([input], rois, output_size, [spatial_scale], sampling_ratio, aligned, mode="route")


class RoIAlign(nn.Module):
    """mmcv.ops.RoIAlign(output_size, spatial_scale=1.0, sampling_ratio=0, pool_mode='avg', aligned=True,
    use_torchvision=False); ``forward(input [N,C,H,W], rois [K,5]) -> [K,C,ph,pw]``."""

    def __init__(self, output_size, spatial_scale: float = 1.0, sampling_ratio: int = 0, pool_mode: str = "avg",
                 aligned: bool = True, use_torchvision: bool = False):
        super().__init__()
        self.output_size = _pair(output_size)
        self.spatial_scale = float(spatial_scale)
        self.sampling_ratio = int(sampling_ratio)
        self.pool_mode = pool_mode
        self.aligned = aligned
        self.use_torchvision = use_torchvision
        if use_torchvision:
            raise NotImplementedError("use_torchvision=True is not a B200-native path")

    def forward(self, input: torch.Tensor, rois: torch.Tensor) -> torch.Tensor:
        return roi_align(input, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.pool_mode, self.aligned)

    def __repr__(self):
        return (f"{self.__class__.__name__}(output_size={self.output_size}, spatial_scale={self.spatial_scale}, "
                f"sampling_ratio={self.sampling_ratio}, pool_mode={self.pool_mode}, aligned={self.aligned}, "
                f"use_torchvision={self.use_torchvision})")


# ----------------------------------------------------------------------------- NMS
_MODE = {"agnostic": L.NMS_AGNOSTIC, "offset": L.NMS_OFFSET, "perclass": L.NMS_PERCLASS,
         "perclass_raw": L.NMS_PERCLASS_RAW}


def nms_groups(boxes: torch.Tensor, scores: torch.Tensor, labels: Optional[torch.Tensor], groups: Optional[torch.Tensor],
               num_groups: int, max_group_size: int, iou_threshold: float, offset: int = 0, mode: str = "agnostic",
               num_classes: int = 0):
    """Batched greedy NMS over independent groups (images), no host sync.

    ``num_classes`` > 0 sorts into (group, class) segments (labels < num_classes): same result, 5x less work for 5
    classes; ``max_group_size`` then is the capacity of one (group, class) segment (the group's own size always works but
    sizes the pair matrix for it).  With mode 'offset' that requires non-negative box coordinates (status 3 otherwise, see the header).

    Returns (keep [N] int64, group_start [G] int64, group_count [G] int64, status [1] int32), all on the device:
    group g's kept original indices, score-descending, are keep[group_start[g] : group_start[g]+group_count[g]]."""
    L.require_cuda(boxes, "boxes")
    N = boxes.size(0)
    dev = boxes.device
    boxes = boxes.to(torch.float32).contiguous()
    scores = scores.to(torch.float32).contiguous()
    assert boxes.dim() == 2 and boxes.size(1) == 4 and scores.numel() == N
    if labels is not None:
        labels = labels.to(torch.int64).contiguous()
    if groups is not None:
        groups = groups.to(torch.int32).contiguous()
    max_group_size = max(1, min(int(max_group_size), max(N, 1)))
    keep = torch.empty(max(N, 1), dtype=torch.int64, device=dev)
    gstart = torch.empty(num_groups, dtype=torch.int64, device=dev)
    gcount = torch.empty(num_groups, dtype=torch.int64, device=dev)
    status = torch.empty(1, dtype=torch.int32, device=dev)
    lib = L.lib()
    ncls = int(num_classes) if mode != "agnostic" else 0
    wsb = lib.nuhtc_nms_workspace_bytes(N, num_groups, max_group_size, ncls)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.nuhtc_nms(boxes.data_ptr(), scores.data_ptr(), L.ptr(labels), L.ptr(groups), N, num_groups, max_group_size,
                           float(iou_threshold), int(offset), _MODE[mode], ncls, keep.data_ptr(), gstart.data_ptr(),
                           gcount.data_ptr(), status.data_ptr(), ws.data_ptr(), wsb, L.stream_ptr(dev))
    L.check(rc, "nms")
    L.count("nms")
    return keep, gstart, gcount, status


def _nms_single(boxes, scores, labels, iou_threshold, offset, mode) -> torch.Tensor:
    N = boxes.size(0)
    if N == 0:
        return torch.empty(0, dtype=torch.int64, device=boxes.device)
    ncls = 0
    if mode in ("perclass", "perclass_raw") and labels is not None:
        # one NMS per class id, exactly mmcv's loop: the ids become sort segments (dense ids 0..n-1 expected; a sparse id
        # space just leaves empty segments)
        top = int(labels.max().item()) + 1
        if int(labels.min().item()) >= 0 and top <= 4096:
            ncls = top
    elif mode == "offset" and labels is not None:
        # below split_thr mmcv runs ONE nms over the offset boxes.  Class segments give the identical result as long as no
        # coordinate is negative (then boxes of different classes cannot overlap after the offset) and do 1/num_classes
        # of the pair tests; the kernel verifies the precondition itself (status 3) and the call is repeated without
        # segments when it does not hold.
        top = int(labels.max().item()) + 1
        if int(labels.min().item()) >= 0 and top <= 4096:
            ncls = top
    keep, _, gcount, status = nms_groups(boxes, scores, labels, None, 1, N, iou_threshold, offset, mode, num_classes=ncls)
    k, st = (int(v) for v in torch.stack([gcount[0], status[0].to(gcount.dtype)]).tolist())  # one D2H: mmcv's op syncs too
    if st == 3 and ncls > 0:   # a negative coordinate: the all-pairs test on the offset boxes is the contract
        keep, _, gcount, status = nms_groups(boxes, scores, labels, None, 1, N, iou_threshold, offset, mode, num_classes=0)
        k, st = (int(v) for v in torch.stack([gcount[0], status[0].to(gcount.dtype)]).tolist())
    if st != 0:
        raise L.NuhtcError(f"nms: device status {st} (1: a sort segment exceeded its capacity, 2: a label outside "
                           f"[0, num_classes), 3: negative coordinate with class segments)")
    return keep[:k]


def nms(boxes, scores, iou_threshold, offset=0, score_threshold=0, max_num=-1):
    """mmcv.ops.nms: returns (dets [k,5], inds [k] int64), score-descending.  Accepts Tensor or ndarray."""
    assert isinstance(boxes, (torch.Tensor, np.ndarray))
    assert isinstance(scores, (torch.Tensor, np.ndarray))
    is_numpy = False
    if isinstance(boxes, np.ndarray):
        is_numpy = True
        boxes = torch.from_numpy(boxes).cuda()
    if isinstance(scores, np.ndarray):
        scores = torch.from_numpy(scores).cuda()
    assert boxes.size(1) == 4
    assert boxes.size(0) == scores.size(0)
    assert offset in (0, 1)
    L.require_cuda(boxes, "boxes")
    b, s = boxes, scores
    valid_inds = None
    if score_threshold > 0:
        valid_mask = scores > score_threshold
        b, s = boxes[valid_mask], scores[valid_mask]
        valid_inds = torch.nonzero(valid_mask, as_tuple=False).squeeze(dim=1)
    inds = _nms_single(b, s, None, iou_threshold, offset, "agnostic")
    if max_num > 0:
        inds = inds[:max_num]
    if valid_inds is not None:
        inds = valid_inds[inds]
    dets = torch.cat((boxes[inds], scores[inds].reshape(-1, 1)), dim=1)
    if is_numpy:
        dets = dets.cpu().numpy()
        inds = inds.cpu().numpy()
    return dets, inds


def batched_nms(boxes: torch.Tensor, scores: torch.Tensor, idxs: torch.Tensor, nms_cfg: Optional[dict],
                class_agnostic: bool = False):
    """mmcv.ops.batched_nms.  The class offset ``idxs * (boxes.max() + 1)`` is applied inside the kernel in
    the same fp32 arithmetic (it perturbs IoUs at the 1e-4 px level, so it is part of the contract); at or
    above ``split_thr`` only same-class pairs are tested, exactly like mmcv's per-class loop."""
    if nms_cfg is None:
        scores, inds = scores.sort(descending=True, stable=True)
        boxes = boxes[inds]
        return torch.cat([boxes, scores[:, None]], -1), inds
    L.require_cuda(boxes, "boxes")
    nms_cfg_ = nms_cfg.copy()
    class_agnostic = nms_cfg_.pop("class_agnostic", class_agnostic)
    nms_type = nms_cfg_.pop("type", "nms")
    if nms_type != "nms":
        raise NotImplementedError(f"nms type {nms_type!r}: NuHTC configures type='nms' only")
    split_thr = nms_cfg_.pop("split_thr", 10000)
    iou_threshold = nms_cfg_.pop("iou_threshold")
    offset = nms_cfg_.pop("offset", 0)
    score_threshold = nms_cfg_.pop("score_threshold", 0)
    max_num = nms_cfg_.pop("max_num", -1)
    if nms_cfg_:
        raise TypeError(f"unexpected nms_cfg keys {sorted(nms_cfg_)}")
    assert boxes.size(-1) == 4, "rotated boxes are outside the NuHTC path"
    b, s, lab = boxes, scores, idxs
    valid_inds = None
    if score_threshold > 0:
        valid_mask = scores > score_threshold
        b, s, lab = boxes[valid_mask], scores[valid_mask], idxs[valid_mask]
        valid_inds = torch.nonzero(valid_mask, as_tuple=False).squeeze(dim=1)
    split = boxes.shape[0] >= split_thr  # mmcv then runs one nms per id in `idxs`, class_agnostic or not
    if class_agnostic:
        mode = "perclass_raw" if split else "agnostic"
    else:
        mode = "perclass" if split else "offset"
        # mmcv takes boxes.max() over the tensor it is given, i.e. before any score filtering
        if valid_inds is not None and b.shape[0] != boxes.shape[0]:
            raise NotImplementedError("score_threshold together with class offsets is not used by NuHTC")
    keep = _nms_single(b, s, None if mode == "agnostic" else lab, iou_threshold, offset, mode)
    if max_num > 0:
        keep = keep[:max_num]
    if valid_inds is not None:
        keep = valid_inds[keep]
    return torch.cat([boxes[keep], scores[keep][:, None]], -1), keep
