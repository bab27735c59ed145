"""The detector's test-time image pipeline on the GPU (the tile loader of SURVEY.md 8f-4).

``inference_detector(model, [np.ndarray]*B)`` (tools/infer_wsi.py:485 -> mmdet/apis/inference.py:90-153) runs the mmdet 2.x
test pipeline per tile on the CPU -- cv2 bilinear upscale, float32, BGR->RGB, (x - mean) / std, pad to a multiple of 32,
HWC->CHW -- and then copies the fp32 batch to the device: 50.3 MB for 16 tiles at 512x512 where the uint8 tiles are 3.1 MB.
Here the uint8 tiles cross PCIe and ONE kernel (``nuhtc_preprocess_tiles``, csrc/preprocess.cu) produces the backbone's
input, bit-identical to what mmdet's pipeline hands the model.

Only the pipeline the NuHTC configs use is supported; ``TilePipeline.from_cfg`` raises ``NotImplementedError`` for anything
else rather than computing something different.  There is no CPU path: host tiles are input only.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from . import _lib as L

__all__ = ["TilePipeline", "inference_detector"]

# Collect's default meta_keys (mmdet/datasets/pipelines/formatting.py)
_META_KEYS = ("filename", "ori_filename", "ori_shape", "img_shape", "pad_shape", "scale_factor", "flip", "flip_direction",
              "img_norm_cfg")


def _unsupported(what: str):
    raise NotImplementedError(f"TilePipeline: {what} is not supported (only the NuHTC test pipeline: MultiScaleFlipAug("
                              "scale_factor=s >= 1, flip=False)[Resize(keep_ratio=True), RandomFlip, Normalize, "
                              "Pad(size_divisor), ImageToTensor / DefaultFormatBundle, Collect(['img'])])")


def _check_only(step, allowed: Dict[str, object]):
    """Every key of the transform dict other than `type` must be in `allowed` and, where a value is given, equal to it."""
    for k, v in step.items():
        if k == "type":
            continue
        if k not in allowed:
            _unsupported(f"{step['type']}({k}=...)")
        if allowed[k] is not None and v != allowed[k] and not (isinstance(allowed[k], tuple) and v in allowed[k]):
            _unsupported(f"{step['type']}({k}={v!r})")


class TilePipeline:
    """uint8 HWC tiles -> (img [B,3,Hp,Wp] fp32 on the device, img_metas list[dict]) as mmdet's test pipeline + collate.

    Host tiles are staged in one reusable pinned buffer and copied with ``Tensor.copy_(non_blocking=True)``; an event
    recorded after the copy is waited on before the buffer is refilled, so a call returns without waiting for the GPU."""

    def __init__(self, scale_factor: float, mean: Sequence[float], std: Sequence[float], to_rgb: bool = True,
                 size_divisor: int = 32):
        if not scale_factor >= 1.0:
            _unsupported(f"scale_factor={scale_factor!r} (< 1 is a downscale: cv2 switches to INTER_AREA there)")
        if int(size_divisor) != size_divisor or size_divisor < 1:
            _unsupported(f"Pad(size_divisor={size_divisor!r})")
        self.scale_factor = float(scale_factor)
        self.mean = np.asarray(mean, dtype=np.float32).reshape(3)   # Normalize.__init__ stores float32 arrays
        self.std = np.asarray(std, dtype=np.float32).reshape(3)
        self.to_rgb = bool(to_rgb)
        self.size_divisor = int(size_divisor)
        self._stage = None      # pinned uint8 staging buffer for host tiles
        self._stage_done = None  # event recorded after the last copy out of it

    @classmethod
    def from_cfg(cls, pipeline_cfg) -> "TilePipeline":
        """Parse ``cfg.data.test.pipeline`` (a list of mmcv transform dicts)."""
        steps = list(pipeline_cfg)
        if len(steps) != 2:
            _unsupported(f"a pipeline of {len(steps)} top-level steps")
        load, aug = steps
        if load.get("type") not in ("LoadImageFromFile", "LoadImageFromWebcam"):
            _unsupported(f"loading step {load.get('type')!r}")
        _check_only(load, dict(to_float32=False, color_type="color", channel_order="bgr", file_client_args=None))
        if aug.get("type") != "MultiScaleFlipAug":
            _unsupported(f"step {aug.get('type')!r}")
        _check_only(aug, dict(transforms=None, img_scale=(None,), scale_factor=None, flip=False, flip_direction=None))
        s = aug.get("scale_factor")
        if isinstance(s, (list, tuple)):
            if len(s) != 1:
                _unsupported("several scale factors (multi-scale aug_test)")
            s = s[0]
        if s is None or isinstance(s, bool) or not isinstance(s, (int, float)):
            _unsupported(f"MultiScaleFlipAug(scale_factor={s!r}) (img_scale lists are not supported)")
        tr = list(aug.get("transforms", []))
        names = [t.get("type") for t in tr]
        if "RandomFlip" in names:
            _check_only(tr.pop(names.index("RandomFlip")), dict(flip_ratio=None, direction=None))
            names = [t.get("type") for t in tr]
        if len(names) != 5 or names[:3] != ["Resize", "Normalize", "Pad"] or \
                names[3] not in ("ImageToTensor", "DefaultFormatBundle") or names[4] != "Collect":
            _unsupported(f"transforms {names}")
        resize, norm, pad, fmt, collect = tr
        _check_only(resize, dict(keep_ratio=True, img_scale=(None,), backend="cv2", interpolation="bilinear",
                                 override=False, multiscale_mode=None, ratio_range=(None,), bbox_clip_border=None))
        _check_only(norm, dict(mean=None, std=None, to_rgb=None))
        _check_only(pad, dict(size_divisor=None, size=(None,), pad_to_square=False, pad_val=None))
        pad_val = pad.get("pad_val", 0)
        if (pad_val.get("img", 0) if isinstance(pad_val, dict) else pad_val) != 0:
            _unsupported(f"Pad(pad_val={pad_val!r})")
        if pad.get("size_divisor") is None:
            _unsupported("Pad without size_divisor")
        if fmt["type"] == "ImageToTensor":
            if list(fmt.get("keys", ["img"])) != ["img"]:
                _unsupported(f"ImageToTensor(keys={fmt.get('keys')!r})")
        else:
            _check_only(fmt, dict())
        if list(collect.get("keys", [])) != ["img"]:
            _unsupported(f"Collect(keys={collect.get('keys')!r})")
        if "meta_keys" in collect and tuple(collect["meta_keys"]) != _META_KEYS:
            _unsupported(f"Collect(meta_keys={collect['meta_keys']!r})")
        return cls(float(s), norm["mean"], norm["std"], norm.get("to_rgb", True), pad["size_divisor"])

    def sizes(self, h: int, w: int):
        """(new_h, new_w, pad_h, pad_w, scale_factor float32 [4]): Resize._random_scale + mmcv.imrescale + Pad."""
        s = self.scale_factor
        scale = (int(w * s), int(h * s))
        f = min(max(scale) / max(h, w), min(scale) / min(h, w))
        new_w, new_h = int(w * f + 0.5), int(h * f + 0.5)
        if new_h < h or new_w < w:
            _unsupported(f"a {h}x{w} tile at scale_factor {s} ({new_h}x{new_w} is a downscale)")
        d = self.size_divisor
        pad_h, pad_w = int(math.ceil(new_h / d)) * d, int(math.ceil(new_w / d)) * d
        sf = np.array([new_w / w, new_h / h, new_w / w, new_h / h], dtype=np.float32)
        return new_h, new_w, pad_h, pad_w, sf

    def _to_device(self, tiles, device) -> torch.Tensor:
        stream = torch.cuda.current_stream(device)
        if isinstance(tiles, torch.Tensor):
            if tiles.dtype != torch.uint8 or tiles.dim() != 4 or tiles.shape[3] != 3:
                raise ValueError(f"tiles must be uint8 [B,h,w,3], got {tuple(tiles.shape)} {tiles.dtype}")
            if tiles.is_cuda:
                return tiles.to(device).contiguous()
            if tiles.is_pinned():
                return tiles.contiguous().to(device, non_blocking=True)
            host = [tiles]
            shape = tuple(tiles.shape)
        else:
            host = [np.asarray(t) for t in tiles]
            if not host:
                raise ValueError("an empty list of tiles has no tile size; pass a uint8 tensor [0,h,w,3]")
            shape0 = host[0].shape
            for t in host:
                if t.dtype != np.uint8 or t.ndim != 3 or t.shape[2] != 3:
                    raise ValueError(f"every tile must be a uint8 HWC array with 3 channels, got {t.shape} {t.dtype}")
                if t.shape != shape0:
                    raise ValueError(f"tiles of one batch must have the same size, got {shape0} and {t.shape}")
            shape = (len(host),) + shape0
        n = int(np.prod(shape))
        if self._stage_done is not None:
            self._stage_done.synchronize()      # the previous copy out of the staging buffer has finished
        if self._stage is None or self._stage.numel() < n:
            self._stage = torch.empty(n, dtype=torch.uint8, pin_memory=True)
            self._stage_done = None
        st = self._stage[:n].view(shape)
        if len(host) == 1 and isinstance(host[0], torch.Tensor):
            st.copy_(host[0])
        else:
            stn = st.numpy()
            for i, t in enumerate(host):
                stn[i] = t
        dev = torch.empty(shape, dtype=torch.uint8, device=device)
        with torch.cuda.stream(stream):
            dev.copy_(st, non_blocking=True)
            if self._stage_done is None:
                self._stage_done = torch.cuda.Event()
            self._stage_done.record(stream)
        return dev

    def __call__(self, tiles, device=None) -> Tuple[torch.Tensor, List[dict]]:
        """tiles: list of equal-size uint8 HWC ndarrays, or a uint8 tensor [B,h,w,3] on the CPU (pinned or not) or on CUDA.
        Returns (img [B,3,Hp,Wp] fp32 on `device` (default: the current CUDA device), img_metas)."""
        if not torch.cuda.is_available():
            raise L.NuhtcError("TilePipeline needs a CUDA device: the pipeline runs on the GPU only (no CPU fallback)")
        device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if device.type != "cuda":
            raise L.NuhtcError(f"TilePipeline runs on a CUDA device, got {device}")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(device):
            x = self._to_device(tiles, device)
            B, h, w = int(x.shape[0]), int(x.shape[1]), int(x.shape[2])
            new_h, new_w, pad_h, pad_w, sf = self.sizes(h, w)
            out = torch.empty((B, 3, pad_h, pad_w), dtype=torch.float32, device=device)
            F3 = ctypes.c_float * 3
            L.check(L.lib().nuhtc_preprocess_tiles(L.ptr(x), B, h, w, new_h, new_w, pad_h, pad_w, int(self.to_rgb),
                                                   F3(*self.mean.tolist()), F3(*self.std.tolist()), L.ptr(out),
                                                   L.stream_ptr(device)), "nuhtc_preprocess_tiles")
            L.count("preprocess")
        return out, self.metas(B, h, w)

    def metas(self, B: int, h: int, w: int) -> List[dict]:
        """`img_metas` of a batch of B (h, w) tiles: Collect's default meta_keys for ndarray input."""
        new_h, new_w, pad_h, pad_w, sf = self.sizes(h, w)
        return [dict(filename=None, ori_filename=None, ori_shape=(h, w, 3), img_shape=(new_h, new_w, 3),
                     pad_shape=(pad_h, pad_w, 3), scale_factor=sf.copy(), flip=False, flip_direction=None,
                     img_norm_cfg=dict(mean=self.mean.copy(), std=self.std.copy(), to_rgb=self.to_rgb))
                for _ in range(B)]


_PIPELINES: Dict[tuple, TilePipeline] = {}


def inference_detector(model, imgs):
    """mmdet.apis.inference_detector (mmdet/apis/inference.py:90-153) for ndarray tiles, with the test pipeline on the GPU.

    Same arguments and return value: one image or a list/tuple of equal-size uint8 HWC images; the model is called as
    ``model(return_loss=False, rescale=True, img=[img], img_metas=[metas])`` under ``torch.no_grad()``.  The pipeline is
    built from ``model.cfg.data.test.pipeline`` and cached per (config, tile size)."""
    is_batch = isinstance(imgs, (list, tuple))
    if not is_batch:
        imgs = [imgs]
    if not all(isinstance(i, np.ndarray) for i in imgs):
        raise NotImplementedError("inference_detector: only ndarray tiles are supported (file loading stays on the host)")
    if not imgs:
        raise ValueError("inference_detector: no images")
    device = next(model.parameters()).device
    if device.type != "cuda":
        raise L.NuhtcError(f"inference_detector: the model is on {device}; the pipeline runs on a CUDA device only")
    pipeline_cfg = model.cfg.data.test.pipeline
    key = (repr(pipeline_cfg), imgs[0].shape)
    pipe = _PIPELINES.get(key)
    if pipe is None:
        pipe = _PIPELINES[key] = TilePipeline.from_cfg(pipeline_cfg)
    img, metas = pipe(imgs, device=device)
    with torch.no_grad():
        results = model(return_loss=False, rescale=True, img=[img], img_metas=[metas])
    return results if is_batch else results[0]
