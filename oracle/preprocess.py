"""CPU oracle for the detector's test-time image pipeline  --  TEST INFRASTRUCTURE ONLY (numpy, no cv2).

Restates what `inference_detector(model, [np.ndarray]*B)` (mmdet/apis/inference.py:90-153, called at
tools/infer_wsi.py:485) does to each tile under the NuHTC test pipeline of mmdet 2.x / mmcv 1.7.2:

    LoadImageFromWebcam -> MultiScaleFlipAug(scale_factor=s, flip=False)[
        Resize(keep_ratio=True) (cv2, bilinear) -> RandomFlip (no-op) -> Normalize(mean, std, to_rgb)
        -> Pad(size_divisor) -> ImageToTensor / DefaultFormatBundle -> Collect(['img'])]

* size rule: `Resize._random_scale` with `scale_factor` -> `mmcv.imrescale` -> `rescale_size` / `_scale_size`
* `cv2.resize(INTER_LINEAR)` on uint8: cv2's fixed-point path (11-bit coefficients, the SIMD vertical formula)
* `mmcv.imnormalize_`: cvtColor(BGR2RGB), cv2.subtract(float64 mean), cv2.multiply(1/float64 std) on float32
* `mmcv.impad_to_multiple(pad_val=0)`, HWC -> CHW, the batch collate and the `Collect` meta keys

The arithmetic is pinned against cv2 (tests/golden/make_golden_preprocess.py, tests/test_preprocess_cpu.py); the transform
order, the `int(x * s)` truncation and the meta keys follow mmdet 2.x as recalled (DESIGN.md section 2).
"""
from __future__ import annotations

import math

import numpy as np

COEF_BITS = 11
COEF_SCALE = 1 << COEF_BITS   # INTER_RESIZE_COEF_SCALE


def size_rule(h: int, w: int, s: float, size_divisor: int = 32):
    """(new_h, new_w, pad_h, pad_w, scale_factor float32 [4]) of a (h, w) tile rescaled by s and padded."""
    scale = (int(w * s), int(h * s))                                        # Resize._random_scale: (w, h)
    f = min(max(scale) / max(h, w), min(scale) / min(h, w))                 # rescale_size
    new_w, new_h = int(w * f + 0.5), int(h * f + 0.5)                       # _scale_size
    pad_h = int(math.ceil(new_h / size_divisor)) * size_divisor
    pad_w = int(math.ceil(new_w / size_divisor)) * size_divisor
    sf = np.array([new_w / w, new_h / h, new_w / w, new_h / h], dtype=np.float32)
    return new_h, new_w, pad_h, pad_w, sf


def _coeffs(n_out: int, n_in: int, reset_border: bool):
    """cv2 resize coefficients along one axis: source index and the two 11-bit weights per output index."""
    scale = 1.0 / (n_out / n_in)
    f = ((np.arange(n_out, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if reset_border:                      # columns only: rows keep their fraction, only the indices are clamped
        lo, hi = s < 0, s >= n_in - 1
        f[lo | hi] = 0
        s[lo] = 0
        s[hi] = n_in - 1
    a1 = np.rint(f * np.float32(COEF_SCALE)).astype(np.int64)                # rint: round half to even, like cvRound
    a0 = np.rint((np.float32(1) - f) * np.float32(COEF_SCALE)).astype(np.int64)
    return s, a0, a1


def resize_linear_u8(src: np.ndarray, new_h: int, new_w: int) -> np.ndarray:
    """`cv2.resize(src, (new_w, new_h), interpolation=cv2.INTER_LINEAR)` for uint8 [h,w,C] (upscaling or identity)."""
    h, w = src.shape[:2]
    S = src.astype(np.int64).reshape(h, w, -1)
    sx, a0, a1 = _coeffs(new_w, w, True)
    sy, b0, b1 = _coeffs(new_h, h, False)
    sx1 = np.minimum(sx + 1, w - 1)
    Hrow = S[:, sx, :] * a0[None, :, None] + S[:, sx1, :] * a1[None, :, None]    # horizontal pass, int32 per channel
    H0 = Hrow[np.clip(sy, 0, h - 1)]
    H1 = Hrow[np.clip(sy + 1, 0, h - 1)]
    b0, b1 = b0[:, None, None], b1[:, None, None]
    out = ((((H0 >> 4) * b0) >> 16) + (((H1 >> 4) * b1) >> 16) + 2) >> 2    # cv2's SIMD vertical pass
    return np.clip(out, 0, 255).astype(np.uint8).reshape((new_h, new_w) + src.shape[2:])


def norm_table(mean, std, to_rgb: bool) -> np.ndarray:
    """[3,256] float32: normalised value of byte v in OUTPUT channel c (the channel after the optional BGR->RGB swap)."""
    mean = np.asarray(mean, dtype=np.float32).astype(np.float64)
    inv = 1.0 / np.asarray(std, dtype=np.float32).astype(np.float64)
    v = np.arange(256, dtype=np.float64)
    return ((v[None, :] - mean[:, None]) * inv[:, None]).astype(np.float32)


def pipeline(tiles, s: float, mean, std, to_rgb: bool, size_divisor: int = 32):
    """tiles: [B,h,w,3] uint8 (array or list of equal-size arrays) -> (img [B,3,Hp,Wp] float32, img_metas list[dict])."""
    tiles = [np.asarray(t) for t in tiles]
    B = len(tiles)
    h, w = tiles[0].shape[:2]
    new_h, new_w, pad_h, pad_w, sf = size_rule(h, w, s, size_divisor)
    lut = norm_table(mean, std, to_rgb)
    img = np.zeros((B, 3, pad_h, pad_w), dtype=np.float32)
    for b, t in enumerate(tiles):
        r = resize_linear_u8(t, new_h, new_w)
        for c in range(3):
            img[b, c, :new_h, :new_w] = lut[c][r[:, :, 2 - c if to_rgb else c]]
    return img, [metas(h, w, new_h, new_w, pad_h, pad_w, sf, mean, std, to_rgb) for _ in range(B)]


def metas(h, w, new_h, new_w, pad_h, pad_w, sf, mean, std, to_rgb):
    """One image's `img_metas` entry as `Collect` (default meta_keys) returns it for an ndarray input."""
    return dict(filename=None, ori_filename=None, ori_shape=(h, w, 3), img_shape=(new_h, new_w, 3),
                pad_shape=(pad_h, pad_w, 3), scale_factor=sf.copy(), flip=False, flip_direction=None,
                img_norm_cfg=dict(mean=np.asarray(mean, dtype=np.float32), std=np.asarray(std, dtype=np.float32),
                                  to_rgb=bool(to_rgb)))


def data(tiles, s: float, mean, std, to_rgb: bool, size_divisor: int = 32):
    """The keyword arguments `inference_detector` passes to the model besides return_loss / rescale."""
    img, m = pipeline(tiles, s, mean, std, to_rgb, size_divisor)
    return dict(img=[img], img_metas=[m])
