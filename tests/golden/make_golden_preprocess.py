#!/usr/bin/env python
"""Golden vectors for the test-time image pipeline (nuhtc_b200/preprocess.py, csrc/preprocess.cu), made with REAL cv2.

The mmcv 1.7.2 bodies the pipeline runs are written out below with their cv2 calls: `imrescale` / `rescale_size` /
`imresize` (cv2.resize, INTER_LINEAR) and `imnormalize_` (cvtColor BGR2RGB, cv2.subtract / cv2.multiply with float64
scalars).  Tiles: one seeded 256x256 tile at s = 2.0, 80/30, 4.0, 1.0 and one 77x100 tile at s = 3.0, both to_rgb values.

Stored compactly: the tiles (wrapping ramps with a random patch, a random row and column and saturated patches) and the
resized uint8 images on a prime-strided sample of rows plus the first and last three, both as uint8 differences along x
(np.cumsum(..., axis=1, dtype=np.uint8) restores them), and the cv2 normalisation of every byte value per channel.  The fp32
output is then fully determined: out[c, y, x] = norm[to_rgb][c, resized[y, x, 2 - c if to_rgb else c]] inside the image,
0 in the pad.

    python tests/golden/make_golden_preprocess.py     (needs cv2)
"""
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MEAN = [123.675, 116.28, 103.53]   # the NuHTC configs' img_norm_cfg
STD = [58.395, 57.12, 57.375]
CASES = [("t256", 2.0), ("t256", 80 / 30), ("t256", 4.0), ("t256", 1.0), ("t77x100", 3.0)]


def tile(h, w, seed):
    g = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    t = np.stack([(xx * (c + 1) + yy * (3 - c) + 80 * c) % 256 for c in range(3)], -1).astype(np.uint8)  # wrapping ramps
    ph, pw = h // 8, w // 8
    t[:ph, :pw] = g.integers(0, 256, (ph, pw, 3), dtype=np.uint8)     # full-entropy patch: every rounding case
    t[-ph:, -pw:] = 255
    t[-ph:, :pw] = 0
    t[h // 2, :] = g.integers(0, 256, (w, 3), dtype=np.uint8)         # one random row and column through the middle
    t[:, w // 2] = g.integers(0, 256, (h, 3), dtype=np.uint8)
    return t


def rescale_size(old_size, scale):
    """mmcv/image/geometric.py rescale_size for a tuple scale (+ _scale_size)."""
    w, h = old_size
    max_long_edge, max_short_edge = max(scale), min(scale)
    scale_factor = min(max_long_edge / max(h, w), max_short_edge / min(h, w))
    return int(w * float(scale_factor) + 0.5), int(h * float(scale_factor) + 0.5)


def resize(img, s):
    """mmdet Resize._random_scale (scale_factor branch) + _resize_img (keep_ratio=True, cv2, bilinear)."""
    scale = tuple([int(x * s) for x in img.shape[:2]][::-1])
    new_size = rescale_size((img.shape[1], img.shape[0]), scale)
    out = cv2.resize(img, new_size, interpolation=cv2.INTER_LINEAR)
    h, w = img.shape[:2]
    sf = np.array([out.shape[1] / w, out.shape[0] / h, out.shape[1] / w, out.shape[0] / h], dtype=np.float32)
    return out, sf


def imnormalize(img, mean, std, to_rgb):
    """mmcv/image/photometric.py imnormalize (copy + astype float32) and imnormalize_."""
    img = img.copy().astype(np.float32)
    mean = np.float64(np.array(mean, dtype=np.float32).reshape(1, -1))
    stdinv = 1 / np.float64(np.array(std, dtype=np.float32).reshape(1, -1))
    if to_rgb:
        cv2.cvtColor(img, cv2.COLOR_BGR2RGB, img)
    cv2.subtract(img, mean, img)
    cv2.multiply(img, stdinv, img)
    return img


def norm_table(to_rgb):
    """[3,256] float32 by OUTPUT channel: every byte value through imnormalize, all three input channels distinct."""
    v = np.arange(256, dtype=np.uint8)
    img = np.stack([v, np.roll(v, 85), np.roll(v, 170)], -1)[None]    # [1,256,3], channel k holds roll(v, 85k)
    out = imnormalize(img, MEAN, STD, to_rgb)[0]                     # [256,3] by output channel
    tab = np.empty((3, 256), np.float32)
    for c in range(3):
        k = 2 - c if to_rgb else c
        tab[c, np.roll(v, 85 * k)] = out[:, c]
    return tab


def delta_x(a):
    """uint8 difference along x (axis -2 of [..., x, 3]) with wraparound: ramps become runs that deflate compresses."""
    return np.diff(a, axis=-2, prepend=np.zeros_like(a[..., :1, :]))


def rows_of(new_h):
    """The three first and last rows (border coefficients) and every 11th row between (11 is prime: all row phases)."""
    return np.unique(np.concatenate([[0, 1, 2, new_h - 3, new_h - 2, new_h - 1], np.arange(3, new_h, 11)])).astype(np.int32)


def main():
    tiles = dict(t256=tile(256, 256, 0), t77x100=tile(77, 100, 1))
    z = dict(mean=np.array(MEAN, np.float32), std=np.array(STD, np.float32), cv2_version=np.array(cv2.__version__),
             norm_rgb=norm_table(True), norm_bgr=norm_table(False), **{f"tile_{k}": delta_x(v) for k, v in tiles.items()})
    for i, (name, s) in enumerate(CASES):
        out, sf = resize(tiles[name], s)
        rows = rows_of(out.shape[0])
        z[f"case{i}_tile"] = np.array(name)
        z[f"case{i}_s"] = np.float64(s)
        z[f"case{i}_new_hw"] = np.array(out.shape[:2], np.int32)
        z[f"case{i}_scale_factor"] = sf
        z[f"case{i}_rows"] = rows
        z[f"case{i}_resized"] = delta_x(out[rows])
    path = os.path.join(HERE, "preprocess.npz")
    np.savez_compressed(path, **z)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
