"""Test-side helpers of the image-pipeline tests: the NuHTC test pipeline config and the golden file's decoding."""
import os

import numpy as np

MEAN = [123.675, 116.28, 103.53]
STD = [58.395, 57.12, 57.375]
SCALES = [2.0, 80 / 30, 4.0, 1.0]
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "preprocess.npz")


def nuhtc_pipeline(s=2.0, to_rgb=True, load="LoadImageFromFile", fmt=None, **aug):
    """cfg.data.test.pipeline of the NuHTC configs with MultiScaleFlipAug.scale_factor = s (tools/infer_wsi.py:416-419)."""
    return [dict(type=load),
            dict(type="MultiScaleFlipAug", img_scale=None, scale_factor=s, flip=False, **aug,
                 transforms=[dict(type="Resize", keep_ratio=True), dict(type="RandomFlip"),
                             dict(type="Normalize", mean=MEAN, std=STD, to_rgb=to_rgb), dict(type="Pad", size_divisor=32),
                             fmt or dict(type="ImageToTensor", keys=["img"]), dict(type="Collect", keys=["img"])])]


def load_golden():
    """dict with tiles {name: [h,w,3] uint8}, norm {to_rgb: [3,256] float32} and cases [(tile, s, new_hw, sf, rows, resized)]."""
    z = np.load(GOLDEN)
    undelta = lambda a: np.cumsum(a, axis=-2, dtype=np.uint8)   # stored as uint8 differences along x
    tiles = {k[5:]: undelta(z[k]) for k in z.files if k.startswith("tile_")}
    cases, i = [], 0
    while f"case{i}_s" in z.files:
        cases.append((str(z[f"case{i}_tile"]), float(z[f"case{i}_s"]), tuple(int(v) for v in z[f"case{i}_new_hw"]),
                      z[f"case{i}_scale_factor"], z[f"case{i}_rows"], undelta(z[f"case{i}_resized"])))
        i += 1
    return dict(tiles=tiles, norm={True: z["norm_rgb"], False: z["norm_bgr"]}, mean=z["mean"], std=z["std"], cases=cases)


def expected_rows(resized_rows, norm, to_rgb, pad_w):
    """[3, R, pad_w] float32 the pipeline must produce on the golden's sampled rows."""
    R, new_w = resized_rows.shape[:2]
    out = np.zeros((3, R, pad_w), np.float32)
    for c in range(3):
        out[c, :, :new_w] = norm[c][resized_rows[:, :, 2 - c if to_rgb else c]]
    return out
