"""CPU: the test-time image pipeline.  The oracle (oracle/preprocess.py) against live cv2 and against the committed golden
made with cv2; the size rule and metas; unsupported configs; the C ABI's argument checks; no CPU fallback."""
import ctypes
import types

import numpy as np
import pytest
import torch

from _preprocess_golden import MEAN, SCALES, STD, expected_rows, load_golden, nuhtc_pipeline
from oracle import preprocess as P

import nuhtc_b200 as nb
from nuhtc_b200 import _lib
from nuhtc_b200.preprocess import TilePipeline

RESIZE_SHAPES = [((256, 256), (512, 512)), ((256, 256), (682, 682)), ((256, 256), (1024, 1024)), ((256, 256), (384, 384)),
                 ((256, 256), (533, 533)), ((256, 256), (640, 640)), ((77, 100), (231, 300)), ((5, 7), (11, 13)),
                 ((256, 256), (256, 256))]


def _random_shapes(n, seed):
    g = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        h, w = (int(v) for v in g.integers(1, 90, 2))
        out.append(((h, w), (int(h * g.uniform(1, 4.5)) or 1, int(w * g.uniform(1, 4.5)) or 1)))
    return [((h, w), (max(nh, h), max(nw, w))) for (h, w), (nh, nw) in out]


@pytest.mark.parametrize("kind", ["random", "zeros", "full255"])
def test_oracle_resize_matches_cv2(kind):
    cv2 = pytest.importorskip("cv2")
    g = np.random.default_rng(1)
    for (h, w), (nh, nw) in RESIZE_SHAPES + _random_shapes(25, 2):
        if kind == "random":
            t = g.integers(0, 256, (h, w, 3), dtype=np.uint8)
        else:
            t = np.full((h, w, 3), 0 if kind == "zeros" else 255, np.uint8)
        ref = cv2.resize(t, (nw, nh), interpolation=cv2.INTER_LINEAR)
        assert np.array_equal(P.resize_linear_u8(t, nh, nw), ref), ((h, w), (nh, nw))


@pytest.mark.parametrize("to_rgb", [True, False])
def test_norm_table_matches_cv2_exhaustively(to_rgb):
    cv2 = pytest.importorskip("cv2")
    v = np.arange(256, dtype=np.uint8)
    img = np.stack([v, np.roll(v, 85), np.roll(v, 170)], -1)[None].astype(np.float32)   # distinct value per channel
    src = img.copy()
    # mmcv.imnormalize_ (mmcv/image/photometric.py)
    if to_rgb:
        cv2.cvtColor(img, cv2.COLOR_BGR2RGB, img)
    cv2.subtract(img, np.float64(np.array(MEAN, np.float32).reshape(1, -1)), img)
    cv2.multiply(img, 1 / np.float64(np.array(STD, np.float32).reshape(1, -1)), img)
    lut = P.norm_table(MEAN, STD, to_rgb)
    for c in range(3):
        got = lut[c][src[0, :, 2 - c if to_rgb else c].astype(np.int64)]
        assert np.array_equal(got.view(np.uint32), img[0, :, c].view(np.uint32)), c


def test_oracle_reproduces_the_golden():
    """preprocess.npz was made with cv2 (tests/golden/make_golden_preprocess.py): pins the oracle without cv2."""
    g = load_golden()
    for to_rgb in (True, False):
        assert np.array_equal(P.norm_table(g["mean"], g["std"], to_rgb).view(np.uint32), g["norm"][to_rgb].view(np.uint32))
    for name, s, new_hw, sf, rows, resized in g["cases"]:
        t = g["tiles"][name]
        new_h, new_w, pad_h, pad_w, sf_o = P.size_rule(t.shape[0], t.shape[1], s)
        assert (new_h, new_w) == new_hw and np.array_equal(sf_o, sf), (name, s)
        assert np.array_equal(P.resize_linear_u8(t, new_h, new_w)[rows], resized), (name, s)
        img, _ = P.pipeline([t], s, MEAN, STD, True)
        assert np.array_equal(img[0][:, rows], expected_rows(resized, g["norm"][True], True, pad_w))


@pytest.mark.parametrize("s,new,pad", [(2.0, 512, 512), (80 / 30, 682, 704), (4.0, 1024, 1024), (1.0, 256, 256)])
def test_size_rule_and_metas(s, new, pad):
    assert P.size_rule(256, 256, s)[:4] == (new, new, pad, pad)
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(s))
    new_h, new_w, pad_h, pad_w, sf = pipe.sizes(256, 256)
    assert (new_h, new_w, pad_h, pad_w) == (new, new, pad, pad)
    assert sf.dtype == np.float32 and np.array_equal(sf, np.full(4, new / 256, np.float32))
    got, ref = pipe.metas(3, 256, 256), P.pipeline(np.zeros((3, 256, 256, 3), np.uint8), s, MEAN, STD, True)[1]
    assert len(got) == 3
    for m, r in zip(got, ref):
        assert list(m) == list(r)
        for k in ("filename", "ori_filename", "ori_shape", "img_shape", "pad_shape", "flip", "flip_direction"):
            assert m[k] == r[k], k
        assert m["scale_factor"].dtype == np.float32 and np.array_equal(m["scale_factor"], r["scale_factor"])
        for k in ("mean", "std"):
            assert m["img_norm_cfg"][k].dtype == np.float32 and np.array_equal(m["img_norm_cfg"][k], r["img_norm_cfg"][k])
        assert m["img_norm_cfg"]["to_rgb"] is True
    assert got[0]["scale_factor"] is not got[1]["scale_factor"]    # one array per image, like the per-image pipeline


def test_non_square_size_rule():
    assert P.size_rule(77, 100, 3.0)[:4] == (231, 300, 256, 320)
    assert TilePipeline(3.0, MEAN, STD).sizes(77, 100)[:4] == (231, 300, 256, 320)
    assert TilePipeline(2.5, MEAN, STD, size_divisor=1).sizes(77, 100)[:4] == P.size_rule(77, 100, 2.5, 1)[:4]


def test_accepted_config_variants():
    for cfg in (nuhtc_pipeline(2.0, load="LoadImageFromWebcam"), nuhtc_pipeline(2.0, fmt=dict(type="DefaultFormatBundle")),
                nuhtc_pipeline([2.0]), nuhtc_pipeline(2, to_rgb=False)):
        p = TilePipeline.from_cfg(cfg)
        assert p.scale_factor == 2.0 and p.size_divisor == 32
    assert TilePipeline.from_cfg(nuhtc_pipeline(2, to_rgb=False)).to_rgb is False


def _edit(fn):
    cfg = nuhtc_pipeline(2.0)
    fn(cfg, {t["type"]: t for t in cfg[1]["transforms"]})
    return cfg


@pytest.mark.parametrize("edit", [
    lambda c, t: c[1].update(flip=True),                                       # aug_test
    lambda c, t: c[1].update(img_scale=[(1333, 800)], scale_factor=None),      # img_scale lists
    lambda c, t: c[1].update(scale_factor=[1.0, 2.0]),                         # multi-scale
    lambda c, t: c[1].update(scale_factor=0.5),                                # downscale
    lambda c, t: t["Resize"].update(keep_ratio=False),
    lambda c, t: t["Resize"].update(backend="pillow"),
    lambda c, t: t["Resize"].update(interpolation="nearest"),
    lambda c, t: t["Pad"].update(size=(512, 512), size_divisor=None),
    lambda c, t: t["Pad"].update(pad_val=255),
    lambda c, t: c[1]["transforms"].insert(1, dict(type="PhotoMetricDistortion")),
    lambda c, t: t["Collect"].update(keys=["img", "gt_bboxes"]),
    lambda c, t: c[0].update(to_float32=True),
    lambda c, t: c.append(dict(type="Collect", keys=["img"])),
])
def test_unsupported_configs_raise(edit):
    with pytest.raises(NotImplementedError):
        TilePipeline.from_cfg(_edit(edit))


def test_abi_rejects_bad_arguments_without_gpu():
    L = _lib.lib()
    F3 = ctypes.c_float * 3
    m, s = F3(*MEAN), F3(*STD)
    fake = ctypes.c_void_p(16)      # never dereferenced: validation fails before any CUDA call
    assert L.nuhtc_preprocess_tiles(None, 2, 256, 256, 512, 512, 512, 512, 1, m, s, None, None) == -1   # null, B > 0
    assert b"null" in L.nuhtc_last_error()
    assert L.nuhtc_preprocess_tiles(fake, 2, 256, 256, 512, 512, 512, 512, 1, None, s, fake, None) == -1  # null mean
    assert L.nuhtc_preprocess_tiles(fake, 2, 256, 256, 128, 128, 128, 128, 1, m, s, fake, None) == -1   # downscale
    assert b"downscaling" in L.nuhtc_last_error()
    assert L.nuhtc_preprocess_tiles(fake, 2, 256, 256, 512, 600, 512, 576, 1, m, s, fake, None) == -1   # pad < new
    assert L.nuhtc_preprocess_tiles(fake, 2, 0, 256, 512, 512, 512, 512, 1, m, s, fake, None) == -1     # size <= 0
    assert L.nuhtc_preprocess_tiles(fake, 2, 256, 256, 512, 512, 512, -4, 1, m, s, fake, None) == -1
    assert L.nuhtc_preprocess_tiles(fake, -1, 256, 256, 512, 512, 512, 512, 1, m, s, fake, None) == -1
    assert L.nuhtc_preprocess_tiles(None, 0, 256, 256, 512, 512, 512, 512, 1, None, None, None, None) == 0  # nothing to do


def test_pipeline_refuses_to_run_without_cuda(monkeypatch):
    """host tiles are input only: no CUDA device means an error, not a CPU computation"""
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(2.0))
    with pytest.raises(nb.NuhtcError):
        pipe([np.zeros((256, 256, 3), np.uint8)])
    with pytest.raises(nb.NuhtcError):
        pipe(torch.zeros(1, 256, 256, 3, dtype=torch.uint8))


def test_inference_detector_refuses_a_cpu_model():
    model = types.SimpleNamespace(parameters=lambda: iter([torch.zeros(1)]),
                                  cfg=types.SimpleNamespace(data=types.SimpleNamespace(test=types.SimpleNamespace(
                                      pipeline=nuhtc_pipeline(2.0)))))
    with pytest.raises(nb.NuhtcError):
        nb.inference_detector(model, [np.zeros((256, 256, 3), np.uint8)])


def test_patch_inference_rebinds_the_script():
    from nuhtc_b200.patch import patch_inference
    mod = types.SimpleNamespace(inference_detector=None, mask_nms="untouched")
    assert patch_inference(mod) == ["infer_wsi.inference_detector"]
    assert mod.inference_detector is nb.inference_detector and mod.mask_nms == "untouched"


@pytest.mark.parametrize("s", SCALES)
def test_oracle_matches_mmdet_compose(s):
    """only where mmdet is importable: the real test pipeline + collate against the oracle's data dict"""
    pytest.importorskip("mmdet")
    from mmcv.parallel import collate
    from mmdet.datasets.pipelines import Compose
    from mmdet.datasets import replace_ImageToTensor
    g = np.random.default_rng(3)
    tiles = [g.integers(0, 256, (256, 256, 3), dtype=np.uint8) for _ in range(2)]
    pipe = Compose(replace_ImageToTensor(nuhtc_pipeline(s, load="LoadImageFromWebcam")))
    data = collate([pipe(dict(img=t)) for t in tiles], samples_per_gpu=2)
    img = data["img"][0].data[0].numpy()
    metas = data["img_metas"][0].data[0]
    ref = P.data(tiles, s, MEAN, STD, True)
    assert np.array_equal(img.view(np.uint32), ref["img"][0].view(np.uint32))
    for m, r in zip(metas, ref["img_metas"][0]):
        assert set(m) == set(r)
        assert m["img_shape"] == r["img_shape"] and m["pad_shape"] == r["pad_shape"]
        assert np.array_equal(m["scale_factor"], r["scale_factor"])
