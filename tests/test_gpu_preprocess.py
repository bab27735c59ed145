"""GPU: the test-time image pipeline kernel (csrc/preprocess.cu) against the cv2-made golden and the oracle, bit for bit;
host and device inputs, B = 0, CUDA-graph capture, and inference_detector against a stand-in model."""
import types

import numpy as np
import pytest
import torch

from _preprocess_golden import MEAN, SCALES, STD, expected_rows, load_golden, nuhtc_pipeline
from oracle import preprocess as P

import nuhtc_b200 as nb
from nuhtc_b200.preprocess import TilePipeline

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bits(x):
    x = torch.as_tensor(x).contiguous()
    return x.view(torch.int32)


def _same(got, ref):
    assert got.dtype == torch.float32 and tuple(got.shape) == tuple(ref.shape)
    assert torch.equal(_bits(got.cpu()), _bits(torch.from_numpy(np.ascontiguousarray(ref))))


@pytest.mark.parametrize("to_rgb", [True, False])
def test_golden(to_rgb):
    g = load_golden()
    for name, s, (new_h, new_w), sf, rows, resized in g["cases"]:
        pipe = TilePipeline(s, g["mean"], g["std"], to_rgb)
        t = torch.from_numpy(g["tiles"][name]).to(DEV)[None]
        img, metas = pipe(t)
        _, _, pad_h, pad_w = img.shape
        assert metas[0]["img_shape"] == (new_h, new_w, 3) and np.array_equal(metas[0]["scale_factor"], sf)
        exp = torch.from_numpy(expected_rows(resized, g["norm"][to_rgb], to_rgb, pad_w))
        assert torch.equal(_bits(img[0][:, torch.from_numpy(rows).long().to(DEV)].cpu()), _bits(exp)), (name, s)
        assert not img[0, :, new_h:].any() and not img[0, :, :, new_w:].any()     # zero pad


_RESIZED = {}


def _oracle_resized(tiles, s, key):
    if key not in _RESIZED:
        new_h, new_w = P.size_rule(tiles.shape[1], tiles.shape[2], s)[:2]
        _RESIZED[key] = np.stack([P.resize_linear_u8(t, new_h, new_w) for t in tiles])
    return _RESIZED[key]


def _oracle_img(resized, pad_h, pad_w, to_rgb):
    lut = P.norm_table(MEAN, STD, to_rgb)
    B, new_h, new_w = resized.shape[:3]
    out = np.zeros((B, 3, pad_h, pad_w), np.float32)
    for c in range(3):
        out[:, c, :new_h, :new_w] = lut[c][resized[..., 2 - c if to_rgb else c]]
    return out


@pytest.mark.parametrize("s", SCALES)
@pytest.mark.parametrize("to_rgb", [True, False])
def test_matches_oracle_b16_every_input_kind(s, to_rgb):
    g = np.random.default_rng(int(s * 1000))
    tiles = g.integers(0, 256, (16, 256, 256, 3), dtype=np.uint8)
    tiles[3] = 0
    tiles[4] = 255
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(s, to_rgb))
    new_h, new_w, pad_h, pad_w, _ = pipe.sizes(256, 256)
    ref = _oracle_img(_oracle_resized(tiles, s, s), pad_h, pad_w, to_rgb)
    inputs = {"list": list(tiles), "pinned": torch.from_numpy(tiles).pin_memory(), "pageable": torch.from_numpy(tiles),
              "cuda": torch.from_numpy(tiles).to(DEV)}
    for kind, x in inputs.items():
        img, metas = pipe(x)
        assert img.device == torch.device(DEV) and len(metas) == 16, kind
        _same(img, ref)
    # the staging buffer is reused: a second host batch right after the first must not see the first one's bytes
    img1, _ = pipe(list(tiles[::-1]))
    img2, _ = pipe(list(tiles))
    _same(img1, ref[::-1])
    _same(img2, ref)


def test_odd_shape_and_unpadded_width():
    """77x100 tiles (231x300 at s = 3, pad 256x320) and size_divisor 1 at s = 2.5 (pad width 249: the scalar-store path)"""
    g = np.random.default_rng(5)
    tiles = g.integers(0, 256, (5, 77, 100, 3), dtype=np.uint8)
    for s, div in ((3.0, 32), (2.5, 1)):
        pipe = TilePipeline(s, MEAN, STD, True, size_divisor=div)
        new_h, new_w, pad_h, pad_w, _ = pipe.sizes(77, 100)
        ref = _oracle_img(np.stack([P.resize_linear_u8(t, new_h, new_w) for t in tiles]), pad_h, pad_w, True)
        img, _ = pipe(list(tiles))
        _same(img, ref)


def test_empty_batch():
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(2.0))
    for x in (torch.zeros(0, 256, 256, 3, dtype=torch.uint8, device=DEV), torch.zeros(0, 256, 256, 3, dtype=torch.uint8)):
        img, metas = pipe(x)
        assert tuple(img.shape) == (0, 3, 512, 512) and img.is_cuda and metas == []


def test_unequal_tiles_raise():
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(2.0))
    with pytest.raises(ValueError):
        pipe([np.zeros((256, 256, 3), np.uint8), np.zeros((256, 240, 3), np.uint8)])


def test_cuda_graph_capture_and_replay():
    pipe = TilePipeline.from_cfg(nuhtc_pipeline(2.0))
    g = np.random.default_rng(7)
    a, b = (torch.from_numpy(g.integers(0, 256, (4, 256, 256, 3), dtype=np.uint8)).to(DEV) for _ in range(2))
    static = a.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        pipe(static)                        # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out, _ = pipe(static)
    static.copy_(b)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(out), _bits(pipe(b)[0]))
    static.copy_(a)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(out), _bits(pipe(a)[0]))


class _StandIn(torch.nn.Module):
    """Records what inference_detector hands the detector and returns a sentinel per image."""

    def __init__(self, pipeline):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1))
        self.cfg = types.SimpleNamespace(data=types.SimpleNamespace(test=types.SimpleNamespace(pipeline=pipeline)))
        self.calls = []

    def forward(self, **kw):
        self.calls.append((kw, torch.is_grad_enabled()))
        return [("result", i) for i in range(len(kw["img_metas"][0]))]


@pytest.mark.parametrize("s", [2.0, 80 / 30])
def test_inference_detector_feeds_the_model_what_mmdet_would(s):
    model = _StandIn(nuhtc_pipeline(s)).to(DEV)
    g = np.random.default_rng(11)
    tiles = [g.integers(0, 256, (256, 256, 3), dtype=np.uint8) for _ in range(6)]
    out = nb.inference_detector(model, tiles)
    assert out == [("result", i) for i in range(6)]
    assert nb.inference_detector(model, tiles[0]) == ("result", 0)        # single image: results[0]
    (kw, grad), _ = model.calls
    assert not grad
    ref = P.data(tiles, s, MEAN, STD, True)
    assert set(kw) == {"return_loss", "rescale"} | set(ref)
    assert kw["return_loss"] is False and kw["rescale"] is True
    assert len(kw["img"]) == 1 and kw["img"][0].is_cuda
    _same(kw["img"][0], ref["img"][0])
    assert len(kw["img_metas"]) == 1 and len(kw["img_metas"][0]) == 6
    for m, r in zip(kw["img_metas"][0], ref["img_metas"][0]):
        assert list(m) == list(r)
        for k, v in r.items():
            if isinstance(v, np.ndarray):
                assert m[k].dtype == v.dtype and np.array_equal(m[k], v), k
            elif isinstance(v, dict):
                assert m[k]["to_rgb"] == v["to_rgb"]
                assert all(m[k][q].dtype == np.float32 and np.array_equal(m[k][q], v[q]) for q in ("mean", "std"))
            else:
                assert m[k] == v and type(m[k]) is type(v), k
