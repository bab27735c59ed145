"""CPU: the float64 RoIAlign / attention-pooling references (tests/_roi_ref64.py) against the fp32 C oracle, the committed
goldens made from the reference's own source, and torchvision.ops.roi_align -- each within the reference's own bound, so
the bound the GPU kernels are held to is known to contain a correct fp32 computation."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import _roi_ref64 as R

G = os.path.join(os.path.dirname(__file__), "golden")


def _rois(K, B, frame_w, frame_h, seed, lo=2.0, hi=120.0):
    g = torch.Generator().manual_seed(seed)
    ctr = torch.rand(K, 2, generator=g) * torch.tensor([frame_w * 1.1, frame_h * 1.1]) - torch.tensor([frame_w, frame_h]) * 0.05
    wh = lo + torch.rand(K, 2, generator=g) * (hi - lo)
    r = torch.cat([torch.randint(0, B, (K, 1), generator=g).float(), ctr - wh / 2, ctr + wh / 2], 1)
    r[0, 1:] = torch.tensor([10.0, 10.0, 10.0, 10.0])                              # zero size
    r[1, 1:] = torch.tensor([-60.0, -60.0, frame_w + 60.0, frame_h + 60.0])        # larger than the frame
    r[2, 1:] = torch.tensor([-500.0, -500.0, -400.0, -400.0])                      # wholly outside
    return r


def _within(out, ref, tol, what):
    R.check(out, ref, tol, what)


@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("sr", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("P", [7, 14])
def test_reference_matches_oracle_roi_align(oracle, aligned, sr, P):
    torch.manual_seed(sr + 10 * P + int(aligned))
    B, C, H, W = 2, 16, 23, 41       # non-square, odd
    x = torch.randn(B, C, H, W)
    rois = _rois(160, B, W * 4, H * 4, seed=P + sr)
    ref, tol = R.roi_align_ref64([x], rois, P, [0.25], sr, aligned)
    out = oracle.roi_align(x, rois, P, 0.25, sr, aligned=aligned)
    _within(out, ref, tol, f"P={P} sr={sr} aligned={aligned}")


def test_reference_matches_oracle_on_tall_and_wide_maps(oracle):
    torch.manual_seed(3)
    for H, W in ((1, 37), (37, 1), (96, 33), (13, 200), (1, 1)):
        x = torch.randn(1, 8, H, W)
        rois = _rois(80, 1, W * 4, H * 4, seed=H * W)
        for P in (7, 14):
            ref, tol = R.roi_align_ref64([x], rois, P, [0.25], 0)
            _within(oracle.roi_align(x, rois, P, 0.25, 0), ref, tol, f"{H}x{W} P={P}")


def test_reference_routes_and_sums_like_the_extractors(oracle):
    from nuhtc_b200 import synth
    feats = synth.fpn_levels(2, 32, frame=256, seed=3)
    rois = synth.proposals(2, 150, "routed", frame=256, seed=4)
    scales = [1 / s for s in synth.FPN_STRIDES]
    assert np.array_equal(R.route_levels(rois, 4), oracle.map_roi_levels(rois, 4).numpy())
    for P in (7, 14):
        ref, tol = R.roi_align_ref64(feats, rois, P, scales, 0, mode="route")
        _within(oracle.single_roi_extract(feats, rois, synth.FPN_STRIDES, P, 0), ref, tol, f"route P={P}")
        ref, tol = R.roi_align_ref64(feats[:2], rois, P, scales[:2], 2, mode="sum")
        _within(oracle.sum_roi_extract(feats[:2], rois, synth.FPN_STRIDES[:2], P, 2), ref, tol, f"sum P={P}")


def test_reference_bias_and_pool2_follow_their_definitions(oracle):
    """sum mode with a bias, and a pool2 level = adaptive_avg_pool2d(RoIAlign(2P, sr=0), P), composed from the oracle."""
    torch.manual_seed(5)
    B, C = 2, 16
    a, s = torch.randn(B, C, 40, 52), torch.randn(B, C, 20, 26)
    g = torch.Generator().manual_seed(6)
    ctr = 8 + torch.rand(120, 2, generator=g) * torch.tensor([190.0, 140.0])
    wh = 3 + torch.rand(120, 2, generator=g) * 60
    rois = torch.cat([torch.randint(0, B, (120, 1), generator=g).float(), ctr - wh / 2, ctr + wh / 2], 1)
    bias = torch.randn(120, C)
    for P in (7, 14):
        ref, tol = R.roi_align_ref64([a, s], rois, P, [0.25, 0.125], 2, mode="sum", bias=bias, pool2=[False, True])
        want = oracle.roi_align(a, rois, P, 0.25, 2) + F.adaptive_avg_pool2d(oracle.roi_align(s, rois, 2 * P, 0.125, 0), P)
        want = want + bias[:, :, None, None]
        _within(want, ref, tol, f"pool2 P={P}")


def test_reference_attention_pool_matches_oracle_and_torch_eps(oracle):
    """the centre cell, the cosine's eps (each norm clamped to 1e-8, as the installed torch does) and the relu threshold"""
    a, b = torch.tensor([[3e-9, 4e-9]]), torch.tensor([[1e-3, 0.0]])
    assert abs(F.cosine_similarity(a, b, dim=1).item() - 0.3) < 1e-6       # (3e-9 / 1e-8) * 1: clamped separately
    torch.manual_seed(7)
    B, C, H, W = 3, 24, 9, 13
    f = torch.randn(B, C, H, W)
    f[0, :, 2, 3] = 0.0                                  # a zero vector
    f[1, :, 4, 4] *= 1e-6                                # a near-zero one (norm ~ 5e-6)
    feats = [torch.zeros(B, C, 4 * H, 4 * W), torch.zeros(B, C, 2 * H, 2 * W), f, torch.randn(B, C, 5, 7)]
    rois = _rois(90, B, 16 * W, 16 * H, seed=8, lo=1.0, hi=300.0)
    rois[3, 0], rois[3, 1:] = 0, torch.tensor([2 * 16 * 3.0, 2 * 16 * 2.0, 0.0, 0.0])   # centre on the zero vector's cell
    rois[4, 0], rois[4, 1:] = 1, torch.tensor([2 * 16 * 4.0, 2 * 16 * 4.0, 0.0, 0.0])
    for thres in (0.0, 0.2, 0.9):
        ref, tol = R.attention_pool_ref64(f, rois, 16, thres)
        want = oracle.attention_roi_extract(feats, rois, (4, 8, 16, 32), 1, 0, start_level=2, thres=thres)
        r3, t3 = R.attention_pool_ref64(feats[3], rois, 32, thres)
        _within(want[:, :, 0, 0], ref + r3, tol + t3 + R.U32 * (ref.abs() + r3.abs()), f"thres={thres}")


@pytest.mark.parametrize("P,sr", [(7, 2), (14, 0)])
def test_reference_attention_extractor_matches_oracle(oracle, P, sr):
    from nuhtc_b200 import synth
    feats = [f[:, :, :, : f.shape[3] * 3 // 4].contiguous() for f in synth.fpn_levels(2, 32, frame=256, seed=9)]   # non-square
    rois = synth.proposals(2, 100, "nuclei", frame=256, seed=10)
    ref, tol = R.attention_extractor_ref64(feats, rois, synth.FPN_STRIDES, P, sr, thres=0.2)
    want = oracle.attention_roi_extract(feats, rois, synth.FPN_STRIDES, P, sr, start_level=2, thres=0.2)
    _within(want, ref, tol, "attention extractor")


def test_reference_matches_attention_golden():
    """tests/golden/attention_extractor.npz: the reference's own AttentionRoIExtractor (make_golden.py), fp32 CPU"""
    from nuhtc_b200 import synth
    z = np.load(os.path.join(G, "attention_extractor.npz"))
    feats = synth.fpn_levels(2, 64, frame=256, seed=21)
    rois = torch.from_numpy(z["rois"])
    ref, tol = R.attention_extractor_ref64(feats, rois, synth.FPN_STRIDES, 7, 2, thres=0.0)
    cs = int(z["channel_stride"])
    _within(torch.from_numpy(z["out"]), ref[:, ::cs], tol[:, ::cs], "golden channels")
    _within(torch.from_numpy(z["out_bin_sum"]), ref.sum((2, 3)), tol.sum((2, 3)) + 49 * R.U32 * ref.abs().sum((2, 3)), "golden bin sums")


def test_reference_routing_matches_level_golden():
    z = np.load(os.path.join(G, "roi_levels.npz"))
    assert np.array_equal(R.route_levels(torch.from_numpy(z["rois"]), 4), z["levels"])


def test_reference_matches_torchvision():
    tv = pytest.importorskip("torchvision.ops")
    torch.manual_seed(11)
    x = torch.randn(2, 8, 30, 45)
    rois = _rois(120, 2, 180, 120, seed=12)
    for aligned in (True, False):
        for sr in (0, 2, 3):
            ref, tol = R.roi_align_ref64([x], rois, 7, [0.25], sr, aligned)
            out = tv.roi_align(x, rois, 7, 0.25, sr, aligned)
            _within(out, ref, tol, f"torchvision aligned={aligned} sr={sr}")


def test_window_geometry_helper():
    """the strip-staging geometry the GPU tests build their edge cases from: a bin of exactly 8 / 9 taps"""
    # scale 1, aligned: start = x1 - 0.5; P = 7 with sr = 1: one sample per bin at start + (p + .5) * bin
    rois = torch.tensor([[0, 0.5, 0.5, 0.5 + 7 * 7.0, 4.0], [0, 0.5, 0.5, 0.5 + 7 * 8.0, 4.0]])
    w = R.windows(rois, [(64, 64)], [1.0], 7, sr=8, mode="sum")
    assert [d["xtaps"] for d in w] == [8, 9] and [d["x0"] for d in w] == [0, 0]
    # a sample exactly on -1 is kept (weight 1 on cell 0); just below it is dropped
    A, lo, taps = R.axis_matrix(np.float32(-1.5), np.float32(1.0), 7, 1, 10)
    assert lo == 0 and A[0, 0] == 1.0 and taps[0] == 2
    A, lo, taps = R.axis_matrix(np.float32(np.nextafter(np.float32(-1.5), np.float32(-2))), np.float32(1.0), 7, 1, 10)
    assert taps[0] == 0 and A[0].sum() == 0
