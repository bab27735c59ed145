"""GPU parity of the RoI-extractor mirrors (same constructor config and forward signature as the reference classes)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
STRIDES = (4, 8, 16, 32)


def _ext_cfg(P, sr, C):
    return dict(roi_layer=dict(type="RoIAlign", output_size=P, sampling_ratio=sr), out_channels=C, featmap_strides=list(STRIDES))


@pytest.mark.parametrize("P,sr", [(7, 2), (14, 0)])
def test_attention_roi_extractor(oracle, P, sr):
    """The extractor of the four shipped NuHTC configs: RoIAlign on levels 0,1 + cosine-attention pooling on 2,3."""
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_extractors import AttentionRoIExtractor
    feats = synth.fpn_levels(3, 64, frame=512, seed=31)
    rois = synth.proposals(3, 150, "nuclei", frame=512, seed=32)
    rois[0, 1:] = torch.tensor([-30.0, -30.0, -10.0, -5.0])      # centre cell clamps to (0, 0)
    rois[1, 1:] = torch.tensor([500.0, 490.0, 600.0, 700.0])     # centre beyond the frame clamps to the last cell
    ext = AttentionRoIExtractor(start_level=2, thres=0, **_ext_cfg(P, sr, 64)).cuda()
    out = ext(tuple(f.cuda() for f in feats), rois.cuda()).cpu()
    ref = oracle.attention_roi_extract(feats, rois, STRIDES, P, sr, start_level=2, thres=0.0)
    assert out.shape == ref.shape
    assert (out - ref).abs().max().item() <= 3e-5   # four summed terms, each to 1e-5
    # a positive threshold exercises the relu
    ext2 = AttentionRoIExtractor(start_level=2, thres=0.2, **_ext_cfg(P, sr, 64)).cuda()
    out2 = ext2(tuple(f.cuda() for f in feats), rois.cuda()).cpu()
    ref2 = oracle.attention_roi_extract(feats, rois, STRIDES, P, sr, start_level=2, thres=0.2)
    assert (out2 - ref2).abs().max().item() <= 3e-5
    # single-level input degenerates to a plain RoIAlign (the semantic extractor, roi_extractors_cus.py:197-198)
    one = ext((feats[0].cuda(),), rois.cuda()).cpu()
    assert (one - oracle.roi_align(feats[0], rois, P, 0.25, sr)).abs().max().item() <= 1e-5
    assert ext(tuple(f.cuda() for f in feats), torch.zeros(0, 5).cuda()).shape == (0, 64, P, P)


def test_attention_pool_golden_from_reference_source(oracle):
    import os
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_extractors import AttentionRoIExtractor
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "attention_extractor.npz"))
    feats = synth.fpn_levels(2, 64, frame=256, seed=21)
    ext = AttentionRoIExtractor(start_level=2, thres=0, **_ext_cfg(7, 2, 64)).cuda()
    out = ext(tuple(f.cuda() for f in feats), torch.from_numpy(z["rois"]).cuda()).cpu()
    assert out.shape == (z["rois"].shape[0], 64, 7, 7)
    # the golden keeps every k-th channel whole and, for every channel, the sum over the 7x7 bins
    assert (out[:, ::int(z["channel_stride"])] - torch.from_numpy(z["out"])).abs().max().item() <= 3e-5
    assert (out.double().sum((2, 3)) - torch.from_numpy(z["out_bin_sum"]).double()).abs().max().item() <= 49 * 3e-5


@pytest.mark.parametrize("C", [64, 256])
def test_single_roi_extractor(oracle, C):
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_extractors import SingleRoIExtractor
    feats = synth.fpn_levels(2, C, frame=256, seed=33)
    rois = synth.proposals(2, 120, "routed", frame=256, seed=34)
    ext = SingleRoIExtractor(finest_scale=56, **_ext_cfg(7, 0, C)).cuda()
    out = ext(tuple(f.cuda() for f in feats), rois.cuda()).cpu()
    ref = oracle.single_roi_extract(feats, rois, STRIDES, 7, 0, 56)
    assert (out - ref).abs().max().item() <= 1e-5
    assert torch.equal(ext.map_roi_levels(rois, 4), oracle.map_roi_levels(rois, 4))
    assert ext.num_inputs == 4 and ext.roi_layers[2].spatial_scale == 1 / 16
    with pytest.raises(NotImplementedError):
        SingleRoIExtractor(roi_layer=dict(type="RoIPool", output_size=7), out_channels=C, featmap_strides=[4])
