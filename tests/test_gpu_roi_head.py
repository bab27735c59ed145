"""GPU parity of the RoI-head drop-in (nuhtc_b200.htc_roi_head) against golden results made by EXECUTING THE REFERENCE'S
simple_test / _bbox_forward source with the same seeded toy heads (tests/golden/make_golden_roi_head.py)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")
B, FRAME = 2, 512


def _inputs():
    from nuhtc_b200 import synth
    import _toy_heads as T
    feats = synth.fpn_levels(B, T.C, frame=FRAME, seed=41)
    props = synth.proposals(B, 150, "nuclei", frame=FRAME, seed=42)
    plist = [torch.cat([props[props[:, 0] == b][:, 1:], torch.ones(int((props[:, 0] == b).sum()), 1)], 1) for b in range(B)]
    metas = [dict(img_shape=(FRAME, FRAME, 3), ori_shape=(256, 256, 3), scale_factor=np.array([2., 2., 2., 2.], dtype=np.float32),
                  flip=False)] * B
    return feats, props, plist, metas


def test_fused_bbox_features_match_reference_bbox_forward():
    """_bbox_forward (htc_roi_head_cus.py:187-203): AttentionRoIExtractor 7x7 sr=2 + adaptive_avg_pool2d of the 14x14 semantic
    RoIAlign, here ONE launch (levels 0,1 + the semantic map pooled at twice the size, attention vector added at the store)."""
    import _toy_heads as T
    from nuhtc_b200 import stage_levels
    from nuhtc_b200.roi_stage import RoIStage, RoIStageConfig, bbox2roi
    z = np.load(os.path.join(G, "roi_head_simple_test.npz"))
    feats, props, plist, _ = _inputs()
    sem = T.ToySemanticHead()
    _, sem_feat = sem(feats)
    cfg = RoIStageConfig(extractor="attention", sum_levels=2, semantic_fusion=("bbox", "mask"), bbox_sampling_ratio=2)
    st = RoIStage(cfg, [None] * 3, None)
    rois = bbox2roi([p[:, :4] for p in plist]).cuda()
    out = st.extract(stage_levels([f.cuda() for f in feats]), rois, 7, 2, stage_levels([sem_feat.cuda()]), "bbox").cpu()
    assert out.shape == (rois.shape[0], T.C, 7, 7)
    # the golden keeps every k-th channel whole and, for every channel, the sum over the 7x7 bins
    sums = out.double().sum((2, 3))
    out = out[:, ::int(z["channel_stride"])]
    ref = torch.from_numpy(z["bbox_feats"])
    assert out.shape == ref.shape
    assert (out - ref).abs().max().item() <= 5e-5      # five summed terms (2 RoIAlign levels, 2 attention levels, semantic)
    assert (sums - torch.from_numpy(z["bbox_feats_bin_sum"]).double()).abs().max().item() <= 49 * 5e-5


def test_simple_test_matches_reference(oracle):
    """simple_test(img, x, proposal_list, img_metas, rescale=True) -> list[(bbox_result, segm_result)]: same detections per
    class in the same order, boxes to 2e-3 px and scores to 5e-5 (the toy heads' GEMMs over 3136 features run on the GPU here
    and on the CPU in the golden run, which moves logits and deltas at the 1e-6 relative level, three cascade stages deep), masks identical except at pixels whose pasted probability is within
    1e-4 of the threshold."""
    import _toy_heads as T
    from nuhtc_b200.htc_roi_head import HybridTaskCascadeRoIHead_Lite, seesaw_activation
    z = np.load(os.path.join(G, "roi_head_simple_test.npz"))
    feats, props, plist, metas = _inputs()
    torch.backends.cudnn.allow_tf32 = False      # the toy heads' convolutions must not run in TF32 (cuDNN's default): this
    torch.backends.cuda.matmul.allow_tf32 = False   # test compares with an fp32 CPU run of the reference
    heads = [T.ToyBBoxHead(i).cuda() for i in range(3)]
    for h in heads:
        h.score_activation = seesaw_activation
    mh, sh = T.ToyMaskHead().cuda(), T.ToySemanticHead().cuda()
    head = HybridTaskCascadeRoIHead_Lite(3, heads, mh, T.TEST_CFG, extractor="attention", start_level=2, thres=0.0,
                                         bbox_roi_layer=dict(type="RoIAlign", output_size=7, sampling_ratio=2),
                                         mask_roi_layer=dict(type="RoIAlign", output_size=14, sampling_ratio=0),
                                         semantic_head=sh, semantic_fusion=("bbox", "mask"))
    res = head.simple_test(torch.zeros(B, 3, FRAME, FRAME), tuple(f.cuda() for f in feats), [p.cuda() for p in plist], metas,
                           rescale=True)
    assert len(res) == B
    for i, (bbox_result, segm_result) in enumerate(res):
        ref = z[f"det_{i}"]
        assert len(bbox_result) == T.NUM_CLASSES and len(segm_result) == T.NUM_CLASSES
        got = np.concatenate([np.concatenate([b, np.full((len(b), 1), c, np.float32)], 1) for c, b in enumerate(bbox_result)])
        assert got.shape == ref.shape, (got.shape, ref.shape)
        assert np.array_equal(got[:, 5], ref[:, 5])                        # same classes in the same order
        assert np.abs(got[:, :4] - ref[:, :4]).max() <= 2e-3               # px; three cascaded decodes of GEMM outputs
        assert np.abs(got[:, 4] - ref[:, 4]).max() <= 5e-5
        masks = np.stack([m for c in segm_result for m in c])
        refm = np.unpackbits(z[f"mask_{i}"], axis=2)[:, :, :256].astype(bool)
        assert masks.dtype == np.bool_ and masks.shape == refm.shape
        diff = masks != refm
        assert diff.mean() < 1e-4, diff.mean()                             # a handful of threshold pixels at most
    # stock signature (no img argument)
    from nuhtc_b200.htc_roi_head import HybridTaskCascadeRoIHead
    stock = HybridTaskCascadeRoIHead(3, heads, mh, T.TEST_CFG, extractor="attention", semantic_head=sh)
    res2 = stock.simple_test(tuple(f.cuda() for f in feats), [p.cuda() for p in plist], metas, rescale=True)
    assert all(np.array_equal(a[0][c], b[0][c]) for a, b in zip(res, res2) for c in range(T.NUM_CLASSES))
    # no proposals at all
    none = head.simple_test(None, tuple(f.cuda() for f in feats), [torch.zeros(0, 5).cuda()] * B, metas, rescale=True)
    assert all(sum(len(b) for b in r[0]) == 0 and all(len(s) == 0 for s in r[1]) for r in none)
