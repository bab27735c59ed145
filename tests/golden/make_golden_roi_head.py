"""Golden results of the RoI head's test path, made by EXECUTING THE REFERENCE'S OWN SOURCE:

  HybridTaskCascadeRoIHead_Lite.simple_test / _bbox_forward      nuhtc/models/htc_roi_head_cus.py:2184-2376, 187-203
  AttentionRoIExtractor.forward                                  nuhtc/models/roi_extractors_cus.py:195-259
  Shared2FCBBoxHeadWithProb.get_bboxes + multiclass_nms          nuhtc/models/bbox_head.py:230-292, 12-102
  SeesawLoss.get_activation / _split_cls_score                   mmdet/models/losses/seesaw_loss.py:138-175
  BBoxHead.regress_by_class                                      mmdet/models/roi_heads/bbox_heads/bbox_head.py:459-496
  delta2bbox, bbox2roi, bbox2result, merge_aug_masks             mmdet/core/...
  FCNMaskHead.get_seg_masks + _do_paste_mask                     mmdet/models/roi_heads/mask_heads/fcn_mask_head.py:179-412

pulled out with `ast` (decorators stripped) and run on the CPU.  The mmcv ops they reach (RoIAlign, batched_nms) are the
oracle's restatements; the heads are the seeded toy modules of tests/_toy_heads.py.  Runs in the build container only.

    python tests/golden/make_golden_roi_head.py
"""
import ast
import os
import sys
from warnings import warn

import numpy as np
import torch
import torch.nn.functional as F

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))


def extract(path, name, cls=None, extra=None):
    src = open(os.path.join(REF, path)).read()
    tree = ast.parse(src)
    body = tree.body
    if cls is not None:
        body = next(n for n in tree.body if isinstance(n, ast.ClassDef) and n.name == cls).body
    fn = next(n for n in body if isinstance(n, ast.FunctionDef) and n.name == name)
    fn.decorator_list = []
    mod = ast.Module(body=[fn], type_ignores=[])
    ns = {"torch": torch, "np": np, "F": F}
    ns.update(extra or {})
    exec(compile(mod, path, "exec"), ns)
    return ns[name]


class Cfg(dict):
    __getattr__ = dict.get


def main():
    import einops
    import types
    from oracle import cpu as O
    from nuhtc_b200 import synth
    import _toy_heads as T

    MM = "thirdparty/mmdetection/mmdet/"
    d2b = extract(MM + "core/bbox/coder/delta_xywh_bbox_coder.py", "delta2bbox")
    bbox2roi = extract(MM + "core/bbox/transforms.py", "bbox2roi")
    bbox2result = extract(MM + "core/bbox/transforms.py", "bbox2result")
    merge_aug_masks = extract(MM + "core/post_processing/merge_augs.py", "merge_aug_masks")
    paste = extract(MM + "models/roi_heads/mask_heads/fcn_mask_head.py", "_do_paste_mask")
    ref_get_seg_masks = extract(MM + "models/roi_heads/mask_heads/fcn_mask_head.py", "get_seg_masks", cls="FCNMaskHead",
                            extra={"_do_paste_mask": paste, "BYTES_PER_FLOAT": 4, "GPU_MEM_LIMIT": 1024 ** 3, "warn": warn})
    mnms = extract("nuhtc/models/bbox_head.py", "multiclass_nms", extra={"batched_nms": O.batched_nms})
    ref_get_bboxes = extract("nuhtc/models/bbox_head.py", "get_bboxes", cls="Shared2FCBBoxHeadWithProb", extra={"multiclass_nms": mnms})
    regress = extract(MM + "models/roi_heads/bbox_heads/bbox_head.py", "regress_by_class", cls="BBoxHead")
    split = extract(MM + "models/losses/seesaw_loss.py", "_split_cls_score", cls="SeesawLoss")
    act = extract(MM + "models/losses/seesaw_loss.py", "get_activation", cls="SeesawLoss")
    att = extract("nuhtc/models/roi_extractors_cus.py", "forward", cls="AttentionRoIExtractor", extra={"einops": einops})
    bbox_forward = extract("nuhtc/models/htc_roi_head_cus.py", "_bbox_forward", cls="HybridTaskCascadeRoIHead_Cus",   # inherited by _Lite
                           extra={"adaptive_avg_pool2d": F.adaptive_avg_pool2d})
    ref_simple_test = extract("nuhtc/models/htc_roi_head_cus.py", "simple_test", cls="HybridTaskCascadeRoIHead_Lite",
                          extra={"bbox2roi": bbox2roi, "bbox2result": bbox2result, "merge_aug_masks": merge_aug_masks})

    class Layer:
        def __init__(self, scale, P, sr):
            self.output_size, self.scale, self.sr = (P, P), scale, sr

        def __call__(self, feat, r):
            return O.roi_align(feat, r, self.output_size[0], self.scale, self.sr, nthreads=8)

    def extractor(P, sr, strides):
        e = types.SimpleNamespace(out_channels=64, start_level=[2, 3], thres=0, aggregation="sum", with_pre=False, with_post=False,
                                  roi_layers=[Layer(1 / s_, P, sr) for s_ in strides], featmap_strides=list(strides))
        e.__call__ = None
        fn = lambda feats, rois, e=e: att(e, feats, rois)
        fn.featmap_strides = list(strides)
        return fn

    class Seesaw:
        num_classes = T.NUM_CLASSES
        _split_cls_score = split
        get_activation = act

    class Coder:
        def __init__(self, stds):
            self.stds = stds

        def decode(self, b, d, max_shape=None):
            return d2b(b, d, (0., 0., 0., 0.), self.stds, max_shape)

    class BHead:
        custom_cls_channels, reg_class_agnostic, num_classes = True, True, T.NUM_CLASSES
        loss_cls = Seesaw()
        regress_by_class = regress
        get_bboxes = ref_get_bboxes

        def __init__(self, i):
            self.m = T.ToyBBoxHead(i)
            self.bbox_coder = Coder(T.STDS[i])

        def __call__(self, f):
            return self.m(f)

    class MHead:
        num_classes, class_agnostic = T.NUM_CLASSES, True
        get_seg_masks = ref_get_seg_masks

        def __init__(self):
            self.m = T.ToyMaskHead()

        def __call__(self, f, last_feat=None):
            return self.m(f), None

    sem = T.ToySemanticHead()

    class Head:
        with_semantic, seg_head, with_watershed_proposal, with_seg, with_mask, mask_info_flow = True, None, False, False, True, True
        num_stages = 3
        semantic_fusion = ("bbox", "mask")
        test_cfg = Cfg(T.TEST_CFG)
        _bbox_forward = bbox_forward
        simple_test = ref_simple_test

        def __init__(self):
            self.bbox_head = [BHead(i) for i in range(3)]
            self.mask_head = [MHead()]
            self.bbox_roi_extractor = [extractor(7, 2, (4, 8, 16, 32))] * 3
            self.mask_roi_extractor = [extractor(14, 0, (4, 8, 16, 32))]
            self.semantic_roi_extractor = extractor(14, 0, (4,))

        def semantic_head(self, x):
            return sem(x)

    B, frame = 2, 512
    feats = synth.fpn_levels(B, T.C, frame=frame, seed=41)
    props = synth.proposals(B, 150, "nuclei", frame=frame, seed=42)
    proposal_list = [torch.cat([props[props[:, 0] == b][:, 1:], torch.ones(int((props[:, 0] == b).sum()), 1)], 1) for b in range(B)]
    metas = [dict(img_shape=(frame, frame, 3), ori_shape=(256, 256, 3), scale_factor=np.array([2., 2., 2., 2.], dtype=np.float32),
                  flip=False)] * B
    out = {}
    with torch.no_grad():
        head = Head()
        # the fused bbox features of stage 0, for the extractor-level test
        sem_pred, sem_feat = sem(feats)
        rois = bbox2roi([p[:, :4] for p in proposal_list])
        bf = head.bbox_roi_extractor[0](feats[:4], rois)
        sf = F.adaptive_avg_pool2d(head.semantic_roi_extractor([sem_feat], rois), (7, 7))
        # every 32nd channel whole + every channel's sum over the 7x7 bins: the full features are 3.7 MB of incompressible floats
        out["bbox_feats"] = (bf + sf)[:, ::32].contiguous().numpy()
        out["channel_stride"] = np.int64(32)
        out["bbox_feats_bin_sum"] = (bf + sf).double().sum((2, 3)).float().numpy()
        res = head.simple_test(torch.zeros(B, 3, frame, frame), tuple(feats), proposal_list, metas, rescale=True)
    for i, (bbox_result, segm_result) in enumerate(res):
        out[f"det_{i}"] = np.concatenate([np.concatenate([b, np.full((len(b), 1), c, np.float32)], 1) for c, b in enumerate(bbox_result)])
        masks = [m for c in segm_result for m in c]
        out[f"mask_{i}"] = np.packbits(np.stack(masks).astype(np.uint8), axis=2) if masks else np.zeros((0, 256, 32), np.uint8)
        print("image", i, "detections", len(out[f"det_{i}"]), "per class", [len(b) for b in bbox_result])
    np.savez_compressed(os.path.join(HERE, "roi_head_simple_test.npz"), **out)
    print("written")


if __name__ == "__main__":
    main()
