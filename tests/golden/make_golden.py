"""Generate golden vectors by EXECUTING THE REFERENCE'S OWN SOURCE for the pure-torch parts of the path.

Runs only in the build container (it reads /root/reference, which does not exist on the GPU box); the .npz
files it writes are committed and are what the test-suite reads.  The functions are pulled out of the
reference files with `ast` (decorators stripped, so neither mmcv nor mmdet has to import) and exec'd
against torch/numpy:

  _do_paste_mask      thirdparty/mmdetection/mmdet/models/roi_heads/mask_heads/fcn_mask_head.py:344-412
  delta2bbox          thirdparty/mmdetection/mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:163-260
  bbox2roi            thirdparty/mmdetection/mmdet/core/bbox/transforms.py:59-78
  map_roi_levels      thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:36-55
  multiclass_nms      nuhtc/models/bbox_head.py:12-102  (its `batched_nms` import is mmcv's: the oracle's
                      restatement is injected, so this pins the wrapper logic around it)

The mmcv / pycocotools / shapely kernels themselves cannot be executed here (not installed, no network):
those boundaries stay "parity unpinned" and are anchored on torchvision CPU ops / brute force instead.

    python tests/golden/make_golden.py
"""
import ast
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))


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


def main():
    from oracle import cpu as O
    from nuhtc_b200 import synth
    g = torch.Generator().manual_seed(0)

    # ---- paste
    paste = extract("thirdparty/mmdetection/mmdet/models/roi_heads/mask_heads/fcn_mask_head.py", "_do_paste_mask")
    boxes, probs, _ = synth.nuclei_masks(24, frame=96, seed=5)
    boxes[0] = torch.tensor([-10.0, -7.5, 14.2, 9.9])
    boxes[1] = torch.tensor([80.3, 70.0, 110.0, 99.0])
    boxes[2] = torch.tensor([30.0, 40.0, 30.0, 60.0])
    boxes[3] = torch.tensor([0.0, 0.0, 96.0, 96.0])
    full, _ = paste(probs, boxes, 96, 96, skip_empty=False)
    part, sl = paste(probs[4:5], boxes[4:5], 96, 96, skip_empty=True)
    np.savez_compressed(os.path.join(HERE, "paste.npz"), boxes=boxes.numpy(), probs=probs.numpy(), full=full.numpy(),
                        part=part.numpy(), part_slices=np.array([sl[0].start, sl[0].stop, sl[1].start, sl[1].stop]))

    # ---- delta2bbox (+ the reference's own known-answer test, tests/test_utils/test_coder.py:27-40)
    d2b = extract("thirdparty/mmdetection/mmdet/core/bbox/coder/delta_xywh_bbox_coder.py", "delta2bbox")
    rois = torch.Tensor([[0., 0., 1., 1.], [0., 0., 1., 1.], [0., 0., 1., 1.], [5., 5., 5., 5.]])
    deltas = torch.Tensor([[0., 0., 0., 0.], [1., 1., 1., 1.], [0., 0., 2., -1.], [0.7, -1.9, -0.5, 0.3]])
    kat = d2b(rois, deltas, max_shape=(32, 32, 3))
    expected = torch.Tensor([[0.0000, 0.0000, 1.0000, 1.0000], [0.1409, 0.1409, 2.8591, 2.8591],
                             [0.0000, 0.3161, 4.1945, 0.6839], [5.0000, 5.0000, 5.0000, 5.0000]])
    assert kat.allclose(expected, atol=1e-4), "reference delta2bbox failed its own KAT?"
    r = synth.proposals(1, 300, "nuclei", seed=3)[:, 1:]
    dl = torch.randn(300, 4, generator=g)
    dec = d2b(r, dl, means=(0., 0., 0., 0.), stds=(0.1, 0.1, 0.2, 0.2), max_shape=(512, 512, 3))
    np.savez_compressed(os.path.join(HERE, "delta2bbox.npz"), kat_rois=rois.numpy(), kat_deltas=deltas.numpy(), kat_out=kat.numpy(),
                        rois=r.numpy(), deltas=dl.numpy(), out=dec.numpy())

    # ---- map_roi_levels / bbox2roi
    class _Self:
        finest_scale = 56
    mrl = extract("thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py", "map_roi_levels",
                  cls="SingleRoIExtractor")
    rr = synth.proposals(4, 500, "routed", seed=8)
    rr[:8, 1:] = torch.tensor([[0, 0, 112, 112], [0, 0, 111.99, 112], [0, 0, 224, 224], [0, 0, 448, 448], [0, 0, 56, 56],
                               [5, 5, 5, 5], [0, 0, 223.9999, 224], [0, 0, 512, 512]], dtype=torch.float32)
    lv = mrl(_Self(), rr, 4)
    b2r = extract("thirdparty/mmdetection/mmdet/core/bbox/transforms.py", "bbox2roi")
    lst = [torch.rand(5, 5, generator=g), torch.zeros(0, 5), torch.rand(3, 4, generator=g)]
    np.savez_compressed(os.path.join(HERE, "roi_levels.npz"), rois=rr.numpy(), levels=lv.numpy(),
                        b2r_in0=lst[0].numpy(), b2r_in2=lst[2].numpy(), b2r_out=b2r(lst).numpy())

    # ---- multiclass_nms (nuhtc copy) with the oracle's batched_nms injected
    mc = extract("nuhtc/models/bbox_head.py", "multiclass_nms", extra={"batched_nms": O.batched_nms})
    n, C = 1000, 5
    bx = synth.nms_boxes(n, seed=12)[0]
    sc = torch.rand(n, C + 1, generator=g)
    sc = sc / sc.sum(1, keepdim=True) * 1.8
    dets, labels, _ = mc(bx, sc, 0.35, dict(type="nms", iou_threshold=0.5), 500, return_inds=True)
    np.savez_compressed(os.path.join(HERE, "multiclass_nms.npz"), boxes=bx.numpy(), scores=sc.numpy(), dets=dets.numpy(),
                        labels=labels.numpy())
    # ---- AttentionRoIExtractor.forward (the extractor of all four shipped configs) with mmcv's RoIAlign layers
    # replaced by the oracle's restatement: pins the attention branch, the centre-cell rule and the level sum
    import einops

    class _Layer:
        def __init__(self, scale, P, sr):
            self.output_size, self.scale, self.sr = (P, P), scale, sr

        def __call__(self, feat, r):
            return O.roi_align(feat, r, self.output_size[0], self.scale, self.sr)

    class _Ext:
        out_channels, start_level, thres, aggregation, with_pre, with_post = 64, [2, 3], 0, "sum", False, False
        roi_layers = [_Layer(1 / s_, 7, 2) for s_ in (4, 8, 16, 32)]

        def roi_rescale(self, r, f):
            raise NotImplementedError

    att = extract("nuhtc/models/roi_extractors_cus.py", "forward", cls="AttentionRoIExtractor", extra={"einops": einops})
    feats = synth.fpn_levels(2, 64, frame=256, seed=21)
    arois = synth.proposals(2, 60, "nuclei", frame=256, seed=22)
    aout = att(_Ext(), feats, arois)
    # every 16th channel whole + every channel's sum over the 7x7 bins: the full output is 1.5 MB of incompressible floats
    np.savez_compressed(os.path.join(HERE, "attention_extractor.npz"), rois=arois.numpy(), out=aout[:, ::16].contiguous().numpy(),
                        channel_stride=np.int64(16), out_bin_sum=aout.double().sum((2, 3)).float().numpy())
    # ---- RPNHead._bbox_post_process from the reference source (bbox_coder.decode = the reference delta2bbox,
    # batched_nms = the oracle's mmcv restatement)
    class _Coder:
        @staticmethod
        def decode(anchors, deltas, max_shape=None):
            return d2b(anchors, deltas, max_shape=max_shape)

    class _Rpn:
        bbox_coder = _Coder()

    class _Cfg(dict):
        __getattr__ = dict.get

    post = extract("thirdparty/mmdetection/mmdet/models/dense_heads/rpn_head.py", "_bbox_post_process", cls="RPNHead",
                   extra={"batched_nms": O.batched_nms})
    n_lv = [600, 300, 150, 75]
    anchors, deltas, sc, ids = [], [], [], []
    for l, n_ in enumerate(n_lv):
        ctr = torch.rand(n_, 2, generator=g) * 512
        wh = (8 * 2 ** l) * (0.5 + torch.rand(n_, 2, generator=g))
        anchors.append(torch.cat([ctr - wh / 2, ctr + wh / 2], 1))
        deltas.append(torch.randn(n_, 4, generator=g) * 0.3)
        sc.append(torch.rand(n_, generator=g))
        ids.append(torch.full((n_,), l, dtype=torch.long))
    rcfg = _Cfg(min_bbox_size=0, nms=dict(type="nms", iou_threshold=0.7), max_per_img=300)
    rdets = post(_Rpn(), sc, deltas, anchors, ids, rcfg, (512, 512, 3))
    np.savez_compressed(os.path.join(HERE, "rpn_post.npz"), anchors=torch.cat(anchors).numpy(), deltas=torch.cat(deltas).numpy(),
                        scores=torch.cat(sc).numpy(), ids=torch.cat(ids).numpy(), dets=rdets.numpy())
    # ---- mask2inst (tools/infer_wsi.py:51-54) with the real cv2 (the function body is the reference's own)
    import cv2
    m2i = extract("tools/infer_wsi.py", "mask2inst", extra={"cv2": cv2, "np": np})
    rng = np.random.default_rng(5)

    def blobs(h, w, n, r):
        m = np.zeros((h, w), np.uint8)
        yy, xx = np.mgrid[:h, :w]
        for _ in range(n):
            cy, cx = rng.uniform(0, h), rng.uniform(0, w)
            a, b = rng.uniform(1, r, 2)
            t = rng.uniform(0, np.pi)
            u = (xx - cx) * np.cos(t) + (yy - cy) * np.sin(t)
            v = -(xx - cx) * np.sin(t) + (yy - cy) * np.cos(t)
            m |= ((u / a) ** 2 + (v / b) ** 2 <= 1).astype(np.uint8)
        return m

    cm = np.zeros((96, 96, 96), np.uint8)
    for i in range(96):
        kind = i % 4
        if kind == 0:
            cm[i, 20:60, 30:70] = rng.random((40, 40)) < rng.uniform(0.2, 0.8)          # noise: nested borders
        elif kind == 1:
            cm[i] = blobs(96, 96, int(rng.integers(1, 4)), 14)                           # nucleus-like
        elif kind == 2:
            cm[i] = (blobs(96, 96, 2, 30) & (1 - blobs(96, 96, 2, 10))) | blobs(96, 96, 1, 3)   # holes, islands, > 64 px
        else:
            cm[i] = cv2.dilate((rng.random((96, 96)) < 0.3).astype(np.uint8), np.ones((2, 2), np.uint8))
        if not cm[i].any():
            cm[i, 5, 7] = 1
    cm[3] = 0; cm[3, 0, 0] = 1                      # single pixel at the corner
    cm[7] = 1                                       # full frame
    cm[11] = 0; cm[11, 40, 10:90] = 1               # 1-px line
    cont = [m2i(m) for m in cm]
    np.savez_compressed(os.path.join(HERE, "contours.npz"), masks=np.packbits(cm, axis=2),
                        points=np.concatenate([c.reshape(-1, 2) for c in cont]).astype(np.int32),
                        offsets=np.cumsum([0] + [c.shape[0] for c in cont]).astype(np.int64), cv2_version=cv2.__version__)
    print("golden vectors written to", HERE)


if __name__ == "__main__":
    main()
