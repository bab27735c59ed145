#!/usr/bin/env python
"""Per-op microbenchmarks on one GPU (CUDA events, L2-exceeding working sets): achieved algorithmic GB/s and the
fraction of the measured HBM peak for every kernel of the RoI stage.  Not the contract bench (that is bench.py)."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import nuhtc_b200 as nb
from nuhtc_b200 import synth


def timeit(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    t = sorted(x.elapsed_time(y) for x, y in evs)
    return float(np.median(t)), t[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=256)
    ap.add_argument("--tiles", type=int, default=16)
    ap.add_argument("--tag", default="")
    ap.add_argument("--only", default="")
    ap.add_argument("--impl", default="auto", choices=["auto", "nhwc"], help="RoIAlign path: strip-shared (CG32) or round-1 per-RoI (NHWC)")
    a = ap.parse_args()
    peak = 6550.7
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    B, C = a.tiles, a.channels
    dev = "cuda"
    feats = [f.to(dev) for f in synth.fpn_levels(B, C)]
    if a.impl == "auto":
        nchw_cl = nb.stage_levels(feats)            # staged once: no layout work inside the timed call
    else:
        nhwc = [nb.to_nhwc(f) for f in feats]
        nchw_cl = [n.permute(0, 3, 1, 2) for n in nhwc]  # channels_last views: no staging inside the timed call
    scales = [1 / s for s in synth.FPN_STRIDES]
    out = []

    def rec(name, ms, best, nbytes, **kw):
        r = dict(op=name, tag=a.tag, ms=round(ms, 4), best_ms=round(best, 4), GBps=round(nbytes / ms / 1e6, 1),
                 frac_of_measured_peak=round(nbytes / ms / 1e6 / peak, 4), bytes=int(nbytes), **kw)
        out.append(r)
        print(json.dumps(r), flush=True)

    def want(n):
        return not a.only or a.only in n or n in a.only

    for dist in ("nuclei", "routed"):
        rois = synth.proposals(B, 1000, dist).to(dev)
        K = rois.shape[0]
        lv = sorted(set(torch.floor(torch.log2(torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2])) / 56 + 1e-6)).clamp(0, 3).long().tolist()))
        inb = sum(feats[l].numel() * 4 for l in lv)
        for P, sr in ((7, 0), (7, 2), (14, 0)):
            if not want(f"roi_align_{P}"):
                continue
            o = torch.empty(K, C, P, P, device=dev)
            ms, best = timeit(lambda: nb.roi_align_levels(nchw_cl, rois, P, scales, sr, mode="route", out=o, impl=a.impl))
            rec(f"roi_align_{P}x{P}_sr{sr}_{dist}", ms, best, K * C * P * P * 4 + inb + K * 20, K=K)
            del o
    if want("sum"):
        rois = synth.proposals(B, 1000, "nuclei").to(dev)
        f64 = [f.to(dev) for f in synth.fpn_levels(B, 64)][:2]
        n64 = nb.stage_levels(f64) if a.impl == "auto" else [nb.to_nhwc(f).permute(0, 3, 1, 2) for f in f64]
        o = torch.empty(rois.shape[0], 64, 7, 7, device=dev)
        ms, best = timeit(lambda: nb.roi_align_levels(n64, rois, 7, [1 / 4, 1 / 8], 2, mode="sum", out=o, impl=a.impl))
        rec("roi_align_7x7_sr2_sum01_C64", ms, best, o.numel() * 4 + sum(f.numel() * 4 for f in f64) + rois.shape[0] * 20)
    if want("nhwc"):
        ms, best = timeit(lambda: [nb.to_nhwc(f) for f in feats])
        rec("nchw_to_nhwc_4levels", ms, best, 2 * sum(f.numel() * 4 for f in feats))
        ms, best = timeit(lambda: [nb.to_cg32(f) for f in feats])
        rec("nchw_to_cg32_4levels", ms, best, 2 * sum(f.numel() * 4 for f in feats))
    boxes, probs, scores = synth.nuclei_masks(8000, seed=0)
    boxes, probs, scores = boxes.to(dev), probs.to(dev), scores.to(dev)
    if want("paste"):
        for kind, per in (("bin", 65536), ("bits", 8192), ("prob", 262144)):
            ms, best = timeit(lambda: nb.paste_masks(probs, boxes, 256, 256, thr=0.5, kind=kind, want_stats=(kind != "prob")))
            rec(f"paste_{kind}_8000", ms, best, 8000 * (per + 28 * 28 * 4 + 16))
    dense = nb.paste_masks(probs, boxes, 256, 256, thr=0.5, kind="bin")
    if want("pack"):
        ms, best = timeit(lambda: nb.pack_masks(dense))
        rec("pack_masks_8000", ms, best, 8000 * (65536 + 8192))
    bits, area, bbox = nb.pack_masks(dense)
    tile = (torch.arange(8000, device=dev) // 500).to(torch.int32)
    if want("mask_nms"):
        ms, best = timeit(lambda: nb.mask_nms_device(bits, area, bbox, scores, 256, 0.05, tile=tile, num_tiles=16, max_tile_size=500))
        rec("mask_nms_16x500", ms, best, 8000 * 8192)
    if want("nms"):
        bs, ss, ls, gs = [], [], [], []
        for g in range(16):
            b_, s_, l_ = synth.nms_boxes(5000, seed=g)
            bs.append(b_); ss.append(s_); ls.append(l_); gs.append(torch.full((5000,), g, dtype=torch.int32))
        Bx, Sx, Lx, Gx = (torch.cat(t).to(dev) for t in (bs, ss, ls, gs))
        Bx = Bx + 20.0
        ms, best = timeit(lambda: nb.nms_groups(Bx, Sx, Lx, Gx, 16, 5000, 0.5, 0, "offset"))
        rec("nms_16x5000_grouped", ms, best, 80000 * 28, boxes_per_s=round(80000 / ms * 1e3))
        ms, best = timeit(lambda: nb.nms_groups(Bx, Sx, Lx, Gx, 16, 5000, 0.5, 0, "offset", num_classes=5))
        rec("nms_16x5000_grouped_class_segments", ms, best, 80000 * 28, boxes_per_s=round(80000 / ms * 1e3))
        for N in (2000, 20000, 200000):
            b_, s_, l_ = (t.to(dev) for t in synth.nms_boxes(N, seed=1))
            cfg = dict(type="nms", iou_threshold=0.5)
            ms, best = timeit(lambda: nb.batched_nms(b_, s_, l_, cfg), iters=5, warm=2)
            rec(f"batched_nms_{N}", ms, best, N * 28, boxes_per_s=round(N / ms * 1e3))
    if want("attention"):
        # AttentionRoIExtractor (PanNuke config): C = 64, levels 2,3 of a 512 px frame, K = 16000 RoIs
        f64 = [f.to(dev) for f in synth.fpn_levels(B, 64)]
        r_ = synth.proposals(B, 1000, "nuclei").to(dev)
        for lvl in (2, 3):
            ms, best = timeit(lambda: nb.mmcv_ops.attention_pool(f64[lvl], r_, float(synth.FPN_STRIDES[lvl]), 0.0))
            hw = f64[lvl].shape[2] * f64[lvl].shape[3]
            rec(f"attention_pool_level{lvl}_C64", ms, best, f64[lvl].numel() * 4 + r_.shape[0] * (20 + 256),
                gflops=round(4 * 64 * hw * r_.shape[0] / ms / 1e6, 1))
    if want("rpn"):
        from nuhtc_b200 import rpn
        g = torch.Generator().manual_seed(0)
        cls, reg, anc = [], [], []
        for s_ in (4, 8, 16, 32):
            h_ = 512 // s_
            cls.append((torch.randn(B, 3, h_, h_, generator=g) * 2).to(dev))
            reg.append((torch.randn(B, 12, h_, h_, generator=g) * 0.25).to(dev))
            ys, xs = torch.meshgrid(torch.arange(h_), torch.arange(h_), indexing="ij")
            ctr = torch.stack([xs, ys], -1).reshape(-1, 1, 2).float() * s_
            wh = torch.tensor([[1.0, 1.0], [1.4, 0.7], [0.7, 1.4]]) * (4.0 * s_)
            anc.append(torch.cat([ctr - wh / 2, ctr + wh / 2], -1).reshape(-1, 4).to(dev))

        class Cfg(dict):
            __getattr__ = dict.get
        rcfg = Cfg(nms_pre=1000, min_bbox_size=0, nms=dict(type="nms", iou_threshold=0.7), max_per_img=1000)
        ms, best = timeit(lambda: rpn.proposals_batched(cls, reg, anc, (512, 512, 3), rcfg), iters=5, warm=2)
        rec(f"rpn_proposals_batched_{B}img_nms_pre1000", ms, best, B * 4000 * 28, images_per_s=round(B / ms * 1e3))
    if want("watershed"):
        # watershed proposals (f4): 16 semantic maps at stride 4 of a 512 px frame -> instances of the hole-filled mask
        from nuhtc_b200 import watershed as ws
        g = torch.Generator().manual_seed(0)
        sem = torch.nn.functional.interpolate(torch.randn(B, 1, 32, 32, generator=g), size=(128, 128), mode="bicubic").to(dev) * 3
        m = ws.semantic_mask(sem, (512, 512), 0.0)
        ms, best = timeit(lambda: ws.semantic_mask(sem, (512, 512), 0.0))
        rec("watershed_semantic_mask_torch_16x512", ms, best, B * 512 * 512 * 4 * 2)
        ms, best = timeit(lambda: ws.mask_components(m))
        bx, cnt = ws.mask_components(m)
        rec("watershed_components_16x512", ms, best, B * 512 * 512 * 5, instances=int(cnt.sum().item()))
    if want("preprocess"):
        # one TilePipeline call from a uint8 CUDA tensor, host overhead included; the output block is reused from call to
        # call, so tools/bench_preprocess.py is where the kernel is timed with an L2-exceeding working set
        from nuhtc_b200.preprocess import TilePipeline
        t = torch.randint(0, 256, (B, 256, 256, 3), dtype=torch.uint8, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
        for s in (2.0, 4.0):
            pipe = TilePipeline(s, [123.675, 116.28, 103.53], [58.395, 57.12, 57.375])
            ph, pw = pipe.sizes(256, 256)[2:4]
            ms, best = timeit(lambda: pipe(t))
            rec(f"preprocess_{B}x256_to_{ph}", ms, best, t.numel() + B * 3 * ph * pw * 4)
    if want("merge"):
        d = synth.slide_nuclei(64, 64, per_tile=23, seed=0)
        xy, voff, sc = (torch.from_numpy(d[k]).to(dev) for k in ("xy", "voff", "score"))
        ms, best = timeit(lambda: nb.merge_arrays(xy, voff, sc, 0.05), iters=5, warm=2)
        rec(f"merge_{sc.numel()}", ms, best, xy.numel() * 8 + sc.numel() * 20, nuclei_per_s=round(sc.numel() / ms * 1e3))


if __name__ == "__main__":
    main()
