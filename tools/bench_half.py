#!/usr/bin/env python
"""Half-precision RoI stage on one GPU: one JSON line per row.

Arms, at bench.py's shape (C = 256, 16 tiles, K = 16 000 'nuclei' proposals, D = 8 000 mask RoIs, SingleRoIExtractor
routing) and at the PanNuke shape (C = 64, AttentionRoIExtractor: levels 0,1 summed + the pooled attention bias):
  fp32      today's fp32 path
  fp16      fp16 levels, native half staging and half stores
  bf16      bf16 levels, native
  fp16_cast fp16 levels through the fp32 kernels with torch casts at the force_fp32 boundaries (levels upcast once per
            batch, RoI features rounded to fp16 after every call): what a half model pays without the native path
Rows: per-op times (staging, the 7x7 call, the 14x14 call) with CUDA events, the algorithmic bytes of each op from its
shapes and element sizes, their share of the device-to-device copy rate measured in the same run, and a RoIStage step
(stand-in heads whose outputs are in the levels' dtype, captured in a CUDA graph).  The fp32 levels at C = 256 (357 MB)
and every 7x7 / 14x14 output exceed the 126 MB L2.  The run asserts that the fp16 arm's RoI features equal the fp16_cast
arm's bit for bit.  The GPU's name and power limit are read in the same run.

    python tools/bench_half.py [--iters 20] [--shape bench|pannuke|both]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch

import nuhtc_b200 as nb
from nuhtc_b200 import synth
from nuhtc_b200.roi_stage import RoIStage, RoIStageConfig
from bench_ops import timeit
from bench_preprocess import gpu_info, hbm_peak_gbs

ARMS = ("fp32", "fp16", "bf16", "fp16_cast")
SCALES = [1 / s for s in synth.FPN_STRIDES]


def level_of(rois):
    s = torch.sqrt((rois[:, 3] - rois[:, 1]) * (rois[:, 4] - rois[:, 2]))
    return sorted(set(torch.floor(torch.log2(s / 56 + 1e-6)).clamp(0, 3).long().tolist()))


def run_shape(name, B, C, K_per, D, attention, iters, peak, info):
    dev = "cuda"
    f32 = [f.to(dev) for f in synth.fpn_levels(B, C, frame=512, seed=0)]
    rois = synth.proposals(B, K_per, "nuclei", frame=512, seed=0).to(dev)
    mrois = synth.proposals(B, D // B, "nuclei", frame=512, seed=1).to(dev)
    K = rois.shape[0]
    g = torch.Generator().manual_seed(2)
    bias = (torch.randn(K, C, generator=g) * 0.1).to(dev) if attention else None
    mbias = (torch.randn(D, C, generator=g) * 0.1).to(dev) if attention else None
    nlev = 2 if attention else 4
    mode = "sum" if attention else "route"
    sr7 = 2 if attention else 0
    levels = {"fp32": f32, "fp16": [f.half() for f in f32], "bf16": [f.bfloat16() for f in f32]}
    levels["fp16_cast"] = levels["fp16"]
    px = sum(f.shape[2] * f.shape[3] for f in f32) * B * C        # staged elements, all levels
    touched7 = sum(f32[l][0].numel() * B for l in (range(nlev) if attention else level_of(rois)))
    touched14 = sum(f32[l][0].numel() * B for l in (range(nlev) if attention else level_of(mrois)))
    outs = {}

    def emit(op, arm, ms, best, nbytes, **kw):
        r = dict(shape=name, op=op, arm=arm, ms=round(ms, 4), best_ms=round(best, 4), bytes=int(nbytes),
                 GBps=round(nbytes / ms / 1e6, 1), frac_of_copy_rate=round(nbytes / ms / 1e6 / peak, 4), **kw, **info)
        print(json.dumps(r), flush=True)

    for arm in ARMS:
        lv = levels[arm]
        es = lv[0].element_size()
        cast = arm == "fp16_cast"
        odt = lv[0].dtype
        # ---- staging: once per batch (the cast arm upcasts the levels with torch first)
        if cast:
            stage = lambda: nb.stage_levels([f.float() for f in lv])
            sbytes = px * (es + 4) + px * (4 + 4)
        else:
            stage = lambda: nb.stage_levels(lv)
            sbytes = px * (es + 4)
        ms, best = timeit(stage, iters)
        emit("staging", arm, ms, best, sbytes)
        st = stage()
        st_lv = st.sub(range(nlev))
        # ---- the two RoIAlign calls
        for P, sr, R, Rb, touched in ((7, sr7, rois, bias, touched7), (14, 0, mrois, mbias, touched14)):
            n = R.shape[0]
            o = torch.empty(n, C, P, P, dtype=torch.float32 if cast else odt, device=dev)
            call = lambda: nb.roi_align_levels(st_lv, R, P, SCALES[:nlev], sr, mode=mode, finest_scale=56.0, out=o, bias=Rb)
            fn = (lambda: call().half()) if cast else call
            obytes = n * C * P * P
            nbytes = obytes * (4 + 4 + 2 if cast else es) + touched * 4 + n * 20 + (n * C * 4 if Rb is not None else 0)
            ms, best = timeit(fn, iters)
            emit(f"roi_align_{P}x{P}_sr{sr}", arm, ms, best, nbytes, K=n, C=C)
            outs[(arm, P)] = fn()
            del o
        # ---- one RoIStage step, CUDA graph (stand-in heads: outputs in the levels' dtype, independent of the features)
        cfg = RoIStageConfig(extractor="attention" if attention else "single", sum_levels=2, bbox_sampling_ratio=sr7,
                             max_per_img=D // B, contour_max_pts=256)
        heads = synth.SyntheticHeads(K, seed=0).to(dev)
        hdt = torch.float16 if cast else odt
        cls = [c.to(hdt) for c in heads.cls]
        reg = [r.to(hdt) for r in heads.reg]
        pool = heads.pool.to(hdt)
        # the cast arm's heads see fp32 RoI features and round them to fp16 first (force_fp32(out_fp16=True))
        pre = (lambda f: f.half()) if cast else (lambda f: f)
        bbox = [(lambda f, i=i: (pre(f), cls[i], reg[i])[1:]) for i in range(3)]
        stg = RoIStage(cfg, bbox, lambda f, cand: (pre(f), pool[cand % heads.pool_n])[1])

        def step():
            return stg.run([f.float() for f in lv] if cast else lv, rois, max_rois_per_tile=K_per)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            res = step()
        ms, best = timeit(graph.replay, iters)
        emit("roi_stage_step", arm, ms, best, 0, K=K, D=D, detections=int(res.det_valid.sum()))
        outs[(arm, "step")] = res
        del graph, st, st_lv
        torch.cuda.empty_cache()
    for P in (7, 14):
        assert outs[("fp16", P)].dtype == torch.float16 and torch.equal(outs[("fp16", P)], outs[("fp16_cast", P)]), \
            f"{name}: native fp16 {P}x{P} differs from the fp32 kernels + casts"
    a, b = outs[("fp16", "step")], outs[("fp16_cast", "step")]
    same = all(torch.equal(getattr(a, k), getattr(b, k)) for k in ("det_boxes", "det_scores", "det_labels", "det_valid", "mask_bits"))
    assert same, f"{name}: native fp16 step differs from the fp32 stage + casts"
    print(json.dumps(dict(shape=name, check="fp16 native == fp32 kernels + casts", roi_align_7=True, roi_align_14=True, step=True,
                          **info)), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--shape", default="both", choices=["bench", "pannuke", "both"])
    a = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    peak = hbm_peak_gbs()
    print(json.dumps(dict(copy_rate_GBps=round(peak, 1), **info)), flush=True)
    if a.shape in ("bench", "both"):
        run_shape("bench", 16, 256, 1000, 8000, False, a.iters, peak, info)
    if a.shape in ("pannuke", "both"):
        run_shape("pannuke", 16, 64, 1000, 8000, True, a.iters, peak, info)


if __name__ == "__main__":
    main()
