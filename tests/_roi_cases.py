"""Seeded RoIAlign inputs shared by tests/test_gpu_roi_reference.py and the child processes it starts for the library's
A/B environment switches (NUHTC_RA_*, read once per process).  Run as a script, this module is such a child:

    python tests/_roi_cases.py --out DIR --cells JSON

runs the cells with whatever NUHTC_RA_* the environment holds, saves each output as DIR/<cell key>.pt and prints one
JSON line {"cells": [...], "kernels": [...]} with the CUDA kernels it launched."""
from __future__ import annotations

import json
import os
import re
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# a 400 x 208 px frame on four FPN levels: non-square, level 0 is 100 cells wide (four strips, the last one partial),
# level 2 has an odd cell count (13 x 25: staged by the line-permutation kernel)
STRIDES = (4, 8, 16, 32)
LEVEL_HW = ((52, 100), (26, 50), (13, 25), (7, 13))
FRAME_W, FRAME_H = 400.0, 208.0
MODES = ("route4", "route1", "sum2b", "sum2p", "sum1p")


def half_exact(x: torch.Tensor) -> torch.Tensor:
    """fp32 values that fp16 and bf16 both hold exactly: the same levels then serve all three dtypes"""
    x = x.bfloat16().float()
    return torch.where(x.abs() < 2.0 ** -14, torch.zeros_like(x), x)


def levels(C: int, B: int = 2, seed: int = 0):
    g = torch.Generator().manual_seed(1000 * C + seed)
    return [half_exact(torch.randn(B, C, h, w, generator=g)) for h, w in LEVEL_HW]


def population(K: int = 80, B: int = 2, seed: int = 0, edges: bool = True) -> torch.Tensor:
    """nucleus-sized and larger RoIs plus RoIs that force every leftover: windows wider than 18 cells and taller than 18
    rows on the multi-strip level, bins of more than 8 taps at 7x7 and at 14x14"""
    g = torch.Generator().manual_seed(77 + seed)
    ctr = torch.rand(K, 2, generator=g) * torch.tensor([FRAME_W * 1.1, FRAME_H * 1.1]) - torch.tensor([FRAME_W, FRAME_H]) * 0.05
    side = torch.where(torch.rand(K, 1, generator=g) < 0.75, 6 + torch.rand(K, 1, generator=g) * 64,
                       60 + torch.rand(K, 1, generator=g) * 440)
    wh = side * (0.5 + torch.rand(K, 2, generator=g))
    r = torch.cat([torch.randint(0, B, (K, 1), generator=g).float(), ctr - wh / 2, ctr + wh / 2], 1)
    forced = [[13.3, 20.7, 113.3, 44.7],       # 25 cells wide on level 0 (routed there: sqrt(w h) < 112)
              [127.1, 101.9, 229.1, 125.9],    # wide, origin inside strip 1
              [300.6, 30.2, 324.6, 130.2],     # 25 rows tall
              [50.4, 60.9, 310.4, 100.9],      # 7x7 bins of ~9 cells: more than 8 taps
              [-40.2, 90.1, 439.8, 110.1],     # 14x14 bins of ~8.6 cells
              [10.5, 170.25, 30.5, 250.25]]    # hangs off the bottom
    if edges:
        forced += [[10.0, 10.0, 10.0, 10.0],                                  # zero size
                   [-60.0, -60.0, FRAME_W + 60.0, FRAME_H + 60.0],           # larger than the frame
                   [-500.0, -500.0, -400.0, -400.0]]                          # wholly outside
    n = len(forced)
    r[:n, 1:] = torch.tensor(forced)
    return r


def cell_key(c: dict) -> str:
    return f"{c['mode']}-C{c['C']}-P{c['P']}-{c['dtype']}-{c['impl']}"


def cell_args(c: dict):
    """(levels, rois, scales, mode, bias, pool2) of a cell, fp32 CPU tensors"""
    C, mode = c["C"], c["mode"]
    lv = levels(C)
    rois = population(edges=mode not in ("sum2p", "sum1p"))
    sc = [1.0 / s for s in STRIDES]
    bias = torch.randn(rois.shape[0], C, generator=torch.Generator().manual_seed(5 + C))
    if mode == "route4":
        return lv, rois, sc, "route", None, None
    if mode == "route1":
        return lv[:1], rois, sc[:1], "route", None, None
    if mode == "sum2b":
        return lv[:2], rois, sc[:2], "sum", bias, None
    sem = half_exact(torch.randn(2, C, *LEVEL_HW[1], generator=torch.Generator().manual_seed(9 + C)))
    if mode == "sum2p":   # FPN levels 0, 1 + the semantic map pooled at twice the size (NuHTC's bbox branch)
        return lv[:2] + [sem], rois, sc[:2] + [1.0 / 8], "sum", bias, [False, False, True]
    return [sem], rois, [1.0 / 8], "sum", bias, [True]      # sum1p: a lone pool2 level


DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


def run_cell(c: dict) -> torch.Tensor:
    import nuhtc_b200 as nb
    lv, rois, sc, mode, bias, pool2 = cell_args(c)
    dt = DTYPES[c["dtype"]]
    feats = [f.cuda().to(dt) for f in lv]
    return nb.roi_align_levels(feats, rois.cuda(), c["P"], sc, c.get("sr", 0), True, mode, 56.0, impl=c["impl"],
                               bias=None if bias is None else bias.cuda(), pool2=pool2)


def kernel_key(name: str) -> str:
    """a kernel's name with template arguments, without namespaces, return type, parameters or spaces, whether it comes
    from the profiler or from cu++filt: 'roi_align_sep_kernel<7,32,1,2,2,float>'"""
    n = name.replace("(anonymous namespace)::", "").replace("<unnamed>::", "").replace("(int)", "")
    n = re.sub(r"^void\s+", "", n.strip())
    n = n.split("(", 1)[0]
    return re.sub(r"\s+", "", n)


def launched(fn):
    """(fn's result, set of kernel keys it launched), recorded with torch.profiler's CUDA activity"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {kernel_key(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    return res, names


def _child(argv):
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cells", required=True)
    a = ap.parse_args(argv)
    cells = json.loads(a.cells)

    def go():
        done = []
        for c in cells:
            torch.save(run_cell(c).cpu(), os.path.join(a.out, cell_key(c) + ".pt"))
            done.append(cell_key(c))
        return done
    done, names = launched(go)
    print(json.dumps({"cells": done, "kernels": sorted(names)}), flush=True)


if __name__ == "__main__":
    _child(sys.argv[1:])
