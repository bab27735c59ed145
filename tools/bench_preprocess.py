#!/usr/bin/env python
"""Test-time image pipeline on one GPU: prints ONE JSON line with

* the kernel time of `nuhtc_preprocess_tiles` at B = 16 for 256 -> 512 and 256 -> 1024 (CUDA events around a CUDA graph of
  launches that rotate over enough input/output sets that the working set is > 4x the 126 MB L2, so every launch writes
  to HBM; the per-kernel mean from torch.profiler in a separate pass), its algorithmic bytes B*h*w*3 + B*3*Hp*Wp*4 and
  their share of the HBM bandwidth measured in the same run (a 2 GiB device-to-device copy);
* per batch of 16 tiles: mmdet's host pipeline (the mmcv bodies with cv2, tests/golden/make_golden_preprocess.py) with cv2
  on one thread and on all threads, plus the fp32 host-to-device copy of the collated batch, against TilePipeline from the
  same list of ndarrays (uint8 staging + host-to-device copy + kernel);
* the GPU's name and power limit, read in the same run.

    python tools/bench_preprocess.py [--iters 20]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctypes

import numpy as np
import torch

from nuhtc_b200 import _lib as L
from nuhtc_b200.preprocess import TilePipeline

MEAN = [123.675, 116.28, 103.53]
STD = [58.395, 57.12, 57.375]
L2_BYTES = 126 * 2 ** 20


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [v.strip() for v in q.split(",")[:2]]
    except Exception as e:  # the number is still reported, with the reason the limit is missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def hbm_peak_gbs():
    n = 2 ** 30
    src, dst = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        dst.copy_(src)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(20):
        dst.copy_(src)
    b.record()
    torch.cuda.synchronize()
    return 2 * n * 20 / (a.elapsed_time(b) * 1e-3) / 1e9


def kernel_time(pipe, B, h, w, iters):
    new_h, new_w, pad_h, pad_w, _ = pipe.sizes(h, w)
    in_b, out_b = B * h * w * 3, B * 3 * pad_h * pad_w * 4
    sets = max(2, -(-4 * L2_BYTES // (in_b + out_b)))
    g = torch.Generator(device="cuda").manual_seed(0)
    ins = [torch.randint(0, 256, (B, h, w, 3), dtype=torch.uint8, device="cuda", generator=g) for _ in range(sets)]
    outs = [torch.empty(B, 3, pad_h, pad_w, device="cuda") for _ in range(sets)]
    F3 = ctypes.c_float * 3
    mean, std = F3(*MEAN), F3(*STD)
    lib = L.lib()

    def launch(i, stream):
        L.check(lib.nuhtc_preprocess_tiles(ins[i].data_ptr(), B, h, w, new_h, new_w, pad_h, pad_w, 1, mean, std,
                                           outs[i].data_ptr(), stream), "nuhtc_preprocess_tiles")

    per_graph = sets * max(1, 32 // sets)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(sets):
            launch(i, s.cuda_stream)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        cs = torch.cuda.current_stream().cuda_stream
        for k in range(per_graph):
            launch(k % sets, cs)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        graph.replay()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b) / per_graph)
    prof_us = None
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for k in range(4 * sets):
                launch(k % sets, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        for e in prof.key_averages():
            if "nuhtc_preprocess_tiles_kernel" in e.key:
                tot = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                prof_us = round(tot / e.count, 2)
    except Exception as e:  # the event timing above stands on its own
        prof_us = f"unavailable ({type(e).__name__})"
    del graph, ins, outs
    torch.cuda.empty_cache()
    return dict(B=B, tile=h, new=new_h, pad=pad_h, sets_rotated=sets, working_set_MB=round(sets * (in_b + out_b) / 1e6, 1),
                us_median=round(statistics.median(ms) * 1e3, 2), us_min=round(min(ms) * 1e3, 2), us_profiler_mean=prof_us,
                bytes=in_b + out_b)


def host_pipeline(tiles, s, threads, iters):
    """mmdet's per-tile host work + collate + the fp32 copy to the device, per batch (ms): (host, h2d)."""
    import cv2
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from make_golden_preprocess import imnormalize, resize
    cv2.setNumThreads(threads)
    host, h2d = [], []
    for _ in range(iters):
        t0 = time.perf_counter()
        imgs = []
        for t in tiles:
            r, _ = resize(t, s)
            n = imnormalize(r, MEAN, STD, True)
            ph, pw = -(-n.shape[0] // 32) * 32, -(-n.shape[1] // 32) * 32
            p = np.zeros((ph, pw, 3), np.float32)       # mmcv.impad_to_multiple, pad_val 0
            p[: n.shape[0], : n.shape[1]] = n
            imgs.append(np.ascontiguousarray(p.transpose(2, 0, 1)))   # ImageToTensor
        batch = torch.from_numpy(np.stack(imgs))                      # collate
        t1 = time.perf_counter()
        batch.to("cuda")                                              # scatter: pageable fp32 host-to-device copy
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        host.append((t1 - t0) * 1e3)
        h2d.append((t2 - t1) * 1e3)
    return round(statistics.median(host), 2), round(statistics.median(h2d), 2)


def device_pipeline(pipe, tiles, iters):
    for _ in range(3):
        pipe(tiles)
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        t0 = time.perf_counter()
        pipe(tiles)
        torch.cuda.synchronize()
        ms.append((time.perf_counter() - t0) * 1e3)
    return round(statistics.median(ms), 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_preprocess needs a CUDA device")
    torch.cuda.set_device(0)
    res = dict(bench="preprocess", **gpu_info())
    peak = hbm_peak_gbs()
    res["hbm_copy_GBps_measured"] = round(peak, 1)
    g = np.random.default_rng(0)
    tiles = [g.integers(0, 256, (256, 256, 3), dtype=np.uint8) for _ in range(16)]
    for s in (2.0, 4.0):
        pipe = TilePipeline(s, MEAN, STD, True)
        k = kernel_time(pipe, 16, 256, 256, a.iters)
        k["GBps"] = round(k["bytes"] / (k["us_median"] * 1e-6) / 1e9, 1)
        k["share_of_measured_hbm"] = round(k["GBps"] / peak, 3)
        k["us_at_measured_hbm"] = round(k["bytes"] / (peak * 1e9) * 1e6, 2)
        k["device_pipeline_ms_per_batch16"] = device_pipeline(pipe, tiles, a.iters)
        try:
            k["host_cv2_1thread_ms"], k["host_fp32_h2d_ms"] = host_pipeline(tiles, s, 1, max(3, a.iters // 4))
            k["host_cv2_allthreads_ms"], _ = host_pipeline(tiles, s, os.cpu_count() or 1, max(3, a.iters // 4))
            k["host_cpus"] = os.cpu_count()
        except ImportError as e:
            k["host_pipeline"] = f"not measured ({e})"
        res[f"s{int(s)}_{k['new']}"] = k
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
