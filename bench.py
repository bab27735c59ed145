#!/usr/bin/env python
"""bench.py -- WSI tiles/sec through the RoI stage + merge (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3                      # our arm
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1      # reference CPU path (oracle port)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step = one batch of 16 synthetic 256x256 tiles through the hot path (BASELINE configs[1]): 3 cascade stages of
multi-level RoIAlign 7x7 on 1000 proposals/tile over a 256-channel FPN (strides 4-32), per-class batched NMS on
the decoded boxes, RoIAlign 14x14 on the kept detections, mask paste + threshold to the tile frame, per-tile mask
NMS; after the K steps the nuclei of the K*16 tiles are merged across tile seams once (tools/nuclei_merge.py),
inside the timed region.  The bbox / mask heads are stock-cuDNN work outside the target: seeded stand-ins supply
their outputs.  Inputs are resident in HBM for `value`; `e2e` repeats the measurement with pinned HOST buffers
copied in every step and the results read back.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

def trace(msg):
    if os.environ.get("NUHTC_BENCH_TRACE") == "1":
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


METRIC = "wsi_tiles_per_sec_roi_stage_plus_merge"
UNIT = "tiles/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--tiles", type=int, default=16, help="tiles per batch (per GPU)")
    p.add_argument("--proposals", type=int, default=1000)
    p.add_argument("--channels", type=int, default=256)
    p.add_argument("--max-per-img", type=int, default=500)
    p.add_argument("--dist", default="nuclei", choices=["nuclei", "routed"], help="proposal size distribution")
    p.add_argument("--lane", default="dense", choices=["dense", "bits"], help="paste output: dense uint8 masks or bit rows")
    p.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    p.add_argument("--cpu-tiles", type=int, default=2, help="tiles in the bounded CPU-baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--host-wc", action="store_true", help="e2e leg: FPN levels in write-combined pinned host memory (A/B for the H2D rate at N > 1)")
    p.add_argument("--no-graph", action="store_true", help="run the timed steps eagerly instead of replaying a CUDA graph")
    p.add_argument("--no-slide", action="store_true", help="skip the whole-slide leg (BASELINE configs[3] + configs[4])")
    p.add_argument("--no-extra", action="store_true", help="skip the extra roofline entries (routed proposals, PanNuke shape)")
    p.add_argument("--inflight", type=int, default=3, help="batches in flight: consecutive steps alternate between this many "
                   "streams (each with its own captured graph), so the latency-bound tail of one batch (NMS scans, mask NMS, "
                   "contours) overlaps the RoIAlign of the next; 1 = strictly one step after another")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write the RoI-stage result of the last step and the merge's kept nuclei as "
                        "DIR/<name>.npy (rank 0), to compare two builds output for output")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    return a


def stage_config(args):
    from nuhtc_b200.roi_stage import RoIStageConfig
    return RoIStageConfig(extractor="single", bbox_sampling_ratio=0, mask_sampling_ratio=0, score_thr=0.05, nms_iou=0.5,
                          max_per_img=args.max_per_img, dense_masks=(args.lane == "dense"), contour_max_pts=256,
                          fused_dense_bits=os.environ.get("NUHTC_STAGE_FUSED_PASTE", "1") != "0")


def workload_name(args):
    return (f"RoI-stage microbench: {args.tiles}x256x256 tiles, {args.proposals} proposals/tile ({args.dist}), "
            f"{args.channels}-ch FPN strides 4-32, 3 cascade stages 7x7 + 14x14 mask RoIAlign, batched_nms 5 classes, "
            f"paste+threshold, mask NMS, mask2inst contours, cross-tile merge")


class ClockSampler:
    """SM clock / throttle reasons of this rank's GPU sampled DURING the timed region.  NVML in-process (initialised before
    the timed region, one light query every 10 ms from a thread, rank 0 only); a per-rank `nvidia-smi -lms` subprocess takes about a second
    to start and holds driver locks while it does, which on an 8-GPU box stalled the launches of the very region it was
    meant to observe.  Falls back to nvidia-smi when pynvml is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, enabled: bool = True):
        self.index = index
        self.lines = []
        self.proc = None
        self.nvml = None
        self.stop = threading.Event()
        self.enabled = enabled
        if not enabled:
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        n = self.nvml
        names = (("hw_slowdown", n.nvmlClocksThrottleReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksThrottleReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksThrottleReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksThrottleReasonSwPowerCap))
        while not self.stop.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                flags = ",".join("Active" if rs & bit else "Not Active" for _, bit in names)
                self.lines.append(f"{self.index},{sm},{self.max_sm},0,0,{flags}")
            except Exception:
                pass
            self.stop.wait(0.010)   # an NVML query takes driver locks: polling faster slows the host side of the merge down

    def __enter__(self):
        if not self.enabled:
            return self
        if self.nvml is not None:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *a):
        if self.nvml is not None:
            self.stop.set()
            self.t.join(timeout=1)
            return
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


class EventTimers:
    """CUDA-event timers on the current stream, keyed by op name."""

    def __init__(self):
        self.pairs = {}
        self.enabled = False

    @contextlib.contextmanager
    def __call__(self, name):
        if not self.enabled:
            yield
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        yield
        b.record()
        self.pairs.setdefault(name, []).append((a, b))

    def ms(self):
        return {k: [a.elapsed_time(b) for a, b in v] for k, v in self.pairs.items()}


def trimmed_mean(v):
    """Mean of the samples within 3x the median: an eager step now and then pays a cudaMalloc / lazy-load stall on the host
    that lands inside an event bracket (the GPU idles meanwhile); those are not kernel time."""
    v = np.asarray(v, dtype=np.float64)
    if v.size == 0:
        return None, 0
    keep = v[v <= 3.0 * np.median(v)]
    return float(keep.mean()), int(v.size - keep.size)


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def roi_align_bytes(K, C, P, feats, levels_touched):
    """SURVEY.md 8(d): output written once + every touched level read once + the RoIs."""
    out = K * C * P * P * 4
    inp = sum(feats[l].numel() * 4 for l in levels_touched)
    return out + inp + K * 20


# ----------------------------------------------------------------------------------------------- reference arm
def cpu_sample(args, nthreads, tiles):
    """The reference CPU path (oracle port of the mmcv / pycocotools / shapely kernels driven by the reference's
    per-image flow) on a bounded sample of the same workload: `tiles` tiles through the RoI stage + their share of the merge."""
    from nuhtc_b200 import synth
    from oracle import cpu as O
    from oracle.stage import roi_stage_cpu
    cfg = stage_config(args)
    feats = synth.fpn_levels(tiles, args.channels, frame=512, seed=0)
    rois = synth.proposals(tiles, args.proposals, args.dist, frame=512, seed=0)
    heads = synth.SyntheticHeads(tiles * args.proposals, seed=0)
    side = max(1, int(round(tiles ** 0.5)))
    d = synth.slide_nuclei(side, max(1, tiles // side), per_tile=23, seed=0)
    t0 = time.perf_counter()
    roi_stage_cpu(feats, rois, heads.bbox_heads(), heads.mask_head, cfg, nthreads=nthreads)
    t1 = time.perf_counter()
    O.merge_overlap_arrays(d["xy"], d["voff"], d["score"], 0.05)
    t2 = time.perf_counter()
    return tiles / (t2 - t0), {"roi_stage_s": t1 - t0, "merge_s": t2 - t1}


def workload_config(args, world):
    """`config` of the JSON line: the workload only (identical for both arms), nothing measured."""
    return {"workload": workload_name(args), "tiles_per_step_per_gpu": args.tiles, "proposals_per_tile": args.proposals,
            "channels": args.channels, "max_per_img": args.max_per_img, "detections_per_step": args.tiles * args.max_per_img,
            "mask_lane": args.lane, "heads": "seeded stand-ins (stock cuDNN heads are outside the target)",
            "merge": "once per run, inside the timed region, over the contours the timed steps traced (mask-NMS survivors of "
                     "all steps*tiles tiles laid out as a slide stripe at stride 192)",
            "l2": "inputs larger than L2 (356 MB FPN levels + 0.8 GB RoIAlign output per launch)",
            "parallelism": f"tile stripes over {world} GPU(s), seam nuclei all-gathered for the merge"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    vals = []
    for i in range(args.warmup + args.steps):
        v, parts = cpu_sample(args, cores, args.cpu_tiles)
        if i >= args.warmup:
            vals.append(v)
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 * args.cpu_tiles / value, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, args.gpus),   # the same workload as our arm; each step is a bounded sample of it (below)
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{args.cpu_tiles} tiles/step through oracle.stage.roi_stage_cpu (RoIAlign/paste split over "
                                       f"{cores} host threads; NMS / mask NMS / merge single-threaded like mmcv, pycocotools, shapely)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch.distributed as dist
    import nuhtc_b200 as nb
    from nuhtc_b200 import _lib, synth
    from nuhtc_b200.roi_stage import RoIStage

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a GPU: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()

    cfg = stage_config(args)
    B, C = args.tiles, args.channels
    K = B * args.proposals
    # ---- synthetic inputs, generated on the host (pinned: the e2e leg copies them every step)
    feats_h = [f.pin_memory() for f in synth.fpn_levels(B, C, frame=512, seed=rank)]
    rois_h = synth.proposals(B, args.proposals, args.dist, frame=512, seed=rank).pin_memory()
    heads_h = synth.SyntheticHeads(K, seed=rank)
    heads_h.cls = [t.pin_memory() for t in heads_h.cls]   # pageable sources would make every "async" copy block the host
    heads_h.reg = [t.pin_memory() for t in heads_h.reg]
    feats = [f.to(dev) for f in feats_h]
    rois = rois_h.to(dev)
    heads = synth.SyntheticHeads(K, seed=rank).to(dev)
    stage = RoIStage(cfg, heads.bbox_heads(), heads.mask_head)
    timers = EventTimers()
    stage.timer = timers
    # the nuclei of the steps*B tiles this rank processes form a stripe of the slide, `B` tiles wide and `steps` tile rows
    # tall: the merge at the end of the timed region runs on the contours the steps themselves traced
    from nuhtc_b200.slide import merge_sharded
    D_slots = B * args.max_per_img
    acc = NucleiAccumulator(args.steps, D_slots, cfg.contour_max_pts, B, rank, world, dev)
    merged = {}

    def one_step():
        # every batch brings new FPN features: RoIStage.run stages the kernel layout itself, once per batch (timed as
        # "stage_layout")
        return stage.run(feats, rois, max_rois_per_tile=args.proposals)

    def merge_step():
        with timers("merge"):
            ring_xy, voff, score, shard = acc.rings()
            merged["nuclei"] = int(score.numel())
            return merge_sharded(ring_xy, voff, score, shard, rank, world, 0.05)

    trace("warm-up steps")
    for i in range(max(args.warmup, 3)):
        res = one_step()
        acc.collect(i % args.steps, res)
    torch.cuda.synchronize()
    trace("warm-up merge")
    merge_step()
    torch.cuda.synchronize()
    trace("capture")

    # The step is launch bound on the host (~150 small torch ops + ~20 C-ABI calls): it is captured once into a CUDA
    # graph and replayed.  The captured work is exactly one_step() (NHWC staging, 4 RoIAlign launches, NMS, paste,
    # mask NMS and the torch glue between them) on the resident inputs.
    graph = None
    _lib.LAUNCHES["n"] = 0
    if not args.no_graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            one_step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        _lib.LAUNCHES["n"] = 0
        graphs, graph_res = [], []
        for _ in range(max(1, args.inflight)):
            _lib.LAUNCHES["n"] = 0
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                res = one_step()
            graphs.append(g)
            graph_res.append(res)
        graph = graphs[0]
        launches_per_step = _lib.LAUNCHES["n"]
        for g in graphs:
            for _ in range(2):
                g.replay()
        torch.cuda.synchronize()
        # warm-up of the merge at its timed size: all `steps` slabs filled, so the allocator and NCCL see the shapes of the
        # timed region (a merge warmed up on 3 steps' nuclei paid cudaMalloc stalls of tens of ms inside the timed merge)
        for i in range(args.steps):
            graphs[i % len(graphs)].replay()
            acc.collect(i, graph_res[i % len(graphs)])
        merge_step()
        torch.cuda.synchronize()
    lanes = [torch.cuda.Stream() for _ in range(max(1, args.inflight))] if (graph is not None and args.inflight > 1) else []

    trace("timed region")
    # ---- timed region: exactly K steps + the one merge
    sampler = ClockSampler(local, enabled=(rank == 0))   # NVML is initialised here, outside the timed region
    _lib.LAUNCHES["n"] = 0
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with sampler as clocks:
        e0.record()
        main = torch.cuda.current_stream()
        for ln in lanes:
            ln.wait_stream(main)
        for i in range(args.steps):
            if lanes:                                   # step i on lane i % inflight; a lane replays its own graph in order
                with torch.cuda.stream(lanes[i % len(lanes)]):
                    graphs[i % len(lanes)].replay()
                    acc.collect(i, graph_res[i % len(lanes)])
            elif graph is not None:
                graph.replay()
                acc.collect(i, graph_res[0])
            else:
                res = one_step()
                acc.collect(i, res)
        for ln in lanes:
            main.wait_stream(ln)
        e_steps = torch.cuda.Event(enable_timing=True)
        e_steps.record()
        kept = merge_step()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
    ms = e0.elapsed_time(e1)
    trace(f"timed region done: {ms:.1f} ms, merged {merged.get('nuclei')} nuclei")
    steps_ms = e0.elapsed_time(e_steps)   # this rank's K steps without the merge (the merge waits for the slowest rank)
    per_rank_steps = [steps_ms]
    if world > 1:
        tl = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(tl, torch.tensor([steps_ms], device=dev, dtype=torch.float64))
        per_rank_steps = [float(t.item()) for t in tl]
    launches = _lib.LAUNCHES["n"] + (launches_per_step * args.steps if graph is not None else 0)
    if args.dump_outputs and rank == 0:
        last = res if graph is None else graph_res[(args.steps - 1) % len(graphs)]
        dump_outputs(args.dump_outputs, last, kept)

    # ---- per-kernel durations (CUDA events cannot bracket nodes inside a graph): the same K steps are repeated eagerly
    # with an event pair around every op; these feed `roofline`, `roofline_other` and `breakdown_ms_per_step` only
    for _ in range(3):      # eager warm-up: the caching allocator re-creates the blocks the graph's private pool took over
        res = one_step()    # (the previous result stays alive while the next step allocates, exactly like the loop below)
    torch.cuda.synchronize()
    timers.enabled = True
    timers.pairs = {}
    torch.cuda.synchronize()
    i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    i0.record()
    for i in range(args.steps):
        res = one_step()
        acc.collect(i, res)
    merge_step()
    i1.record()
    torch.cuda.synchronize()
    timers.enabled = False
    eager_ms = i0.elapsed_time(i1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches = int(lt.item())
    total_tiles = args.steps * B * world
    value = total_tiles / (ms / 1000.0)
    op_ms = timers.ms()

    # ---- roofline of the dominant kernel: the 7x7 RoIAlign launch (stages 2 and 3 of every step: NHWC staging is
    # timed separately, so these brackets contain the RoIAlign kernel alone)
    peak, peak_src = measured_peak_gbs()
    lv = sorted(set(nb_levels(rois_h)))
    ra = op_ms.get("roi_align_bbox", [])
    ra_ms, ra_dropped = trimmed_mean(ra)
    alg = roi_align_bytes(K, C, 7, feats_h, lv)
    roofline = None
    if ra_ms:
        ach = alg / (ra_ms * 1e-3) / 1e9
        roofline = {"kernel": "roi_align_strip7_kernel + its 3 prepass launches (7x7 bbox RoIAlign, K=%d, C=%d)" % (K, C), "bound": "hbm",
                    "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    # NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch of the strip kernel
                    # on this workload, from the `ncu --set full` capture summarised in profiles/r02_roialign_strip.md
                    # (291.2 MB + 748.5 MB); null for any other shape
                    "traffic": 1046130432 if (K == 16000 and C == 256 and args.dist == "nuclei") else None,
                    "traffic_source": "profiles/r02_roialign_strip.md (ncu capture of the same launch shape, not this run)",
                    "algorithmic_bytes_per_launch": alg, "avg_launch_ms": ra_ms, "launches_timed": len(ra) - ra_dropped,
                    "host_stall_samples_dropped": ra_dropped, "peak_source": peak_src}
    paste = op_ms.get("paste", [])
    D = int(res.det_boxes.shape[0])
    extra = {}
    if paste:
        # dense frame (+ the bit rows when both come from the one-evaluation kernel) + the 28x28 map + the box
        pbytes = D * (256 * 256 * (1 if args.lane == "dense" else 0.125) + (256 * 256 // 8 if cfg.fused_dense_bits else 0) + 28 * 28 * 4 + 16)
        pms, _ = trimmed_mean(paste)
        extra["paste"] = {"achieved": pbytes / (pms * 1e-3) / 1e9, "unit": "GB/s", "frac": pbytes / (pms * 1e-3) / 1e9 / peak,
                          "algorithmic_bytes_per_launch": pbytes, "avg_launch_ms": pms, "masks_per_launch": D}
    rm = op_ms.get("roi_align_mask", [])
    if rm:
        mbytes = roi_align_bytes(D, C, 14, feats_h, lv)
        mms, _ = trimmed_mean(rm)
        extra["roi_align_mask"] = {"achieved": mbytes / (mms * 1e-3) / 1e9, "unit": "GB/s", "frac": mbytes / (mms * 1e-3) / 1e9 / peak,
                                   "algorithmic_bytes_per_launch": mbytes, "avg_launch_ms": mms}
    tr = op_ms.get("stage_layout", [])
    if tr:
        tbytes = 2 * sum(f.numel() * 4 for f in feats_h)
        tms, _ = trimmed_mean(tr)
        extra["stage_layout"] = {"achieved": tbytes / (tms * 1e-3) / 1e9, "unit": "GB/s", "frac": tbytes / (tms * 1e-3) / 1e9 / peak,
                                 "avg_launch_ms": tms}
    # per step: (trimmed) mean bracket x brackets per step
    breakdown = {k: trimmed_mean(v)[0] * len(v) / args.steps for k, v in op_ms.items() if len(v)}

    # ---- extra roofline entries (N = 1 only): the routed proposal distribution and the shipping PanNuke shape
    if rank == 0 and world == 1 and not args.no_extra:
        trace("extra rooflines")
        extra.update(extra_rooflines(args, feats, feats_h, dev, peak))
    # ---- whole-slide leg: BASELINE configs[3] (43 264 tiles of a 40k x 40k slide, batches of 16 per GPU) + configs[4]
    # (cross-tile merge of the ~1.7 M nuclei of that slide), once per rank
    slide_leg = None
    if not args.no_slide and graph is not None:
        trace("slide leg")
        slide_leg = run_slide(args, graphs, lanes, dev, rank, world)
    trace("e2e")

    # ---- e2e: pinned host inputs copied every step, results read back every step
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, stage, feats_h, rois_h, heads_h, heads, feats, rois, dev, world, rank)

    # ---- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, parts = cpu_sample(args, 1, args.cpu_tiles)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{args.cpu_tiles} tiles through oracle.stage.roi_stage_cpu + their merge share, single thread "
                         f"(roi_stage {parts['roi_stage_s']:.2f}s, merge {parts['merge_s']:.3f}s)"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": workload_config(args, world),
                "run": {"nuclei_merged_per_gpu": merged.get("nuclei"), "nuclei_kept": int(kept.numel()) if kept is not None else None},
                "roofline": roofline, "roofline_other": extra, "slide": slide_leg, "breakdown_ms_per_step": breakdown,
                "per_rank_steps_ms": [round(v, 3) for v in per_rank_steps],
                "timing": {"timed_region": ("cuda graph replay of the captured step" + (f", {len(lanes)} batches in flight on {len(lanes)} streams"
                                                                                          if lanes else "")) if graph is not None else "eager",
                           "eager_instrumented_ms_per_step": eager_ms / args.steps,
                           "per_kernel_numbers": "CUDA events around every op in an eager repeat of the same steps, right after the timed region; "
                                                 "brackets above 3x their median (host stalls of the eager loop) are left out of the means"},
                "cpu_baseline": cpu,
                "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, res, kept, big_cap=24 << 20):
    """What the timed path hands its caller, as out_dir/<name>.npy: the RoI-stage result of one step with the padding slots
    dropped (RoIStageResult.compact()) and the merge's kept nuclei.  Integers become float32 (float64 when they are int64);
    contour points past a detection's count are zeroed (unwritten).  The two per-detection arrays that can be large, dense
    masks and contours, are limited to `big_cap` bytes each by a seeded row sample (the same rows for every build when the
    detection count agrees); `*_rows` names the rows kept."""
    os.makedirs(out_dir, exist_ok=True)
    r = res.compact()
    n = int(r.det_boxes.shape[0])
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))

    def rows(row_bytes):
        return perm[: min(n, big_cap // row_bytes)].sort().values

    H, words = r.mask_bits.shape[1:]
    mrows = rows(H * words * 64 * 4)
    if r.masks is not None:
        masks = r.masks[mrows.to(r.masks.device)]
    else:                                                   # bit rows only: bit x % 64 of word x // 64 is pixel x
        bits = r.mask_bits[mrows.to(r.mask_bits.device)]
        masks = ((bits.unsqueeze(-1) >> torch.arange(64, device=bits.device)) & 1).flatten(-2).to(torch.uint8)
    out = {"det_boxes": r.det_boxes, "det_scores": r.det_scores, "det_labels": r.det_labels, "det_tile": r.det_tile,
           "det_cand": r.det_cand, "mask_area": r.mask_area, "keep": r.keep, "tile_start": r.tile_start,
           "tile_count": r.tile_count, "masks_sample": masks, "masks_sample_rows": mrows, "merge_kept": kept}
    if r.contour_xy is not None:
        xy, cnt = r.contour_xy, r.contour_count
        xy = xy * (torch.arange(xy.shape[1], device=xy.device)[None, :] < cnt[:, None]).unsqueeze(-1).to(xy.dtype)
        crows = rows(xy.shape[1] * 2 * 4)
        out.update(contour_count=cnt, contour_xy_sample=xy[crows.to(xy.device)], contour_xy_sample_rows=crows)
    for name, t in out.items():
        if t is None:
            continue
        a = t.detach().cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64 if a.dtype == np.int64 else np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), a)


class NucleiAccumulator:
    """The nuclei the timed steps produce, kept on the device for the cross-tile merge: after every step the traced
    contours of the mask-NMS survivors (RoIStageResult.contour_xy / contour_count), their scores and tile indices are
    copied into the slab of that step.  Step s of rank r is tile row r*steps + s of the slide, `tiles` tiles wide at
    stride 192 (infer_wsi.py: --patch_size 256 --step_size 192), so nuclei of neighbouring tiles meet in the 64 px overlap."""

    def __init__(self, steps, D, max_pts, tiles, rank, world, dev, stride=192, tile=256):
        self.steps, self.D, self.tiles, self.rank, self.world, self.stride, self.tile = steps, D, tiles, rank, world, stride, tile
        self.xy = torch.zeros((steps, D, max_pts, 2), dtype=torch.int32, device=dev)
        self.cnt = torch.zeros((steps, D), dtype=torch.int32, device=dev)
        self.score = torch.zeros((steps, D), dtype=torch.float32, device=dev)
        self.tile_idx = torch.full((steps, D), -1, dtype=torch.int32, device=dev)
        self.row = (rank * steps + torch.arange(steps, device=dev, dtype=torch.int32))[:, None].expand(steps, D)

    def collect(self, step, res):
        self.xy[step].copy_(res.contour_xy, non_blocking=True)
        self.cnt[step].copy_(res.contour_count, non_blocking=True)
        self.score[step].copy_(res.det_scores, non_blocking=True)
        self.tile_idx[step].copy_(res.det_tile, non_blocking=True)

    def rings(self):
        """-> (ring_xy fp64 [sumV,2], voff [n+1], score fp64 [n], shard meta for the multi-GPU merge)."""
        import nuhtc_b200 as nb
        n_all = self.steps * self.D
        t = self.tile_idx.reshape(-1)
        origin = torch.stack([t.clamp(min=0) * self.stride, self.row.reshape(-1) * self.stride], dim=1).to(torch.int32).contiguous()
        sel = (t >= 0) & (self.cnt.reshape(-1) > 0)
        ring_xy, voff, index = nb.rings_for_merge(self.xy.reshape(n_all, -1, 2), self.cnt.reshape(-1), select=sel, origin=origin)
        # scores of different steps repeat (the stand-in heads are seeded tensors): a 1e-12-scale term keyed on the global
        # nucleus index makes them distinct, as the merge contract asks (ties are the only thing it leaves open)
        gid = index + self.rank * n_all
        score = self.score.reshape(-1)[index].to(torch.float64) + gid.to(torch.float64) * 1e-12
        tile_id = (self.row.reshape(-1)[index].to(torch.int64) * self.tiles + t[index].to(torch.int64))
        shard = dict(gid=gid, tile_id=tile_id, tiles_x=self.tiles, tiles_y=self.steps * self.world, stride=self.stride, tile=self.tile,
                     rows=(self.rank * self.steps, (self.rank + 1) * self.steps))
        return ring_xy, voff, score, shard


def _time_ms(fn, iters=10, warm=3):
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
    return float(np.median([x.elapsed_time(y) for x, y in evs]))


def extra_rooflines(args, feats, feats_h, dev, peak):
    """Roofline entries beside the headline one, timed alone with CUDA events (median of 10 launches after 3 warm-ups):
    the 'routed' proposal distribution (all four FPN levels, windows up to the whole map) and the shipping PanNuke shape
    (configs/nuhtc/htc_lite_swin_pytorch_fpn_PanNuke_seasaw_CAS.py: AttentionRoIExtractor, 64 channels, 7x7, sampling_ratio 2:
    RoIAlign of levels 0,1 summed + cosine-attention pooling of levels 2,3 added at the store)."""
    import nuhtc_b200 as nb
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_extractors import AttentionRoIExtractor
    out = {}
    B, C = args.tiles, args.channels
    scales = [1 / s for s in synth.FPN_STRIDES]
    staged = nb.stage_levels(feats)
    rois = synth.proposals(B, args.proposals, "routed", frame=512, seed=1).to(dev)
    K = rois.shape[0]
    o = torch.empty(K, C, 7, 7, device=dev)
    ms = _time_ms(lambda: nb.roi_align_levels(staged, rois, 7, scales, 0, mode="route", out=o))
    nbytes = roi_align_bytes(K, C, 7, feats_h, sorted(set(nb_levels(rois.cpu()))))
    out["roi_align_bbox_routed"] = {"achieved": nbytes / ms / 1e6, "unit": "GB/s", "frac": nbytes / ms / 1e6 / peak,
                                    "algorithmic_bytes_per_launch": nbytes, "avg_launch_ms": ms,
                                    "note": "side log-U(16,512) px: every FPN level, windows up to the whole map (large windows take the per-RoI kernel)"}
    del o, staged
    f64 = [f.to(dev) for f in synth.fpn_levels(B, 64, frame=512, seed=2)]
    rois_n = synth.proposals(B, args.proposals, "nuclei", frame=512, seed=2).to(dev)
    ext = AttentionRoIExtractor(roi_layer=dict(type="RoIAlign", output_size=7, sampling_ratio=2), out_channels=64,
                                featmap_strides=list(synth.FPN_STRIDES), start_level=2, thres=0)
    ms = _time_ms(lambda: ext(f64, rois_n))
    nbytes = rois_n.shape[0] * 64 * 49 * 4 + sum(f.numel() * 4 for f in f64) + rois_n.shape[0] * 20
    out["pannuke_attention_extractor"] = {"achieved": nbytes / ms / 1e6, "unit": "GB/s", "frac": nbytes / ms / 1e6 / peak,
                                          "algorithmic_bytes_per_launch": nbytes, "avg_launch_ms": ms,
                                          "note": "whole AttentionRoIExtractor.forward (layout staging + 2 attention-pool launches + "
                                                  "level-sum RoIAlign with the pooled bias), C=64, 7x7, sampling_ratio=2, K=%d" % rois_n.shape[0]}
    return out


def run_slide(args, graphs, lanes, dev, rank, world):
    """BASELINE configs[3]: a 40k x 40k slide = 208 x 208 tiles of 256 px at stride 192 (43 264 tiles, 2 704 batches of 16),
    sharded by tile rows; every rank replays its share of batches through the captured RoI-stage step (stage layout, 3 + 1
    RoIAlign, NMS, paste, mask NMS, contours).  configs[4]: the cross-tile merge of the slide's ~1.7 M synthetic nuclei
    (duplicates in the 64 px overlap bands), each rank holding its stripe, seam nuclei exchanged over NCCL."""
    import torch.distributed as dist
    import nuhtc_b200 as nb
    from nuhtc_b200 import synth
    from nuhtc_b200.slide import merge_sharded, stripe_rows
    tiles_side = 208
    r0, r1 = stripe_rows(tiles_side, rank, world)
    my_tiles = (r1 - r0) * tiles_side
    batches = (my_tiles + args.tiles - 1) // args.tiles
    slide = synth.slide_nuclei(tiles_side, tiles_side, per_tile=23, seed=208)
    shard = nb.slide.shard_by_rows(slide, rank, world)
    xy, voff, score = (torch.from_numpy(shard[k]).to(dev) for k in ("xy", "voff", "score"))
    total_nuclei = int(len(slide["score"]))
    del slide
    merge_sharded(xy, voff, score, shard, rank, world, 0.05)   # warm-up (allocator, NCCL channels)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    main = torch.cuda.current_stream()
    e0.record()
    for ln in lanes:
        ln.wait_stream(main)
    for i in range(batches):
        if lanes:
            with torch.cuda.stream(lanes[i % len(lanes)]):
                graphs[i % len(lanes)].replay()
        else:
            graphs[0].replay()
    for ln in lanes:
        main.wait_stream(ln)
    e1.record()
    kept = merge_sharded(xy, voff, score, shard, rank, world, 0.05)
    e2.record()
    torch.cuda.synchronize()
    t_stage, t_merge = e0.elapsed_time(e1), e1.elapsed_time(e2)
    nk = torch.tensor([int(kept.numel())], device=dev, dtype=torch.int64)
    if world > 1:
        t = torch.tensor([t_stage, t_merge], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_stage, t_merge = float(t[0]), float(t[1])
        dist.all_reduce(nk)
    tiles = tiles_side * tiles_side
    return {"workload": "configs[3] 208x208 tiles (43264) through the RoI stage, batches of %d per GPU, + configs[4] merge of %d nuclei" % (args.tiles, total_nuclei),
            "tiles": tiles, "batches_per_gpu": batches, "roi_stage_ms": t_stage, "merge_ms": t_merge,
            "tiles_per_s": tiles / ((t_stage + t_merge) / 1e3), "merge_nuclei_per_s": total_nuclei / (t_merge / 1e3),
            "nuclei": total_nuclei, "nuclei_kept": int(nk.item()),
            "note": "every batch replays the same resident synthetic batch (inputs in HBM); max over ranks"}


def nb_levels(rois_h, finest=56.0, L=4):
    """which FPN levels the synthetic RoIs touch (bytes accounting only; same rule as map_roi_levels)"""
    scale = torch.sqrt((rois_h[:, 3] - rois_h[:, 1]) * (rois_h[:, 4] - rois_h[:, 2]))
    return torch.floor(torch.log2(scale / finest + 1e-6)).clamp(0, L - 1).long().tolist()


def wc_pinned_like(t):
    """Copy of a host tensor in write-combined pinned memory (cudaHostAlloc): the device reads it without snooping the CPU caches."""
    import ctypes
    from cuda.bindings import runtime as rt
    nbytes = t.numel() * t.element_size()
    err, ptr = rt.cudaHostAlloc(nbytes, rt.cudaHostAllocWriteCombined | rt.cudaHostAllocPortable)
    if int(err) != 0:
        raise RuntimeError(f"cudaHostAlloc failed: {err}")
    buf = (ctypes.c_byte * nbytes).from_address(int(ptr))
    out = torch.frombuffer(buf, dtype=t.dtype).view(t.shape)
    out.copy_(t)
    return out


def run_e2e(args, stage, feats_h, rois_h, heads_h, heads, feats, rois, dev, world, rank):
    """Same step through the public API with HOST buffers.  Every step copies the FPN levels, the proposals and the head
    outputs from pinned host memory (H2D) and reads the per-tile results back into pinned host memory (D2H: detection
    slots, kept lists and the bit-row masks).  Two device buffer sets alternate so that the H2D of step i+1 and the D2H of
    step i-1 overlap the kernels of step i (copy engines on their own streams); the timed region still contains every
    copy of every step."""
    import torch.distributed as dist
    import nuhtc_b200 as nb
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_stage import RoIStage
    from nuhtc_b200.slide import merge_sharded
    steps = args.e2e_steps or min(args.steps, 10)
    K = rois_h.shape[0]
    if args.host_wc:
        feats_h = [wc_pinned_like(f) for f in feats_h]
    main = torch.cuda.current_stream()
    h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
    sets = []
    for i in range(2):
        f = [torch.empty_like(x, device=dev) for x in feats_h]
        r = torch.empty_like(rois_h, device=dev)
        hd = synth.SyntheticHeads(K, seed=0).to(dev)
        st = RoIStage(stage.cfg, hd.bbox_heads(), hd.mask_head)
        sets.append(dict(feats=f, rois=r, heads=hd, stage=st, graph=None, res=None, ev_in=torch.cuda.Event(), ev_done=torch.cuda.Event(),
                         ev_out=torch.cuda.Event(), host=None))
    h2d = sum(f.numel() * 4 for f in feats_h) + rois_h.numel() * 4 + sum(t.numel() * 4 for t in heads_h.cls + heads_h.reg)

    def upload(S):
        for dst, src in zip(S["feats"], feats_h):
            dst.copy_(src, non_blocking=True)
        S["rois"].copy_(rois_h, non_blocking=True)
        for dst, src in zip(S["heads"].cls + S["heads"].reg, heads_h.cls + heads_h.reg):
            dst.copy_(src, non_blocking=True)

    def compute(S):
        return S["stage"].run(S["feats"], S["rois"], max_rois_per_tile=args.proposals)

    def outputs(r):
        # what the tile loop hands on (infer_wsi.py:528-566): detections, kept lists and the traced contours; the masks
        # themselves stay on the device
        return [r.det_boxes, r.det_scores, r.det_labels, r.det_tile, r.contour_xy, r.contour_count, r.keep, r.tile_start,
                r.tile_count]

    for S in sets:  # warm up (and capture) each buffer set
        upload(S)
        torch.cuda.synchronize()
        for _ in range(2):
            S["res"] = compute(S)
        torch.cuda.synchronize()
        if not args.no_graph:
            side = torch.cuda.Stream()
            side.wait_stream(main)
            with torch.cuda.stream(side):
                compute(S)
            main.wait_stream(side)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                S["res"] = compute(S)
            S["graph"] = g
        S["host"] = [torch.empty(o.shape, dtype=o.dtype, pin_memory=True) for o in outputs(S["res"])]
    d2h = sum(o.numel() * o.element_size() for o in sets[0]["host"])
    acc = NucleiAccumulator(steps, sets[0]["res"].det_boxes.shape[0], stage.cfg.contour_max_pts, args.tiles, rank, world, dev)
    # warm-up of the merge at the size of this leg's timed region (allocator blocks, NCCL buffers of these shapes)
    for i in range(steps):
        S = sets[i % 2]
        if S["graph"] is not None:
            S["graph"].replay()
        else:
            S["res"] = compute(S)
        acc.collect(i, S["res"])
    merge_sharded(*acc.rings(), rank, world, 0.05)
    torch.cuda.synchronize()
    # what the link gives for exactly these buffers (pure copies, nothing else running): the floor of an e2e step
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(3):
        upload(sets[0])
    p1.record()
    torch.cuda.synchronize()
    h2d_ms = p0.elapsed_time(p1) / 3
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    with torch.cuda.stream(h2d_stream):
        h2d_stream.wait_stream(main)
        upload(sets[0])
        sets[0]["ev_in"].record(h2d_stream)
    for i in range(steps):
        cur, nxt = sets[i % 2], sets[(i + 1) % 2]
        if i + 1 < steps:
            with torch.cuda.stream(h2d_stream):
                if i >= 1:
                    h2d_stream.wait_event(nxt["ev_done"])   # the kernels of step i-1 are done with this buffer set
                upload(nxt)
                nxt["ev_in"].record(h2d_stream)
        main.wait_event(cur["ev_in"])
        if i >= 2:
            main.wait_event(cur["ev_out"])                  # its previous results have left for the host
        if cur["graph"] is not None:
            cur["graph"].replay()
        else:
            cur["res"] = compute(cur)
        acc.collect(i, cur["res"])
        cur["ev_done"].record(main)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(cur["ev_done"])
            for dst, src in zip(cur["host"], outputs(cur["res"])):
                dst.copy_(src, non_blocking=True)
            cur["ev_out"].record(d2h_stream)
    main.wait_stream(d2h_stream)
    ring_xy, voff, score, shard = acc.rings()
    kept = merge_sharded(ring_xy, voff, score, shard, rank, world, 0.05)
    kept.cpu()
    e1.record()
    torch.cuda.synchronize()
    for S in sets:
        S["res"].check()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {"value": steps * args.tiles * world / (ms / 1000.0), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "steps": steps, "ms_per_step": ms / steps,
            "h2d_only_ms_per_step": h2d_ms, "h2d_gbs": h2d / h2d_ms / 1e6,
            "host_memory": "write-combined pinned" if args.host_wc else "pinned", "overlap": "H2D of step i+1 and D2H of step i-1 overlap the kernels of step i (two buffer sets, copy streams)"}


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
