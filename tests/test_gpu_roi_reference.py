"""GPU: every RoIAlign and attention-pooling kernel the library can route to, held to the float64 references of
tests/_roi_ref64.py within their first-order fp32 bounds.

  * the dispatch matrix: C x P x mode x dtype (+ the NHWC kernels), each cell with RoIs that force every leftover;
  * geometry: aligned=False, sampling ratios, odd / thin / tall maps, samples exactly on -1, 0, D-1 and D, window origins
    at strip-core edges, windows of exactly 18 / 19 cells, bins of exactly 8 / 9 taps, per-channel scales from 1e-3 to
    1e3, both sides of the strip binning's size limit, all RoIs in one image, K = 1 and K = 70 000;
  * the NUHTC_RA_* A/B switches, each in a child process (the library reads them once per process);
  * attention pooling over C, map shapes, batch layouts, clamp edges, thresholds and degenerate vectors;
  * coverage: every roi_align / strip / CG32-staging / attention kernel in the library was launched by a passing case.
"""
import concurrent.futures as cf
import json
import os
import re
import shutil
import subprocess
import sys

import pytest
import torch

import _roi_cases as RC
import _roi_ref64 as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

LAUNCHED: set = set()     # kernel keys launched by cases that passed
_REFS: dict = {}


def _run(fn):
    """(fn(), the kernels it launched): they count as covered only once the caller's checks have passed"""
    return RC.launched(fn)


def _ref(c: dict):
    key = (c["C"], c["P"], c["mode"], c.get("sr", 0))
    if key not in _REFS:
        lv, rois, sc, mode, bias, pool2 = RC.cell_args(c)
        _REFS[key] = R.roi_align_ref64(lv, rois, c["P"], sc, c.get("sr", 0), True, mode, 56.0, bias, pool2)
    return _REFS[key]


def _tol(c: dict, tol, ref):
    dt = RC.DTYPES[c["dtype"]]
    return tol + R.half_ulp(ref.abs() + tol, dt) if dt != torch.float32 else tol


# ----------------------------------------------------------------------------- 1. the dispatch matrix
@pytest.mark.parametrize("mode", RC.MODES)
@pytest.mark.parametrize("P", [7, 14])
@pytest.mark.parametrize("C", [32, 64, 96, 128, 192, 256, 384, 512])
def test_dispatch_matrix_vs_reference(C, P, mode):
    cells = [dict(C=C, P=P, mode=mode, dtype=d, impl="auto") for d in ("f32", "f16", "bf16")]
    if C % 64 == 0 and mode not in ("sum2p", "sum1p"):
        cells.append(dict(C=C, P=P, mode=mode, dtype="f32", impl="nhwc"))
    outs, names = _run(lambda: [RC.run_cell(c) for c in cells])
    ref, tol = _ref(cells[0])
    for c, o in zip(cells, outs):
        assert o.dtype == RC.DTYPES[c["dtype"]]
        R.check(o, ref, _tol(c, tol, ref), RC.cell_key(c))
    for c, o in zip(cells[1:3], outs[1:3]):   # half levels: the fp32 result on the (exact) upcast levels, rounded once
        assert torch.equal(o, outs[0].to(o.dtype)), RC.cell_key(c)
    LAUNCHED.update(names)


# ----------------------------------------------------------------------------- 2. geometry
GEOM_CELLS = [(7, 64), (7, 256), (14, 64), (14, 256)]


def _check_levels(levels_cpu, rois, P, scales, sr=0, aligned=True, mode="route", what="", impls=("auto", "direct")):
    import nuhtc_b200 as nb
    ref, tol = R.roi_align_ref64(levels_cpu, rois, P, scales, sr, aligned, mode)
    feats = [f.cuda() for f in levels_cpu]
    outs, names = _run(lambda: [nb.roi_align_levels(feats, rois.cuda(), P, scales, sr, aligned, mode, impl=i) for i in impls])
    for i, o in zip(impls, outs):
        R.check(o, ref, tol, f"{what} impl={i}")
    LAUNCHED.update(names)
    return outs, names


@pytest.mark.parametrize("P,C", GEOM_CELLS)
def test_aligned_false_and_sampling_ratios(P, C):
    lv = RC.levels(C)
    rois = RC.population(seed=3)
    sc = [1.0 / s for s in RC.STRIDES]
    for aligned, sr in ((False, 0), (False, 2), (True, 1), (True, 3), (True, 4), (True, 6)):
        _check_levels(lv, rois, P, sc, sr, aligned, what=f"aligned={aligned} sr={sr}", impls=("auto",))
        _check_levels(lv[:1], rois, P, sc[:1], sr, aligned, what=f"one level aligned={aligned} sr={sr}", impls=("auto",))


MAPS = [(1, 1), (1, 37), (37, 1), (7, 48), (7, 49), (20, 79), (96, 33), (13, 200)]


@pytest.mark.parametrize("P,C", GEOM_CELLS)
def test_map_shapes(P, C):
    """one map each: a single cell, one row / column, one strip or several (W = 48 / 49), three strips with a partial last
    one (W = 79), tall, wide; RoIs all over and around it"""
    g = torch.Generator().manual_seed(P + C)
    for H, W in MAPS:
        x = RC.half_exact(torch.randn(2, C, H, W, generator=g))
        K = 60
        ctr = torch.rand(K, 2, generator=g) * torch.tensor([4.0 * W + 16, 4.0 * H + 16]) - 8
        wh = 1 + torch.rand(K, 2, generator=g) * torch.tensor([4.0 * W, 4.0 * H]) * 0.6
        rois = torch.cat([torch.randint(0, 2, (K, 1), generator=g).float(), ctr - wh / 2, ctr + wh / 2], 1)
        _check_levels([x], rois, P, [0.25], what=f"map {H}x{W}")


def _edge_rois(P, D):
    """scale 1/4, aligned, one sample per bin at start + p + 0.5 (bin = 1 cell): samples exactly on -1, 0 (first bins) and
    on D-1, D (last bins), and the same shifted half a cell outwards (-1.5, D + 0.5: rejected)"""
    rows = []
    for lo_shift in (0.0, -0.5):
        x1 = 4.0 * (-0.5 + lo_shift)          # start = -1.5 (+ shift): samples -1, 0, 1, ...
        rows.append([x1, x1, x1 + 4.0 * P, x1 + 4.0 * P])
        x1 = 4.0 * (D - P + 1 - lo_shift)     # start = D - P + 0.5: the last two samples are D - 1 and D
        rows.append([x1, x1, x1 + 4.0 * P, x1 + 4.0 * P])
        rows.append([4.0 * (-0.5 + lo_shift), 4.0 * (D - P + 1 - lo_shift), 4.0 * (-0.5 + lo_shift) + 4.0 * P,
                     4.0 * (D - P + 1 - lo_shift) + 4.0 * P])
    return torch.tensor([[0.0] + r for r in rows])


def _strip_targets(P, H, W, seed):
    """RoIs on an H x W level (scale 1/4) picked by their staged window: origins at s*31 - 1, s*31, s*31 + 1, windows of
    exactly 18 and 19 cells wide and tall, bins of exactly 8 and 9 taps on each axis"""
    g = torch.Generator().manual_seed(seed)
    N = 3000
    want = {("x0", v) for s in (1, 2) for v in (31 * s - 1, 31 * s, 31 * s + 1)}
    want |= {("ww", 18), ("ww", 19), ("hh", 18), ("hh", 19), ("xtaps", 8), ("xtaps", 9), ("ytaps", 8), ("ytaps", 9)}
    x1 = torch.rand(N, generator=g) * 4 * (W - 4)
    y1 = torch.rand(N, generator=g) * 4 * (H - 4)
    big = 4 * P * torch.tensor([6.0, 7.0]).mean()
    kind = torch.randint(0, 3, (N, 2), generator=g)
    wh = torch.where(kind == 0, 4 * (15 + torch.rand(N, 2, generator=g) * 6),                  # 18 / 19 cell windows
                     torch.where(kind == 1, big * (0.85 + 0.3 * torch.rand(N, 2, generator=g)),   # 8 / 9 tap bins
                                 4 * (2 + torch.rand(N, 2, generator=g) * 10)))                  # small: origins
    cand = torch.stack([torch.zeros(N), x1, y1, x1 + wh[:, 0], y1 + wh[:, 1]], 1)
    win = R.windows(cand, [(H, W)], [0.25], P, mode="sum")
    picked, found = [], set()
    for k, d in enumerate(win):
        hit = {(f, d[f]) for f in ("x0", "ww", "hh", "xtaps", "ytaps")} & (want - found)
        if hit:
            picked.append(k)
            found |= hit
    assert found == want, f"no candidate for {sorted(want - found)}"
    return cand[picked]


@pytest.mark.parametrize("P,C", GEOM_CELLS)
def test_exact_edges_and_strip_boundaries(P, C):
    D = 100        # a square map of four strips: the x edges and the y edges are both at D
    g = torch.Generator().manual_seed(7 * P + C)
    x = RC.half_exact(torch.randn(1, C, D, D, generator=g))
    rois = torch.cat([_edge_rois(P, D), _strip_targets(P, D, D, seed=P * C)])
    for sr in (0, 1):
        _check_levels([x], rois, P, [0.25], sr, what=f"edges and strip targets sr={sr}")


@pytest.mark.parametrize("P,C", GEOM_CELLS)
def test_per_channel_scales(P, C):
    """channels scaled from 1e-3 to 1e3: the bound follows each channel, so a channel mix-up cannot hide"""
    g = torch.Generator().manual_seed(11)
    s = 10.0 ** (torch.rand(C, generator=g) * 6 - 3)
    lv = [f * s[None, :, None, None] for f in RC.levels(C)]
    _check_levels(lv, RC.population(seed=4), P, [1.0 / t for t in RC.STRIDES], what="scaled channels", impls=("auto", "nhwc"))


@pytest.mark.parametrize("P", [7, 14])
def test_strip_binning_limit_both_sides(P):
    """B = 1, C = 32, one 48-wide level: 51 200 rows give nkeys * 4 == 200 KiB, the largest map the strip binning takes;
    51 201 rows go to the per-RoI kernel for every RoI.  Both against the reference, and the route asserted."""
    g = torch.Generator(device="cuda").manual_seed(5)
    K = 120
    gc = torch.Generator().manual_seed(6)
    for H, strip in ((51200, True), (51201, False)):
        x = torch.randn(1, 32, H, 48, device="cuda", generator=g)
        ctr = torch.rand(K, 2, generator=gc) * torch.tensor([192.0, 4.0 * H])
        ctr[:8, 1] = 4.0 * H - torch.rand(8, generator=gc) * 40      # the last rows
        wh = 4 + torch.rand(K, 2, generator=gc) * 60
        rois = torch.cat([torch.zeros(K, 1), ctr - wh / 2, ctr + wh / 2], 1)
        xc = x.cpu()
        _, names = _check_levels([xc], rois, P, [0.25], what=f"H={H}", impls=("auto",))
        assert any(n.startswith(f"roi_align_strip{P}_kernel") for n in names) == strip, (H, sorted(names))
        del x, xc
        torch.cuda.empty_cache()


def test_all_rois_in_one_image_k1_and_k70000():
    import nuhtc_b200 as nb
    sc = [1.0 / s for s in RC.STRIDES]
    g = torch.Generator().manual_seed(12)
    lv8 = [RC.half_exact(torch.randn(8, 64, h, w, generator=g)) for h, w in RC.LEVEL_HW]
    rois = RC.population(K=120, B=8, seed=5)
    rois[:, 0] = 5
    for P in (7, 14):
        _check_levels(lv8, rois, P, sc, what=f"B=8 one image P={P}")
        _check_levels(lv8, rois[9:10], P, sc, what=f"K=1 P={P}")
    # K = 70 000 at C = 32: every RoI against the literal kernel, every 10th against the reference
    lv = RC.levels(32, B=4)
    big = RC.population(K=70000, B=4, seed=6)
    feats = [f.cuda() for f in lv]
    for P in (7, 14):
        (fast, lit), names = _run(lambda: [nb.roi_align_levels(feats, big.cuda(), P, sc, 0, impl=i) for i in ("auto", "direct")])
        idx = torch.arange(0, 70000, 10)
        ref, tol = R.roi_align_ref64(lv, big[idx], P, sc, 0)
        R.check(fast[idx.cuda()], ref, tol, f"K=70000 P={P}")
        assert (fast - lit).abs().max().item() <= 1e-5
        LAUNCHED.update(names)


def test_lone_pool2_level_is_pooled_at_twice_the_size():
    """sum mode over one pool2 level (a channel-group shape the strip kernels would otherwise take): the 2P pooling"""
    for C in (32, 256):
        for P in (7, 14):
            c = dict(C=C, P=P, mode="sum1p", dtype="f32", impl="auto")
            out, names = _run(lambda: RC.run_cell(c))
            ref, tol = _ref(c)
            R.check(out, ref, tol, RC.cell_key(c))
            LAUNCHED.update(names)


# ----------------------------------------------------------------------------- 3. A/B switches in child processes
def _cells(Cs, Ps, modes, impl, dtypes=("f32",)):
    return [dict(C=C, P=P, mode=m, dtype=d, impl=impl) for C in Cs for P in Ps for m in modes for d in dtypes]


AB = {
    ("NUHTC_RA_PIPE", "0"): _cells((64, 128, 256), (7, 14), ("route4", "sum2p"), "auto") + _cells((64, 128, 256), (7, 14), ("route4",), "nhwc")
                             + _cells((128,), (7,), ("route4",), "auto", ("f16",)),
    ("NUHTC_RA_STRIP", "0"): _cells((32, 64, 256), (7, 14), ("route4", "route1"), "auto") + _cells((256,), (14,), ("route1",), "auto", ("bf16",)),
    ("NUHTC_RA_VEC", "1"): _cells((128, 192, 256, 384, 512), (7, 14), ("route4",), "nhwc"),
    ("NUHTC_RA_VEC", "3"): _cells((192, 256, 384, 512), (7, 14), ("route4",), "nhwc"),
    ("NUHTC_RA_TMAP", "1"): _cells((128, 192, 256, 384, 512), (14,), ("route4", "route1"), "nhwc"),
    ("NUHTC_RA_TMAP", "2"): _cells((128, 192, 256, 384, 512), (14,), ("route4", "route1"), "nhwc"),
    ("NUHTC_RA_BULK", "0"): _cells((64, 128, 256), (7, 14), ("route4",), "auto") + _cells((64, 128, 256), (7, 14), ("route4",), "nhwc"),
    ("NUHTC_RA_BULK", "3"): _cells((64, 128, 256), (7, 14), ("route4",), "auto") + _cells((64, 128, 256), (7, 14), ("route4",), "nhwc"),
    ("NUHTC_RA_YROWS", "8"): _cells((64, 256), (7, 14), ("route4", "route1"), "auto"),
    ("NUHTC_RA_YROWS", "64"): _cells((64, 256), (7, 14), ("route4", "route1"), "auto"),
}
# the knob changes how data moves, never a RoI's accumulation order: the outputs must equal the default run's bytes
# (BULK: how the pipelined kernel's tile leaves shared memory; YROWS: how RoIs are binned into strip work units)
BYTE_IDENTICAL = {"NUHTC_RA_BULK", "NUHTC_RA_YROWS"}


def _child(setting, cells, out_dir):
    env = {k: v for k, v in os.environ.items() if not k.startswith("NUHTC_RA_")}
    env[setting[0]] = setting[1]
    flags = ["-s"] if sys.flags.no_user_site else []
    p = subprocess.run([sys.executable, *flags, os.path.join(ROOT, "tests", "_roi_cases.py"), "--out", out_dir,
                        "--cells", json.dumps(cells)], env=env, cwd=ROOT, capture_output=True, text=True, timeout=240)
    assert p.returncode == 0, f"{setting}: exit {p.returncode}\n{p.stderr[-3000:]}"
    return json.loads(p.stdout.strip().splitlines()[-1])


def test_ab_switches_in_child_processes(tmp_path):
    dirs = {s: tmp_path / f"{s[0]}_{s[1]}" for s in AB}
    for d in dirs.values():
        d.mkdir()
    with cf.ThreadPoolExecutor(max_workers=5) as ex:
        futs = {s: ex.submit(_child, s, cells, str(dirs[s])) for s, cells in AB.items()}
        results = {s: f.result() for s, f in futs.items()}
    default_ok = not any(k.startswith("NUHTC_RA_") for k in os.environ)
    for s, cells in AB.items():
        res = results[s]
        assert res["cells"] == [RC.cell_key(c) for c in cells]
        for c in cells:
            out = torch.load(dirs[s] / (RC.cell_key(c) + ".pt"))
            ref, tol = _ref(c)
            R.check(out, ref, _tol(c, tol, ref), f"{s[0]}={s[1]} {RC.cell_key(c)}")
            if s[0] in BYTE_IDENTICAL and default_ok:
                assert torch.equal(out, RC.run_cell(c).cpu()), f"{s[0]}={s[1]} changed the bytes of {RC.cell_key(c)}"
        LAUNCHED.update(res["kernels"])


# ----------------------------------------------------------------------------- 4. attention pooling
def _attn_rois(B, H, W, stride, per_image, seed, empty_images=()):
    """per_image RoIs per image (none in empty_images): centres all over the map, exactly on and beyond every clamp edge"""
    g = torch.Generator().manual_seed(seed)
    rows = []
    for b in range(B):
        if b in empty_images:
            continue
        n = per_image
        ctr = (torch.rand(n, 2, generator=g) * 1.4 - 0.2) * torch.tensor([W * stride, H * stride])
        edge = torch.tensor([[0.0, 0.0], [W * stride - 0.01, H * stride - 0.01], [W * stride, H * stride], [-0.01, -0.01],
                             [(W - 1) * stride, (H - 1) * stride], [-5.0 * stride, 3e4], [3e4, -5.0 * stride]])
        m = min(n, len(edge))
        ctr[:m] = edge[:m]
        wh = torch.rand(n, 2, generator=g) * 6 * stride
        wh[:m] = 0.0                  # x1 + x2 == 2 * centre exactly
        rows.append(torch.cat([torch.full((n, 1), float(b)), ctr - wh / 2, ctr + wh / 2], 1))
    r = torch.cat(rows)
    return r[torch.randperm(len(r), generator=g)]


ATT_MAPS = [(1, 1), (1, 64), (5, 13), (13, 5), (9, 7), (65, 1), (33, 40), (64, 64)]


@pytest.mark.parametrize("H,W", ATT_MAPS)
def test_attention_pool_vs_reference(H, W):
    from nuhtc_b200.mmcv_ops import attention_pool
    stride = 16
    g = torch.Generator().manual_seed(H * 100 + W)
    names_all = set()
    for C in (1, 7, 32, 63, 64):
        for B, per_image, empty in ((1, 1, ()), (3, 63, (1,)), (5, 65, (0, 3)), (3, 64, (2,)), (1, 200, ())):
            f = torch.randn(B, C, H, W, generator=g)
            flat = f.view(B, C, -1)
            if H * W > 2:
                flat[:, :, 0] = 0.0                      # a zero vector at the first position of every image
                flat[:, :, -1] *= 1e-5                   # a near-zero one (norm < 1e-4) at the last
            rois = _attn_rois(B, H, W, stride, per_image, seed=C + B, empty_images=empty)
            fc, rc = f.cuda(), rois.cuda()
            for thres in (0.0, 0.2, 0.9):
                ref, tol = R.attention_pool_ref64(f, rois, stride, thres)
                out, names = _run(lambda: attention_pool(fc, rc, stride, thres))
                R.check(out, ref, tol, f"attention {H}x{W} C={C} B={B} n={per_image} thres={thres}")
                names_all |= names
            # out=: the result is added to what the buffer holds
            pre = torch.randn(rois.shape[0], C, generator=g)
            acc = attention_pool(fc, rc, stride, 0.2, out=pre.cuda())
            ref, tol = R.attention_pool_ref64(f, rois, stride, 0.2)
            R.check(acc, ref + pre.double(), tol + R.U32 * (ref.abs() + pre.double().abs()), f"attention out= {H}x{W} C={C}")
    LAUNCHED.update(names_all)


def test_attention_extractor_on_non_square_levels():
    from nuhtc_b200.roi_extractors import AttentionRoIExtractor
    g = torch.Generator().manual_seed(21)
    feats = [torch.randn(3, 64, h, w, generator=g) for h, w in RC.LEVEL_HW]
    rois = RC.population(K=150, B=3, seed=8, edges=False)
    rois[:, 0] = torch.where(rois[:, 0] == 1, torch.zeros_like(rois[:, 0]), rois[:, 0])   # image 1 holds no RoIs
    for P, sr in ((7, 2), (14, 0)):
        ext = AttentionRoIExtractor(start_level=2, thres=0.2, roi_layer=dict(type="RoIAlign", output_size=P, sampling_ratio=sr),
                                    out_channels=64, featmap_strides=list(RC.STRIDES)).cuda()
        out, names = _run(lambda: ext(tuple(f.cuda() for f in feats), rois.cuda()))
        ref, tol = R.attention_extractor_ref64(feats, rois, RC.STRIDES, P, sr, thres=0.2)
        R.check(out, ref, tol, f"AttentionRoIExtractor P={P}")
        LAUNCHED.update(names)


# ----------------------------------------------------------------------------- 5. coverage (runs last)
COVERED = re.compile(r"^(roi_align_\w+|strip\w*|\w*_to_cg32\w*|attn_\w+|nchw_to_nhwc\w*)(<|$)")


def _library_kernels():
    from nuhtc_b200 import _lib
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    bindir = os.path.dirname(nvcc)
    obj = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=bindir)
    filt = shutil.which("cu++filt") or shutil.which("cu++filt", path=bindir)
    if not obj or not filt:
        pytest.skip("cuobjdump / cu++filt unavailable")
    res = subprocess.run([obj, "--dump-resource-usage", _lib.LIB_PATH], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    mangled = re.findall(r"Function (\S+):", res.stdout)
    dem = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, timeout=60).stdout.splitlines()
    return {RC.kernel_key(n) for n in dem}


def test_zz_every_roi_kernel_launched_and_passed():
    lib = {k for k in _library_kernels() if COVERED.match(k)}
    assert len(lib) >= 40, sorted(lib)
    if not LAUNCHED:
        pytest.skip("no kernel launches recorded: run the whole file (or the profiler yields no CUDA kernel events here)")
    missing = sorted(lib - LAUNCHED)
    assert not missing, f"{len(missing)} of {len(lib)} kernels never launched by a passing case: {missing}"
