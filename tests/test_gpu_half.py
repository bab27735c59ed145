"""GPU: fp16 / bf16 feature maps through the RoI stage.

Contract (mmcv's force_fp32(out_fp16=True), extended to bf16): half levels are upcast exactly while they are staged,
everything is computed in fp32 as for fp32 levels, and every RoI feature is rounded once to the levels' dtype.  So the
native half path must equal, bit for bit, the fp32 path on the upcast levels followed by ``.to(dtype)``."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DTYPES = [torch.float16, torch.bfloat16]
STRIDES = (4, 8, 16, 32)
SCALES = [1.0 / s for s in STRIDES]


def _levels(B, C, dtype, seed, frame=512):
    from nuhtc_b200 import synth
    return [f.cuda().to(dtype) for f in synth.fpn_levels(B, C, frame=frame, seed=seed)]


def _rois(B, n_per, dist, seed, frame=512):
    from nuhtc_b200 import synth
    return synth.proposals(B, n_per, dist, frame=frame, seed=seed).cuda()


def _native_equals_cast(levels, rois, P, scales, sr, **kw):
    import nuhtc_b200 as nb
    dtype = levels[0].dtype
    out = nb.roi_align_levels(levels, rois, P, scales, sr, **kw)
    ref = nb.roi_align_levels([f.float() for f in levels], rois, P, scales, sr, **kw)
    assert out.dtype == dtype and out.shape == ref.shape
    assert torch.isfinite(ref).all()
    assert torch.equal(out, ref.to(dtype))
    return out


def _extreme_map(shape, dtype, seed):
    """randn values, plus a share of values in the dtype's subnormal range and near its largest finite value."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g)
    fi = torch.finfo(dtype)
    pick = torch.randint(0, 6, shape, generator=g)
    x = torch.where(pick == 0, x.sign() * fi.tiny * torch.rand(shape, generator=g), x)     # subnormals (and zeros)
    x = torch.where(pick == 1, x.sign() * fi.max * (0.5 + 0.5 * torch.rand(shape, generator=g)), x)
    return x.to(dtype).cuda()


# ----------------------------------------------------------------------------------------------------------- staging
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("layout,H,W", [("nchw", 32, 40), ("channels_last", 32, 40), ("nchw", 13, 11)])
def test_staging_equals_upcast(dtype, layout, H, W):
    import nuhtc_b200 as nb
    x = _extreme_map((2, 64, H, W), dtype, seed=H * W)
    sub = (x.float().abs() < torch.finfo(dtype).tiny) & (x != 0)
    assert sub.any() and (x.float().abs() > torch.finfo(dtype).max / 2).any()
    if layout == "channels_last":
        x = x.contiguous(memory_format=torch.channels_last)
    got = nb.to_cg32(x)
    ref = nb.to_cg32(x.float())
    assert got.dtype == torch.float32 and got.shape == (2, 2, H, W, 32)
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32))


# ------------------------------------------------------------------------------------- RoIAlign: native == cast
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [64, 256])
@pytest.mark.parametrize("P,sr", [(7, 0), (7, 2), (14, 0), (14, 2)])
def test_route_native_equals_cast(dtype, C, P, sr):
    levels = _levels(2, C, dtype, seed=P + sr)
    rois = _rois(2, 400, "nuclei", seed=C + P)
    _native_equals_cast(levels, rois, P, SCALES, sr, mode="route", finest_scale=56.0)


def _leftover_count(levels, rois, P, sr, dtype):
    """One direct C-ABI call: how many RoIs the strip kernels left to the per-RoI kernel (workspace counter 2)."""
    import nuhtc_b200 as nb
    from nuhtc_b200 import _lib as L
    st = nb.stage_levels(levels)
    nl, K = len(levels), rois.shape[0]
    Hs = (ctypes.c_int * nl)(*[h for h, _ in st.shapes])
    Ws = (ctypes.c_int * nl)(*[w for _, w in st.shapes])
    sc = (ctypes.c_float * nl)(*SCALES[:nl])
    ptrs = (ctypes.c_void_p * nl)(*[b.data_ptr() for b in st.cg32])
    lib = L.lib()
    wsb = lib.nuhtc_roi_align_workspace_bytes(Hs, Ws, nl, st.B, K, P, P)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    out = torch.empty((K, st.C, P, P), dtype=dtype, device="cuda")
    L.check(lib.nuhtc_roi_align_cg32_dt(ptrs, Hs, Ws, sc, nl, st.B, st.C, rois.data_ptr(), K, P, P, sr, 1, L.ROI_ROUTE, 56.0, None,
                                        out.data_ptr(), L.DTYPE_CODES[dtype], None, ws.data_ptr(), wsb, L.stream_ptr()), "cg32_dt")
    return int(ws[8:12].view(torch.int32).item())


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("P,sr", [(7, 2), (14, 0)])
def test_routed_with_leftovers_native_equals_cast(dtype, P, sr):
    levels = _levels(2, 256, dtype, seed=7)
    rois = _rois(2, 600, "routed", seed=8)
    assert _leftover_count(levels, rois, P, sr, dtype) > 0   # the per-RoI kernel writes half of these outputs too
    _native_equals_cast(levels, rois, P, SCALES, sr, mode="route", finest_scale=56.0)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [64, 256])
@pytest.mark.parametrize("P,sr", [(7, 2), (14, 0)])
def test_sum_bias_and_semantic_native_equals_cast(dtype, C, P, sr):
    import nuhtc_b200 as nb
    levels = _levels(2, C, dtype, seed=11)
    rois = _rois(2, 300, "nuclei", seed=12)
    g = torch.Generator().manual_seed(13)
    bias = torch.randn(rois.shape[0], C, generator=g).cuda()
    _native_equals_cast(levels[:2], rois, P, SCALES[:2], sr, mode="sum", bias=bias)
    # the semantic level of the bbox branch: RoIAlign at 2P x 2P, 2x2-averaged, inside the same launch
    sem = (torch.randn(2, C, 128, 128, generator=g) * 0.5).cuda().to(dtype)
    lv = nb.stage_levels(levels[:2]).cat(nb.stage_levels([sem]))
    out = nb.roi_align_levels(lv, rois, P, SCALES[:2] + [0.25], sr, mode="sum", bias=bias, pool2=[False, False, True])
    ref = nb.roi_align_levels(nb.stage_levels([f.float() for f in levels[:2] + [sem]]), rois, P, SCALES[:2] + [0.25], sr,
                              mode="sum", bias=bias, pool2=[False, False, True])
    assert out.dtype == dtype and torch.equal(out, ref.to(dtype))


@pytest.mark.parametrize("dtype", DTYPES)
def test_empty_and_caller_out(dtype):
    import nuhtc_b200 as nb
    levels = _levels(1, 64, dtype, seed=21)
    e = nb.roi_align_levels(levels, torch.zeros(0, 5, device="cuda"), 7, SCALES, 0, mode="route")
    assert e.shape == (0, 64, 7, 7) and e.dtype == dtype
    rois = _rois(1, 100, "nuclei", seed=22)
    buf = torch.full((100, 64, 7, 7), float("nan"), dtype=dtype, device="cuda")
    got = nb.roi_align_levels(levels, rois, 7, SCALES, 2, mode="route", out=buf)
    assert got.data_ptr() == buf.data_ptr()
    assert torch.equal(buf, nb.roi_align_levels([f.float() for f in levels], rois, 7, SCALES, 2, mode="route").to(dtype))
    with pytest.raises(AssertionError):
        nb.roi_align_levels(levels, rois, 7, SCALES, 2, mode="route", out=buf.float())


@pytest.mark.parametrize("dtype", DTYPES)
def test_cast_paths_native_equals_cast(dtype):
    """C = 24 has no channel-group kernel and impl='direct' is the literal kernel: fp32 between one cast each way."""
    levels = _levels(2, 24, dtype, seed=31)
    rois = _rois(2, 120, "routed", seed=32)
    _native_equals_cast(levels, rois, 7, SCALES, 2, mode="route", finest_scale=56.0)
    levels = _levels(2, 64, dtype, seed=33)
    _native_equals_cast(levels, rois, 14, SCALES, 0, mode="route", finest_scale=56.0, impl="direct")


# ----------------------------------------------------------------------------------------------- against the oracle
def _ulp(v, dtype):
    """spacing of `dtype` at |v| (fp32 tensor), the subnormal spacing below the normal range"""
    mant, emin = (10, -14) if dtype == torch.float16 else (7, -126)
    e = torch.floor(torch.log2(v.abs())).clamp(min=emin)
    return torch.exp2(e - mant)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("P,sr", [(7, 2), (14, 0)])
def test_against_oracle(oracle, dtype, P, sr):
    import nuhtc_b200 as nb
    g = torch.Generator().manual_seed(41)
    x = torch.randn(2, 64, 32, 32, generator=g).to(dtype)
    rois = _rois(2, 100, "nuclei", seed=42, frame=128).cpu()
    o32 = oracle.roi_align(x.float(), rois, P, 0.25, sr)
    ref = o32.to(dtype)
    lit = nb.roi_align_levels([x.cuda()], rois.cuda(), P, [0.25], sr, True, impl="direct").cpu()
    assert lit.dtype == dtype and torch.equal(lit, ref)
    out = nb.roi_align(x.cuda(), rois.cuda(), P, 0.25, sr, "avg", True).cpu()
    s32 = nb.roi_align(x.float().cuda(), rois.cuda(), P, 0.25, sr, "avg", True).cpu()
    dev = (s32 - o32).abs()
    assert dev.max().item() <= 1e-5
    # each side is rounded once: apart from one spacing of the output type, only what the fp32 results differ by
    d = (out.float() - ref.float()).abs()
    assert (d <= _ulp(torch.maximum(out.float().abs(), ref.float().abs()), dtype) + dev).all()
    assert (out != ref).float().mean().item() < 0.01


# ------------------------------------------------------------------------------------------------------ extractors
@pytest.mark.parametrize("dtype", DTYPES)
def test_extractors_return_feats_dtype(dtype):
    from nuhtc_b200.roi_extractors import AttentionRoIExtractor, SingleRoIExtractor
    feats = _levels(2, 64, dtype, seed=51)
    rois = _rois(2, 200, "routed", seed=52)

    def cfg(P, sr):
        return dict(roi_layer=dict(type="RoIAlign", output_size=P, sampling_ratio=sr), out_channels=64, featmap_strides=list(STRIDES))
    exts = [AttentionRoIExtractor(start_level=2, thres=0, **cfg(7, 2)), SingleRoIExtractor(finest_scale=56, **cfg(7, 0)),
            AttentionRoIExtractor(start_level=2, thres=0, **cfg(14, 0))]
    for ext in exts:
        ext.fp16_enabled = True                      # what mmcv's wrap_fp16_model sets
        for kw in (dict(), dict(roi_scale_factor=1.5)):
            got = ext(feats, rois, **kw)
            ref = ext([f.float() for f in feats], rois, **kw)
            assert got.dtype == dtype and ref.dtype == torch.float32
            assert torch.equal(got, ref.to(dtype))
        assert ext(feats, rois[:0]).dtype == dtype
    only_attn = AttentionRoIExtractor(start_level=0, thres=0, **cfg(7, 2))
    assert torch.equal(only_attn(feats, rois), only_attn([f.float() for f in feats], rois).to(dtype))


# ------------------------------------------------------------------------------------------------------ end to end
class _CastIn(torch.nn.Module):
    """A half head behind a callable that takes fp32 input: the force_fp32 boundary of an fp32 extractor."""

    def __init__(self, m, dtype, upcast_second=False):
        super().__init__()
        self.m, self.dtype, self.upcast_second = m, dtype, upcast_second
        for a in ("num_classes", "target_stds", "score_activation"):
            if hasattr(m, a):
                setattr(self, a, getattr(m, a))

    def forward(self, x):
        if isinstance(x, (list, tuple)):
            p, f = self.m([t.to(self.dtype) for t in x])
            return p, (f.float() if self.upcast_second else f)
        return self.m(x.to(self.dtype))


@pytest.mark.parametrize("dtype", DTYPES)
def test_simple_test_half_equals_fp32_stage_with_casts(dtype):
    import _toy_heads as T
    from nuhtc_b200 import synth
    from nuhtc_b200.htc_roi_head import HybridTaskCascadeRoIHead_Lite, seesaw_activation
    B, FRAME = 2, 512
    x = tuple(f.cuda().to(dtype) for f in synth.fpn_levels(B, T.C, frame=FRAME, seed=61))
    props = synth.proposals(B, 150, "nuclei", frame=FRAME, seed=62)
    plist = [torch.cat([props[props[:, 0] == b][:, 1:], torch.ones(int((props[:, 0] == b).sum()), 1)], 1).cuda() for b in range(B)]
    metas = [dict(img_shape=(FRAME, FRAME, 3), ori_shape=(256, 256, 3), scale_factor=np.array([2.] * 4, dtype=np.float32))] * B
    heads = [T.ToyBBoxHead(i).cuda().to(dtype) for i in range(3)]
    for h in heads:
        h.score_activation = seesaw_activation
    mh, sh = T.ToyMaskHead().cuda().to(dtype), T.ToySemanticHead().cuda().to(dtype)
    kw = dict(extractor="attention", start_level=2, thres=0.0, bbox_roi_layer=dict(type="RoIAlign", output_size=7, sampling_ratio=2),
              mask_roi_layer=dict(type="RoIAlign", output_size=14, sampling_ratio=0), semantic_fusion=("bbox", "mask"))
    half = HybridTaskCascadeRoIHead_Lite(3, heads, mh, T.TEST_CFG, semantic_head=sh, **kw)
    cast = HybridTaskCascadeRoIHead_Lite(3, [_CastIn(h, dtype) for h in heads], _CastIn(mh, dtype), T.TEST_CFG,
                                         semantic_head=_CastIn(sh, dtype, upcast_second=True), **kw)
    got = half.simple_test(None, x, plist, metas, rescale=True)
    ref = cast.simple_test(None, tuple(f.float() for f in x), plist, metas, rescale=True)
    n = 0
    for (gb, gs), (rb, rs) in zip(got, ref):
        for c in range(T.NUM_CLASSES):
            assert gb[c].dtype == np.float32 and np.array_equal(gb[c], rb[c])
            assert len(gs[c]) == len(rs[c]) and all(a.dtype == np.bool_ and np.array_equal(a, b) for a, b in zip(gs[c], rs[c]))
            n += len(gb[c])
    assert n > 0
    with pytest.raises(NotImplementedError):
        HybridTaskCascadeRoIHead_Lite(3, heads, mh, T.TEST_CFG, semantic_head=sh, watershed_proposal=True,
                                      **kw).simple_test(None, x, plist, metas, rescale=True)


def test_simple_test_under_autocast():
    """fp32 heads, the whole test path under torch.autocast(bfloat16): bf16 levels in, the reference result format out."""
    import _toy_heads as T
    from nuhtc_b200 import synth
    from nuhtc_b200.htc_roi_head import HybridTaskCascadeRoIHead_Lite, seesaw_activation
    B, FRAME = 2, 512
    heads = [T.ToyBBoxHead(i).cuda() for i in range(3)]
    for h in heads:
        h.score_activation = seesaw_activation
    head = HybridTaskCascadeRoIHead_Lite(3, heads, T.ToyMaskHead().cuda(), T.TEST_CFG, semantic_head=T.ToySemanticHead().cuda())
    props = synth.proposals(B, 150, "nuclei", frame=FRAME, seed=62)
    plist = [torch.cat([props[props[:, 0] == b][:, 1:], torch.ones(int((props[:, 0] == b).sum()), 1)], 1).cuda() for b in range(B)]
    metas = [dict(img_shape=(FRAME, FRAME, 3), ori_shape=(256, 256, 3), scale_factor=np.array([2.] * 4, dtype=np.float32))] * B
    lin = torch.nn.Conv2d(T.C, T.C, 1).cuda()          # stands in for the neck: its output is bf16 under autocast
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        x = tuple(lin(f.cuda()) for f in synth.fpn_levels(B, T.C, frame=FRAME, seed=61))
        assert all(f.dtype == torch.bfloat16 for f in x)
        res = head.simple_test(None, x, plist, metas, rescale=True)
    n = 0
    for bbox_result, segm_result in res:
        for c in range(T.NUM_CLASSES):
            assert bbox_result[c].dtype == np.float32 and bbox_result[c].shape[1] == 5
            assert len(segm_result[c]) == len(bbox_result[c]) and all(m.dtype == np.bool_ for m in segm_result[c])
            n += len(bbox_result[c])
    assert n > 0


# ---------------------------------------------------------------------------------------------------- graph capture
@pytest.mark.parametrize("dtype", DTYPES)
def test_stage_graph_replay_equals_eager(dtype):
    from nuhtc_b200 import synth
    from nuhtc_b200.roi_stage import RoIStage, RoIStageConfig
    B, n_per = 2, 300
    cfg = RoIStageConfig(extractor="attention", sum_levels=2, semantic_fusion=("bbox", "mask"), bbox_sampling_ratio=2,
                         max_per_img=100, contour_max_pts=64)
    heads = synth.SyntheticHeads(B * n_per, seed=71).to("cuda")
    bbox = [(lambda f, i=i: (heads.cls[i].to(f.dtype), heads.reg[i].to(f.dtype))) for i in range(3)]
    st = RoIStage(cfg, bbox, lambda f, cand: heads.mask_head(f, cand).to(f.dtype))
    feats = _levels(B, 64, dtype, seed=72)
    sem = _levels(B, 64, dtype, seed=73)[0]
    rois = _rois(B, n_per, "nuclei", seed=74)

    def run():
        return st.run(feats, rois, max_rois_per_tile=n_per, semantic_feat=sem)

    eager = run()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        cap = run()
    g.replay()
    torch.cuda.synchronize()
    assert int(eager.det_valid.sum()) > 0
    for a in ("det_boxes", "det_scores", "det_labels", "det_valid", "masks", "mask_bits", "tile_start", "tile_count", "contour_count"):
        assert torch.equal(getattr(cap, a), getattr(eager, a)), a
    # only the listed entries of `keep` and the traced points of `contour_xy` are defined
    assert all(torch.equal(x, y) for x, y in zip(cap.kept_indices(), eager.kept_indices()))
    live = torch.arange(cfg.contour_max_pts, device="cuda")[None, :] < eager.contour_count[:, None].long()
    assert torch.equal(cap.contour_xy[live], eager.contour_xy[live])
