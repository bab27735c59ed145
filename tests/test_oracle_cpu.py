"""CPU: pin the oracle.  (1) golden vectors produced by executing the reference's own source
(tests/golden/make_golden.py); (2) torchvision CPU ops, which share mmcv's Detectron lineage; (3) brute force /
exact rational arithmetic for the pycocotools and shapely boundaries."""
import os
from fractions import Fraction

import numpy as np
import pytest
import torch
import torchvision

from nuhtc_b200 import synth

G = os.path.join(os.path.dirname(__file__), "golden")


# ------------------------------------------------------------------ golden vectors from the reference source
def test_golden_paste(oracle):
    z = np.load(os.path.join(G, "paste.npz"))
    boxes, probs = torch.from_numpy(z["boxes"]), torch.from_numpy(z["probs"])
    out = oracle.paste_masks(probs, boxes, 96, 96)
    assert torch.equal(out, torch.from_numpy(z["full"]))          # same torch ops on the same grid: bit-exact
    y0, y1, x0, x1 = z["part_slices"]
    assert torch.equal(out[4:5, y0:y1, x0:x1], torch.from_numpy(z["part"]))  # skip_empty region == full-frame values
    c = oracle.paste_masks_c(probs, boxes, 96, 96)
    assert (c - torch.from_numpy(z["full"])).abs().max().item() <= 1e-6


def test_golden_delta2bbox(oracle):
    z = np.load(os.path.join(G, "delta2bbox.npz"))
    kat = oracle.delta2bbox(torch.from_numpy(z["kat_rois"]), torch.from_numpy(z["kat_deltas"]), max_shape=(32, 32, 3))
    expected = torch.Tensor([[0.0000, 0.0000, 1.0000, 1.0000], [0.1409, 0.1409, 2.8591, 2.8591],
                             [0.0000, 0.3161, 4.1945, 0.6839], [5.0000, 5.0000, 5.0000, 5.0000]])
    assert kat.allclose(expected, atol=1e-4)  # the reference's own KAT (mmdet tests/test_utils/test_coder.py:27-40)
    assert torch.equal(kat, torch.from_numpy(z["kat_out"]))
    out = oracle.delta2bbox(torch.from_numpy(z["rois"]), torch.from_numpy(z["deltas"]), stds=(0.1, 0.1, 0.2, 0.2), max_shape=(512, 512, 3))
    assert torch.equal(out, torch.from_numpy(z["out"]))


def test_golden_roi_levels(oracle):
    z = np.load(os.path.join(G, "roi_levels.npz"))
    lv = oracle.map_roi_levels(torch.from_numpy(z["rois"]), 4)
    assert torch.equal(lv, torch.from_numpy(z["levels"]))
    assert set(np.unique(z["levels"])) == {0, 1, 2, 3}


def test_cpu_log2_is_correctly_rounded_near_level_boundaries():
    """The kernels route with float(log2(double(v))) (roi_common.cuh:route_level); that equals torch's CPU log2 -- the
    reference's map_roi_levels on the CPU path -- on every float within +-200 000 ulps of the level boundaries."""
    for k in (1, 2, 3):
        c = torch.tensor(2.0 ** k, dtype=torch.float32)
        v = (c.view(torch.int32) + torch.arange(-200000, 200001, dtype=torch.int32)).view(torch.float32)
        assert torch.equal(torch.floor(torch.log2(v)), torch.floor(torch.log2(v.double()).float()))
    v = torch.nextafter(torch.tensor(8.0), torch.tensor(0.0))
    assert float(torch.floor(torch.log2(v))) == 3.0   # the fp32 logarithm rounds up across the boundary


def test_golden_multiclass_nms(oracle):
    z = np.load(os.path.join(G, "multiclass_nms.npz"))
    dets, labels, _ = oracle.multiclass_nms(torch.from_numpy(z["boxes"]), torch.from_numpy(z["scores"]), 0.35,
                                            dict(type="nms", iou_threshold=0.5), 500)
    assert torch.equal(dets, torch.from_numpy(z["dets"])) and torch.equal(labels, torch.from_numpy(z["labels"]))


# ------------------------------------------------------------------ torchvision CPU cross-checks
@pytest.mark.parametrize("P,sr,scale", [(7, 0, 0.25), (7, 2, 0.25), (14, 0, 0.25), (14, 2, 0.125), (7, 0, 1 / 32)])
def test_roi_align_equals_torchvision(oracle, P, sr, scale):
    torch.manual_seed(0)
    x = torch.randn(2, 6, 32, 32)
    K = 150
    ctr = torch.rand(K, 2) * 128
    wh = torch.rand(K, 2) * 100
    rois = torch.cat([torch.randint(0, 2, (K, 1)).float(), ctr - wh / 2, ctr + wh / 2], 1)
    rois[0, 1:] = torch.tensor([10., 10., 10., 10.])
    rois[1, 1:] = torch.tensor([-50., -50., 200., 200.])
    rois[2, 1:] = torch.tensor([120., 120., 140., 140.])
    a = oracle.roi_align(x, rois, P, scale, sr)
    b = torchvision.ops.roi_align(x, rois, P, scale, sr, aligned=True)
    assert torch.equal(a, b)
    assert torch.equal(oracle.roi_align(x, rois, P, scale, sr, nthreads=3), a)


@pytest.mark.parametrize("N", [10, 1000, 6000])
def test_nms_equals_torchvision(oracle, N):
    boxes, scores, labels = synth.nms_boxes(N, seed=N)
    _, k = oracle.nms(boxes, scores, 0.5)
    assert torch.equal(k, torchvision.ops.nms(boxes, scores, 0.5))
    _, kb = oracle.batched_nms(boxes, scores, labels, dict(type="nms", iou_threshold=0.5))
    assert torch.equal(kb, torchvision.ops.batched_nms(boxes, scores, labels, 0.5))


def test_batched_nms_split_equals_per_class_reference_loop(oracle):
    boxes, scores, labels = synth.nms_boxes(3000, seed=4)
    cfg = dict(type="nms", iou_threshold=0.5, split_thr=100)
    d, k = oracle.batched_nms(boxes, scores, labels, cfg)
    # above split_thr the result is the union of per-class NMS on the offset boxes, score-sorted
    off = boxes + (labels.float() * (boxes.max() + 1))[:, None]
    parts = []
    for c in labels.unique():
        idx = (labels == c).nonzero().squeeze(1)
        parts.append(idx[torchvision.ops.nms(off[idx], scores[idx], 0.5)])
    allk = torch.cat(parts)
    allk = allk[scores[allk].argsort(descending=True)]
    assert torch.equal(k, allk)
    assert torch.equal(d[:, :4], boxes[k])


# ------------------------------------------------------------------ pycocotools boundary: integer exactness
def test_mask_iou_equals_pixel_counts(oracle):
    rng = np.random.default_rng(0)
    n, H, W = 40, 48, 64
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((n, H, W), np.uint8)
    for i in range(n):
        cy, cx = rng.uniform(5, 43, 2)
        a, b = rng.uniform(3, 12, 2)
        masks[i] = (((yy - cy) / a) ** 2 + ((xx - cx) / b) ** 2 <= 1)
    masks[3] = 0
    masks[4] = 1
    iou = oracle.mask_iou(masks)
    inter = (masks[:, None].astype(np.int64) * masks[None]).sum((2, 3))
    area = masks.sum((1, 2)).astype(np.int64)
    union = area[:, None] + area[None] - inter
    ref = np.where(inter > 0, inter / np.maximum(union, 1), 0.0)
    assert (iou == ref).all()
    assert (oracle.mask_area(masks) == area).all()
    keep = oracle.mask_nms(masks, rng.permutation(n).astype(np.float32), thr=0.05)
    sub = iou[np.ix_(keep, keep)]
    assert (sub[np.triu_indices(len(keep), 1)] <= 0.05).all()


# ------------------------------------------------------------------ shapely boundary: exact area of intersection
def _outline(m):
    """boundary polygon (pixel-edge ring) of a 4-connected hole-free blob: area(A∩B) is then a pixel count"""
    H, W = m.shape
    nxt = {}
    for y in range(H):
        for x in range(W):
            if not m[y, x]:
                continue
            if y == 0 or not m[y - 1, x]:
                nxt[(x, y)] = (x + 1, y)
            if x == W - 1 or not m[y, x + 1]:
                nxt[(x + 1, y)] = (x + 1, y + 1)
            if y == H - 1 or not m[y + 1, x]:
                nxt[(x + 1, y + 1)] = (x, y + 1)
            if x == 0 or not m[y, x - 1]:
                nxt[(x, y + 1)] = (x, y)
    start = next(iter(nxt))
    pts, cur = [start], nxt[start]
    while cur != start:
        pts.append(cur)
        cur = nxt[cur]
    assert len(pts) == len(nxt)
    return np.array(pts, dtype=np.float64)


def test_polygon_intersection_equals_pixel_count(oracle):
    rng = np.random.default_rng(1)
    yy, xx = np.mgrid[0:64, 0:64]
    for _ in range(120):
        m = []
        for _k in range(2):
            cy, cx = rng.uniform(20, 44, 2)
            a, b = rng.uniform(4, 12, 2)
            m.append(((((yy - cy) / a) ** 2 + ((xx - cx) / b) ** 2) <= 1).astype(np.uint8))
        p, q = _outline(m[0]), _outline(m[1])
        assert oracle.poly_area(p) == m[0].sum()
        inter = (m[0] & m[1]).sum()
        assert oracle.poly_inter_area(p, q) == inter                      # heavy collinear overlap, still exact
        assert oracle.poly_inter_area(p[::-1].copy(), q) == inter        # orientation-independent
        assert oracle.poly_inter_area(q, p) == inter


def _exact_inter(P, Q):
    """the same trapezoid identity in exact rational arithmetic"""
    def edges(R):
        n = len(R)
        return [(R[i], R[(i + 1) % n]) for i in range(n)]

    def area2(R):
        return sum(a[0] * b[1] - b[0] * a[1] for a, b in edges(R))
    P = [(Fraction(int(x)), Fraction(int(y))) for x, y in P]
    Q = [(Fraction(int(x)), Fraction(int(y))) for x, y in Q]
    oy = min(y for _, y in P + Q)
    tot = Fraction(0)
    for (e0, e1) in edges(P):
        if e0[0] == e1[0]:
            continue
        se = 1
        if e0[0] > e1[0]:
            e0, e1, se = e1, e0, -1
        for (f0, f1) in edges(Q):
            if f0[0] == f1[0]:
                continue
            sf = 1
            if f0[0] > f1[0]:
                f0, f1, sf = f1, f0, -1
            xa, xb = max(e0[0], f0[0]), min(e1[0], f1[0])
            if xb <= xa:
                continue
            le = lambda x: e0[1] - oy + (e1[1] - e0[1]) * (x - e0[0]) / (e1[0] - e0[0])
            lf = lambda x: f0[1] - oy + (f1[1] - f0[1]) * (x - f0[0]) / (f1[0] - f0[0])
            d0, d1 = le(xa) - lf(xa), le(xb) - lf(xb)
            xs = [xa, xb]
            if d0 * d1 < 0:
                xs = [xa, xa + (xb - xa) * d0 / (d0 - d1), xb]
            for u, v in zip(xs[:-1], xs[1:]):
                mid = (u + v) / 2
                lo = le if le(mid) <= lf(mid) else lf
                tot += se * sf * (lo(u) + lo(v)) / 2 * (v - u)
    if (area2(P) < 0) != (area2(Q) < 0):
        tot = -tot
    return tot


def test_polygon_iou_close_to_exact_rational(oracle):
    d = synth.slide_nuclei(3, 3, per_tile=12, seed=3)
    rings = [d["xy"][d["voff"][i]:d["voff"][i + 1]] for i in range(len(d["score"]))]
    checked = 0
    for i in range(len(rings)):
        for j in range(i + 1, len(rings)):
            a, b = rings[i], rings[j]
            if a[:, 0].max() < b[:, 0].min() or b[:, 0].max() < a[:, 0].min() or a[:, 1].max() < b[:, 1].min() or b[:, 1].max() < a[:, 1].min():
                continue
            ex = _exact_inter(a, b)
            got = oracle.poly_inter_area(a, b)
            assert abs(got - float(ex)) <= 1e-9
            checked += 1
    assert checked > 30


def test_merge_oracle_equals_naive_greedy(oracle):
    d = synth.slide_nuclei(4, 3, per_tile=15, seed=6)
    N = len(d["score"])
    rings = [d["xy"][d["voff"][i]:d["voff"][i + 1]] for i in range(N)]
    order = sorted(range(N), key=lambda i: (-d["score"][i], i))
    dead, kept = set(), []
    for a_i, a in enumerate(order):
        if a in dead:
            continue
        kept.append(a)
        for b in order[a_i + 1:]:
            if b not in dead and oracle.poly_iou(rings[a], rings[b]) > 0.05:
                dead.add(b)
    got = oracle.merge_overlap_arrays(d["xy"], d["voff"], d["score"], 0.05, "probability")
    assert got.tolist() == kept
    area = oracle.merge_overlap_arrays(d["xy"], d["voff"], d["score"], 0.05, "area")
    assert len(area) == len(kept) and set(area.tolist()) != set(kept)


def _blob_rings(rng, count, size=64):
    """Contour-shaped rings: smooth non-convex blobs (thresholded sums of Gaussians) traced by the contour oracle,
    closed like infer_wsi.py:53 does.  Rings the tracer returns with a pinch point (not simple) are dropped."""
    yy, xx = np.mgrid[0:size, 0:size]
    rings = []
    while len(rings) < count:
        f = np.zeros((size, size))
        for _ in range(rng.integers(2, 5)):
            cy, cx = rng.uniform(22, size - 22, 2)
            sy, sx = rng.uniform(4, 9, 2)
            f += np.exp(-(((yy - cy) / sy) ** 2 + ((xx - cx) / sx) ** 2))
        m = (f > 0.55).astype(np.uint8)
        if m.sum() < 30:
            continue
        from oracle import cpu as O
        r = O.mask2inst(m).reshape(-1, 2).astype(np.float64)
        if len(r) < 4 or len(np.unique(r[:-1], axis=0)) != len(r) - 1:   # a vertex visited twice: self-touching ring
            continue
        rings.append(r)
    return rings


def test_polygon_area_second_anchor_slab_decomposition(oracle):
    """The trapezoid-identity oracle (whose summation order follows the GPU's 32-lane butterfly) against an independent
    algorithm -- vertical slab decomposition with the even-odd rule -- on > 1e4 pairs: the duplicated, jittered ellipse
    contours of the synthetic slide and cv2-style contours of non-convex blobs.  Areas agree to 1e-9 relative and every
    IoU > 0.05 decision (the only thing the merge consumes) is identical."""
    from scipy.spatial import cKDTree
    d = synth.slide_nuclei(24, 24, per_tile=23, seed=31)
    N = len(d["score"])
    rings = [d["xy"][d["voff"][i]:d["voff"][i + 1]] for i in range(N)]
    ctr = np.array([r.mean(0) for r in rings])
    pairs = sorted(cKDTree(ctr).query_pairs(22.0))
    rng = np.random.default_rng(7)
    blobs = _blob_rings(rng, 400)
    cases = [(rings[i], rings[j]) for i, j in pairs[:9000]]
    for _ in range(3000):
        a, b = blobs[rng.integers(len(blobs))], blobs[rng.integers(len(blobs))]
        cases.append((a, b + rng.integers(-14, 15, 2).astype(np.float64)))
    assert len(cases) >= 12000
    overlapping = decided = 0
    for a, b in cases:
        t = oracle.poly_inter_area(a, b)
        s = oracle.poly_inter_area_slab(a, b)
        aa, ab = oracle.poly_area(a), oracle.poly_area(b)
        assert abs(t - s) <= 1e-9 * max(1.0, min(aa, ab)), (t, s)
        if t > 0:
            overlapping += 1
            iou_t, iou_s = t / (aa + ab - t), s / (aa + ab - s)
            if abs(iou_t - 0.05) > 1e-9:       # the contract excludes |IoU - thr| < 1e-9
                decided += 1
                assert (iou_t > 0.05) == (iou_s > 0.05)
    assert overlapping > 6000 and decided > 6000


def test_merge_oracle_equals_all_pairs_search_and_slab_area(oracle):
    """The grid-accelerated oracle against (1) an O(N^2) candidate search (every envelope pair, what STRtree.query
    yields) and (2) the same greedy loop on the slab-decomposition area, at ~10k and ~170k nuclei."""
    d = synth.slide_nuclei(16, 16, per_tile=23, seed=11)
    for strat in ("probability", "area"):
        ref = oracle.merge_overlap_arrays(d["xy"], d["voff"], d["score"], 0.05, strat)
        assert np.array_equal(ref, oracle.merge_overlap_arrays_check(d["xy"], d["voff"], d["score"], 0.05, strat, naive=True))
        assert np.array_equal(ref, oracle.merge_overlap_arrays_check(d["xy"], d["voff"], d["score"], 0.05, strat, naive=True, slab=True))
    assert 9000 < len(d["score"]) < 11000
    from _slides import load_case
    _, d, thr = load_case(1)   # 66 x 66 tiles, the exact-threshold pairs dropped (the two areas round those differently)
    ref = oracle.merge_overlap_arrays(d["xy"], d["voff"], d["score"], thr)
    assert np.array_equal(ref, oracle.merge_overlap_arrays_check(d["xy"], d["voff"], d["score"], thr, naive=False, slab=True))


@pytest.mark.parametrize("case", [0, 1, 2])
def test_merge_golden_hashes(oracle, case):
    """Committed kept-id hashes at 15k / 170k / 1.7M nuclei (tests/golden/merge_large.json, BASELINE cfg 5): the oracle
    reproduces them here; tests/test_gpu_merge.py holds the CUDA merge to the same hashes.  No decisive pair of a golden
    case is closer than 1e-9 to the threshold (the exact 1/20 ties of the raw slides were dropped)."""
    from _slides import load_case, sha
    c, d, thr = load_case(case)
    k, margin, ties = oracle.merge_overlap_arrays_check(d["xy"], d["voff"], d["score"], thr, naive=False, with_margin=True)
    assert len(ties) == 0 and margin > 1e-9
    assert len(k) == c["probability"]["kept"] and sha(k.astype(np.int64)) == c["probability"]["kept_ids_sha256"]
    assert np.array_equal(k, oracle.merge_overlap_arrays(d["xy"], d["voff"], d["score"], thr))


def test_threshold_ties_exist_and_are_dropped(oracle):
    """IoU of integer-vertex rings is rational and does hit 1/20 exactly: the raw 66x66 slide holds such decisive pairs,
    the slab and trapezoid areas round them to different sides, and drop_threshold_ties removes exactly the nuclei the
    golden file lists."""
    from _slides import golden
    c = golden()["cases"][1]
    d = synth.slide_nuclei(c["tiles"][0], c["tiles"][1], per_tile=23, seed=c["seed"])
    _, margin, ties = oracle.merge_overlap_arrays_check(d["xy"], d["voff"], d["score"], 0.05, naive=False, with_margin=True)
    assert margin < 1e-12 and len(ties) >= 1
    _, removed = oracle.drop_threshold_ties(d, 0.05)
    assert removed.tolist() == c["removed_out_of_contract"]
    assert {int(a) for a, b in ties} | {int(b) for a, b in ties} & set(removed.tolist())


def test_golden_cases_hold_no_identical_rings():
    """Out of contract (DESIGN.md 2): the reference keys a dict by the shapely polygon (nuclei_merge.py:101-103), so two
    nuclei with IDENTICAL rings collide and it keeps the LOWER-scored copy.  The raw synthetic slides do hold a few such
    twins (4 pairs in 171k nuclei); the golden cases drop the lower-scored copy, like the exact-threshold pairs."""
    from _slides import load_case
    raw = synth.slide_nuclei(66, 66, per_tile=23, seed=66)
    keys = {raw["xy"][raw["voff"][i]:raw["voff"][i + 1]].tobytes() for i in range(len(raw["score"]))}
    assert len(keys) < len(raw["score"])
    _, d, _ = load_case(1)
    keys = {d["xy"][d["voff"][i]:d["voff"][i + 1]].tobytes() for i in range(len(d["score"]))}
    assert len(keys) == len(d["score"])


def test_golden_attention_extractor(oracle):
    """AttentionRoIExtractor.forward executed from the reference source (mmcv RoIAlign layers -> oracle) vs the restatement."""
    z = np.load(os.path.join(G, "attention_extractor.npz"))
    feats = synth.fpn_levels(2, 64, frame=256, seed=21)
    out = oracle.attention_roi_extract(feats, torch.from_numpy(z["rois"]), (4, 8, 16, 32), 7, 2, start_level=2, thres=0.0)
    assert out.shape == (z["rois"].shape[0], 64, 7, 7)
    # the golden keeps every k-th channel whole and, for every channel, the sum over the 7x7 bins
    assert torch.equal(out[:, ::int(z["channel_stride"])], torch.from_numpy(z["out"]))
    assert torch.allclose(out.double().sum((2, 3)), torch.from_numpy(z["out_bin_sum"]).double(), rtol=1e-6, atol=1e-6)


def test_rpn_post_process_golden(oracle):
    """RPNHead._bbox_post_process (rpn_head.py:189-236): golden made by executing the reference method."""
    z = np.load(os.path.join(G, "rpn_post.npz"))
    t = lambda k: torch.from_numpy(z[k])
    d = oracle.rpn_bbox_post_process(t("scores"), t("deltas"), t("anchors"), t("ids"), (512, 512, 3),
                                     dict(type="nms", iou_threshold=0.7), 300)
    assert torch.equal(d, t("dets"))


def _golden_contours():
    z = np.load(os.path.join(G, "contours.npz"))
    cm = np.unpackbits(z["masks"], axis=2)[:, :, :96]
    return cm, z["points"], z["offsets"]


def test_contour_golden(oracle):
    """mask2inst (tools/infer_wsi.py:51-54): golden made by running the reference function body on the real cv2."""
    cm, pts, off = _golden_contours()
    for i, m in enumerate(cm):
        assert np.array_equal(oracle.mask2inst(m).reshape(-1, 2), pts[off[i]: off[i + 1]]), i


def test_contour_live_cv2(oracle):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(12)
    for it in range(400):
        h, w = rng.integers(1, 48, 2)
        m = (rng.random((h, w)) < rng.uniform(0.1, 0.9)).astype(np.uint8)
        if it % 3 == 0:
            m = cv2.dilate(m, np.ones((2, 2), np.uint8))
        for simple, flag in ((True, cv2.CHAIN_APPROX_SIMPLE), (False, cv2.CHAIN_APPROX_NONE)):
            c, _ = cv2.findContours(m, cv2.RETR_TREE, flag)
            ref = c[0].reshape(-1, 2) if len(c) else np.zeros((0, 2), np.int32)
            assert np.array_equal(oracle.contour0(m, simple), ref)
