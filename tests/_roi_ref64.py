"""Float64 references for RoIAlign (mmcv 1.7.2 ``roi_align_forward``, avg, as the RoI extractors drive it) and for the
cosine-attention pooling of AttentionRoIExtractor, with a rigorous first-order error bound for an fp32 implementation.

The geometry is the contract and is computed exactly as the reference computes it, in fp32 (numpy float32 scalars round
every operation to nearest, like the reference's CPU code): level routing, the RoI's start / extent / bin / sample count
and every sample coordinate.  Everything after the coordinates is float64.  mmcv's validity test (reject a sample outside
(-1, D) on EITHER axis) and its bilinear weights factor per axis, so one RoI on one level is

    ref[c] = Ay . F[b, c] . Ax^T / max(gh * gw, 1)          Ay in R^{P x H}, Ax in R^{P x W}

with Ay / Ax the per-axis sums of the sample weights.  The matrices are cropped to the window rows / columns the RoI
reaches, so a RoI on a 51 201-row map costs no more than one on a 32-row map.

Acceptance (``bound``): an fp32 result passes when |out - ref| <= (4 gh gw + 16) u absbound + 1e-30 with u = 2^-24 and
absbound = |Ay| |F| |Ax|^T / count, the first-order bound of the literal kernel's sequential fp32 sum (4 products and
3 adds per sample, one add into the accumulator, one division); in sum mode the levels' bounds add up, and a 16-bit
output adds half an ulp of its type.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn.functional as F

U32 = 2.0 ** -24
f32 = np.float32


# ----------------------------------------------------------------------------- geometry (fp32, the reference's op order)
def route_levels(rois: torch.Tensor, L: int, finest: float = 56.0) -> np.ndarray:
    """SingleRoIExtractor.map_roi_levels evaluated by torch on the CPU in fp32 (single_level_roi_extractor.py:51-55)."""
    r = rois.detach().cpu().float()
    scale = torch.sqrt((r[:, 3] - r[:, 1]) * (r[:, 4] - r[:, 2]))
    return torch.floor(torch.log2(scale / finest + 1e-6)).clamp(min=0, max=L - 1).long().numpy()


def roi_geom(roi, scale: float, P: int, sr: int, aligned: bool, pool2: bool = False):
    """(start_w, start_h, bin_w, bin_h, gw, gh, count) of one RoI on one level, fp32 as mmcv computes them.
    pool2: the geometry of the level's 2P x 2P RoIAlign with sampling_ratio 0 (the semantic branch's definition)."""
    s = f32(scale)
    off = f32(0.5) if aligned else f32(0.0)
    x1, y1, x2, y2 = (f32(v) for v in roi[1:5])
    sw, sh = x1 * s - off, y1 * s - off
    rw, rh = (x2 * s - off) - sw, (y2 * s - off) - sh
    if not aligned:
        rw, rh = max(rw, f32(1.0)), max(rh, f32(1.0))
    PP = 2 * P if pool2 else P
    bw, bh = rw / f32(PP), rh / f32(PP)
    if pool2:
        sr = 0
    gw = sr if sr > 0 else int(math.ceil(rw / f32(PP)))
    gh = sr if sr > 0 else int(math.ceil(rh / f32(PP)))
    return sw, sh, bw, bh, gw, gh, max(gh * gw, 1), PP


def _coords(start, bin_, PP: int, g: int) -> np.ndarray:
    """[PP, g] fp32 sample coordinates (start + p*bin) + ((i + .5)*bin)/g."""
    p = np.arange(PP, dtype=np.float32)[:, None]
    i = np.arange(max(g, 0), dtype=np.float32)[None, :] + f32(0.5)
    return (f32(start) + p * f32(bin_)) + (i * f32(bin_)) / f32(g if g > 0 else 1)


def axis_matrix(start, bin_, PP: int, g: int, D: int):
    """Per-axis weights of the bins: (A [PP, n] float64 over cells lo..lo+n-1, lo, taps [PP] per-bin tap count as the
    kernels' tap tables count it: last valid sample's upper cell - first valid sample's lower cell + 1, 0 if none)."""
    c = _coords(start, bin_, PP, g)
    valid = ~((c < -1.0) | (c > f32(D)))
    cc = np.where(c <= 0, f32(0), c)
    lo = cc.astype(np.int64)                    # (int)c: truncation of a non-negative value
    top = lo >= D - 1
    lo = np.where(top, D - 1, lo)
    hi = np.where(top, D - 1, lo + 1)
    cc = np.where(top, lo.astype(np.float32), cc)
    lw = cc.astype(np.float64) - lo             # float64: the exact weights of the fp32 coordinate
    hw = 1.0 - lw
    if not valid.any():
        return np.zeros((PP, 0)), 0, np.zeros(PP, dtype=np.int64)
    a = int(lo[valid].min())
    b = int(hi[valid].max())
    A = np.zeros((PP, b - a + 1))
    rows = np.broadcast_to(np.arange(PP)[:, None], c.shape)
    np.add.at(A, (rows[valid], lo[valid] - a), hw[valid])
    np.add.at(A, (rows[valid], hi[valid] - a), lw[valid])
    rowany = valid.any(axis=1)
    first = np.argmax(valid, axis=1)
    last = valid.shape[1] - 1 - np.argmax(valid[:, ::-1], axis=1)
    pr = np.arange(PP)
    taps = np.where(rowany, hi[pr, last] - lo[pr, first] + 1, 0)
    return A, a, taps


def windows(rois: torch.Tensor, level_hw: Sequence[tuple], scales: Sequence[float], P: int, sr: int = 0,
            aligned: bool = True, mode: str = "route", finest: float = 56.0) -> list:
    """Per RoI (route mode: on its routed level; sum mode: on level 0) the window the strip kernels stage:
    dict(level, x0, ww, y0, hh, xtaps, ytaps) -- x0/y0 the first cell, ww/hh the extent, *taps the largest tap count of a
    bin on that axis (> 8: the RoI takes the literal path)."""
    r = rois.detach().cpu().float().numpy()
    lv = route_levels(rois, len(level_hw), finest) if mode == "route" else np.zeros(len(r), np.int64)
    out = []
    for k in range(len(r)):
        l = int(lv[k])
        H, W = level_hw[l]
        sw, sh, bw, bh, gw, gh, cnt, PP = roi_geom(r[k], scales[l], P, sr, aligned)
        Ax, x0, tx = axis_matrix(sw, bw, PP, gw, W)
        Ay, y0, ty = axis_matrix(sh, bh, PP, gh, H)
        out.append(dict(level=l, x0=x0, ww=Ax.shape[1], y0=y0, hh=Ay.shape[1], xtaps=int(tx.max()), ytaps=int(ty.max())))
    return out


# ----------------------------------------------------------------------------- RoIAlign reference
def _pool_one(Fb: torch.Tensor, Fab: torch.Tensor, roi, scale, P, sr, aligned, pool2, H, W):
    """(value [C,P,P], absbound [C,P,P], coordinate-shift allowance [C,P,P]) of one RoI on one level, float64."""
    sw, sh, bw, bh, gw, gh, cnt, PP = roi_geom(roi, scale, P, sr, aligned, pool2)
    C = Fb.shape[0]
    Ax, x0, _ = axis_matrix(sw, bw, PP, gw, W)
    Ay, y0, _ = axis_matrix(sh, bh, PP, gh, H)
    if Ax.shape[1] == 0 or Ay.shape[1] == 0:
        z = torch.zeros(C, P, P, dtype=torch.float64)
        return z, z.clone(), z.clone()
    ax, ay = torch.from_numpy(Ax), torch.from_numpy(Ay)
    win = Fb[:, y0:y0 + Ay.shape[1], x0:x0 + Ax.shape[1]]
    awin = Fab[:, y0:y0 + Ay.shape[1], x0:x0 + Ax.shape[1]]
    val = ay @ (win @ ax.T) / cnt
    ab = ay @ (awin @ ax.T) / cnt
    grow = (4 * gh * gw + 16) * U32
    if pool2:   # adaptive_avg_pool2d(2P -> P): the mean of each 2x2 block of the 2P x 2P result
        val = val.view(C, P, 2, P, 2).mean(dim=(2, 4))
        ab = ab.view(C, P, 2, P, 2).mean(dim=(2, 4))
        # The kernel pools the level directly at P x P with 2g samples per bin, whose coordinates round differently from
        # these (same real positions): allow each coordinate 8 ulps of the RoI's extent, times the largest weight change
        # that moves (2 max|F| per unit of coordinate on each axis).
        ext = max(abs(float(sw)), abs(float(sh))) + max(float(bw), float(bh)) * PP + 2.0
        shift = 2.0 * 8 * U32 * ext * 2.0 * awin.amax(dim=(1, 2))[:, None, None].expand(C, P, P)
        grow = (16 * gh * gw + 16) * U32        # the kernel sums (2 gh) x (2 gw) samples per output bin
        return val, grow * ab, shift.clone()
    return val, grow * ab, torch.zeros_like(val)


def roi_align_ref64(levels: Sequence[torch.Tensor], rois: torch.Tensor, P: int, scales: Sequence[float], sr: int = 0,
                    aligned: bool = True, mode: str = "route", finest: float = 56.0, bias: Optional[torch.Tensor] = None,
                    pool2: Optional[Sequence[bool]] = None, out_dtype: torch.dtype = torch.float32):
    """float64 (ref [K,C,P,P], tol [K,C,P,P]): the RoIAlign result and the acceptance bound, the largest |out - ref| an
    fp32 kernel with the reference's accumulation may show: per level (4 gh gw + 16) u absbound (+ the coordinate
    allowance of a ``pool2`` level), summed over the levels, + 2 u |bias|, + half an ulp of a 16-bit ``out_dtype``.  ``levels`` [B,C,H_l,W_l] of any
    float dtype are taken exactly (upcast); ``rois`` [K,5] are used as fp32."""
    r = rois.detach().cpu().float().numpy()
    K = len(r)
    L = len(levels)
    lv64 = [f.detach().cpu().double() for f in levels]
    lva = [f.abs() for f in lv64]
    C = lv64[0].shape[1]
    pool2 = list(pool2) if pool2 is not None else [False] * L
    ref = torch.zeros(K, C, P, P, dtype=torch.float64)
    tol = torch.zeros(K, C, P, P, dtype=torch.float64)
    route = route_levels(rois, L, finest) if mode == "route" else None
    for k in range(K):
        b = int(r[k, 0])
        lvls = [int(route[k])] if mode == "route" else range(L)
        for l in lvls:
            H, W = lv64[l].shape[2], lv64[l].shape[3]
            v, t, s = _pool_one(lv64[l][b], lva[l][b], r[k], scales[l], P, sr, aligned, pool2[l], H, W)
            ref[k] += v
            tol[k] += t + s
    if bias is not None:
        bz = bias.detach().cpu().double()[:, :, None, None]
        ref += bz
        tol += 2 * U32 * bz.abs()
    tol += 1e-30
    if out_dtype in (torch.float16, torch.bfloat16):
        tol += half_ulp(ref.abs() + tol, out_dtype)
    return ref, tol


def half_ulp(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """half the spacing of ``dtype`` values at magnitude x (float64 in, float64 out)."""
    fi = torch.finfo(dtype)
    mant = {torch.float16: 10, torch.bfloat16: 7}[dtype]
    e = torch.floor(torch.log2(x.clamp(min=fi.tiny)))
    return torch.exp2(e - mant - 1)


def check(out: torch.Tensor, ref: torch.Tensor, tol: torch.Tensor, what: str = "") -> None:
    """assert |out - ref| <= tol everywhere; the message names the worst element."""
    o = out.detach().cpu().double()
    assert o.shape == ref.shape, (what, tuple(o.shape), tuple(ref.shape))
    err = (o - ref).abs()
    bad = ~(err <= tol)
    if bad.any():
        ratio = torch.where(tol > 0, err / tol, torch.full_like(err, float("inf")))
        i = int(torch.argmax(torch.where(bad, ratio, torch.zeros_like(ratio))))
        idx = np.unravel_index(i, tuple(o.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements out of bound; worst at {tuple(int(j) for j in idx)}: "
                             f"out {o.flatten()[i].item():.9g} ref {ref.flatten()[i].item():.9g} err {err.flatten()[i].item():.3g} "
                             f"bound {tol.flatten()[i].item():.3g}")


# ----------------------------------------------------------------------------- attention pooling reference
def attention_centres(rois: torch.Tensor, stride: float, H: int, W: int):
    """the RoI's centre cell: torch.div(x1 + x2, 2 * stride, rounding_mode='floor') in fp32, clamped to the map."""
    r = rois.detach().cpu().float()
    cx = torch.div(r[:, 1] + r[:, 3], 2 * stride, rounding_mode="floor").clamp(0, W - 1).long()
    cy = torch.div(r[:, 2] + r[:, 4], 2 * stride, rounding_mode="floor").clamp(0, H - 1).long()
    return r[:, 0].long(), cy, cx


def attention_pool_ref64(feat: torch.Tensor, rois: torch.Tensor, stride: float, thres: float):
    """float64 (ref [K,C], tol [K,C]) of AttentionRoIExtractor's pooling of one level (roi_extractors_cus.py:220-238):
    sim = relu(cos(f[b,:,cy,cx], f[b,:,h,w]) - thres) + thres, out = mean_{h,w} f[b,:,h,w] * sim.  Cosine as torch's
    F.cosine_similarity: each norm clamped to eps = 1e-8 separately, then <x1/n1, x2/n2>."""
    f = feat.detach().cpu().double()
    B, C, H, W = f.shape
    HW = H * W
    b, cy, cx = attention_centres(rois, stride, H, W)
    ref = torch.zeros(len(b), C, dtype=torch.float64)
    tol = torch.zeros_like(ref)
    for i in range(B):
        sel = (b == i).nonzero().flatten()
        if len(sel) == 0:
            continue
        pos = f[i].reshape(C, HW).T                                         # [HW, C]
        vec = f[i][:, cy[sel], cx[sel]].T                                   # [k, C]
        cos = (vec / vec.norm(dim=1, keepdim=True).clamp(min=1e-8)) @ (pos / pos.norm(dim=1, keepdim=True).clamp(min=1e-8)).T
        sim = F.relu(cos - thres) + thres                                   # [k, HW]
        ref[sel] = sim @ pos / HW
        apos = pos.abs()
        tol[sel] = U32 * ((HW + 4) * (sim.abs() @ apos) / HW + (C + 8) * apos.mean(dim=0)[None, :])
    return ref, tol + 1e-30


def attention_extractor_ref64(feats: Sequence[torch.Tensor], rois: torch.Tensor, strides: Sequence[int], P: int, sr: int,
                              start_level: int = 2, thres: float = 0.0):
    """AttentionRoIExtractor (aggregation='sum', roi_extractors_cus.py:195-259) composed from the two references: the
    RoIAlign sum of the levels below ``start_level`` plus, broadcast over the bins, the attention pooling of the others
    (level stride 4 * 2**i as the reference hard-codes it).  float64 (ref, tol)."""
    pooled = [i for i in range(len(feats)) if i < start_level]
    bias = torch.zeros(rois.shape[0], feats[0].shape[1], dtype=torch.float64)
    btol = torch.zeros_like(bias)
    for i in range(start_level, len(feats)):
        a, t = attention_pool_ref64(feats[i], rois, 4 * 2 ** i, thres)
        bias += a
        btol += t + U32 * bias.abs()            # the running fp32 sum of the levels' vectors
    ref, tol = roi_align_ref64([feats[i] for i in pooled], rois, P, [1.0 / strides[i] for i in pooled], sr, mode="sum")
    return ref + bias[:, :, None, None], tol + (btol + 2 * U32 * bias.abs())[:, :, None, None]
