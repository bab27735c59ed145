// Multi-level RoIAlign forward for sm_100a.
//
// Replaces mmcv-full 1.7.2 `roi_align_forward` (avg pool) as driven per FPN level by
//   /root/reference/thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:58-115
//   /root/reference/nuhtc/models/roi_extractors_cus.py:195-218,246
// with ONE launch that covers every level (per-RoI level routing, or level sum).
//
// Two kernels:
//  * roi_align_sep_kernel  -- the fast path.  RoIAlign's sample grid is a tensor product, so
//      out[ph][pw] = sum_y sum_x Wy[ph][y] * Wx[pw][x] * V[y][x]     (avg pool, bilinear)
//    with per-bin tap weights Wx/Wy that depend only on the RoI.  A CTA owns (RoI, channel chunk);
//    the tap tables are built once per RoI in shared memory ("staging of sampling coordinates"),
//    every thread then owns 4 contiguous channels (one 128-bit NHWC gather per tap) and one output
//    column pw, sweeps the window rows once, and keeps its P outputs in registers.  The [CC,P,P]
//    result is transposed through shared memory and leaves as coalesced 128-bit streaming stores
//    of the contiguous NCHW chunk.  Reads per RoI drop from 4*gh*gw*P*P to (rows * x-taps) per
//    column, which is what lets the kernel run at the HBM write rate instead of the L1 rate.
//  * roi_align_direct_kernel -- literal per-sample restatement (any layout / shape), same float op
//    order as the CPU reference; used as fallback and as an on-device cross-check.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "roi_common.cuh"
#include "roi_strip.cuh"

// ---------------------------------------------------------------------------------------------
// literal kernel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float direct_one(const float *plane, long sy, long sx, int H, int W, const RoiGeom &g,
                                            int ph, int pw) {
    float acc = 0.f;
    for (int iy = 0; iy < g.gh; ++iy) {
        const float y = sample_coord(g.start_h, g.bin_h, ph, iy, g.gh);
        for (int ix = 0; ix < g.gw; ++ix) {
            const float x = sample_coord(g.start_w, g.bin_w, pw, ix, g.gw);
            int yl, yh, xl, xh;
            float ly, hy, lx, hx;
            // the reference rejects the sample if EITHER axis is out of range
            const bool oky = axis_sample(y, H, yl, yh, ly, hy);
            const bool okx = axis_sample(x, W, xl, xh, lx, hx);
            if (!(oky && okx)) continue;
            const float w1 = __fmul_rn(hy, hx), w2 = __fmul_rn(hy, lx), w3 = __fmul_rn(ly, hx), w4 = __fmul_rn(ly, lx);
            const float v1 = __ldg(plane + yl * sy + xl * sx), v2 = __ldg(plane + yl * sy + xh * sx);
            const float v3 = __ldg(plane + yh * sy + xl * sx), v4 = __ldg(plane + yh * sy + xh * sx);
            const float s = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, v1), __fmul_rn(w2, v2)), __fmul_rn(w3, v3)),
                                      __fmul_rn(w4, v4));
            acc = __fadd_rn(acc, s);
        }
    }
    return __fdiv_rn(acc, g.count);
}

__global__ void __launch_bounds__(256) roi_align_direct_kernel(RoiLevels lv, int C, int layout, const float *__restrict__ rois,
                                                               long total, int PH, int PW, int sr, int aligned, int mode,
                                                               float finest, float *__restrict__ out, const float *__restrict__ bias) {
    for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int pw = (int)(idx % PW);
        const int ph = (int)((idx / PW) % PH);
        const int c = (int)((idx / ((long)PW * PH)) % C);
        const long k = idx / ((long)PW * PH * C);
        const float *roi = rois + k * 5;
        float r = 0.f;
        int l0 = 0, l1 = lv.L;
        if (mode == NUHTC_ROI_ROUTE) {
            l0 = route_level(roi, lv.L, finest);
            l1 = l0 + 1;
        }
        for (int l = l0; l < l1; ++l) {
            const int H = lv.H[l], W = lv.W[l];
            const RoiGeom g = roi_geom(roi, lv.scale[l], PH, PW, sr, aligned, lv.pool2[l]);
            const float *plane;
            long sy, sx;
            if (layout == NUHTC_LAYOUT_NCHW) {
                plane = lv.data[l] + ((long)g.b * C + c) * H * W;
                sy = W;
                sx = 1;
            } else {
                plane = lv.data[l] + (long)g.b * H * W * C + c;
                sy = (long)W * C;
                sx = C;
            }
            const float f = direct_one(plane, sy, sx, H, W, g, ph, pw);
            r = (mode == NUHTC_ROI_ROUTE) ? f : __fadd_rn(r, f);
        }
        out[idx] = bias ? __fadd_rn(r, __ldg(bias + k * C + c)) : r;
    }
}

// ---------------------------------------------------------------------------------------------
// separable fast kernel (NHWC input)
// ---------------------------------------------------------------------------------------------
template <int P>
struct SepCfg {
    static constexpr int PP = P * P;
    // channel stride of the staging tile: == 1 (mod 8) makes the rotated column writes conflict-free
    static constexpr int S = (PP % 8 == 1) ? PP : (PP + ((9 - PP % 8) % 8));
};

// One sweep over the window rows [y0, y1) for a thread that owns output column pw (NX x-taps starting at
// the pointer) and PB output rows: t = sum_j wx[j] * V[y][xs+j] per row, then acc[i] += wy[i][y-ys[i]] * t.
// pix = float stride between neighbouring pixels (C for NHWC, 32 for the channel-group layout), slice = float stride
// between the VEC channel slices of a thread.
template <int NX, int PB, int VEC>
__device__ __forceinline__ void sweep_rows(const float *__restrict__ rowp, size_t rstride, size_t pix, size_t slice, int y0, int y1,
                                           const float *__restrict__ s_wxp, const float *__restrict__ s_wyp, const int (&ys)[PB],
                                           const int (&ny)[PB], float2 (&acc)[PB][VEC][2], int nx_rt = 0) {
    constexpr int NXR = NX > 0 ? NX : 1;
    float wx[NXR];
#pragma unroll
    for (int j = 0; j < NX; ++j) wx[j] = s_wxp[j];
#pragma unroll 2
    for (int y = y0; y < y1; ++y, rowp += rstride) {
        float2 t[VEC][2];
#pragma unroll
        for (int u = 0; u < VEC; ++u) {
            t[u][0] = make_float2(0.f, 0.f);
            t[u][1] = make_float2(0.f, 0.f);
        }
        if (NX > 0) {
            // all NX*VEC gathers are issued before the first FMA consumes one
            float4 v[NXR][VEC];
#pragma unroll
            for (int j = 0; j < NX; ++j)
#pragma unroll
                for (int u = 0; u < VEC; ++u) v[j][u] = ldg_f4(rowp + (size_t)j * pix + u * slice);
#pragma unroll
            for (int j = 0; j < NX; ++j)
#pragma unroll
                for (int u = 0; u < VEC; ++u) {
                    t[u][0] = ffma2(wx[j], make_float2(v[j][u].x, v[j][u].y), t[u][0]);
                    t[u][1] = ffma2(wx[j], make_float2(v[j][u].z, v[j][u].w), t[u][1]);
                }
        } else {
            // wide bins (5..kMaxTap taps): runtime tap count, weights from shared memory
#pragma unroll 2
            for (int j = 0; j < nx_rt; ++j) {
                const float w = s_wxp[j];
#pragma unroll
                for (int u = 0; u < VEC; ++u) {
                    const float4 vv = ldg_f4(rowp + (size_t)j * pix + u * slice);
                    t[u][0] = ffma2(w, make_float2(vv.x, vv.y), t[u][0]);
                    t[u][1] = ffma2(w, make_float2(vv.z, vv.w), t[u][1]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < PB; ++i) {
            const int jj = y - ys[i];
            if ((unsigned)jj < (unsigned)ny[i]) {
                const float w = s_wyp[i * kMaxTap + jj];
#pragma unroll
                for (int u = 0; u < VEC; ++u) {
                    acc[i][u][0] = ffma2(w, t[u][0], acc[i][u][0]);
                    acc[i][u][1] = ffma2(w, t[u][1], acc[i][u][1]);
                }
            }
        }
    }
}

// P output size; NQ channel quads per VEC slice; PHS: the P output rows are split over PHS thread groups;
// VEC: float4 slices per thread (a thread owns channels 4q..4q+3 of each slice).  CTA = (RoI, CC channels).
// OutT: output element type; the tile stays fp32 and every value is rounded once on its way out.
template <int P, int NQ, int PHS, int VEC, int MINB, typename OutT>
__global__ void __launch_bounds__(NQ *P *PHS, MINB) roi_align_sep_kernel(RoiLevels lv, int C, const float *__restrict__ rois, int sr,
                                                                    int aligned, int mode, float finest,
                                                                    OutT *__restrict__ out, const float *__restrict__ bias,
                                                                    int cg32, const int *__restrict__ list,
                                                                    const int *__restrict__ list_count) {
    constexpr int CC = NQ * 4 * VEC;
    constexpr int PP = SepCfg<P>::PP;
    constexpr int S = SepCfg<P>::S;
    constexpr int NT = NQ * P * PHS;
    constexpr int PB = P / PHS;
    static_assert(P % PHS == 0, "row split must divide P");
    static_assert(NT >= 32 + P, "tap builders sit on warps 0 and 1");
    extern __shared__ __align__(128) float smem[];
    float *s_tile = smem;                // [CC][S]
    float *s_wx = s_tile + CC * S;       // [P][kMaxTap]
    float *s_wy = s_wx + P * kMaxTap;    // [P][kMaxTap], already divided by the sample count
    int *s_xs = (int *)(s_wy + P * kMaxTap);
    int *s_nx = s_xs + P;
    int *s_ys = s_nx + P;
    int *s_ny = s_ys + P;
    int *s_meta = s_ny + P;              // [0] level, [1] batch index

    // with a RoI list (the strip kernel's leftovers: windows too large to stage) a small grid walks the device-side list
    const int n_items = list ? *list_count : (int)gridDim.x;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    if (item != (int)blockIdx.x) __syncthreads();   // the previous item's tile and tables are still being read
    const int k = list ? list[item] : item;
    const int c0 = blockIdx.y * CC;
    const int tid = threadIdx.x;
    const int q = tid % NQ;
    const int pw = (tid / NQ) % P;
    const int ph0 = (tid / (NQ * P)) * PB; // first output row owned by this thread
    const float *roi = rois + (size_t)k * 5;

    float2 acc[PB][VEC][2];
#pragma unroll
    for (int i = 0; i < PB; ++i)
#pragma unroll
        for (int u = 0; u < VEC; ++u) acc[i][u][0] = acc[i][u][1] = make_float2(0.f, 0.f);

    const int nlev = mode == NUHTC_ROI_ROUTE ? 1 : lv.L;
    for (int it = 0; it < nlev; ++it) {
        if (it) __syncthreads(); // the previous level's tables are still being read
        // ---- phase A: the RoI geometry and the tap tables are computed by 2P threads only (x bins on warp 0,
        // y bins on warp 1); everybody else waits at the barrier instead of redoing the divisions
        const bool xb = tid < P, yb = tid >= 32 && tid < 32 + P;
        if (xb || yb) {
            const int l = mode == NUHTC_ROI_ROUTE ? route_level(roi, lv.L, finest) : it;
            const RoiGeom g = roi_geom(roi, lv.scale[l], P, P, sr, aligned, lv.pool2[l]);
            if (xb) {
                build_axis_taps(g.start_w, g.bin_w, g.gw, tid, lv.W[l], 1.0f, s_wx + tid * kMaxTap, s_xs + tid, s_nx + tid);
                if (tid == 0) {
                    s_meta[0] = l;
                    s_meta[1] = g.b;
                }
            } else {
                const int p = tid - 32;
                build_axis_taps(g.start_h, g.bin_h, g.gh, p, lv.H[l], g.count, s_wy + p * kMaxTap, s_ys + p, s_ny + p);
            }
        }
        __syncthreads();
        const int l = s_meta[0], b = s_meta[1];
        const int H = lv.H[l], W = lv.W[l];
        const int nx = s_nx[pw];
        int ys[PB], ny[PB];
        bool slow = nx < 0;
        int y0 = 1 << 30, y1 = -1;
#pragma unroll
        for (int i = 0; i < PB; ++i) {
            ys[i] = s_ys[ph0 + i];
            ny[i] = s_ny[ph0 + i];
            slow = slow || ny[i] < 0;
            if (ny[i] > 0) {
                y0 = min(y0, ys[i]);
                y1 = max(y1, ys[i] + ny[i]);
            }
        }
        // NHWC: [b][y][x][C]; channel-group layout: [b][C/32][y][x][32] (the thread's quad never straddles a group)
        const int cq = c0 + 4 * q;
        const size_t plane = (size_t)H * W * 32;
        const size_t pix = cg32 ? 32 : (size_t)C;
        const size_t slice = cg32 ? (size_t)(NQ * 4 / 32) * plane : (size_t)NQ * 4;
        const float *img = cg32 ? lv.data[l] + (size_t)b * H * W * C + (size_t)(cq >> 5) * plane + (cq & 31)
                                : lv.data[l] + (size_t)b * H * W * C + cq;
        if (!slow) {
            if (nx > 0 && y1 > y0) {
                const float *rowp = img + ((size_t)y0 * W + s_xs[pw]) * pix;
                const size_t rstride = (size_t)W * pix;
                const float *wxp = s_wx + pw * kMaxTap, *wyp = s_wy + ph0 * kMaxTap;
                switch (nx) {
                    case 1: sweep_rows<1, PB, VEC>(rowp, rstride, pix, slice, y0, y1, wxp, wyp, ys, ny, acc); break;
                    case 2: sweep_rows<2, PB, VEC>(rowp, rstride, pix, slice, y0, y1, wxp, wyp, ys, ny, acc); break;
                    case 3: sweep_rows<3, PB, VEC>(rowp, rstride, pix, slice, y0, y1, wxp, wyp, ys, ny, acc); break;
                    case 4: sweep_rows<4, PB, VEC>(rowp, rstride, pix, slice, y0, y1, wxp, wyp, ys, ny, acc); break;
                    default: sweep_rows<0, PB, VEC>(rowp, rstride, pix, slice, y0, y1, wxp, wyp, ys, ny, acc, nx); break;
                }
            }
        } else {
            // ---- a bin of this thread is wider than the tap table (very large RoI): literal per-sample path
            const RoiGeom g = roi_geom(roi, lv.scale[l], P, P, sr, aligned, lv.pool2[l]);
#pragma unroll 1
            for (int pi = 0; pi < PB; ++pi) {
                const int ph = ph0 + pi;
                float a[VEC][4];
#pragma unroll
                for (int u = 0; u < VEC; ++u) a[u][0] = a[u][1] = a[u][2] = a[u][3] = 0.f;
                for (int iy = 0; iy < g.gh; ++iy) {
                    int yl, yh;
                    float ly, hy;
                    const bool oky = axis_sample(sample_coord(g.start_h, g.bin_h, ph, iy, g.gh), H, yl, yh, ly, hy);
                    for (int ix = 0; ix < g.gw; ++ix) {
                        int xl, xh;
                        float lx, hx;
                        const bool okx = axis_sample(sample_coord(g.start_w, g.bin_w, pw, ix, g.gw), W, xl, xh, lx, hx);
                        if (!(oky && okx)) continue;
                        const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;
#pragma unroll
                        for (int u = 0; u < VEC; ++u) {
                            const float *pu = img + u * slice;
                            const float4 v1 = ldg_f4(pu + ((size_t)yl * W + xl) * pix), v2 = ldg_f4(pu + ((size_t)yl * W + xh) * pix);
                            const float4 v3 = ldg_f4(pu + ((size_t)yh * W + xl) * pix), v4 = ldg_f4(pu + ((size_t)yh * W + xh) * pix);
                            a[u][0] += w1 * v1.x + w2 * v2.x + w3 * v3.x + w4 * v4.x;
                            a[u][1] += w1 * v1.y + w2 * v2.y + w3 * v3.y + w4 * v4.y;
                            a[u][2] += w1 * v1.z + w2 * v2.z + w3 * v3.z + w4 * v4.z;
                            a[u][3] += w1 * v1.w + w2 * v2.w + w3 * v3.w + w4 * v4.w;
                        }
                    }
                }
                // acc is indexed statically: fold this bin into the matching registers
#pragma unroll
                for (int pp = 0; pp < PB; ++pp) {
                    if (pp == pi) {
#pragma unroll
                        for (int u = 0; u < VEC; ++u) {
                            acc[pp][u][0].x += __fdiv_rn(a[u][0], g.count);
                            acc[pp][u][0].y += __fdiv_rn(a[u][1], g.count);
                            acc[pp][u][1].x += __fdiv_rn(a[u][2], g.count);
                            acc[pp][u][1].y += __fdiv_rn(a[u][3], g.count);
                        }
                    }
                }
            }
        }
    }

    // ---- transpose [channels of this thread][ph][pw] into the [CC][S] staging tile.
    // Lanes of a warp hold consecutive channel quads (stride 4*S words == 4 mod 32), so the four
    // channels are written in a lane-rotated order that spreads the 32 lanes over all 32 banks.
    const int lane = tid & 31;
    const int rot = (lane >> 3) - (lane / NQ);
#pragma unroll
    for (int i = 0; i < PB; ++i) {
#pragma unroll
        for (int u = 0; u < VEC; ++u) {
            float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
            if (bias) bz = ldg_f4(bias + (size_t)k * C + c0 + u * NQ * 4 + 4 * q);
            const float a0 = acc[i][u][0].x + bz.x, a1 = acc[i][u][0].y + bz.y, a2 = acc[i][u][1].x + bz.z, a3 = acc[i][u][1].y + bz.w;
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int j = (jj + rot) & 3;
                const float v = j == 0 ? a0 : (j == 1 ? a1 : (j == 2 ? a2 : a3));
                s_tile[(u * NQ * 4 + 4 * q + j) * S + (ph0 + i) * P + pw] = v;
            }
        }
    }
    __syncthreads();
    OutT *outp = out + ((size_t)k * C + c0) * PP;
    constexpr int N4 = CC * PP / 4;
    for (int i = tid; i < N4; i += NT) {
        float4 v;
        if (S == PP) {
            v = *reinterpret_cast<const float4 *>(s_tile + 4 * i);
        } else {
            int c = (4 * i) / PP, e = 4 * i - c * PP;
            float t[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                t[u] = s_tile[c * S + e];
                if (++e == PP) {
                    e = 0;
                    ++c;
                }
            }
            v = make_float4(t[0], t[1], t[2], t[3]);
        }
        st_stream4(outp + 4 * i, to_out<OutT>(v.x), to_out<OutT>(v.y), to_out<OutT>(v.z), to_out<OutT>(v.w));
    }
    }   // item loop
}

template <int P, int NQ, int VEC>
static size_t sep_smem_bytes() {
    return sizeof(float) * (NQ * 4 * VEC * SepCfg<P>::S + 2 * P * kMaxTap) + sizeof(int) * (4 * P + 4);
}

template <int P, int NQ, int PHS, int VEC, int MINB, typename OutT>
static int launch_sep(const RoiLevels &lv, int C, const float *rois, int K, int sr, int aligned, int mode, float finest,
                      OutT *out, const float *bias, cudaStream_t st, int cg32 = 0, const int *list = nullptr,
                      const int *list_count = nullptr) {
    static bool attr_done[kNuhtcMaxDevices] = {false};
    const int dev = nuhtc_device();
    const size_t smem = sep_smem_bytes<P, NQ, VEC>();
    if (!attr_done[dev]) {
        NUHTC_CUDA(cudaFuncSetAttribute(roi_align_sep_kernel<P, NQ, PHS, VEC, MINB, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    // every RoI: one CTA each; a RoI list: a resident grid that walks the list (its length is only known on the device)
    const int gx = list ? (K < 4 * nuhtc_sm_count() ? K : 4 * nuhtc_sm_count()) : K;
    dim3 grid(gx, C / (NQ * 4 * VEC));
    roi_align_sep_kernel<P, NQ, PHS, VEC, MINB, OutT><<<grid, NQ * P * PHS, smem, st>>>(lv, C, rois, sr, aligned, mode, finest, out, bias,
                                                                                  cg32, list, list_count);
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}

// ---------------------------------------------------------------------------------------------
// pipelined fast kernel: persistent CTAs, one producer warp + NQ*P*PHS consumer threads
// ---------------------------------------------------------------------------------------------
// The v2 kernel above exposes one L2 round trip per window row to every consumer warp.  Here a producer
// warp runs ahead of the consumers: for every work item (RoI, channel chunk, level) it builds the tap
// tables into a double-buffered slot and streams the window rows [y0,y1) x [x0,x0+ww) of the NHWC level
// into a shared-memory ring with TMA bulk copies (cp.async.bulk, completion on an mbarrier).  The consumer
// warps wait on the row's "full" barrier, take their taps with conflict-free LDS.128, and release the
// row to the producer through its "empty" barrier.  Window rows wider than the ring stage, or bins with
// more than kMaxTap taps, fall back to the direct global-load sweep of the v2 kernel inside the same CTA.
constexpr int kPipeMaxRows = 40; // staged windows taller than this take the direct path

// 2-D TMA tensor maps of the NHWC levels: dim0 = channels, dim1 = pixels (B*H*W); box = {CC channels, WBOX pixels}.
// They let a CTA that owns only CC of the C channels fetch a window row with ONE instruction (cp.async.bulk.tensor,
// UTMALDG) instead of one small bulk copy per pixel.
constexpr int kTmapLevels = 4;
constexpr int kTmapBoxes = 4;
__host__ __device__ constexpr int tmap_box_px(int v) { return 8 * (v + 1); } // 8, 16, 24, 32 pixels
struct RoiTmaps {
    CUtensorMap m[kTmapLevels][kTmapBoxes];
};
__device__ __forceinline__ void tma_tensor2d_g2s(uint32_t dst, const CUtensorMap *map, int c0, int p0, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(map), "r"(c0), "r"(p0), "r"(bar)
                 : "memory");
}

template <int P>
struct PipeSlot { // tap tables + geometry of one work item
    float wx[P][kMaxTap];
    float wy[P][kMaxTap]; // already divided by the sample count
    int xs[P], nx[P], ys[P], ny[P];
    int mode;   // 0 staged rows, 1 direct global sweep, 2 literal (a bin exceeds the tap table)
    int x0, ww; // staged column range
    int y0, y1; // window rows
    int level, batch, k, c0, last, pad0, pad1;
    // dense y weights of the staged rows: wyd[y - y0][bin] (0 where the bin does not touch the row), 8 floats per
    // group of up to 7 bins so that a consumer takes its weights of a row with two LDS.128 and no compares
    float wyd[kPipeMaxRows][(P + 6) / 7 * 8];
};

enum { kPipeStaged = 0, kPipeDirect = 1, kPipeLiteral = 2 };
constexpr int kPipeSlots = 4;

// position in the row ring: stage index and the parity of its current use
struct RingPos {
    unsigned stage, parity;
    template <int NS>
    __device__ __forceinline__ void next() {
        if (++stage == NS) {
            stage = 0;
            parity ^= 1u;
        }
    }
};

// consumer: staged rows for a thread with NX x-taps (NX == 0: runtime count, weights from the slot) and PB (<= 14)
// output rows whose dense weights sit at wyd[row][0..7] (rows 0..6) and wyd[row][8..15] (rows 7..13)
template <int NX, int PB, int NS, int WYS>
__device__ __forceinline__ void staged_rows(const float *ring, int stage_floats, int pixs, int y0, int y1, int toff,
                                            const float *s_wxp, const float *s_wyd, float2 (&acc)[PB][1][2], uint32_t full0,
                                            uint32_t empty0, RingPos &rp, int nx_rt, int my0, int my1) {
    constexpr int NXR = NX > 0 ? NX : 1;
    float wx[NXR];
#pragma unroll
    for (int j = 0; j < NX; ++j) wx[j] = s_wxp[j];
    const int lane = threadIdx.x & 31;
    for (int y = y0; y < y1; ++y, s_wyd += WYS) {
        mbar_wait(full0 + 8 * rp.stage, rp.parity);
        if (y >= my0 && y < my1) {
            const float *row = ring + (size_t)rp.stage * stage_floats + toff; // toff: the thread's first tap of this row
            float2 t0 = make_float2(0.f, 0.f), t1 = make_float2(0.f, 0.f);
            if (NX > 0) {
#pragma unroll
                for (int j = 0; j < NX; ++j) {
                    const float4 v = *reinterpret_cast<const float4 *>(row + (size_t)j * pixs);
                    t0 = ffma2(wx[j], make_float2(v.x, v.y), t0);
                    t1 = ffma2(wx[j], make_float2(v.z, v.w), t1);
                }
            } else {
                for (int j = 0; j < nx_rt; ++j) {
                    const float4 v = *reinterpret_cast<const float4 *>(row + (size_t)j * pixs);
                    const float w = s_wxp[j];
                    t0 = ffma2(w, make_float2(v.x, v.y), t0);
                    t1 = ffma2(w, make_float2(v.z, v.w), t1);
                }
            }
            constexpr int NG = (PB + 6) / 7; // groups of up to 7 output rows, 8 weight floats each
            float w[NG * 8];
#pragma unroll
            for (int gI = 0; gI < NG; ++gI) {
                const float4 wa = *reinterpret_cast<const float4 *>(s_wyd + 8 * gI), wb = *reinterpret_cast<const float4 *>(s_wyd + 8 * gI + 4);
                w[8 * gI + 0] = wa.x; w[8 * gI + 1] = wa.y; w[8 * gI + 2] = wa.z; w[8 * gI + 3] = wa.w;
                w[8 * gI + 4] = wb.x; w[8 * gI + 5] = wb.y; w[8 * gI + 6] = wb.z; w[8 * gI + 7] = wb.w;
            }
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                acc[i][0][0] = ffma2(w[i / 7 * 8 + i % 7], t0, acc[i][0][0]);
                acc[i][0][1] = ffma2(w[i / 7 * 8 + i % 7], t1, acc[i][0][1]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8 * rp.stage);
        rp.next<NS>();
    }
}

// Warp roles: [0, NCONS) consumers, warp NCONS/32 builds tap tables (kPipeSlots items ahead), warp NCONS/32+1 streams rows.
// OutT: output element type; values are rounded to it in registers, so the tile and the bulk store hold OutT.
template <int P, int NQ, int PHS, int NS, int WMAX, int MINB, typename OutT>
__global__ void __launch_bounds__((NQ *P *PHS + 31) / 32 * 32 + 64, MINB)
    roi_align_pipe_kernel(RoiLevels lv, int C, const float *__restrict__ rois, int K, int sr, int aligned, int mode, float finest,
                          OutT *__restrict__ out, const float *__restrict__ bias, int bulk_store_flag,
                          const __grid_constant__ RoiTmaps tm, int cg32, const int *__restrict__ list,
                          const int *__restrict__ list_count) {
    constexpr int CC = NQ * 4;
    constexpr int PP = SepCfg<P>::PP;
    // tile stride: the padded one is conflict-free for the transposition; the dense one (== PP) leaves as ONE asynchronous
    // bulk store.  P = 14 with 128-channel chunks takes the dense stride although its transposition then is 4-way
    // conflicted (channel rows must stay 16-byte aligned for the bulk copy): the store overlaps the next chunk's rows.
    constexpr bool kDenseTile = (P == 14 && NQ == 32);
    constexpr int S = kDenseTile ? PP : SepCfg<P>::S;
    const bool kBulkStore = (S == PP) && (bulk_store_flag & 1) != 0;            // contiguous tile == contiguous global chunk
    constexpr int NWORK = NQ * P * PHS;              // consumer threads that own outputs
    constexpr int NCONS = (NWORK + 31) / 32 * 32;    // padded to whole warps: the tail threads only keep the barriers company
    constexpr int CONS_WARPS = NCONS / 32;
    constexpr int PB = P / PHS;
    constexpr int STAGE_FLOATS = WMAX * CC;
    static_assert(P <= 16, "x bins on lanes 0..15, y bins on lanes 16..31 of the tap warp");
    extern __shared__ __align__(128) float smem[];
    float *s_ring = smem;                                   // [NS][WMAX][CC]
    float *s_tile_raw = s_ring + (size_t)NS * STAGE_FLOATS; // [CC][S] OutT (sized for fp32)
    OutT *s_tile = reinterpret_cast<OutT *>(s_tile_raw);
    PipeSlot<P> *s_slot = reinterpret_cast<PipeSlot<P> *>(s_tile_raw + CC * S); // [kPipeSlots]
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_slot + kPipeSlots);    // full[NS], empty[NS], tfull[slots], tempty[slots]
    const uint32_t full0 = smem_u32(s_bar), empty0 = full0 + 8 * NS, tfull0 = empty0 + 8 * NS, tempty0 = tfull0 + 8 * kPipeSlots;

    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < NS; ++s) {
            mbar_init(full0 + 8 * s, 1);
            mbar_init(empty0 + 8 * s, CONS_WARPS);
        }
        for (int s = 0; s < kPipeSlots; ++s) {
            mbar_init(tfull0 + 8 * s, 32);
            mbar_init(tempty0 + 8 * s, CONS_WARPS + 1); // every consumer warp + the copy warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int nchunk = C / CC;
    const int nlev = mode == NUHTC_ROI_ROUTE ? 1 : lv.L;
    // a unit = one RoI (of the device-side list when there is one: the strip kernel's leftovers): its levels are consecutive
    // items, its channel chunks share the item's tables (nchunk > 1 is only launched with nlev == 1)
    const long nunits = list ? *list_count : K;
    // channel-group layout [b][C/32][y][x][32]: a stage holds the CC/32 groups of a row one after the other, [g][WMAX][32]
    constexpr int GPC = CC / 32 > 0 ? CC / 32 : 1;
    unsigned itemctr = 0;
    constexpr int WYS = (P + 6) / 7 * 8;
    static_assert(PB <= 7 || (PB == P && P <= 14), "a consumer owns at most 7 output rows, or all of them");

    if (tid >= NCONS + 32) {
        // =========================== copy warp: streams the window rows of every staged item ===========================
        const int lane = tid - NCONS - 32;
        RingPos rp{0u, 0u};
        for (long unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
            for (int it = 0; it < nlev; ++it, ++itemctr) {
                const unsigned slot = itemctr % kPipeSlots, use = itemctr / kPipeSlots;
                mbar_wait(tfull0 + 8 * slot, use & 1);
                const PipeSlot<P> &sl = s_slot[slot];
                const int md = sl.mode, x0 = sl.x0, ww = sl.ww, y0 = sl.y0, y1 = sl.y1, l = sl.level, b = sl.batch;
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty0 + 8 * slot); // the slot's geometry is in registers now
                if (md == kPipeStaged && y1 > y0) {
                    const int H = lv.H[l], W = lv.W[l];
                    const size_t rstride = (size_t)W * C;
                    const int bv = (ww + 7) / 8 - 1; // smallest tensor-map box that covers the row
                    for (int chunk = 0; chunk < nchunk; ++chunk) {
                        const int c0 = chunk * CC;
                        const float *src0 = lv.data[l] + (((size_t)b * H + y0) * W + x0) * (size_t)C + c0;
                        const int pix0 = (b * H + y0) * W + x0;
                        // channel-group layout: lane g < GPC copies the row segment of group chunk*GPC + g (ww * 128 contiguous bytes)
                        const float *srcg = lv.data[l] + ((((size_t)b * (C / 32) + chunk * GPC + (lane < GPC ? lane : 0)) * H + y0) * W + x0) * 32;
                        for (int y = y0; y < y1; ++y, rp.next<NS>()) {
                            const unsigned stage = rp.stage;
                            mbar_wait(empty0 + 8 * stage, rp.parity ^ 1u);
                            const uint32_t dst = smem_u32(s_ring + (size_t)stage * STAGE_FLOATS);
                            if (cg32) {
                                if (lane == 0) mbar_arrive_expect_tx(full0 + 8 * stage, (uint32_t)ww * 128u * GPC);
                                __syncwarp();
                                if (lane < GPC)
                                    tma_bulk_g2s(dst + (uint32_t)lane * WMAX * 128u, srcg + (size_t)(y - y0) * W * 32, (uint32_t)ww * 128u,
                                                 full0 + 8 * stage);
                            } else if (lane == 0) {
                                if (nchunk == 1) { // the row segment is contiguous in NHWC: one plain bulk copy
                                    mbar_arrive_expect_tx(full0 + 8 * stage, (uint32_t)ww * CC * 4);
                                    tma_bulk_g2s(dst, src0 + (size_t)(y - y0) * rstride, (uint32_t)ww * CC * 4, full0 + 8 * stage);
                                } else {           // CC of the C channels: one 2-D tensor copy of {CC, box} elements
                                    mbar_arrive_expect_tx(full0 + 8 * stage, (uint32_t)tmap_box_px(bv) * CC * 4);
                                    tma_tensor2d_g2s(dst, &tm.m[l][bv], c0, pix0 + (y - y0) * W, full0 + 8 * stage);
                                }
                            }
                        }
                    }
                }
            }
        }
        return;
    }
    if (tid >= NCONS) {
        // =========================== tap warp: tables + window geometry, kPipeSlots items ahead ===========================
        const int lane = tid - NCONS;
        for (long unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
            const int k = list ? list[unit] : (int)unit;
            const float *roi = rois + (size_t)k * 5;
            for (int it = 0; it < nlev; ++it, ++itemctr) {
                const unsigned slot = itemctr % kPipeSlots, use = itemctr / kPipeSlots;
                mbar_wait(tempty0 + 8 * slot, (use & 1) ^ 1);
                PipeSlot<P> &sl = s_slot[slot];
                const int l = mode == NUHTC_ROI_ROUTE ? route_level(roi, lv.L, finest) : it;
                const RoiGeom g = roi_geom(roi, lv.scale[l], P, P, sr, aligned, lv.pool2[l]);
                const int H = lv.H[l], W = lv.W[l];
                int first = 0, n = 0;
                if (lane < P) {
                    build_axis_taps(g.start_w, g.bin_w, g.gw, lane, W, 1.0f, sl.wx[lane], &first, &n);
                    sl.xs[lane] = first;
                    sl.nx[lane] = n;
                } else if (lane >= 16 && lane < 16 + P) {
                    build_axis_taps(g.start_h, g.bin_h, g.gh, lane - 16, H, g.count, sl.wy[lane - 16], &first, &n);
                    sl.ys[lane - 16] = first;
                    sl.ny[lane - 16] = n;
                }
                // window = union of the bins' tap ranges: reductions over the x half (lanes 0..15) and the y half (16..31)
                const bool has = ((lane < P) || (lane >= 16 && lane < 16 + P)) && n > 0;
                const bool bad = ((lane < P) || (lane >= 16 && lane < 16 + P)) && n < 0;
                int lo = has ? first : (1 << 30), hi = has ? first + n : -1;
#pragma unroll
                for (int o = 8; o; o >>= 1) {
                    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
                    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
                }
                const int x0 = __shfl_sync(0xffffffffu, lo, 0), x1 = __shfl_sync(0xffffffffu, hi, 0);
                const int y0 = __shfl_sync(0xffffffffu, lo, 16), y1 = __shfl_sync(0xffffffffu, hi, 16);
                const bool lit = __any_sync(0xffffffffu, bad);
                const bool empty = x1 <= x0 || y1 <= y0;
                const int ww = empty ? 0 : x1 - x0;
                const bool staged = !lit && ww <= WMAX && (empty || y1 - y0 <= kPipeMaxRows);
                if (staged && !empty) {
                    // dense y weights: lane r owns window rows r, r+32
                    __syncwarp(); // the bin lanes' wy / ys / ny are in the slot
                    for (int r = lane; r < y1 - y0; r += 32) {
                        float w[WYS];
#pragma unroll
                        for (int i = 0; i < WYS; ++i) w[i] = 0.f;
#pragma unroll
                        for (int p = 0; p < P; ++p) {
                            const int jj = y0 + r - sl.ys[p];
                            if ((unsigned)jj < (unsigned)sl.ny[p]) w[p / 7 * 8 + p % 7] = sl.wy[p][jj];
                        }
#pragma unroll
                        for (int i = 0; i < WYS; i += 4)
                            *reinterpret_cast<float4 *>(&sl.wyd[r][i]) = make_float4(w[i], w[i + 1], w[i + 2], w[i + 3]);
                    }
                }
                if (lane == 0) {
                    sl.mode = lit ? kPipeLiteral : (staged ? kPipeStaged : kPipeDirect);
                    sl.x0 = empty ? 0 : x0;
                    sl.ww = ww;
                    sl.y0 = empty ? 0 : y0;
                    sl.y1 = empty ? 0 : y1;
                    sl.level = l;
                    sl.batch = g.b;
                    sl.k = k;
                    sl.c0 = 0;
                    sl.last = it == nlev - 1;
                }
                mbar_arrive(tfull0 + 8 * slot); // all 32 lanes arrive: each releases its own table writes
            }
        }
        return;
    }

    // =========================== consumer warps ===========================
    const bool worker = tid < NWORK;
    const int wt = worker ? tid : 0;
    const int q = wt % NQ;
    const int pw = (wt / NQ) % P;
    const int ph0 = (wt / (NQ * P)) * PB;
    const int lane = tid & 31;
    float2 acc[PB][1][2];
#pragma unroll
    for (int i = 0; i < PB; ++i) acc[i][0][0] = acc[i][0][1] = make_float2(0.f, 0.f);
    RingPos rp{0u, 0u};
    // flush constants of this thread: the lane-rotated channel order and the tile offsets that go with it
    const int rot = kDenseTile ? ((q >> 1) & 3) : (lane >> 3) - (lane / NQ);
    const bool rot1 = (rot & 1) != 0, rot2 = (rot & 2) != 0;
    int toff[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) toff[jj] = (4 * q + ((jj + rot) & 3)) * S + ph0 * P + pw;
    // ---- flush: transpose the accumulators into the tile (lane-rotated channel order: conflict-free), stream it out
    auto flush = [&](int k, int c0) {
        asm volatile("bar.sync 1, %0;" ::"n"(NCONS) : "memory"); // the previous flush has left the tile (thread 0 waited on its store)
        if (worker) {
#pragma unroll
            float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
            if (bias) bz = ldg_f4(bias + (size_t)k * C + c0 + 4 * q);
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                const float a0 = acc[i][0][0].x + bz.x, a1 = acc[i][0][0].y + bz.y, a2 = acc[i][0][1].x + bz.z, a3 = acc[i][0][1].y + bz.w;
                // rotate (a0..a3) left by rot with two conditional stages (the predicates are per-thread constants)
                const float b0 = rot2 ? a2 : a0, b1 = rot2 ? a3 : a1, b2 = rot2 ? a0 : a2, b3 = rot2 ? a1 : a3;
                s_tile[toff[0] + i * P] = to_out<OutT>(rot1 ? b1 : b0);
                s_tile[toff[1] + i * P] = to_out<OutT>(rot1 ? b2 : b1);
                s_tile[toff[2] + i * P] = to_out<OutT>(rot1 ? b3 : b2);
                s_tile[toff[3] + i * P] = to_out<OutT>(rot1 ? b0 : b3);
                acc[i][0][0] = acc[i][0][1] = make_float2(0.f, 0.f);
            }
        }
        OutT *outp = out + ((size_t)k * C + c0) * PP;
        if (kBulkStore) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // my tile writes become visible to the TMA engine
            asm volatile("bar.sync 1, %0;" ::"n"(NCONS) : "memory");
            if (tid == 0) {
                tma_bulk_s2g(outp, smem_u32(s_tile), CC * PP * sizeof(OutT));   // 16-bit: CC >= 32, still a multiple of 16 B
                tma_store_wait_read(); // only this thread waits; the others are already on the next unit's rows
            }
        } else {
            asm volatile("bar.sync 1, %0;" ::"n"(NCONS) : "memory");
            constexpr int N4 = CC * PP / 4;
            if (bulk_store_flag & 2) { // A/B: conflict-free scalar reads of the padded tile, 32-bit coalesced stores
                for (int e = tid; e < CC * PP; e += NCONS) {
                    const int c = e / PP;
                    st_stream1(outp + e, s_tile[c * S + (e - c * PP)]);
                }
            } else
            for (int i = tid; i < N4; i += NCONS) {
                int c = (4 * i) / PP, e = 4 * i - c * PP;
                OutT t[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    t[u] = s_tile[c * S + e];
                    if (++e == PP) {
                        e = 0;
                        ++c;
                    }
                }
                st_stream4(outp + 4 * i, t[0], t[1], t[2], t[3]);
            }
        }
    };
    for (long unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        int k = 0, c0 = 0;
        for (int it = 0; it < nlev; ++it, ++itemctr) {
            const unsigned slot = itemctr % kPipeSlots, use = itemctr / kPipeSlots;
            mbar_wait(tfull0 + 8 * slot, use & 1);
            const PipeSlot<P> &sl = s_slot[slot];
            const int md = sl.mode, y0 = sl.y0, y1 = sl.y1, l = sl.level;
            k = sl.k;
            const int nx = sl.nx[pw];
            int ys[PB], ny[PB];
            int my0 = 1 << 30, my1 = -1;
#pragma unroll
            for (int i = 0; i < PB; ++i) {
                ys[i] = sl.ys[ph0 + i];
                ny[i] = sl.ny[ph0 + i];
                if (ny[i] > 0) {
                    my0 = min(my0, ys[i]);
                    my1 = max(my1, ys[i] + ny[i]);
                }
            }
            const float *wxp = sl.wx[pw], *wyp = sl.wy[ph0];
            if (!worker) { my0 = 0; my1 = 0; }
            for (int chunk = 0; chunk < nchunk; ++chunk) {
                c0 = chunk * CC;
                if (md == kPipeStaged) {
                    if (y1 > y0) {
                        const int xoff = sl.xs[pw] - sl.x0;
                        if (nx <= 0) { my0 = 0; my1 = 0; } // no valid sample in this column: still take part in the row barriers
                        const float *wyd = &sl.wyd[0][ph0 / 7 * 8];
                        const int pixs = cg32 ? 32 : CC;
                        const int toff = cg32 ? (q >> 3) * (WMAX * 32) + xoff * 32 + 4 * (q & 7) : xoff * CC + 4 * q;
                        switch (nx) {
                            case 1: staged_rows<1, PB, NS, WYS>(s_ring, STAGE_FLOATS, pixs, y0, y1, toff, wxp, wyd, acc, full0, empty0, rp, nx, my0, my1); break;
                            case 2: staged_rows<2, PB, NS, WYS>(s_ring, STAGE_FLOATS, pixs, y0, y1, toff, wxp, wyd, acc, full0, empty0, rp, nx, my0, my1); break;
                            case 3: staged_rows<3, PB, NS, WYS>(s_ring, STAGE_FLOATS, pixs, y0, y1, toff, wxp, wyd, acc, full0, empty0, rp, nx, my0, my1); break;
                            case 4: staged_rows<4, PB, NS, WYS>(s_ring, STAGE_FLOATS, pixs, y0, y1, toff, wxp, wyd, acc, full0, empty0, rp, nx, my0, my1); break;
                            default: staged_rows<0, PB, NS, WYS>(s_ring, STAGE_FLOATS, pixs, y0, y1, toff, wxp, wyd, acc, full0, empty0, rp, nx > 0 ? nx : 0, my0, my1); break;
                        }
                    }
                } else if (worker) {
                    const int H = lv.H[l], W = lv.W[l];
                    const int cq = c0 + 4 * q;
                    const size_t pix = cg32 ? 32 : (size_t)C;
                    const float *img = cg32 ? lv.data[l] + (size_t)sl.batch * H * W * C + (size_t)(cq >> 5) * H * W * 32 + (cq & 31)
                                            : lv.data[l] + (size_t)sl.batch * H * W * C + cq;
                    if (md == kPipeDirect) {
                        if (nx > 0 && my1 > my0) {
                            const float *rowp = img + ((size_t)my0 * W + sl.xs[pw]) * pix;
                            sweep_rows<0, PB, 1>(rowp, (size_t)W * pix, pix, 0, my0, my1, wxp, wyp, ys, ny, acc, nx);
                        }
                    } else {
                        const float *roi = rois + (size_t)k * 5;
                        const RoiGeom g = roi_geom(roi, lv.scale[l], P, P, sr, aligned, lv.pool2[l]);
    #pragma unroll 1
                        for (int pi = 0; pi < PB; ++pi) {
                            const int ph = ph0 + pi;
                            float a[4] = {0.f, 0.f, 0.f, 0.f};
                            for (int iy = 0; iy < g.gh; ++iy) {
                                int yl, yh;
                                float ly, hy;
                                const bool oky = axis_sample(sample_coord(g.start_h, g.bin_h, ph, iy, g.gh), H, yl, yh, ly, hy);
                                for (int ix = 0; ix < g.gw; ++ix) {
                                    int xl, xh;
                                    float lx, hx;
                                    const bool okx = axis_sample(sample_coord(g.start_w, g.bin_w, pw, ix, g.gw), W, xl, xh, lx, hx);
                                    if (!(oky && okx)) continue;
                                    const float w1 = hy * hx, w2 = hy * lx, w3 = ly * hx, w4 = ly * lx;
                                    const float4 v1 = ldg_f4(img + ((size_t)yl * W + xl) * pix), v2 = ldg_f4(img + ((size_t)yl * W + xh) * pix);
                                    const float4 v3 = ldg_f4(img + ((size_t)yh * W + xl) * pix), v4 = ldg_f4(img + ((size_t)yh * W + xh) * pix);
                                    a[0] += w1 * v1.x + w2 * v2.x + w3 * v3.x + w4 * v4.x;
                                    a[1] += w1 * v1.y + w2 * v2.y + w3 * v3.y + w4 * v4.y;
                                    a[2] += w1 * v1.z + w2 * v2.z + w3 * v3.z + w4 * v4.z;
                                    a[3] += w1 * v1.w + w2 * v2.w + w3 * v3.w + w4 * v4.w;
                                }
                            }
    #pragma unroll
                            for (int pp = 0; pp < PB; ++pp) {
                                if (pp == pi) {
                                    acc[pp][0][0].x += __fdiv_rn(a[0], g.count);
                                    acc[pp][0][0].y += __fdiv_rn(a[1], g.count);
                                    acc[pp][0][1].x += __fdiv_rn(a[2], g.count);
                                    acc[pp][0][1].y += __fdiv_rn(a[3], g.count);
                                }
                            }
                        }
                    }
                }
                if (nchunk > 1) flush(k, c0); // every channel chunk of the RoI is its own output tile
            }
            // the slot can be rebuilt as soon as every consumer warp has its taps out of it
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty0 + 8 * slot);
        }

        if (nchunk == 1) flush(k, 0);
    }
    if (kBulkStore && tid == 0) tma_store_wait_all(); // global writes complete before the CTA retires
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() { // resolved through the runtime: no link-time dependency on libcuda
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// maps of every level for a CTA that owns CC channels; false if the driver entry point is unavailable
static bool build_tmaps(const RoiLevels &lv, int B, int C, int CC, RoiTmaps *tm) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc || lv.L > kTmapLevels) return false;
    for (int l = 0; l < lv.L; ++l)
        for (int v = 0; v < kTmapBoxes; ++v) {
            const cuuint64_t gdim[2] = {(cuuint64_t)C, (cuuint64_t)B * lv.H[l] * lv.W[l]};
            const cuuint64_t gstride[1] = {(cuuint64_t)C * 4};
            const cuuint32_t box[2] = {(cuuint32_t)CC, (cuuint32_t)tmap_box_px(v)};
            const cuuint32_t estr[2] = {1, 1};
            if (enc(&tm->m[l][v], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void *)lv.data[l], gdim, gstride, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                return false;
        }
    return true;
}

template <int P, int NQ, int PHS, int NS, int WMAX, int MINB, typename OutT>
static int launch_pipe(const RoiLevels &lv, int B, int C, const float *rois, int K, int sr, int aligned, int mode, float finest,
                       OutT *out, const float *bias, cudaStream_t st, int cg32 = 0, const int *list = nullptr,
                       const int *list_count = nullptr) {
    static int grid_cache[kNuhtcMaxDevices] = {0};
    int &grid_cached = grid_cache[nuhtc_device()];
    static_assert(WMAX <= tmap_box_px(kTmapBoxes - 1) || true, "");
    // the CTA's NQ * 4 channels must tile C: with C = 192 and 128-channel chunks, nchunk = 1 would read each pixel's
    // 192 channels as 128 (NUHTC_RA_TMAP=2)
    if (C % (NQ * 4) != 0) return 1; // caller falls back
    RoiTmaps tm;
    memset(&tm, 0, sizeof tm);
    if (C / (NQ * 4) > 1 && !cg32) {
        if (WMAX > tmap_box_px(kTmapBoxes - 1) || !build_tmaps(lv, B, C, NQ * 4, &tm)) return 1; // caller falls back
    }
    if (cg32 && (NQ * 4) % 32 != 0) return 1;
    const size_t smem = sizeof(float) * ((size_t)NS * WMAX * NQ * 4 + NQ * 4 * ((P == 14 && NQ == 32) ? P * P : SepCfg<P>::S)) +
                        kPipeSlots * sizeof(PipeSlot<P>) +
                        sizeof(uint64_t) * (2 * NS + 2 * kPipeSlots) + 128;
    auto kern = roi_align_pipe_kernel<P, NQ, PHS, NS, WMAX, MINB, OutT>;
    constexpr int nthreads = (NQ * P * PHS + 31) / 32 * 32 + 64;
    if (!grid_cached) {
        NUHTC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        NUHTC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nthreads, smem));
        if (per_sm < 1) {
            nuhtc_set_error("roi_align pipe kernel does not fit on an SM (smem %zu)", smem);
            return NUHTC_ECUDA;
        }
        grid_cached = per_sm * nuhtc_sm_count(); // persistent: every CTA resident, a multiple of the SM count
    }
    const long nunits = K;
    const int grid = (int)(nunits < grid_cached ? nunits : grid_cached);
    static const int bulk = getenv("NUHTC_RA_BULK") ? atoi(getenv("NUHTC_RA_BULK")) : 1;
    kern<<<grid, nthreads, smem, st>>>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, bulk, tm, cg32, list, list_count);
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}

static int ra_pipe() { // NUHTC_RA_PIPE=0 selects the v2 (non-pipelined) kernel for A/B runs
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("NUHTC_RA_PIPE");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v;
}

// tuning knob (A/B on the GPU box): NUHTC_RA_VEC=1 keeps one float4 slice per thread
static int ra_vec() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("NUHTC_RA_VEC");
        v = (e && e[0] >= '1' && e[0] <= '3') ? e[0] - '0' : 2; // 1: one slice/thread; 2: two slices, 2 CTAs/SM; 3: two slices, 3 CTAs/SM
    }
    return v;
}

NUHTC_API int nuhtc_roi_align_fwd(const float *const *feats, const int *H, const int *W, const float *scale, int L, int B,
                                  int C, int layout, const float *rois, int K, int PH, int PW, int sampling_ratio,
                                  int aligned, int mode, float finest_scale, int impl, float *out, const float *bias,
                                  void *stream) {
    NUHTC_CHECK_ARG(L >= 1 && L <= NUHTC_MAX_LEVELS, "roi_align: L=%d out of range", L);
    NUHTC_CHECK_ARG(B >= 0 && C >= 1 && PH >= 1 && PW >= 1 && K >= 0, "roi_align: bad sizes B=%d C=%d PH=%d PW=%d K=%d", B, C,
                    PH, PW, K);
    NUHTC_CHECK_ARG(layout == NUHTC_LAYOUT_NCHW || layout == NUHTC_LAYOUT_NHWC, "roi_align: bad layout %d", layout);
    NUHTC_CHECK_ARG(mode == NUHTC_ROI_ROUTE || mode == NUHTC_ROI_SUM, "roi_align: bad mode %d", mode);
    NUHTC_CHECK_ARG(finest_scale > 0.f || L == 1 || mode == NUHTC_ROI_SUM, "roi_align: finest_scale must be > 0");
    if (K == 0) return NUHTC_OK;
    NUHTC_CHECK_ARG(feats && H && W && scale && rois && out, "roi_align: null pointer");
    RoiLevels lv;
    lv.L = L;
    for (int l = 0; l < L; ++l) {
        NUHTC_CHECK_ARG(feats[l] != nullptr && H[l] >= 1 && W[l] >= 1, "roi_align: bad level %d", l);
        lv.data[l] = feats[l];
        lv.H[l] = H[l];
        lv.W[l] = W[l];
        lv.scale[l] = scale[l];
        lv.pool2[l] = 0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    bool aligned16 = true;
    for (int l = 0; l < L; ++l) aligned16 = aligned16 && (((uintptr_t)feats[l]) % 16 == 0);
    aligned16 = aligned16 && (((uintptr_t)out) % 16 == 0);
    const bool fast_ok = impl == NUHTC_IMPL_AUTO && layout == NUHTC_LAYOUT_NHWC && PH == PW && (PH == 7 || PH == 14) &&
                         C % 64 == 0 && aligned16;
    if (fast_ok && ra_pipe()) {
        const int sr = sampling_ratio;
        int rc = 1; // 1 = not handled by the pipelined kernel
        if (PH == 7) { // the CTA owns every channel of the level: one plain bulk copy per window row
            // ring shape A/B on the box (K = 16000): 5 x 32 px stages 0.457 ms nuclei / 0.867 ms routed; 8 x 20 px 0.444 / 1.595;
            // 10 x 16 px 0.543 / 1.757; 6 x 26 px 0.451 / 1.135 -- more, narrower stages do not help (the kernel is not short
            // of loads in flight) and send wide windows down the direct path
            if (C == 256) rc = launch_pipe<7, 64, 1, 5, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
            else if (C == 128) rc = launch_pipe<7, 32, 1, 8, 24, 1>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
            else if (C == 64) rc = launch_pipe<7, 16, 1, 8, 24, 2>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
        } else if (C == 64) {
            rc = launch_pipe<14, 16, 2, 8, 24, 1>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
        } else if ((mode == NUHTC_ROI_ROUTE || L == 1) && getenv("NUHTC_RA_TMAP")) {
            // Channel chunks fetched through 2-D tensor maps (cp.async.bulk.tensor), opt-in.  K=16000, C=256 on the box:
            //   =1  64-channel chunks, two row halves per thread column      1.81 ms nuclei / 3.51 ms routed
            //   =2  128-channel chunks, dense tile + one async bulk store    1.47 ms nuclei / 4.42 ms routed
            //   non-pipelined roi_align_sep_kernel<14,8,2,2,2> (default)     1.55 ms nuclei / 2.16 ms routed
            // =2 wins 5 % on nucleus-sized windows but its 24-px ring rows send the wide windows of large RoIs down the
            // direct-load path, so the non-pipelined kernel stays the default for the mask branch.
            if (getenv("NUHTC_RA_TMAP")[0] == '2')   // 128-channel halves, every thread owns all 14 rows of its column
                rc = launch_pipe<14, 32, 1, 8, 24, 1>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
            else
                rc = launch_pipe<14, 16, 2, 12, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
        }
        if (rc != 1) return rc;
    }
    if (fast_ok) {
        const int sr = sampling_ratio;
        const bool v2 = ra_vec() >= 2;
        if (PH == 7) {
            if (C % 256 == 0) {
                if (ra_vec() == 3) return launch_sep<7, 32, 1, 2, 3>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
                if (v2) return launch_sep<7, 32, 1, 2, 2>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
                return launch_sep<7, 64, 1, 1, 2>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
            }
            if (C % 128 == 0) {
                if (v2) return launch_sep<7, 16, 1, 2, 4>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
                return launch_sep<7, 32, 1, 1, 4>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
            }
            return launch_sep<7, 16, 1, 1, 8>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
        }
        // A/B on the box (K = 16000, nuclei): <14,8,2,2,2> 1.55 ms; one slice per thread at 4 CTAs/SM 1.94 ms, at 3 CTAs/SM
        // 1.85 ms; a dense 196-float tile stride with float4 copy-out (no read conflicts) 2.35 ms
        if (v2) return launch_sep<14, 8, 2, 2, 2>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
        return launch_sep<14, 16, 2, 1, 2>(lv, C, rois, K, sr, aligned, mode, finest_scale, out, bias, st);
    }
    const long total = (long)K * C * PH * PW;
    const int threads = 256;
    long blocks = (total + threads - 1) / threads;
    const long cap = (long)nuhtc_sm_count() * 32;
    if (blocks > cap) blocks = cap;
    roi_align_direct_kernel<<<(unsigned)blocks, threads, 0, st>>>(lv, C, layout, rois, total, PH, PW, sampling_ratio, aligned,
                                                                  mode, finest_scale, out, bias);
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}


// per-RoI kernel on the channel-group layout: every RoI (list == nullptr) or the RoIs of a device-side list
template <typename OutT>
static int launch_sep_cg32(const RoiLevels &lv, int B, int C, const float *rois, int K, int P, int sr, int aligned, int mode,
                           float finest, OutT *out, const float *bias, cudaStream_t st, const int *list,
                           const int *list_count) {
    // Pipelined kernel first: the window rows arrive through bulk copies (one per channel group and row), so a RoI's
    // latency is one ring fill instead of a chain of dependent global loads per row.  NUHTC_RA_PIPE=0: A/B switch.
    if (ra_pipe()) {
        const int nlev = mode == NUHTC_ROI_ROUTE ? 1 : lv.L;
        int rc = 1;
        if (P == 7) {
            if (C == 256) rc = launch_pipe<7, 64, 1, 5, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
            else if (C == 128) rc = launch_pipe<7, 32, 1, 8, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
            // C = 64 (the PanNuke configs' two-level sum): measured 0.72 ms pipelined vs 0.29 ms per-RoI on K = 16000 -> per-RoI
        } else if (C % 128 == 0 && (C == 128 || nlev == 1)) { // 128-channel chunks: a chunk is its own output tile, so no level sum across chunks
            rc = launch_pipe<14, 32, 1, 6, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
        } else if (C == 64) {
            rc = launch_pipe<14, 16, 2, 8, 32, 1>(lv, B, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
        }
        if (rc != 1) return rc;
    }
    if (P == 7) {
        if (C % 256 == 0) return launch_sep<7, 32, 1, 2, 2>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
        if (C % 128 == 0) return launch_sep<7, 16, 1, 2, 4>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
        if (C % 64 == 0) return launch_sep<7, 16, 1, 1, 8>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
        return launch_sep<7, 8, 1, 1, 8>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
    }
    if (C % 64 == 0) return launch_sep<14, 8, 2, 2, 2>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
    return launch_sep<14, 8, 2, 1, 2>(lv, C, rois, K, sr, aligned, mode, finest, out, bias, st, 1, list, list_count);
}

NUHTC_API size_t nuhtc_roi_align_workspace_bytes(const int *H, const int *W, int L, int B, int K, int PH, int PW) {
    if (L < 1 || L > NUHTC_MAX_LEVELS || !H || !W || PH != PW || (PH != 7 && PH != 14) || K <= 0) return 256;
    return roi_strip_workspace_bytes(H, W, L, B, K, PH);
}

static size_t dtype_size(int dtype) {   // 0: not a NUHTC_DTYPE_* code
    return dtype == NUHTC_DTYPE_F32 ? 4 : (dtype == NUHTC_DTYPE_F16 || dtype == NUHTC_DTYPE_BF16) ? 2 : 0;
}

NUHTC_API int nuhtc_to_cg32_dt(const void *in, int in_dtype, float *out, int B, int C, int H, int W, int channels_last, void *stream) {
    const size_t es = dtype_size(in_dtype);
    NUHTC_CHECK_ARG(es != 0, "to_cg32: unknown dtype code %d", in_dtype);
    NUHTC_CHECK_ARG(B >= 0 && C >= 32 && C % 32 == 0 && H >= 1 && W >= 1, "to_cg32: bad sizes (C must be a multiple of 32)");
    if (B == 0) return NUHTC_OK;
    // the staging kernels read four input elements at a time and write 16-byte vectors
    NUHTC_CHECK_ARG(in && out && ((uintptr_t)in % (4 * es) == 0) && ((uintptr_t)out % 16 == 0), "to_cg32: null or misaligned pointer");
    NUHTC_CHECK_ARG(channels_last || (H * W) % 4 == 0, "to_cg32: H*W must be a multiple of 4 for an NCHW source");
    NUHTC_CHECK_ARG(C / 32 <= 65535 && B <= 65535, "to_cg32: C or B too large");
    return roi_to_cg32(in, in_dtype, out, B, C, H, W, channels_last, (cudaStream_t)stream);
}

NUHTC_API int nuhtc_to_cg32(const float *in, float *out, int B, int C, int H, int W, int channels_last, void *stream) {
    return nuhtc_to_cg32_dt(in, NUHTC_DTYPE_F32, out, B, C, H, W, channels_last, stream);
}

template <typename OutT>
static int roi_align_cg32_run(const RoiLevels &lv, int B, int C, const float *rois, int K, int PH, int PW, int sampling_ratio,
                              int aligned, int mode, float finest_scale, OutT *out, int out_dtype, const float *bias, void *ws,
                              size_t ws_bytes, cudaStream_t st) {
    static const bool no_strip = getenv("NUHTC_RA_STRIP") && getenv("NUHTC_RA_STRIP")[0] == '0';   // A/B: per-RoI kernel only
    // the strip prepass builds its tap tables at the output size: a pool2 level (a lone one in sum mode) needs the
    // per-RoI kernels, which pool it with 2g samples per bin
    bool pool2 = false;
    for (int l = 0; l < lv.L; ++l) pool2 = pool2 || lv.pool2[l] != 0;
    if (roi_strip_supported(C, PH, PW, mode, lv.L) && !no_strip && !pool2) {
        const int *left = nullptr, *left_count = nullptr;
        const int rc = roi_strip_forward(lv, B, C, rois, K, PH, sampling_ratio, aligned, mode, finest_scale, out, out_dtype, bias, ws,
                                         ws_bytes, st, &left, &left_count);
        if (rc == NUHTC_OK)
            return launch_sep_cg32(lv, B, C, rois, K, PH, sampling_ratio, aligned, mode, finest_scale, out, bias, st, left, left_count);
        if (rc != 1) return rc;   // 1: the levels are too large for the strip binning -> every RoI through the per-RoI kernel
    }
    return launch_sep_cg32(lv, B, C, rois, K, PH, sampling_ratio, aligned, mode, finest_scale, out, bias, st, nullptr, nullptr);
}

NUHTC_API int nuhtc_roi_align_cg32_dt(const float *const *feats, const int *H, const int *W, const float *scale, int L, int B,
                                      int C, const float *rois, int K, int PH, int PW, int sampling_ratio, int aligned, int mode,
                                      float finest_scale, const int *pool2, void *out, int out_dtype, const float *bias, void *ws,
                                      size_t ws_bytes, void *stream) {
    NUHTC_CHECK_ARG(dtype_size(out_dtype) != 0, "roi_align_cg32: unknown dtype code %d", out_dtype);
    NUHTC_CHECK_ARG(L >= 1 && L <= NUHTC_MAX_LEVELS, "roi_align_cg32: L=%d out of range", L);
    NUHTC_CHECK_ARG(PH == PW && (PH == 7 || PH == 14) && C >= 32 && C % 32 == 0 && B >= 0 && K >= 0,
                    "roi_align_cg32: needs PH == PW in {7, 14} and C %% 32 == 0 (PH=%d PW=%d C=%d)", PH, PW, C);
    NUHTC_CHECK_ARG(mode == NUHTC_ROI_ROUTE || mode == NUHTC_ROI_SUM, "roi_align_cg32: bad mode %d", mode);
    NUHTC_CHECK_ARG(finest_scale > 0.f || L == 1 || mode == NUHTC_ROI_SUM, "roi_align_cg32: finest_scale must be > 0");
    if (K == 0) return NUHTC_OK;
    NUHTC_CHECK_ARG(feats && H && W && scale && rois && out, "roi_align_cg32: null pointer");
    RoiLevels lv;
    lv.L = L;
    for (int l = 0; l < L; ++l) {
        NUHTC_CHECK_ARG(feats[l] != nullptr && H[l] >= 1 && W[l] >= 1 && ((uintptr_t)feats[l] % 128 == 0), "roi_align_cg32: bad level %d", l);
        lv.data[l] = feats[l];
        lv.H[l] = H[l];
        lv.W[l] = W[l];
        lv.scale[l] = scale[l];
        lv.pool2[l] = pool2 ? pool2[l] : 0;
        NUHTC_CHECK_ARG(lv.pool2[l] == 0 || mode == NUHTC_ROI_SUM, "roi_align_cg32: pool2 levels need mode SUM");
    }
    NUHTC_CHECK_ARG((uintptr_t)out % 16 == 0, "roi_align_cg32: out must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    switch (out_dtype) {
        case NUHTC_DTYPE_F16:
            return roi_align_cg32_run(lv, B, C, rois, K, PH, PW, sampling_ratio, aligned, mode, finest_scale, static_cast<__half *>(out),
                                      out_dtype, bias, ws, ws_bytes, st);
        case NUHTC_DTYPE_BF16:
            return roi_align_cg32_run(lv, B, C, rois, K, PH, PW, sampling_ratio, aligned, mode, finest_scale,
                                      static_cast<__nv_bfloat16 *>(out), out_dtype, bias, ws, ws_bytes, st);
        default:
            return roi_align_cg32_run(lv, B, C, rois, K, PH, PW, sampling_ratio, aligned, mode, finest_scale, static_cast<float *>(out),
                                      out_dtype, bias, ws, ws_bytes, st);
    }
}

NUHTC_API int nuhtc_roi_align_cg32(const float *const *feats, const int *H, const int *W, const float *scale, int L, int B,
                                   int C, const float *rois, int K, int PH, int PW, int sampling_ratio, int aligned, int mode,
                                   float finest_scale, const int *pool2, float *out, const float *bias, void *ws, size_t ws_bytes,
                                   void *stream) {
    return nuhtc_roi_align_cg32_dt(feats, H, W, scale, L, B, C, rois, K, PH, PW, sampling_ratio, aligned, mode, finest_scale, pool2,
                                   out, NUHTC_DTYPE_F32, bias, ws, ws_bytes, stream);
}

// ---------------------------------------------------------------------------------------------
// NCHW -> NHWC (once per level per batch; HBM-bound transpose through a padded smem tile)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const float *__restrict__ in, float *__restrict__ out, int C,
                                                           int HW) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x, ty = threadIdx.y; // (32, 8)
    const float *src = in + (size_t)b * C * HW;
    float *dst = out + (size_t)b * C * HW;
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        const int c = c0 + ty + i, hw = hw0 + tx;
        if (c < C && hw < HW) tile[ty + i][tx] = __ldg(src + (size_t)c * HW + hw);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        const int hw = hw0 + ty + i, c = c0 + tx;
        if (c < C && hw < HW) dst[(size_t)hw * C + c] = tile[tx][ty + i];
    }
}

// 64 x 64 tile, 128-bit global accesses on both sides (HW % 4 == 0, C % 4 == 0, 16-byte aligned pointers): 16 KB per CTA
// instead of 4 KB and four independent 16-byte loads per thread in flight
__global__ void __launch_bounds__(256) nchw_to_nhwc_vec_kernel(const float *__restrict__ in, float *__restrict__ out, int C,
                                                               int HW) {
    __shared__ float tile[64][65];
    const int b = blockIdx.z;
    const int hw0 = blockIdx.x * 64, c0 = blockIdx.y * 64;
    const int t = threadIdx.x;
    const int r = t >> 4, q = (t & 15) * 4;
    const float *src = in + (size_t)b * C * HW;
    float *dst = out + (size_t)b * C * HW;
    float4 v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + r + 16 * k, hw = hw0 + q;
        v[k] = (c < C && hw < HW) ? ldg_f4(src + (size_t)c * HW + hw) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float *row = &tile[r + 16 * k][q];
        row[0] = v[k].x;
        row[1] = v[k].y;
        row[2] = v[k].z;
        row[3] = v[k].w;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int hw = hw0 + r + 16 * k, c = c0 + q;
        if (hw < HW && c < C) {
            const float4 o = make_float4(tile[q][r + 16 * k], tile[q + 1][r + 16 * k], tile[q + 2][r + 16 * k], tile[q + 3][r + 16 * k]);
            *reinterpret_cast<float4 *>(dst + (size_t)hw * C + c) = o;
        }
    }
}

NUHTC_API int nuhtc_nchw_to_nhwc(const float *in, float *out, int B, int C, int H, int W, void *stream) {
    NUHTC_CHECK_ARG(B >= 0 && C >= 1 && H >= 1 && W >= 1, "nchw_to_nhwc: bad sizes");
    if (B == 0) return NUHTC_OK;
    NUHTC_CHECK_ARG(in && out, "nchw_to_nhwc: null pointer");
    const int HW = H * W;
    static const bool vec_ok_env = !(getenv("NUHTC_NHWC_VEC") && getenv("NUHTC_NHWC_VEC")[0] == '0');
    if (vec_ok_env && HW % 4 == 0 && C % 4 == 0 && ((uintptr_t)in % 16 == 0) && ((uintptr_t)out % 16 == 0)) {
        dim3 g64((HW + 63) / 64, (C + 63) / 64, B);
        NUHTC_CHECK_ARG(g64.y <= 65535 && g64.z <= 65535, "nchw_to_nhwc: C or B too large");
        nchw_to_nhwc_vec_kernel<<<g64, 256, 0, (cudaStream_t)stream>>>(in, out, C, HW);
        NUHTC_LAUNCH_CHECK();
        return NUHTC_OK;
    }
    dim3 grid((HW + 31) / 32, (C + 31) / 32, B);
    NUHTC_CHECK_ARG(grid.y <= 65535 && grid.z <= 65535, "nchw_to_nhwc: C or B too large");
    nchw_to_nhwc_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(in, out, C, HW);
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}
