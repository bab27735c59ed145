// Strip-shared RoIAlign forward for sm_100a -- the default path for 7x7 / 14x14 outputs (C % 32 == 0).
//
// Replaces mmcv-full 1.7.2 `roi_align_forward` (avg pool, aligned) as driven per FPN level by
//   /root/reference/thirdparty/mmdetection/mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:58-115
// for ALL levels and RoIs in one launch sequence, like roi_align.cu, but organised around the FEATURE MAP instead of
// the RoI.  Round 1's kernel pulled every RoI's own window through L2 (16 000 windows x 121 KB = 1.9 GB for a 0.27 GB
// level: each cell crossed the L2->SM fabric ~7 times, profiles/r01_roialign_pipe.md) and was bound by the L2 slices.
// Here a CTA owns a vertical STRIP of one image for one group of 32 channels and marches down it once:
//
//   layout   levels are staged as [B][C/32][H][W][32] fp32 ("CG32": one 128-byte line per cell and channel group), so a
//            strip row is ONE contiguous segment and a CTA that owns 32 channels still moves whole lines;
//   prepass  (3 small launches) bins the RoIs by (level, image, strip, y-part), orders every bin by window top, and writes
//            one record per RoI -- x tap tables and dense per-row y weights in the reference's fp32 op order ("staging of
//            sampling coordinates") -- at its sorted position; windows that cannot be staged go to a leftover list;
//   ring     the producer warp streams the strip's rows top to bottom into a shared-memory ring with one TMA bulk copy per
//            row (cp.async.bulk, full/empty mbarriers); the ring runs on across unit boundaries, so the next unit's first
//            rows land while the teams finish the current one;
//   teams    NT teams of 8*P threads (thread = 4 channels x output column) pop RoIs in window-top order, wait for the rows
//            [y0, y0+hh) they need, run the separable pooling out of shared memory (LDS.128 + packed FFMA2), transpose
//            their [32][P][P] result through a team tile and send it off with one asynchronous bulk store; a row is
//            released to the producer once every team has moved past it.
// Each level row is fetched by (strips x channel groups) CTAs once (+ the x halo, ~1.4x at W = 128) instead of once per
// overlapping RoI.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"
#include "roi_common.cuh"
#include "roi_strip.cuh"

namespace {

constexpr int kCG = 32;                               // channels per group: 32 floats = one 128-byte line per cell
constexpr int kBW = 48;                               // cells per staged row (ring row = 6144 B)
constexpr int kXH = 18;                               // widest window staged on a level that needs several strips
constexpr int kCore = kBW - kXH + 1;                  // 31: strip s owns window origins [s*kCore, (s+1)*kCore)
constexpr int kRMax = 18;                             // tallest staged window
constexpr int kNU = 4;                                // unit descriptors in flight
constexpr int kRowFloats = kBW * kCG;
constexpr int kSmemMax = 232448;                      // 227 KB opt-in shared memory per CTA
constexpr int kScanSmemMax = 200 * 1024;              // the scan kernel stages the key histogram in shared memory

// One record per staged RoI, written by the prepass at the RoI's sorted position and fetched with one bulk copy: the x tap
// tables and the dense per-row y weights in the reference's fp32 op order ("staging of sampling coordinates").
// The consumers sweep the window rows once (x taps first), and the y pass is sparse at the granularity of groups of four
// output rows: gs[g] / ge[g] bound the window rows that reach group g (bins 4g .. 4g+3), which cuts the sweep into counted
// loops whose bodies only touch the accumulators of one group or of two neighbouring groups.
template <int P>
struct __align__(16) StripRec {
    static constexpr int WYS = (P + 3) / 4 * 4;
    int k, y0, hh, x0;
    unsigned char xs[16];   // per output column: first x tap - x0
    signed char nx[16];     // per output column: x taps (0: no valid sample)
    unsigned char gs[4], ge[4];   // per bin group: first / one-past-last window row that reaches it
    unsigned char sB, eA;         // 7x7 shorthand: gs[1], ge[0]
    unsigned char gdense, nxmax;  // a row reaches three groups: sweep every row into every bin; max x taps of a column
    int pad[1];
    float wx[P][kMaxTap];
    float wyd[kRMax][WYS];  // [window row][bin]: y weight / sample count, 0 where the bin misses the row
};
static_assert(sizeof(StripRec<7>) == 64 + 7 * 32 + kRMax * 32 && sizeof(StripRec<14>) == 64 + 14 * 32 + kRMax * 64, "record layout");

struct StripLevel {
    const float *data;
    int H, W;
    float scale;
    int nstrips, nyp, ypart_rows;
    int key0, bin0;
};

struct StripUnit {   // one per non-empty bin; the unit proper is (bin, channel group)
    int level, b, X0, BW, Y0, Y1, item_begin, item_count;
};

struct StripArgs {
    StripLevel lv[NUHTC_MAX_LEVELS];
    int L, B, C, K;
    int sr, aligned, mode;
    float finest;
    int nkeys, nbins;
    int dbg;           // measurement switches (NUHTC_RA_DBG): 1 skip the pooling arithmetic + stores, 2 skip the stores only
    const float *rois;
    void *out;         // [K][C][P][P] elements of the kernel's OutT
    const float *bias;
    // workspace
    int *item_key;     // [K] sort key of the item, -1: leftover
    int *hist;         // [nkeys + 1] -> exclusive offsets
    int *cursor;       // [nkeys]
    int *bin_ymax;     // [nbins]
    StripUnit *units;  // [nbins]
    int *counters;     // [0] nunits (bins x channel groups), [1] unit cursor, [2] leftover count
    int *leftover;     // [K]
    void *records;     // [K] StripRec<P>
};

// ---------------------------------------------------------------------------------------------
// prepass
// ---------------------------------------------------------------------------------------------
struct ItemGeom {
    int level, b;
    int x0, ww, y0, hh;   // window
    bool lit;             // a bin exceeds the tap table
    bool empty;           // no valid sample at all
};

// A warp evaluates the tap tables of one RoI: lanes [0, P) the x bins, lanes [16, 16 + P) the y bins.
// Returns the lane's table (w, first, n) and the window geometry (all lanes).
template <int P>
__device__ __forceinline__ ItemGeom item_tables(const StripArgs &a, int k, int lane, float (&w)[kMaxTap], int &first, int &n,
                                                float &count) {
    const float *roi = a.rois + (size_t)k * 5;
    ItemGeom g;
    g.level = a.mode == NUHTC_ROI_ROUTE ? route_level(roi, a.L, a.finest) : 0;
    const StripLevel &lv = a.lv[g.level];
    const RoiGeom rg = roi_geom(roi, lv.scale, P, P, a.sr, a.aligned);
    g.b = rg.b;
    count = rg.count;
    first = 0;
    n = 0;
    const bool xb = lane < P, yb = lane >= 16 && lane < 16 + P;
    if (xb) build_axis_taps(rg.start_w, rg.bin_w, rg.gw, lane, lv.W, 1.0f, w, &first, &n);
    else if (yb) build_axis_taps(rg.start_h, rg.bin_h, rg.gh, lane - 16, lv.H, rg.count, w, &first, &n);
    const bool has = (xb || yb) && n > 0, bad = (xb || yb) && n < 0;
    int lo = has ? first : (1 << 30), hi = has ? first + n : -1;
#pragma unroll
    for (int o = 8; o; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    const int x0 = __shfl_sync(0xffffffffu, lo, 0), x1 = __shfl_sync(0xffffffffu, hi, 0);
    const int y0 = __shfl_sync(0xffffffffu, lo, 16), y1 = __shfl_sync(0xffffffffu, hi, 16);
    g.lit = __any_sync(0xffffffffu, bad);
    g.empty = x1 <= x0 || y1 <= y0;
    g.x0 = g.empty ? 0 : x0;
    g.ww = g.empty ? 0 : x1 - x0;
    g.y0 = g.empty ? 0 : y0;
    g.hh = g.empty ? 0 : y1 - y0;
    return g;
}

__device__ __forceinline__ bool item_staged(const StripArgs &a, const ItemGeom &g) {
    if (g.lit || g.empty || g.hh > kRMax) return false;
    if (g.b < 0 || g.b >= a.B) return false;
    const StripLevel &lv = a.lv[g.level];
    return lv.nstrips == 1 ? lv.W <= kBW : g.ww <= kXH;
}

// K1: sort key of every RoI (warp per RoI), histogram of the keys, lowest window bottom of every bin
template <int P>
__global__ void __launch_bounds__(256) strip_keys_kernel(StripArgs a) {
    const int lane = threadIdx.x & 31;
    const int k = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (k >= a.K) return;
    float w[kMaxTap];
    int first, n;
    float count;
    const ItemGeom g = item_tables<P>(a, k, lane, w, first, n, count);
    if (lane != 0) return;
    int key = -1;
    if (item_staged(a, g)) {
        const StripLevel &lv = a.lv[g.level];
        const int s = lv.nstrips == 1 ? 0 : min(g.x0 / kCore, lv.nstrips - 1);
        // the last strip of a level is cut at the map edge: its windows reach at most W, which fits by construction
        key = lv.key0 + (g.b * lv.nstrips + s) * lv.H + g.y0;
        const int bin = lv.bin0 + (g.b * lv.nstrips + s) * lv.nyp + g.y0 / lv.ypart_rows;
        atomicAdd(a.hist + key, 1);
        atomicMax(a.bin_ymax + bin, g.y0 + g.hh);
    }
    a.item_key[k] = key;
}

// K2: one CTA.  Exclusive scan of the key histogram (-> sorted positions), then one descriptor per non-empty bin.
__global__ void __launch_bounds__(1024) strip_scan_kernel(StripArgs a) {
    __shared__ int s_warp[32];
    __shared__ int s_carry, s_units;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) {
        s_carry = 0;
        s_units = 0;
    }
    __syncthreads();
    extern __shared__ int s_h[];
    {   // the histogram is staged in shared memory (coalesced both ways); every thread owns a contiguous run of keys:
        // local sum, one block scan of the 1024 partial sums, local write-back
        for (int i = tid; i < a.nkeys; i += 1024) s_h[i] = a.hist[i];
        __syncthreads();
        const int per = (a.nkeys + 1023) / 1024;
        const int k0 = min(a.nkeys, tid * per), k1 = min(a.nkeys, k0 + per);
        int sum = 0;
        for (int i = k0; i < k1; ++i) sum += s_h[i];
        int x = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_warp[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int t = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            s_warp[lane] = t;
        }
        __syncthreads();
        int run = (wid ? s_warp[wid - 1] : 0) + x - sum;
        for (int i = k0; i < k1; ++i) {
            const int v = s_h[i];
            s_h[i] = run;
            run += v;
        }
        if (tid == 1023) s_carry = s_warp[31];
        __syncthreads();
        for (int i = tid; i < a.nkeys; i += 1024) {
            const int v = s_h[i];
            a.hist[i] = v;
            a.cursor[i] = v;
        }
    }
    if (tid == 0) a.hist[a.nkeys] = s_carry;
    __syncthreads();
    // bins -> units, in (level, image, strip, y-part) order so that neighbouring units share rows and records in L2
    for (int base = 0; base < a.nbins; base += 1024) {
        const int bin = base + tid;
        int cnt = 0, begin = 0, Y0 = 0, level = 0, b = 0, s = 0;
        if (bin < a.nbins) {
            level = a.L - 1;
            while (level > 0 && bin < a.lv[level].bin0) --level;
            const StripLevel &lv = a.lv[level];
            const int r = bin - lv.bin0;
            const int yp = r % lv.nyp, bs = r / lv.nyp;
            s = bs % lv.nstrips;
            b = bs / lv.nstrips;
            const int ka = lv.key0 + bs * lv.H + yp * lv.ypart_rows;
            const int kb = lv.key0 + bs * lv.H + min(lv.H, (yp + 1) * lv.ypart_rows);
            // the scanned histogram is still in shared memory (entry nkeys = the total): the walk below is a chain of
            // dependent reads, 32 L2 round trips per bin when it went through a.hist
            const int total = s_carry;
            auto Hs = [&](int i) { return i < a.nkeys ? s_h[i] : total; };
            begin = Hs(ka);
            cnt = Hs(kb) - begin;
            if (cnt > 0) {
                int kk = ka;
                while (Hs(kk + 1) == begin) ++kk;   // first non-empty key of the bin = smallest window top
                Y0 = kk - (lv.key0 + bs * lv.H);
            }
        }
        const unsigned m = __ballot_sync(0xffffffffu, cnt > 0);
        if (lane == 0) s_warp[wid] = __popc(m);
        __syncthreads();
        if (wid == 0) {
            int t = s_warp[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            s_warp[lane] = t;
        }
        __syncthreads();
        if (cnt > 0) {
            const int slot = s_units + (wid ? s_warp[wid - 1] : 0) + __popc(m & ((1u << lane) - 1));
            const StripLevel &lv = a.lv[level];
            StripUnit u;
            u.level = level;
            u.b = b;
            u.X0 = lv.nstrips == 1 ? 0 : s * kCore;
            u.BW = min(kBW, lv.W - u.X0);
            u.Y0 = Y0;
            u.Y1 = a.bin_ymax[bin];
            u.item_begin = begin;
            u.item_count = cnt;
            a.units[slot] = u;
        }
        __syncthreads();
        if (tid == 0) s_units += s_warp[31];
        __syncthreads();
    }
    if (tid == 0) a.counters[0] = s_units;
}

// K3: records at their sorted positions (warp per RoI); RoIs that cannot be staged go to the leftover list
template <int P>
__global__ void __launch_bounds__(256) strip_records_kernel(StripArgs a) {
    // (record layout: StripRec<P>)
    const int lane = threadIdx.x & 31;
    const int k = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    if (k >= a.K) return;
    const int key = a.item_key[k];
    if (key < 0) {
        if (lane == 0) a.leftover[atomicAdd(a.counters + 2, 1)] = k;
        return;
    }
    float w[kMaxTap];
    int first, n;
    float count;
    const ItemGeom g = item_tables<P>(a, k, lane, w, first, n, count);
    int pos = 0;
    if (lane == 0) pos = atomicAdd(a.cursor + key, 1);
    pos = __shfl_sync(0xffffffffu, pos, 0);
    StripRec<P> *rec = reinterpret_cast<StripRec<P> *>(a.records) + pos;
    if (lane == 0) {
        rec->k = k;
        rec->y0 = g.y0;
        rec->hh = g.hh;
        rec->x0 = g.x0;
    }
    if (lane < 16) {
        rec->xs[lane] = (unsigned char)((lane < P && n > 0) ? first - g.x0 : 0);
        rec->nx[lane] = (signed char)(lane < P ? n : 0);
    }
    int nxmax = lane < P ? n : 0;
#pragma unroll
    for (int o = 8; o; o >>= 1) nxmax = max(nxmax, __shfl_xor_sync(0xffffffffu, nxmax, o));
    nxmax = __shfl_sync(0xffffffffu, nxmax, 0);
    if (lane < P) {
        *reinterpret_cast<float4 *>(&rec->wx[lane][0]) = make_float4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<float4 *>(&rec->wx[lane][4]) = make_float4(w[4], w[5], w[6], w[7]);
    }
    // dense y weights: wyd[r][p] = w_p[y0 + r - first_p] where bin p reaches window row r, else 0.  The bin lanes park
    // their tables in shared memory; then lane r assembles window row r and writes it with 128-bit stores.
    constexpr int WYS = StripRec<P>::WYS;
    __shared__ float s_wy[8][P][kMaxTap];
    __shared__ int s_fn[8][P][2];
    const int wib = threadIdx.x >> 5;
    const bool ybin = lane >= 16 && lane < 16 + P;
    if (ybin) {
        const int p = lane - 16;
#pragma unroll
        for (int j = 0; j < kMaxTap; ++j) s_wy[wib][p][j] = w[j];
        s_fn[wib][p][0] = first - g.y0;
        s_fn[wib][p][1] = n;
    }
    __syncwarp();
    if (lane < g.hh) {
        float row[WYS];
#pragma unroll
        for (int p = 0; p < WYS; ++p) {
            row[p] = 0.f;
            if (p < P) {
                const int jj = lane - s_fn[wib][p][0];
                if ((unsigned)jj < (unsigned)s_fn[wib][p][1]) row[p] = s_wy[wib][p][jj];
            }
        }
#pragma unroll
        for (int p = 0; p < WYS; p += 4) *reinterpret_cast<float4 *>(&rec->wyd[lane][p]) = make_float4(row[p], row[p + 1], row[p + 2], row[p + 3]);
    }
    // bin groups: rows [gs, ge) reach group g = bins 4g .. 4g+3
    int gs[4], ge[4];
    bool dense = false;
#pragma unroll
    for (int gI = 0; gI < 4; ++gI) {
        const bool in = ybin && n > 0 && (lane - 16) / 4 == gI;
        int lo = in ? first - g.y0 : 255, hi = in ? first + n - g.y0 : 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (hi <= lo) {   // no bin of the group has a valid sample: an empty stretch at the end of the previous group
            lo = gI ? ge[gI - 1] : 0;
            hi = lo;
        }
        if (gI && lo < gs[gI - 1]) lo = gs[gI - 1];   // the row ranges of the bins ascend; keep the bounds monotone
        if (gI && hi < ge[gI - 1]) hi = ge[gI - 1];
        gs[gI] = lo;
        ge[gI] = hi;
        if (gI >= 2 && gs[gI] < ge[gI - 2]) dense = true;   // a row reaches three groups
    }
    if (lane == 0) {
#pragma unroll
        for (int gI = 0; gI < 4; ++gI) {
            rec->gs[gI] = (unsigned char)gs[gI];
            rec->ge[gI] = (unsigned char)ge[gI];
        }
        rec->sB = (unsigned char)gs[1];
        rec->eA = (unsigned char)ge[0];
        rec->gdense = dense ? 1 : 0;
        rec->nxmax = (unsigned char)nxmax;
    }
}

// ---------------------------------------------------------------------------------------------
// strip kernel
// ---------------------------------------------------------------------------------------------
struct __align__(16) UnitSlot {
    StripUnit u;
    int cg;        // channel group
    int row_base;  // position of row Y0 in the ring's running row count
    int next_item; // shared pop counter of the consumers
    int valid;     // 0: no more units
};

// ---- pieces shared by the two strip kernels ---------------------------------------------------------------------------
struct StripBars {
    uint32_t full0, empty0, ufull0, uempty0, rfull0;
};

template <int NR>
__device__ __forceinline__ void strip_producer(const StripArgs &a, UnitSlot *s_unit, float *s_ring, const StripBars &B) {
    const int ncg = a.C / kCG;
    const int nunits = a.counters[0] * ncg;
    unsigned g = 0;   // running row count of this CTA's ring
    for (unsigned uc = 0;; ++uc) {
        const unsigned us = uc % kNU;
        mbar_wait(B.uempty0 + 8 * us, ((uc / kNU) & 1) ^ 1);
        const int u = atomicAdd(a.counters + 1, 1);
        UnitSlot &S = s_unit[us];
        if (u >= nunits) {
            S.valid = 0;
            mbar_arrive(B.ufull0 + 8 * us);
            break;
        }
        const StripUnit d = a.units[u / ncg];
        S.u = d;
        S.cg = u % ncg;
        S.row_base = (int)g;
        S.next_item = 0;
        S.valid = 1;
        mbar_arrive(B.ufull0 + 8 * us);   // release: the slot's contents are visible to whoever acquires the phase
        const StripLevel &lv = a.lv[d.level];
        const float *src = lv.data + ((((size_t)d.b * ncg + S.cg) * lv.H + d.Y0) * lv.W + d.X0) * kCG;
        const uint32_t bytes = (uint32_t)d.BW * kCG * 4;
        const size_t rstride = (size_t)lv.W * kCG;
        for (int y = d.Y0; y < d.Y1; ++y, ++g, src += rstride) {
            const unsigned slot = g % NR;
            mbar_wait(B.empty0 + 8 * slot, ((g / NR) & 1) ^ 1);
            mbar_arrive_expect_tx(B.full0 + 8 * slot, bytes);
            tma_bulk_g2s(smem_u32(s_ring + (size_t)slot * kRowFloats), src, bytes, B.full0 + 8 * slot);
        }
    }
}

// Rows [from, to) of the current unit are behind this consumer: one arrival per row on its slot's `empty` barrier (by the
// consumer's warp 0 when `arrive`).  A slot's barrier only moves on to its next use once ALL consumers have arrived, and
// the producer refills the slot only then -- so before arriving for a row the lane first sees that row's `full` phase
// complete: that proves the slot's previous use has been released by everybody and this arrival is counted for the right
// phase (a consumer that skips more than NR rows would otherwise arrive twice in one phase).  EVERY warp walks the skipped
// rows' `full` phases: a parity wait can tell the current phase from the next one but not from the one after, so a warp
// must have seen row g - NR land before it may wait for row g -- otherwise the wait passes at once and the warp reads a
// slot that was never filled.  16 rows at a time: distinct slots per round.
template <int NR>
__device__ __forceinline__ void strip_release_rows(int from, int to, int row_base, int Y0, int lane, bool arrive, const StripBars &B) {
    for (int base = from; base < to; base += 16) {
        const int r = base + (lane & 15);
        if (lane < 16 && r < to) {
            const unsigned gg = (unsigned)(row_base + r - Y0);
            mbar_wait(B.full0 + 8 * (gg % NR), (gg / NR) & 1);
            if (arrive) mbar_arrive(B.empty0 + 8 * (gg % NR));
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// 7x7: one warp per (RoI, channel group)
// ---------------------------------------------------------------------------------------------
// lane = (channel-quad column q < 4, output column pw < 7), 28 active lanes, no barrier between warps anywhere.  A lane
// owns two float4 slices of the 32 channels (channels 4q.. and 16+4q..).  LDS.128 is served a quarter-warp at a time (8
// lanes = 2 output columns x 4 quads): lanes of an odd column load their HIGH slice first, so the two columns of a phase
// cover banks 0-15 and 16-31 and every tap load is conflict-free although the two columns read different cells.
// Row-major, x first: t = sum_j wx[j] * V[row][xs + j], then the row feeds the output rows it reaches.  The y pass is
// sparse at the granularity of two bin groups (bins 0-3, bins 4-6): the window rows split into a stretch that feeds only
// the first group, a stretch that feeds both and a stretch that feeds only the second -- three counted loops with
// statically named accumulators, no per-row control flow.
struct Strip7Cfg {
    static constexpr int NW = 15;                     // consumer warps (+ the producer warp = 512 threads, 128 registers each)
    static constexpr int NTHREADS = 32 * (NW + 1);
    static constexpr int TILE_FLOATS = 16 * 49;       // one 16-channel slice of a RoI: 3136 B, contiguous in the output
    static constexpr int FIXED = NW * (TILE_FLOATS * 4 + 2 * (int)sizeof(StripRec<7>)) + kNU * (int)sizeof(UnitSlot) + 16 * NW + 16 * kNU + 256;
    static constexpr int NR_RAW = (kSmemMax - FIXED) / (kRowFloats * 4 + 16);
    static constexpr int NR = NR_RAW > 32 ? 32 : NR_RAW;
    static_assert(NR >= kRMax + 2, "the ring must hold the tallest window plus some slack");
};

template <typename OutT>
__global__ void __launch_bounds__(Strip7Cfg::NTHREADS, 1) roi_align_strip7_kernel(const __grid_constant__ StripArgs a) {
    using Cfg = Strip7Cfg;
    using Rec = StripRec<7>;
    constexpr int P = 7, PP = 49, NW = Cfg::NW, NR = Cfg::NR;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *s_ring = reinterpret_cast<float *>(smem_raw);                              // [NR][kBW][32]
    float *s_tile = s_ring + (size_t)NR * kRowFloats;                                 // [NW][TILE_FLOATS]
    Rec *s_rec = reinterpret_cast<Rec *>(s_tile + NW * Cfg::TILE_FLOATS);            // [NW][2]
    UnitSlot *s_unit = reinterpret_cast<UnitSlot *>(s_rec + NW * 2);                  // [kNU]
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_unit + kNU);                     // full[NR], empty[NR], ufull[kNU], uempty[kNU], rfull[NW*2]
    StripBars B;
    B.full0 = smem_u32(s_bar);
    B.empty0 = B.full0 + 8 * NR;
    B.ufull0 = B.empty0 + 8 * NR;
    B.uempty0 = B.ufull0 + 8 * kNU;
    B.rfull0 = B.uempty0 + 8 * kNU;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < NR; ++s) {
            mbar_init(B.full0 + 8 * s, 1);
            mbar_init(B.empty0 + 8 * s, NW);
        }
        for (int s = 0; s < kNU; ++s) {
            mbar_init(B.ufull0 + 8 * s, 1);
            mbar_init(B.uempty0 + 8 * s, NW);
        }
        for (int s = 0; s < NW * 2; ++s) mbar_init(B.rfull0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid < 32) {
        if (tid == 0) strip_producer<NR>(a, s_unit, s_ring, B);
        return;
    }
    const int cw = (tid >> 5) - 1, lane = tid & 31;
    const bool worker = lane < 28;
    const int q = lane & 3, pw = worker ? lane >> 2 : 0;
    // this lane keeps its HIGH slice in register set 0; the four idle lanes share a quarter-warp with column 6 (even: low
    // half of its cell) and must read a high half, or that phase of every tap load is a 2-way bank conflict
    const bool odd = worker ? (pw & 1) != 0 : true;
    OutT *tile = reinterpret_cast<OutT *>(s_tile + cw * Cfg::TILE_FLOATS);   // a 16-bit tile fills half of its slot
    Rec *recs = s_rec + cw * 2;
    const uint32_t rf0 = B.rfull0 + 8 * (cw * 2);
    unsigned rec_uses[2] = {0u, 0u};
    bool store_pending = false;

    for (unsigned uc = 0;; ++uc) {
        const unsigned us = uc % kNU;
        mbar_wait(B.ufull0 + 8 * us, (uc / kNU) & 1);
        UnitSlot &S = s_unit[us];
        if (!S.valid) break;
        const StripUnit d = S.u;
        const int cg = S.cg, row_base = S.row_base;
        const Rec *gtab = reinterpret_cast<const Rec *>(a.records) + d.item_begin;
        int passed = d.Y0;   // first row of this unit the warp has not released yet
        auto fetch = [&](int item, int buf) {   // lane 0 only: the whole fixed-size record with one bulk copy
            mbar_arrive_expect_tx(rf0 + 8 * buf, (uint32_t)sizeof(Rec));
            tma_bulk_g2s(smem_u32(&recs[buf]), gtab + item, (uint32_t)sizeof(Rec), rf0 + 8 * buf);
        };
        int cur = 0, curbuf = 0;
        if (lane == 0) {
            cur = atomicAdd(&S.next_item, 1);
            if (cur < d.item_count) fetch(cur, 0);
        }
        cur = __shfl_sync(0xffffffffu, cur, 0);
        while (cur < d.item_count) {
            // ---- next item: pop + prefetch its record into the other buffer
            int nxt = 0;
            if (lane == 0) {
                nxt = atomicAdd(&S.next_item, 1);
                if (nxt < d.item_count) fetch(nxt, curbuf ^ 1);
            }
            nxt = __shfl_sync(0xffffffffu, nxt, 0);
            // ---- this item's record
            mbar_wait(rf0 + 8 * curbuf, rec_uses[curbuf] & 1);
            ++rec_uses[curbuf];
            const Rec &R = recs[curbuf];
            const int k = R.k, y0 = R.y0, hh = R.hh;
            // ---- release the rows above this window
            strip_release_rows<NR>(passed, y0, row_base, d.Y0, lane, true, B);
            const unsigned pos0 = (unsigned)(row_base + y0 - d.Y0);   // ring position of the window's first row
            // The window's rows are waited for four at a time while the sweep advances, and released as soon as neither
            // this item nor the warp's NEXT item (whose window top is read from its record once that has landed) needs
            // them: a warp then holds a few rows instead of its whole window for the whole item, which is what lets the
            // producer run ahead (with whole-window holds the 15 warps pinned spread + window = the entire ring and every
            // row load was exposed latency: 65 M spins on `full` barriers, profiles/r02_roialign_strip.md).
            const int nxu = R.nxmax;             // warp-uniform tap count: columns with fewer taps pad with weight 0
            const bool single = nxu <= 4 && !(a.dbg & 4);   // one sweep only: rows can be released behind it
            int rel = 0;                         // rows [0, rel) of the window are released
            int hold = 0;                        // rows < hold may be released once swept
            bool hold_known = false;
            if (nxt >= d.item_count) {
                hold = hh;
                hold_known = true;
            }
            float2 acc[2][P][2];   // [register set][output row][channel pair]
#pragma unroll
            for (int s = 0; s < 2; ++s)
#pragma unroll
                for (int i = 0; i < P; ++i) acc[s][i][0] = acc[s][i][1] = make_float2(0.f, 0.f);
            if (nxu > 0 && !(a.dbg & 1)) {
                const int nx = worker ? (int)R.nx[pw] : 0;
                const int xoff = R.x0 - d.X0 + (worker ? (int)R.xs[pw] : 0);
                const float *wxp = R.wx[pw];
                // register set 0 reads this float offset inside a cell, set 1 the other half of the 128-byte line.  All
                // addresses are 32-bit shared-window addresses (explicit ld.shared: no generic-pointer conversion per load)
                const uint32_t col0 = smem_u32(s_ring) + (uint32_t)((xoff * kCG + (odd ? 16 : 0) + 4 * q) * 4);
                const int d1 = odd ? -64 : 64;
                const uint32_t wyd0 = smem_u32(&R.wyd[0][0]);
                const int sB = R.sB, eA = R.eA;   // rows [sB, hh) feed bins 4-6, rows [0, eA) feed bins 0-3
                // ONE row loop per tap width (3 or 4: a lane with fewer taps repeats its own last cell with weight 0, so a
                // padded tap never touches memory the lane does not own): the code the 15 warps run at their different
                // places has to fit the instruction cache -- twelve specialised sweeps did not (26 % of the stall samples
                // were instruction fetches, profiles/r02_roialign_strip.md).  The bin group a row feeds is a warp-uniform
                // run-time test.
                auto sweep = [&](auto NXC, int j0) {
                    constexpr int NX = decltype(NXC)::value;
                    float wx[NX];
                    int toff[NX];
#pragma unroll
                    for (int j = 0; j < NX; ++j) {
                        const bool ok = j0 + j < nx;
                        wx[j] = ok ? wxp[j0 + j] : 0.f;
                        toff[j] = (ok ? j0 + j : (nx > 0 ? nx - 1 : 0)) * kCG * 4;
                    }
                    unsigned sl = pos0 % NR;
                    uint32_t rowp = col0 + sl * (uint32_t)(kRowFloats * 4);
                    uint32_t wyp = wyd0;
#pragma unroll 1
                    for (int rc = 0; rc < hh; rc += 4) {
                        const int nrow = min(4, hh - rc);
                        if (lane < nrow) {
                            const unsigned gg = pos0 + rc + lane;
                            mbar_wait(B.full0 + 8 * (gg % NR), (gg / NR) & 1);
                        }
                        __syncwarp();
#pragma unroll 1
                        for (int r = rc; r < rc + nrow; ++r) {
                            const bool gA = r < eA, gB = r >= sB;
                            if (gA || gB) {
                                float4 v[2][NX];
#pragma unroll
                                for (int s = 0; s < 2; ++s)
#pragma unroll
                                    for (int j = 0; j < NX; ++j) v[s][j] = lds_f4(rowp + toff[j] + s * d1);
                                float2 t[2][2];
#pragma unroll
                                for (int s = 0; s < 2; ++s) {
                                    t[s][0] = t[s][1] = make_float2(0.f, 0.f);
#pragma unroll
                                    for (int j = 0; j < NX; ++j) {
                                        t[s][0] = ffma2(wx[j], make_float2(v[s][j].x, v[s][j].y), t[s][0]);
                                        t[s][1] = ffma2(wx[j], make_float2(v[s][j].z, v[s][j].w), t[s][1]);
                                    }
                                }
                                if (gA) {
                                    const float4 wa = lds_f4(wyp);
#pragma unroll
                                    for (int s = 0; s < 2; ++s)
#pragma unroll
                                        for (int h = 0; h < 2; ++h) {
                                            acc[s][0][h] = ffma2(wa.x, t[s][h], acc[s][0][h]);
                                            acc[s][1][h] = ffma2(wa.y, t[s][h], acc[s][1][h]);
                                            acc[s][2][h] = ffma2(wa.z, t[s][h], acc[s][2][h]);
                                            acc[s][3][h] = ffma2(wa.w, t[s][h], acc[s][3][h]);
                                        }
                                }
                                if (gB) {
                                    const float4 wb = lds_f4(wyp + 16);
#pragma unroll
                                    for (int s = 0; s < 2; ++s)
#pragma unroll
                                        for (int h = 0; h < 2; ++h) {
                                            acc[s][4][h] = ffma2(wb.x, t[s][h], acc[s][4][h]);
                                            acc[s][5][h] = ffma2(wb.y, t[s][h], acc[s][5][h]);
                                            acc[s][6][h] = ffma2(wb.z, t[s][h], acc[s][6][h]);
                                        }
                                }
                            }
                            rowp += kRowFloats * 4;
                            wyp += 32;
                            if (++sl == NR) {
                                sl = 0;
                                rowp -= (uint32_t)NR * kRowFloats * 4;
                            }
                        }
                        // ---- rows behind the sweep go back to the producer
                        if (single) {
                            if (!hold_known) {
                                // ONE lane probes the next record's barrier and reads its window top; the warp takes that
                                // lane's answer (32 separate probes can straddle the phase flip and disagree, and a warp
                                // that disagrees about `rel` falls apart at the next __syncwarp)
                                int h = -1;
                                if (lane == 0 && mbar_test(rf0 + 8 * (curbuf ^ 1), rec_uses[curbuf ^ 1] & 1)) h = recs[curbuf ^ 1].y0 - y0;
                                h = __shfl_sync(0xffffffffu, h, 0);
                                if (h >= 0) {
                                    hold = h;
                                    hold_known = true;
                                }
                            }
                            const int lim = min(rc + nrow, hold);
                            __syncwarp();   // every lane has read the rows
                            if (lim > rel) {   // at most 4 + what an earlier chunk could not release yet: 16 lanes suffice twice over
                                for (int r2 = rel + lane; r2 < lim; r2 += 32) mbar_arrive(B.empty0 + 8 * ((pos0 + r2) % NR));
                                rel = lim;
                            }
                        }
                    }
                };
                // bins wider than 4 taps take further sweeps over taps 4.., 8.. (one call site: the sweep code exists once)
#pragma unroll 1
                for (int j0 = 0; j0 < nxu; j0 += 4) {
                    if (nxu - j0 <= 3) sweep(std::integral_constant<int, 3>{}, j0);
                    else sweep(std::integral_constant<int, 4>{}, j0);
                }
            }
            passed = max(passed, y0 + rel);
            // ---- flush: two 16-channel slices through the warp's tile, one asynchronous bulk store each (the values are
            // rounded to OutT in registers: a 16-bit slice is 1568 B, still a multiple of the bulk copy's 16 bytes)
            OutT *outp = static_cast<OutT *>(a.out) + ((size_t)k * a.C + (size_t)cg * kCG) * PP;
            auto flush = [&](auto HASBIAS) {
                constexpr bool kBias = decltype(HASBIAS)::value;
#pragma unroll
                for (int f = 0; f < 2; ++f) {
                    if (lane == 0 && store_pending) tma_store_wait_read();   // the previous store has read the tile
                    __syncwarp();
                    if (worker && !(a.dbg & 2)) {
                        const bool hi = odd != (f == 1);   // slice f sits in register set f ^ odd
                        float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (kBias) bz = ldg_f4(a.bias + (size_t)k * a.C + cg * kCG + 16 * f + 4 * q);
                        OutT *tp = tile + (4 * q) * PP + pw;
#pragma unroll
                        for (int i = 0; i < P; ++i) {
                            float a0 = hi ? acc[1][i][0].x : acc[0][i][0].x, a1 = hi ? acc[1][i][0].y : acc[0][i][0].y;
                            float a2 = hi ? acc[1][i][1].x : acc[0][i][1].x, a3 = hi ? acc[1][i][1].y : acc[0][i][1].y;
                            if (kBias) {
                                a0 += bz.x; a1 += bz.y; a2 += bz.z; a3 += bz.w;
                            }
                            tp[i * P] = to_out<OutT>(a0);
                            tp[i * P + PP] = to_out<OutT>(a1);
                            tp[i * P + 2 * PP] = to_out<OutT>(a2);
                            tp[i * P + 3 * PP] = to_out<OutT>(a3);
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        tma_bulk_s2g(outp + (size_t)f * Cfg::TILE_FLOATS, smem_u32(tile), Cfg::TILE_FLOATS * sizeof(OutT));
                        store_pending = true;
                    }
                }
            };
            if (a.bias) flush(std::true_type{});
            else flush(std::false_type{});
            cur = nxt;
            curbuf ^= 1;
        }
        // ---- unit done for this warp: release its remaining rows and the unit slot
        strip_release_rows<NR>(passed, d.Y1, row_base, d.Y0, lane, true, B);
        if (lane == 0) mbar_arrive(B.uempty0 + 8 * us);
    }
    if (lane == 0 && store_pending) tma_store_wait_all();
}

static size_t strip7_smem_bytes() {
    return (size_t)Strip7Cfg::NR * kRowFloats * 4 + Strip7Cfg::FIXED + 16 * Strip7Cfg::NR;
}

// ---------------------------------------------------------------------------------------------
// 14x14: a team of 4 warps per (RoI, channel group)
// ---------------------------------------------------------------------------------------------
// thread = (channel quad q < 8, output column pw < 14): 112 threads, 4 channels each; a quarter-warp reads the 8 quads of
// ONE cell (128 contiguous bytes), so the tap loads are conflict-free.  Same row-major sweep as the 7x7 kernel with four
// bin groups (0-3, 4-7, 8-11, 12-13): a row feeds one group or two neighbouring ones, which gives seven counted loops.
// The [32][14][14] result leaves in ONE pass through the team tile (25 KB) and one bulk store (see the flush).
struct Strip14Cfg {
    static constexpr int NT = 3, TW = 4, TEAM = TW * 32;
    static constexpr int NTHREADS = 32 + NT * TEAM;
    static constexpr int TILE_FLOATS = 32 * 196;      // the whole [32][14][14] result of a record: ONE bulk store
    static constexpr int FIXED = NT * (TILE_FLOATS * 4 + 2 * (int)sizeof(StripRec<14>)) + kNU * (int)sizeof(UnitSlot) + 64 * NT + 16 * kNU + 256;
    static constexpr int NR_RAW = (kSmemMax - FIXED) / (kRowFloats * 4 + 16);
    static constexpr int NR = NR_RAW > 32 ? 32 : NR_RAW;
    static_assert(NR >= kRMax + 2, "the ring must hold the tallest window plus some slack");
};

template <typename OutT>
__global__ void __launch_bounds__(Strip14Cfg::NTHREADS, 1) roi_align_strip14_kernel(const __grid_constant__ StripArgs a) {
    using Cfg = Strip14Cfg;
    using Rec = StripRec<14>;
    constexpr int P = 14, PP = 196, NT = Cfg::NT, TEAM = Cfg::TEAM, NR = Cfg::NR;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *s_ring = reinterpret_cast<float *>(smem_raw);                              // [NR][kBW][32]
    float *s_tile = s_ring + (size_t)NR * kRowFloats;                                 // [NT][TILE_FLOATS]
    Rec *s_rec = reinterpret_cast<Rec *>(s_tile + NT * Cfg::TILE_FLOATS);            // [NT][2]
    UnitSlot *s_unit = reinterpret_cast<UnitSlot *>(s_rec + NT * 2);                  // [kNU]
    int *s_pop = reinterpret_cast<int *>(s_unit + kNU);                               // [NT][2] broadcast of the popped item
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(s_pop + 8);                        // full[NR], empty[NR], ufull[kNU], uempty[kNU], rfull[NT*2]
    StripBars B;
    B.full0 = smem_u32(s_bar);
    B.empty0 = B.full0 + 8 * NR;
    B.ufull0 = B.empty0 + 8 * NR;
    B.uempty0 = B.ufull0 + 8 * kNU;
    B.rfull0 = B.uempty0 + 8 * kNU;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < NR; ++s) {
            mbar_init(B.full0 + 8 * s, 1);
            mbar_init(B.empty0 + 8 * s, NT);
        }
        for (int s = 0; s < kNU; ++s) {
            mbar_init(B.ufull0 + 8 * s, 1);
            mbar_init(B.uempty0 + 8 * s, NT);
        }
        for (int s = 0; s < NT * 2; ++s) mbar_init(B.rfull0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid < 32) {
        if (tid == 0) strip_producer<NR>(a, s_unit, s_ring, B);
        return;
    }
    const int ct = tid - 32;
    const int team = ct / TEAM, tt = ct % TEAM, twarp = tt >> 5, lane = tt & 31;
    const bool worker = tt < 8 * P;
    const int q = tt & 7, pw = worker ? tt >> 3 : 0;
    OutT *tile = reinterpret_cast<OutT *>(s_tile + team * Cfg::TILE_FLOATS);   // a 16-bit tile fills half of its slot
    Rec *recs = s_rec + team * 2;
    const uint32_t rf0 = B.rfull0 + 8 * (team * 2);
    const int bar_id = 1 + team;
    auto team_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(TEAM) : "memory"); };
    const bool r2 = (q & 2) != 0;   // quads 2,3 of a flush phase (see the flush)
    unsigned rec_uses[2] = {0u, 0u};
    bool store_pending = false;

    for (unsigned uc = 0;; ++uc) {
        const unsigned us = uc % kNU;
        mbar_wait(B.ufull0 + 8 * us, (uc / kNU) & 1);
        UnitSlot &S = s_unit[us];
        if (!S.valid) break;
        const StripUnit d = S.u;
        const int cg = S.cg, row_base = S.row_base;
        const Rec *gtab = reinterpret_cast<const Rec *>(a.records) + d.item_begin;
        int passed = d.Y0;
        auto fetch = [&](int item, int buf) {   // tt == 0 only
            mbar_arrive_expect_tx(rf0 + 8 * buf, (uint32_t)sizeof(Rec));
            tma_bulk_g2s(smem_u32(&recs[buf]), gtab + item, (uint32_t)sizeof(Rec), rf0 + 8 * buf);
        };
        int cur = 0, curbuf = 0;
        unsigned it = 0;   // s_pop is double buffered: the pop of iteration i+1 is written while iteration i's is still read
        if (tt == 0) {
            cur = atomicAdd(&S.next_item, 1);
            s_pop[team * 2] = cur;
            if (cur < d.item_count) fetch(cur, 0);
        }
        team_sync();
        cur = s_pop[team * 2];
        while (cur < d.item_count) {
            if (tt == 0) {
                const int nxt = atomicAdd(&S.next_item, 1);
                s_pop[team * 2 + ((it + 1) & 1)] = nxt;
                if (nxt < d.item_count) fetch(nxt, curbuf ^ 1);
            }
            mbar_wait(rf0 + 8 * curbuf, rec_uses[curbuf] & 1);
            ++rec_uses[curbuf];
            const Rec &R = recs[curbuf];
            const int k = R.k, y0 = R.y0, hh = R.hh;
            // every warp of the team first walks the `full` phases of the rows it leaves behind; only when ALL of them have
            // (team barrier) does warp 0 hand the rows back.  An arrival that ran ahead of a slower warp would let the
            // producer refill the slot twice before that warp looks at it, and a parity wait cannot tell phase n from n + 2.
            // 16 rows at a time: a longer stretch waited for as a whole would wait for slots this very team still holds.
            for (int base = passed; base < y0; base += 16) {
                const int hi = min(base + 16, y0);
                strip_release_rows<NR>(base, hi, row_base, d.Y0, lane, false, B);
                team_sync();
                if (twarp == 0 && base + lane < hi) mbar_arrive(B.empty0 + 8 * ((unsigned)(row_base + base + lane - d.Y0) % NR));
            }
            passed = max(passed, y0);
            {
                const unsigned gg = (unsigned)(row_base + y0 - d.Y0) + (lane < hh ? lane : 0);
                mbar_wait(B.full0 + 8 * (gg % NR), (gg / NR) & 1);
                __syncwarp();
            }
            float2 acc[P][2];
#pragma unroll
            for (int i = 0; i < P; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
            const int nxu = R.nxmax;   // team-uniform tap count: columns with fewer taps pad with weight 0 (no divergence)
            if (nxu > 0 && !(a.dbg & 1)) {
                const int nx = worker ? (int)R.nx[pw] : 0;
                const int xoff = R.x0 - d.X0 + (worker ? (int)R.xs[pw] : 0);
                const float *wxp = R.wx[pw];
                const unsigned slot0 = (unsigned)(row_base + y0 - d.Y0) % NR;
                // 32-bit shared-window addresses (explicit ld.shared: no generic-pointer conversion per load)
                const uint32_t col0 = smem_u32(s_ring) + (uint32_t)((xoff * kCG + 4 * q) * 4);
                const uint32_t wyd0 = smem_u32(&R.wyd[0][0]);
                // GRP bit g: bins 4g .. 4g+3
                auto rows = [&](auto NXC, auto GRPC, const float *wx, const int *toff, int r0, int r1_) {
                    constexpr int NX = decltype(NXC)::value, GRP = decltype(GRPC)::value;
                    unsigned sl = slot0 + r0;
                    if (sl >= NR) sl -= NR;
                    uint32_t rowp = col0 + sl * (uint32_t)(kRowFloats * 4);
                    uint32_t wyp = wyd0 + (uint32_t)r0 * 64;
#pragma unroll 1
                    for (int r = r0; r < r1_; ++r) {
                        float4 v[NX];
#pragma unroll
                        for (int j = 0; j < NX; ++j) v[j] = lds_f4(rowp + toff[j]);
                        float2 t0 = make_float2(0.f, 0.f), t1 = make_float2(0.f, 0.f);
#pragma unroll
                        for (int j = 0; j < NX; ++j) {
                            t0 = ffma2(wx[j], make_float2(v[j].x, v[j].y), t0);
                            t1 = ffma2(wx[j], make_float2(v[j].z, v[j].w), t1);
                        }
#pragma unroll
                        for (int gI = 0; gI < 4; ++gI) {
                            if (GRP & (1 << gI)) {
                                const float4 w = lds_f4(wyp + 16 * gI);
                                const float ws[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                                for (int e = 0; e < 4; ++e) {
                                    if (4 * gI + e < P) {
                                        acc[(4 * gI + e) % P][0] = ffma2(ws[e], t0, acc[(4 * gI + e) % P][0]);
                                        acc[(4 * gI + e) % P][1] = ffma2(ws[e], t1, acc[(4 * gI + e) % P][1]);
                                    }
                                }
                            }
                        }
                        rowp += kRowFloats * 4;
                        wyp += 64;
                        if (++sl == NR) {
                            sl = 0;
                            rowp -= (uint32_t)NR * kRowFloats * 4;
                        }
                    }
                };
                auto sweep = [&](auto NXC, int j0) {
                    constexpr int NX = decltype(NXC)::value;
                    float wx[NX];   // the x taps of this pass: set up once, shared by the (up to seven) row stretches
                    int toff[NX];
#pragma unroll
                    for (int j = 0; j < NX; ++j) {
                        const bool ok = j0 + j < nx;
                        wx[j] = ok ? wxp[j0 + j] : 0.f;
                        toff[j] = (ok ? j0 + j : (nx > 0 ? nx - 1 : 0)) * kCG * 4;   // a padded tap repeats the lane's own last cell
                    }
                    if (R.gdense) {   // a row feeds three groups (very small RoIs): every row feeds every bin
                        rows(NXC, std::integral_constant<int, 15>{}, wx, toff, 0, hh);
                        return;
                    }
                    const int s1 = R.gs[1], s2 = R.gs[2], s3 = R.gs[3], e0 = R.ge[0], e1 = R.ge[1], e2 = R.ge[2];
                    rows(NXC, std::integral_constant<int, 1>{}, wx, toff, 0, min(e0, s1));
                    rows(NXC, std::integral_constant<int, 3>{}, wx, toff, s1, e0);
                    rows(NXC, std::integral_constant<int, 2>{}, wx, toff, max(e0, s1), min(e1, s2));
                    rows(NXC, std::integral_constant<int, 6>{}, wx, toff, s2, e1);
                    rows(NXC, std::integral_constant<int, 4>{}, wx, toff, max(e1, s2), min(e2, s3));
                    rows(NXC, std::integral_constant<int, 12>{}, wx, toff, s3, e2);
                    rows(NXC, std::integral_constant<int, 8>{}, wx, toff, max(e2, s3), hh);
                };
#pragma unroll 1
                for (int j0 = 0; j0 < nxu; j0 += 4) {   // one call site: the sweep code exists once
                    switch (nxu - j0 < 4 ? nxu - j0 : 4) {
                        case 1: sweep(std::integral_constant<int, 1>{}, j0); break;
                        case 2: sweep(std::integral_constant<int, 2>{}, j0); break;
                        case 3: sweep(std::integral_constant<int, 3>{}, j0); break;
                        default: sweep(std::integral_constant<int, 4>{}, j0); break;
                    }
                }
            }
            // ---- flush: the [32][196] result through the team tile, one pass, one bulk store.  A channel row is 196 floats =
            // 4 banks, so the 8 quads of an output column sit 16 banks apart: quads 2,3 (mod 4) store their channel pairs in
            // swapped order (a rotation by two = a renaming of acc[.][0] / acc[.][1], one select per value), which leaves quad q
            // and q + 4 on the same bank -- a 2-way conflict, i.e. as many wavefronts as two half-warp passes would take at
            // half the issue slots (every warp holds quads of both halves, so a split pass is issued twice by every warp).
            OutT *outp = static_cast<OutT *>(a.out) + ((size_t)k * a.C + (size_t)cg * kCG) * PP;
            auto flush = [&](auto HASBIAS) {
                constexpr bool kBias = decltype(HASBIAS)::value;
                if (tt == 0 && store_pending) tma_store_wait_read();
                team_sync();
                if (worker && !(a.dbg & 2)) {
                    const int cl = 4 * q;
                    float4 bz = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (kBias) bz = ldg_f4(a.bias + (size_t)k * a.C + cg * kCG + 4 * q);
                    OutT *tp = tile + pw;
                    OutT *tlo = tp + (cl + (r2 ? 2 : 0)) * PP, *thi = tp + (cl + (r2 ? 0 : 2)) * PP;
#pragma unroll
                    for (int i = 0; i < P; ++i) {
                        float a0 = acc[i][0].x, a1 = acc[i][0].y, a2 = acc[i][1].x, a3 = acc[i][1].y;
                        if (kBias) {
                            a0 += bz.x; a1 += bz.y; a2 += bz.z; a3 += bz.w;
                        }
                        // first instruction pair: channels cl+0,1 for quads 0,1 (mod 4), cl+2,3 for quads 2,3
                        tlo[i * P] = to_out<OutT>(r2 ? a2 : a0);
                        tlo[i * P + PP] = to_out<OutT>(r2 ? a3 : a1);
                        thi[i * P] = to_out<OutT>(r2 ? a0 : a2);
                        thi[i * P + PP] = to_out<OutT>(r2 ? a1 : a3);
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                team_sync();
                if (tt == 0) {
                    tma_bulk_s2g(outp, smem_u32(tile), Cfg::TILE_FLOATS * sizeof(OutT));
                    store_pending = true;
                }
            };
            if (a.bias) flush(std::true_type{});
            else flush(std::false_type{});
            ++it;
            cur = s_pop[team * 2 + (it & 1)];   // written before the team barriers of the flush
            curbuf ^= 1;
        }
        for (int base = passed; base < d.Y1; base += 16) {
            const int hi = min(base + 16, d.Y1);
            strip_release_rows<NR>(base, hi, row_base, d.Y0, lane, false, B);
            team_sync();
            if (twarp == 0 && base + lane < hi) mbar_arrive(B.empty0 + 8 * ((unsigned)(row_base + base + lane - d.Y0) % NR));
        }
        team_sync();
        if (tt == 0) mbar_arrive(B.uempty0 + 8 * us);
    }
    if (tt == 0 && store_pending) tma_store_wait_all();
}

static size_t strip14_smem_bytes() {
    return (size_t)Strip14Cfg::NR * kRowFloats * 4 + Strip14Cfg::FIXED + 16 * Strip14Cfg::NR;
}

// ---------------------------------------------------------------------------------------------
// layout staging: NCHW / channels_last -> [B][C/32][H][W][32]
// ---------------------------------------------------------------------------------------------
// 32 channels x 64 pixels per CTA: reads 64 contiguous elements per channel, writes one contiguous 8 KB chunk.  InT: fp32,
// or fp16 / bf16 upcast exactly on the way in (the staged buffer is fp32 whatever the source type)
template <typename InT>
__global__ void __launch_bounds__(256) nchw_to_cg32_kernel(const InT *__restrict__ in, float *__restrict__ out, int C, int HW) {
    __shared__ float tile[32][65];
    const int b = blockIdx.z, cg = blockIdx.y, hw0 = blockIdx.x * 64;
    const int t = threadIdx.x;
    const InT *src = in + ((size_t)b * C + cg * 32) * HW;
    {   // thread = (channel r + 16k, pixel quad q): 128-bit loads (64-bit for 16-bit sources)
        const int r = t >> 4, q = (t & 15) * 4;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int c = r + 16 * k, hw = hw0 + q;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (hw + 3 < HW) v = ldg_in4(src + (size_t)c * HW + hw);
            else
                for (int e = 0; e < 4; ++e)
                    if (hw + e < HW) (&v.x)[e] = ldg_in1(src + (size_t)c * HW + hw + e);
            tile[c][q] = v.x; tile[c][q + 1] = v.y; tile[c][q + 2] = v.z; tile[c][q + 3] = v.w;
        }
    }
    __syncthreads();
    float *dst = out + (((size_t)b * (C / 32) + cg) * HW + hw0) * 32;
    {   // thread = (pixel p + 32k, channel quad q): 128-bit stores, a warp writes 4 pixels x 128 B
        const int p = t >> 3, q = (t & 7) * 4;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int px = p + 32 * k;
            if (hw0 + px < HW)
                *reinterpret_cast<float4 *>(dst + (size_t)px * 32 + q) = make_float4(tile[q][px], tile[q + 1][px], tile[q + 2][px], tile[q + 3][px]);
        }
    }
}

// channels_last source: [B][HW][C] -> [B][C/32][HW][32], a pure 128-byte-line permutation
template <typename InT>
__global__ void __launch_bounds__(256) nhwc_to_cg32_kernel(const InT *__restrict__ in, float *__restrict__ out, int C, long HW, long total4) {
    for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total4; i += (long)gridDim.x * blockDim.x) {
        // i indexes float4s of the OUTPUT: ((b*CG + cg)*HW + hw)*8 + q
        const int q = (int)(i & 7);
        const long r = i >> 3;
        const long hw = r % HW;
        const long bc = r / HW;
        const int cg = (int)(bc % (C / 32));
        const long b = bc / (C / 32);
        const float4 v = ldg_in4(in + ((size_t)(b * HW + hw)) * C + cg * 32 + q * 4);
        *reinterpret_cast<float4 *>(out + (size_t)i * 4) = v;
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int strip_nyp_env() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("NUHTC_RA_YROWS");
        v = e ? atoi(e) : 32;
        if (v < 8) v = 8;
    }
    return v;
}

static void strip_plan(const int *H, const int *W, int L, int B, StripLevel *lv, int *nkeys, int *nbins) {
    int key = 0, bin = 0;
    for (int l = 0; l < L; ++l) {
        lv[l].H = H[l];
        lv[l].W = W[l];
        lv[l].nstrips = W[l] <= kBW ? 1 : (W[l] + kCore - 1) / kCore;
        lv[l].ypart_rows = strip_nyp_env();
        lv[l].nyp = (H[l] + lv[l].ypart_rows - 1) / lv[l].ypart_rows;
        lv[l].key0 = key;
        lv[l].bin0 = bin;
        key += B * lv[l].nstrips * H[l];
        bin += B * lv[l].nstrips * lv[l].nyp;
    }
    *nkeys = key;
    *nbins = bin;
}

struct StripWs {
    size_t item_key, hist, cursor, bin_ymax, units, counters, leftover, records, total;
};
static StripWs strip_ws_layout(int K, int nkeys, int nbins, int P) {
    StripWs w;
    size_t o = 0;
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o = align_up(o + bytes, 256);
        return at;
    };
    w.counters = take(64);
    w.hist = take(sizeof(int) * ((size_t)nkeys + 1));
    w.bin_ymax = take(sizeof(int) * (size_t)nbins);
    // everything up to here is zeroed by one memset per call
    w.cursor = take(sizeof(int) * (size_t)nkeys);
    w.item_key = take(sizeof(int) * (size_t)K);
    w.units = take(sizeof(StripUnit) * (size_t)nbins);
    w.leftover = take(sizeof(int) * (size_t)K);
    w.records = take((P == 7 ? sizeof(StripRec<7>) : sizeof(StripRec<14>)) * (size_t)K);
    w.total = o;
    return w;
}

size_t roi_strip_workspace_bytes(const int *H, const int *W, int L, int B, int K, int P) {
    StripLevel lv[NUHTC_MAX_LEVELS];
    int nkeys, nbins;
    strip_plan(H, W, L, B, lv, &nkeys, &nbins);
    return strip_ws_layout(K, nkeys, nbins, P).total;
}

bool roi_strip_supported(int C, int PH, int PW, int mode, int L) {
    return PH == PW && (PH == 7 || PH == 14) && C % 32 == 0 && C >= 32 && (mode == NUHTC_ROI_ROUTE || L == 1);
}

template <int P, typename OutT>
static int strip_launch(StripArgs &a, const RoiLevels &lv, cudaStream_t st, const StripWs &w, char *ws) {
    static bool attr_done[kNuhtcMaxDevices] = {false};
    const int dev = nuhtc_device();
    const size_t smem = P == 7 ? strip7_smem_bytes() : strip14_smem_bytes();
    if (!attr_done[dev]) {
        if (P == 7) NUHTC_CUDA(cudaFuncSetAttribute(roi_align_strip7_kernel<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else NUHTC_CUDA(cudaFuncSetAttribute(roi_align_strip14_kernel<OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[dev] = true;
    }
    NUHTC_CUDA(cudaMemsetAsync(ws + w.counters, 0, w.cursor - w.counters, st));
    const int warps_per_block = 8;
    const unsigned gblocks = (unsigned)((a.K + warps_per_block - 1) / warps_per_block);
    strip_keys_kernel<P><<<gblocks, 256, 0, st>>>(a);
    NUHTC_LAUNCH_CHECK();
    static bool scan_attr[kNuhtcMaxDevices] = {false};
    if (!scan_attr[dev]) {
        NUHTC_CUDA(cudaFuncSetAttribute(strip_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmemMax));
        scan_attr[dev] = true;
    }
    strip_scan_kernel<<<1, 1024, (size_t)a.nkeys * sizeof(int), st>>>(a);
    NUHTC_LAUNCH_CHECK();
    strip_records_kernel<P><<<gblocks, 256, 0, st>>>(a);
    NUHTC_LAUNCH_CHECK();
    if (P == 7) roi_align_strip7_kernel<OutT><<<nuhtc_sm_count(), Strip7Cfg::NTHREADS, smem, st>>>(a);
    else roi_align_strip14_kernel<OutT><<<nuhtc_sm_count(), Strip14Cfg::NTHREADS, smem, st>>>(a);
    NUHTC_LAUNCH_CHECK();
    (void)lv;
    return NUHTC_OK;
}

// Fills `a` and runs prepass + strip kernel; the caller then runs its per-RoI kernel over the leftover list
// (*leftover, *leftover_count are device pointers into the workspace).
int roi_strip_forward(const RoiLevels &lv, int B, int C, const float *rois, int K, int P, int sr, int aligned, int mode,
                      float finest, void *out, int out_dtype, const float *bias, void *ws_, size_t ws_bytes, cudaStream_t st,
                      const int **leftover, const int **leftover_count) {
    StripArgs a;
    memset(&a, 0, sizeof a);
    int H[NUHTC_MAX_LEVELS], W[NUHTC_MAX_LEVELS];
    for (int l = 0; l < lv.L; ++l) {
        H[l] = lv.H[l];
        W[l] = lv.W[l];
    }
    strip_plan(H, W, lv.L, B, a.lv, &a.nkeys, &a.nbins);
    for (int l = 0; l < lv.L; ++l) {
        a.lv[l].data = lv.data[l];
        a.lv[l].scale = lv.scale[l];
    }
    if ((size_t)a.nkeys * sizeof(int) > (size_t)kScanSmemMax) return 1;   // maps too large for the binning: per-RoI kernel
    const StripWs w = strip_ws_layout(K, a.nkeys, a.nbins, P);
    if (ws_bytes < w.total || !ws_) {
        nuhtc_set_error("roi_align: workspace %zu < %zu bytes", ws_bytes, w.total);
        return NUHTC_EWORKSPACE;
    }
    char *ws = (char *)ws_;
    static const int dbg = getenv("NUHTC_RA_DBG") ? atoi(getenv("NUHTC_RA_DBG")) : 0;
    a.dbg = dbg;
    a.L = lv.L;
    a.B = B;
    a.C = C;
    a.K = K;
    a.sr = sr;
    a.aligned = aligned;
    a.mode = mode;
    a.finest = finest;
    a.rois = rois;
    a.out = out;
    a.bias = bias;
    a.item_key = (int *)(ws + w.item_key);
    a.hist = (int *)(ws + w.hist);
    a.cursor = (int *)(ws + w.cursor);
    a.bin_ymax = (int *)(ws + w.bin_ymax);
    a.units = (StripUnit *)(ws + w.units);
    a.counters = (int *)(ws + w.counters);
    a.leftover = (int *)(ws + w.leftover);
    a.records = ws + w.records;
    *leftover = a.leftover;
    *leftover_count = a.counters + 2;
    switch (out_dtype) {
        case NUHTC_DTYPE_F16: return P == 7 ? strip_launch<7, __half>(a, lv, st, w, ws) : strip_launch<14, __half>(a, lv, st, w, ws);
        case NUHTC_DTYPE_BF16:
            return P == 7 ? strip_launch<7, __nv_bfloat16>(a, lv, st, w, ws) : strip_launch<14, __nv_bfloat16>(a, lv, st, w, ws);
        default: return P == 7 ? strip_launch<7, float>(a, lv, st, w, ws) : strip_launch<14, float>(a, lv, st, w, ws);
    }
}

template <typename InT>
static int to_cg32_launch(const InT *in, float *out, int B, int C, int H, int W, int channels_last, cudaStream_t st) {
    const int HW = H * W;
    if (channels_last) {
        const long total4 = (long)B * C * HW / 4;
        long blocks = (total4 + 255) / 256;
        const long cap = (long)nuhtc_sm_count() * 16;
        if (blocks > cap) blocks = cap;
        nhwc_to_cg32_kernel<InT><<<(unsigned)blocks, 256, 0, st>>>(in, out, C, HW, total4);
    } else {
        dim3 grid((HW + 63) / 64, C / 32, B);
        nchw_to_cg32_kernel<InT><<<grid, 256, 0, st>>>(in, out, C, HW);
    }
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}

int roi_to_cg32(const void *in, int in_dtype, float *out, int B, int C, int H, int W, int channels_last, cudaStream_t st) {
    switch (in_dtype) {
        case NUHTC_DTYPE_F16: return to_cg32_launch(static_cast<const __half *>(in), out, B, C, H, W, channels_last, st);
        case NUHTC_DTYPE_BF16: return to_cg32_launch(static_cast<const __nv_bfloat16 *>(in), out, B, C, H, W, channels_last, st);
        default: return to_cg32_launch(static_cast<const float *>(in), out, B, C, H, W, channels_last, st);
    }
}
