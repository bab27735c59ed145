// Device helpers shared by the RoIAlign kernels (roi_align.cu, roi_strip.cu): level routing, RoI geometry in the
// reference's fp32 op order, per-axis tap tables, packed fp32x2 FMA, mbarrier / TMA bulk-copy wrappers.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

struct RoiLevels {
    const float *data[NUHTC_MAX_LEVELS];
    int H[NUHTC_MAX_LEVELS];
    int W[NUHTC_MAX_LEVELS];
    float scale[NUHTC_MAX_LEVELS];
    int pool2[NUHTC_MAX_LEVELS];   // != 0: this level is pooled at twice the output size and 2x2-averaged (see roi_geom)
    int L;
};

// SingleRoIExtractor.map_roi_levels (single_level_roi_extractor.py:51-55):
//   torch.floor(torch.log2(sqrt(w*h)/finest + 1e-6)).clamp(0, L-1)
// The reference evaluates log2 in fp32, so a value just below a power of two can round UP to the integer and land one
// level higher than the exact logarithm would put it (v = nextbelow(8.0f): log2 = 3 - 8.6e-8 rounds to 3.0f).  The
// contract is the reference's CPU path (the oracle): IEEE sub/mul/sqrt/div/add, and torch's CPU log2, which is the
// correctly rounded fp32 logarithm on every float within +-200 000 ulps of the boundaries 2, 4, 8 (checked against
// float(log2(double)) in tests/test_oracle_cpu.py) -- reproduced here as float(log2(double(v))).  torch's CUDA ops differ from
// its CPU ops at this point (x / 56 becomes x * (1/56), log2f is libdevice's), so the reference itself routes a handful of
// boundary boxes differently on the two devices; tests/test_gpu_roi_align.py reports that count.
__device__ __forceinline__ int route_level(const float *roi, int L, float finest) {
    const float s = __fsqrt_rn(__fmul_rn(__fsub_rn(roi[3], roi[1]), __fsub_rn(roi[4], roi[2])));
    const float v = __fadd_rn(__fdiv_rn(s, finest), 1e-6f);
    const float f = floorf((float)log2((double)v));   // NaN (negative area) clamps to level 0
    int l = 0;
    if (f >= 1.0f) l = f >= (float)(L - 1) ? L - 1 : (int)f;
    return l;
}

struct RoiGeom {
    float start_w, start_h, bin_w, bin_h;
    int gw, gh;
    float count;
    int b;
};

// pool2: the level enters as `adaptive_avg_pool2d(RoIAlign(2PH x 2PW, sampling_ratio=0), (PH, PW))` -- the semantic branch of
// NuHTC's _bbox_forward (nuhtc/models/htc_roi_head_cus.py:193-199).  Averaging the 2x2 bins of a (2PH x 2PW) RoIAlign with g
// samples per bin and axis IS a (PH x PW) RoIAlign with 2g samples per bin and axis (same sample positions, one division by
// 4*g*g), so the level is pooled directly at the output size with g = 2 * ceil(roi_extent / (2P)).
__device__ __forceinline__ RoiGeom roi_geom(const float *roi, float scale, int PH, int PW, int sr, int aligned, int pool2 = 0) {
    RoiGeom g;
    const float off = aligned ? 0.5f : 0.0f;
    g.start_w = __fsub_rn(__fmul_rn(roi[1], scale), off);
    g.start_h = __fsub_rn(__fmul_rn(roi[2], scale), off);
    const float ew = __fsub_rn(__fmul_rn(roi[3], scale), off);
    const float eh = __fsub_rn(__fmul_rn(roi[4], scale), off);
    float rw = __fsub_rn(ew, g.start_w), rh = __fsub_rn(eh, g.start_h);
    if (!aligned) {
        rw = fmaxf(rw, 1.0f);
        rh = fmaxf(rh, 1.0f);
    }
    g.bin_h = __fdiv_rn(rh, (float)PH);
    g.bin_w = __fdiv_rn(rw, (float)PW);
    if (pool2) {
        g.gh = 2 * (int)ceilf(__fdiv_rn(rh, (float)(2 * PH)));
        g.gw = 2 * (int)ceilf(__fdiv_rn(rw, (float)(2 * PW)));
    } else {
        g.gh = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rh, (float)PH));
        g.gw = sr > 0 ? sr : (int)ceilf(__fdiv_rn(rw, (float)PW));
    }
    int c = g.gh * g.gw;
    if (c < 1) c = 1;
    g.count = (float)c;
    g.b = (int)roi[0];
    return g;
}

// sample coordinate, same association as the CPU reference: (start + p*bin) + ((i+.5)*bin)/g
__device__ __forceinline__ float sample_coord(float start, float bin, int p, int i, int g) {
    return __fadd_rn(__fadd_rn(start, __fmul_rn((float)p, bin)),
                     __fdiv_rn(__fmul_rn((float)i + 0.5f, bin), (float)g));
}

// one axis of the bilinear sample: false if the sample is outside (-1, D)
__device__ __forceinline__ bool axis_sample(float c, int D, int &lo, int &hi, float &l, float &h) {
    if (c < -1.0f || c > (float)D) return false;
    if (c <= 0.f) c = 0.f;
    lo = (int)c;
    if (lo >= D - 1) {
        hi = lo = D - 1;
        c = (float)lo;
    } else {
        hi = lo + 1;
    }
    l = __fsub_rn(c, (float)lo);
    h = __fsub_rn(1.0f, l);
    return true;
}

constexpr int kMaxTap = 8; // taps per bin per axis held in the tables; larger bins take the literal path

// per-axis tap table for bin p: accumulated bilinear weights over the g samples of the bin, each
// divided by `div` (1 for x, the sample count for y).  n = -1 flags a bin with more than kMaxTap taps.
__device__ __forceinline__ void build_axis_taps(float start, float bin, int g, int p, int D, float div, float *w, int *first,
                                                int *n) {
#pragma unroll
    for (int j = 0; j < kMaxTap; ++j) w[j] = 0.f;
    int base = -1, last = -1;
    bool ok = true;
    for (int i = 0; i < g; ++i) {
        const float c = sample_coord(start, bin, p, i, g);
        int lo, hi;
        float l, h;
        if (!axis_sample(c, D, lo, hi, l, h)) continue;
        if (base < 0) base = lo;
        const int a = lo - base, b = hi - base;
        if (b >= kMaxTap) {
            ok = false;
            break;
        }
        w[a] += h;
        w[b] += l;
        last = b;
    }
    if (ok && div != 1.0f) {
#pragma unroll
        for (int j = 0; j < kMaxTap; ++j) w[j] = __fdiv_rn(w[j], div);
    }
    *first = base < 0 ? 0 : base;
    *n = ok ? last + 1 : -1;
}

// two fp32 FMAs in one instruction (Blackwell FFMA2): d = a * {b.x, b.y} + c
__device__ __forceinline__ float2 ffma2(float a, float2 b, float2 c) {
    unsigned long long ra, rb, rc, rd;
    asm("mov.b64 %0, {%1, %1};" : "=l"(ra) : "f"(a));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
    return d;
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
#ifdef NUHTC_WATCHDOG
// debug build: a wait that lasts longer than ~2 s reports itself and traps (which barrier, which thread)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    const long long t0 = clock64();
    for (;;) {
        uint32_t ok;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(bar), "r"(parity)
            : "memory");
        if (ok) return;
        if (clock64() - t0 > 4000000000LL) {
            printf("STUCK block %d thread %d bar +0x%x parity %u\n", blockIdx.x, threadIdx.x, bar & 0x3ffff, parity);
            __trap();
        }
    }
}
#else
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
#endif
// 128-bit load from a 32-bit shared-window address
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
// one non-blocking probe of a phase (true: the phase with this parity has completed)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}

__device__ __forceinline__ void tma_bulk_s2g(void *dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }


// ---- element types (NUHTC_DTYPE_*) --------------------------------------------------------------------------------------
// Half-precision levels are upcast exactly while they are staged; every RoIAlign kernel computes in fp32 and rounds each
// output value once, round-to-nearest-even, to the output type at its final store (mmcv's force_fp32(out_fp16=True)).
template <typename T> __device__ __forceinline__ T to_out(float v);
template <> __device__ __forceinline__ float to_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __half to_out<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 to_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

__device__ __forceinline__ uint32_t bits16(__half v) { return __half_as_ushort(v); }
__device__ __forceinline__ uint32_t bits16(__nv_bfloat16 v) { return __bfloat16_as_ushort(v); }

// four consecutive output elements, streaming store: 16 bytes for fp32, 8 bytes for the 16-bit types
__device__ __forceinline__ void st_stream4(float *p, float a, float b, float c, float d) { st_stream_f4(p, make_float4(a, b, c, d)); }
template <typename T>
__device__ __forceinline__ void st_stream4(T *p, T a, T b, T c, T d) {
    asm volatile("st.global.cs.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(bits16(a) | bits16(b) << 16), "r"(bits16(c) | bits16(d) << 16)
                 : "memory");
}
__device__ __forceinline__ void st_stream1(float *p, float v) { __stcs(p, v); }
template <typename T>
__device__ __forceinline__ void st_stream1(T *p, T v) {
    asm volatile("st.global.cs.u16 [%0], %1;" ::"l"(p), "h"((unsigned short)bits16(v)) : "memory");
}

// four consecutive input elements, upcast exactly to fp32 (bf16: a 16-bit shift, so subnormals stay exact)
__device__ __forceinline__ float4 ldg_in4(const float *p) { return ldg_f4(p); }
__device__ __forceinline__ float4 ldg_in4(const __half *p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    const float2 lo = __half22float2(*reinterpret_cast<const __half2 *>(&u.x)), hi = __half22float2(*reinterpret_cast<const __half2 *>(&u.y));
    return make_float4(lo.x, lo.y, hi.x, hi.y);
}
__device__ __forceinline__ float4 ldg_in4(const __nv_bfloat16 *p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2 *>(p));
    return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xffff0000u), __uint_as_float(u.y << 16),
                       __uint_as_float(u.y & 0xffff0000u));
}
__device__ __forceinline__ float ldg_in1(const float *p) { return __ldg(p); }
__device__ __forceinline__ float ldg_in1(const __half *p) { return __half2float(__ushort_as_half(__ldg(reinterpret_cast<const unsigned short *>(p)))); }
__device__ __forceinline__ float ldg_in1(const __nv_bfloat16 *p) {
    return __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short *>(p)) << 16);
}
