// The detector's test-time image pipeline for sm_100a: what `inference_detector` (mmdet/apis/inference.py:90-153) does
// to every tile on the CPU -- cv2 bilinear upscale, BGR->RGB, (x - mean) / std, zero pad to the size divisor, HWC->CHW --
// as ONE launch from uint8 tiles [B,h,w,3] to the fp32 batch [B,3,Hp,Wp] the backbone reads.
//
// Bit-exact with cv2 4.x / mmcv 1.7.2:
//   * resize coefficients: fx = (float)((dx + 0.5) * scale - 0.5) in double, floor, 11-bit weights rint((1 - f) * 2048),
//     rint(f * 2048); columns clamp index AND fraction at the borders, rows clamp only the indices (cv2's resize setup);
//   * horizontal pass in int32, vertical pass in cv2's SIMD form ((H0 >> 4) * b0 >> 16) + ((H1 >> 4) * b1 >> 16) + 2 >> 2;
//   * normalisation: a per-CTA 3x256 table (float)(((double)v - mean) * (1.0 / (double)std)), exactly what cv2.subtract /
//     cv2.multiply with float64 scalars give (the resized byte is the only input, so a table is the whole operation).
// Every double step is an explicit __d*_rn so nvcc cannot contract it into an FMA the CPU did not execute.
//
// Work split: one thread per (image, band of up to kMaxBandRows output rows, 4 output columns).  A warp writes 512
// contiguous bytes of each channel plane per row with streaming 128-bit stores; the kernel writes 16x the bytes it reads.
// Walking down its band the thread keeps the horizontal pass of the current source row pair in registers, so each source
// byte it needs is loaded (from L1) once per band rather than once per output row.
#include <climits>

#include "common.cuh"

namespace {

constexpr int kMaxBandRows = 8;   // output rows per thread, at most

__device__ __forceinline__ void coeff(int d, double scale, int n_in, bool reset_border, int &s, int &a0, int &a1) {
    float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
    const float fl = floorf(f);
    s = (int)fl;
    f = __fsub_rn(f, fl);
    if (reset_border) {
        if (s < 0) s = 0, f = 0.f;
        if (s >= n_in - 1) s = n_in - 1, f = 0.f;
    }
    a1 = __float2int_rn(__fmul_rn(f, 2048.f));
    a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
}

// H[j][k] = (S[p0[j] + k] * a0[j] + S[p1[j] + k] * a1[j]) >> 4 for the thread's 4 columns of one source row (the >> 4 is
// the first step of cv2's vertical pass)
__device__ __forceinline__ void hrow(const uint8_t *__restrict__ row, const int (&p0)[4], const int (&p1)[4], const int (&a0)[4],
                                     const int (&a1)[4], int (&H)[4][3]) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int k = 0; k < 3; ++k) H[j][k] = ((int)__ldg(row + p0[j] + k) * a0[j] + (int)__ldg(row + p1[j] + k) * a1[j]) >> 4;
}

}  // namespace

// Outside the anonymous namespace and with builtin parameter types: the kernel's name is the same in every build.
__global__ void __launch_bounds__(256) nuhtc_preprocess_tiles_kernel(const uint8_t *__restrict__ tiles, int B, int h, int w,
                                                                     int new_h, int new_w, int pad_h, int pad_w, int to_rgb,
                                                                     int vec, int band_rows, float3 mean, float3 stdv, double scale_y,
                                                                     double scale_x, float *__restrict__ out) {
    __shared__ float lut[3][256];
    for (int i = threadIdx.x; i < 3 * 256; i += blockDim.x) {
        const int c = i >> 8, v = i & 255;
        const float m = c == 0 ? mean.x : c == 1 ? mean.y : mean.z, sd = c == 0 ? stdv.x : c == 1 ? stdv.y : stdv.z;
        const double inv = __ddiv_rn(1.0, (double)sd);
        lut[c][v] = __double2float_rn(__dmul_rn(__dsub_rn((double)v, (double)m), inv));
    }
    __syncthreads();

    const int nq = (pad_w + 3) >> 2, nbands = (pad_h + band_rows - 1) / band_rows;
    const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= (int64_t)B * nbands * nq) return;
    const int q = (int)(item % nq);
    const int64_t bb = item / nq;
    const int band = (int)(bb % nbands), b = (int)(bb / nbands);
    const int x0 = q * 4;

    // the thread's 4 columns: source byte offsets and weights (fixed down the band)
    int p0[4], p1[4], a0[4], a1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int sx;
        coeff(x0 + j, scale_x, w, true, sx, a0[j], a1[j]);
        p0[j] = sx * 3;
        p1[j] = min(sx + 1, w - 1) * 3;
        if (x0 + j >= new_w) p0[j] = p1[j] = a0[j] = a1[j] = 0;   // pad column: never stored
    }
    const uint8_t *img = tiles + (size_t)b * h * w * 3;
    // horizontal pass of source rows sy and sy + 1, kept in registers while the band walks down: with s >= 1 the source
    // row advances by at most one per output row, so each source row is read once per band
    int H0[4][3], H1[4][3];
    int cur = INT_MIN;
    const size_t plane = (size_t)pad_h * pad_w;
    const int y_end = min((band + 1) * band_rows, pad_h);
    for (int y = band * band_rows; y < y_end; ++y) {
        float v[3][4];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int j = 0; j < 4; ++j) v[c][j] = 0.f;
        if (y < new_h) {
            int sy, b0, b1;
            coeff(y, scale_y, h, false, sy, b0, b1);
            if (sy != cur) {
                const bool step = sy == cur + 1;
                if (step) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int k = 0; k < 3; ++k) H0[j][k] = H1[j][k];
                } else {
                    hrow(img + (size_t)min(max(sy, 0), h - 1) * w * 3, p0, p1, a0, a1, H0);
                }
                hrow(img + (size_t)min(max(sy + 1, 0), h - 1) * w * 3, p0, p1, a0, a1, H1);
                cur = sy;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    // H >> 4 <= 32655 and b0 + b1 <= 2049 keep r in [0, 255] (cv2's saturation never acts); the min only
                    // guards the table index
                    const int r = min((((H0[j][k] * b0) >> 16) + ((H1[j][k] * b1) >> 16) + 2) >> 2, 255);
                    v[k][j] = x0 + j < new_w ? lut[to_rgb ? 2 - k : k][r] : 0.f;   // v by SOURCE channel (registers)
                }
        }
        if (to_rgb) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float t = v[0][j];
                v[0][j] = v[2][j];
                v[2][j] = t;
            }
        }
        float *o = out + (size_t)b * 3 * plane + (size_t)y * pad_w + x0;
        if (vec) {
#pragma unroll
            for (int c = 0; c < 3; ++c) st_stream_f4(o + c * plane, make_float4(v[c][0], v[c][1], v[c][2], v[c][3]));
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c)
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (x0 + j < pad_w) o[c * plane + j] = v[c][j];
        }
    }
}

NUHTC_API int nuhtc_preprocess_tiles(const uint8_t *tiles, int B, int h, int w, int new_h, int new_w, int pad_h, int pad_w,
                                     int to_rgb, const float *mean3, const float *std3, float *out, void *stream) {
    NUHTC_CHECK_ARG(B >= 0, "preprocess_tiles: B=%d < 0", B);
    NUHTC_CHECK_ARG(h > 0 && w > 0 && new_h > 0 && new_w > 0 && pad_h > 0 && pad_w > 0,
                    "preprocess_tiles: sizes must be > 0 (h=%d w=%d new=%dx%d pad=%dx%d)", h, w, new_h, new_w, pad_h, pad_w);
    NUHTC_CHECK_ARG(new_h >= h && new_w >= w, "preprocess_tiles: new size %dx%d < tile %dx%d (downscaling is not supported)",
                    new_h, new_w, h, w);
    NUHTC_CHECK_ARG(pad_h >= new_h && pad_w >= new_w, "preprocess_tiles: pad %dx%d < new size %dx%d", pad_h, pad_w, new_h, new_w);
    NUHTC_CHECK_ARG((int64_t)B * pad_h * ((pad_w + 3) / 4) < (int64_t)INT32_MAX * 256,
                    "preprocess_tiles: batch too large (B=%d, pad %dx%d)", B, pad_h, pad_w);
    if (B == 0) return NUHTC_OK;
    NUHTC_CHECK_ARG(tiles && out && mean3 && std3, "preprocess_tiles: null tiles / out / mean3 / std3 with B=%d", B);
    const float3 mean = make_float3(mean3[0], mean3[1], mean3[2]), stdv = make_float3(std3[0], std3[1], std3[2]);
    const double scale_y = 1.0 / ((double)new_h / h), scale_x = 1.0 / ((double)new_w / w);  // cv2: 1 / inv_scale
    const int vec = (pad_w % 4 == 0) && ((uintptr_t)out % 16 == 0);  // 128-bit stores need aligned rows
    // the longest band that still gives two waves of resident threads (3 CTAs of 256 per SM): longer bands read each
    // source row fewer times, shorter ones fill the GPU on small batches
    int band_rows = kMaxBandRows;
    const int64_t quads = (int64_t)B * ((pad_w + 3) / 4);
    while (band_rows > 1 && quads * ((pad_h + band_rows - 1) / band_rows) < 2LL * nuhtc_sm_count() * 768) band_rows /= 2;
    const int64_t items = quads * ((pad_h + band_rows - 1) / band_rows);
    const unsigned grid = (unsigned)((items + 255) / 256);
    nuhtc_preprocess_tiles_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(tiles, B, h, w, new_h, new_w, pad_h, pad_w, to_rgb,
                                                                          vec, band_rows, mean, stdv, scale_y, scale_x, out);
    NUHTC_LAUNCH_CHECK();
    return NUHTC_OK;
}
