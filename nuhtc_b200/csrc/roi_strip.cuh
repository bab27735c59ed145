// Host interface of the strip-shared RoIAlign path (roi_strip.cu), used by the C ABI in roi_align.cu.
#pragma once
#include "roi_common.cuh"

size_t roi_strip_workspace_bytes(const int *H, const int *W, int L, int B, int K, int P);
bool roi_strip_supported(int C, int PH, int PW, int mode, int L);
// prepass + strip kernel on levels in the [B][C/32][H][W][32] layout.  RoIs whose windows cannot be staged are listed in
// *leftover[0 .. **leftover_count) (device memory inside the workspace) for the caller's per-RoI kernel.
// `out` holds elements of `out_dtype` (NUHTC_DTYPE_*).
int roi_strip_forward(const RoiLevels &lv, int B, int C, const float *rois, int K, int P, int sr, int aligned, int mode,
                      float finest, void *out, int out_dtype, const float *bias, void *ws, size_t ws_bytes, cudaStream_t st,
                      const int **leftover, const int **leftover_count);
int roi_to_cg32(const void *in, int in_dtype, float *out, int B, int C, int H, int W, int channels_last, cudaStream_t st);
