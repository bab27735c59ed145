/*
 * nuhtc_b200.h -- C ABI of libnuhtc_b200.so: the B200 (sm_100a) RoI stage + merge of NuHTC.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream (passed as void*,
 * a cudaStream_t).  No entry point allocates device memory or synchronises the stream unless
 * its comment says so: the caller owns inputs, outputs and workspaces (sizes come from the
 * *_workspace_bytes helpers).  All return 0 on success or a negative NUHTC_E* code;
 * nuhtc_last_error() gives a thread-local message for the last failure.
 *
 * The reference interface each entry point replaces is cited as file:line under
 * /root/reference (boyden/NuHTC).  mmcv-full 1.7.2 itself is not vendored there; its FFI
 * (`ext_module.roi_align_forward`, `ext_module.nms`) is what these mirror.
 */
#ifndef NUHTC_B200_H
#define NUHTC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NUHTC_OK 0
#define NUHTC_EINVAL (-1)     /* bad argument */
#define NUHTC_ECUDA (-2)      /* a CUDA runtime call or launch failed */
#define NUHTC_EWORKSPACE (-3) /* workspace too small */
#define NUHTC_EOVERFLOW (-4)  /* a device-side capacity bound was exceeded (see status words) */

#define NUHTC_MAX_LEVELS 8

int nuhtc_abi_version(void);
const char *nuhtc_last_error(void);

/* ---- layout ------------------------------------------------------------------------------
 * FPN levels arrive NCHW fp32 (the mmcv contract).  The RoIAlign gather wants the channel axis
 * contiguous, so each level is re-laid out once per batch: in [B,C,H,W] -> out [B,H,W,C]. */
int nuhtc_nchw_to_nhwc(const float *in, float *out, int B, int C, int H, int W, void *stream);

/* ---- RoIAlign ------------------------------------------------------------------------------
 * Replaces mmcv `ext_module.roi_align_forward(input, rois, output, argmax_y, argmax_x,
 * pooled_height, pooled_width, spatial_scale, sampling_ratio, pool_mode='avg', aligned)` as
 * called per level by mmdet/models/roi_heads/roi_extractors/single_level_roi_extractor.py:79,
 * 96,103 and nuhtc/models/roi_extractors_cus.py:198,218 -- but for ALL levels in one launch.
 *
 *   feats[l]   device pointer of level l, fp32, layout NUHTC_LAYOUT_*; H[l], W[l], scale[l]
 *              (= 1/stride) are host arrays of length L (1..NUHTC_MAX_LEVELS)
 *   rois       [K,5] fp32 (batch_idx, x1, y1, x2, y2), device
 *   out        [K,C,PH,PW] fp32, device, caller-allocated, fully overwritten
 *   mode       NUHTC_ROI_ROUTE: each RoI is pooled on ONE level chosen like
 *              SingleRoIExtractor.map_roi_levels (single_level_roi_extractor.py:36-55) with
 *              `finest_scale`; L==1 degenerates to a plain roi_align.
 *              NUHTC_ROI_SUM: every RoI is pooled on every level and the results are summed in
 *              level order (AttentionRoIExtractor, roi_extractors_cus.py:213-218,246).
 *   impl       NUHTC_IMPL_AUTO picks the separable fast kernel when its preconditions hold
 *              (NHWC, C%4==0, PH==PW in {7,14}); NUHTC_IMPL_DIRECT forces the literal
 *              per-sample kernel (either layout, any shape), which follows the reference's
 *              accumulation order exactly. */
#define NUHTC_LAYOUT_NCHW 0
#define NUHTC_LAYOUT_NHWC 1
#define NUHTC_ROI_ROUTE 0
#define NUHTC_ROI_SUM 1
#define NUHTC_IMPL_AUTO 0
#define NUHTC_IMPL_DIRECT 1
/*   bias       NULL, or [K,C] fp32 added to every bin of (RoI k, channel c) after the level sum -- the broadcast
 *              attention vector of AttentionRoIExtractor (roi_extractors_cus.py:238,246), fused into the store. */
int nuhtc_roi_align_fwd(const float *const *feats, const int *H, const int *W, const float *scale, int L,
                        int B, int C, int layout, const float *rois, int K, int PH, int PW,
                        int sampling_ratio, int aligned, int mode, float finest_scale, int impl, float *out,
                        const float *bias, void *stream);

/* ---- RoIAlign, strip-shared path (the default for 7x7 / 14x14 outputs, C % 32 == 0) ------------------------------
 * Same operation and arguments as nuhtc_roi_align_fwd, on levels staged in the channel-group layout
 * [B][C/32][H][W][32] (nuhtc_to_cg32; 128-byte aligned): one 128-byte line per (cell, group of 32 channels), so a CTA that
 * owns 32 channels of a vertical strip of one image streams whole rows and serves every RoI of the strip from shared
 * memory -- each level row crosses L2->SM once per strip and channel group instead of once per overlapping RoI.
 * mode ROUTE (any L) or L == 1 take the strip kernels; RoIs whose sampling window cannot be staged (wider than 18 cells
 * on a level wider than 48 cells, taller than 18 rows, a bin with more than 8 taps) and mode SUM with L > 1 go
 * through the per-RoI kernel inside the same call.  Results do not depend on the path (same fp32 tap tables).
 *   nuhtc_to_cg32: channels_last != 0: `in` is [B,H,W,C] (a channels_last tensor's memory), else [B,C,H,W].
 *   ws/ws_bytes from nuhtc_roi_align_workspace_bytes; no host synchronisation, CUDA-graph capturable.
 *   pool2      NULL, or L host ints (mode SUM only): level l with pool2[l] != 0 enters the sum as
 *              adaptive_avg_pool2d(RoIAlign(2PH x 2PW, sampling_ratio = 0), (PH, PW)) -- the semantic-feature branch of
 *              NuHTC's _bbox_forward (nuhtc/models/htc_roi_head_cus.py:193-199) -- pooled directly at the output size
 *              (the 2x2 average of bins with g samples per axis is one bin with 2g samples per axis). */
#define NUHTC_LAYOUT_CG32 2
int nuhtc_to_cg32(const float *in, float *out, int B, int C, int H, int W, int channels_last, void *stream);
size_t nuhtc_roi_align_workspace_bytes(const int *H, const int *W, int L, int B, int K, int PH, int PW);
int nuhtc_roi_align_cg32(const float *const *feats, const int *H, const int *W, const float *scale, int L, int B, int C,
                         const float *rois, int K, int PH, int PW, int sampling_ratio, int aligned, int mode,
                         float finest_scale, const int *pool2, float *out, const float *bias, void *ws, size_t ws_bytes,
                         void *stream);

/* ---- cosine-attention pooling (AttentionRoIExtractor, levels >= start_level) ---------------------------------------
 * Replaces nuhtc/models/roi_extractors_cus.py:220-238 for one level: for RoI k with centre cell
 * (b, floor((y1+y2)/(2*stride)), floor((x1+x2)/(2*stride))) (clamped to the map),
 *   out[k,:] (+)= mean_{h,w}( feat[b,:,h,w] * (relu(cos(feat[b,:,cy,cx], feat[b,:,h,w]) - thres) + thres) ).
 *   feat_nhwc [B,H,W,C] fp32 (C <= 64), rois [K,5], out [K,C]; accumulate != 0 adds to out (second level).
 *   status [1] int32: 2 = a RoI's batch index is outside [0,B). */
size_t nuhtc_attention_pool_workspace_bytes(int K, int B);
int nuhtc_attention_pool(const float *feat_nhwc, int B, int H, int W, int C, const float *rois, int K, float stride,
                         float thres, int accumulate, float *out, int32_t *status, void *ws, size_t ws_bytes,
                         void *stream);

/* ---- NMS -----------------------------------------------------------------------------------
 * Replaces mmcv `ext_module.nms(boxes, scores, iou_threshold, offset)` and the class-offset
 * arithmetic of mmcv.ops.batched_nms (call sites nuhtc/models/bbox_head.py:93,208;
 * nuhtc/core/post_processing/bbox_nms.py:83; mmdet/core/post_processing/bbox_nms.py:86;
 * mmdet/models/dense_heads/rpn_head.py:232), batched over independent groups (images).
 *
 *   boxes [N,4] fp32, scores [N] fp32, device.
 *   labels [N] int64 or NULL; groups [N] int32 or NULL (NULL = one group).  Only boxes of the
 *          same group interact.  Groups must be < num_groups; a NEGATIVE group marks a box that
 *          is not a candidate at all (e.g. score <= score_thr): it is skipped without a
 *          host-side compaction.
 *   mode   NUHTC_NMS_AGNOSTIC : IoU on the raw coordinates (labels ignored).
 *          NUHTC_NMS_OFFSET   : coordinates + float(label)*(max_coord_of_group+1) in fp32, all
 *                               pairs tested (batched_nms below split_thr).
 *          NUHTC_NMS_PERCLASS : same offset coordinates, only same-label pairs tested
 *                               (batched_nms at/above split_thr: one nms per class).
 *   Suppression test: inter/(area_i+area_j-inter) > iou_thr with IEEE fp32 division, areas
 *   (x2-x1+offset)*(y2-y1+offset); order = score descending, ties lower index first.
 *   max_group_size  upper bound on the number of boxes in any one sort segment: a group, or with
 *          num_classes > 0 one (group, class) list (the group bound always works; N if unknown).
 *          It sizes the pair matrix, so a tight bound matters.
 *   keep   [N] int64 out: group g's kept ORIGINAL indices, score-descending, are
 *          keep[group_start[g] .. group_start[g]+group_count[g])
 *   group_start, group_count  [num_groups] int64 out (device)
 *   status [1] int32 out (device): 0 ok, 1 = a segment exceeded max_group_size.
 *   ws/ws_bytes from nuhtc_nms_workspace_bytes(N, num_groups, max_group_size). */
#define NUHTC_NMS_AGNOSTIC 0
#define NUHTC_NMS_OFFSET 1
#define NUHTC_NMS_PERCLASS 2
#define NUHTC_NMS_PERCLASS_RAW 3 /* raw coordinates, only same-label pairs: batched_nms(class_agnostic=True) at/above split_thr */
/*   num_classes  0: one sort segment per group.  > 0 (labels must be < num_classes): one segment per (group, class) --
 *          5x fewer pair tests and scans that run in parallel; the per-group list is the merge of its class lists.
 *          Exactly equivalent for PERCLASS / PERCLASS_RAW.  For OFFSET it is equivalent iff no candidate coordinate
 *          is negative (then boxes of different classes cannot overlap after the offset); status 3 reports a
 *          violated precondition and the caller must repeat the call with num_classes = 0. */
size_t nuhtc_nms_workspace_bytes(int64_t N, int num_groups, int64_t max_group_size, int num_classes);
int nuhtc_nms(const float *boxes, const float *scores, const int64_t *labels, const int32_t *groups, int64_t N,
              int num_groups, int64_t max_group_size, float iou_thr, int offset, int mode, int num_classes,
              int64_t *keep, int64_t *group_start, int64_t *group_count, int32_t *status, void *ws, size_t ws_bytes,
              void *stream);

/* ---- mask paste ----------------------------------------------------------------------------
 * Replaces `_do_paste_mask(masks, boxes, img_h, img_w, skip_empty=False)` + the `>= thr`
 * of FCNMaskHead.get_seg_masks (mmdet/models/roi_heads/mask_heads/fcn_mask_head.py:344-412,
 * 292-306): bilinear resample (grid_sample, zeros padding, align_corners=False) of each
 * [mh,mw] probability map into the image frame under its box.
 *   probs [N,mh,mw] fp32 (already sigmoid), boxes [N,4] fp32 (x0,y0,x1,y1 in image px).
 *   out_kind NUHTC_PASTE_PROB : out fp32  [N,img_h,img_w]  resampled probabilities
 *            NUHTC_PASTE_BIN  : out uint8 [N,img_h,img_w]  (prob >= thr), 0/1  (the dense contract)
 *            NUHTC_PASTE_BITS : out uint64 [N,img_h,ceil(img_w/64)] bit x%64 of word x/64
 *   area  [N] int32 or NULL: number of set pixels per mask (BIN/BITS kinds)
 *   bbox  [N,4] int32 or NULL: tight x0,y0,x1,y1 (exclusive max) of set pixels; 0,0,0,0 if empty */
#define NUHTC_PASTE_PROB 0
#define NUHTC_PASTE_BIN 1
#define NUHTC_PASTE_BITS 2
int nuhtc_paste_masks(const float *probs, const float *boxes, int N, int mh, int mw, int img_h, int img_w,
                      float thr, int out_kind, void *out, int32_t *area, int32_t *bbox, void *stream);
/* Both binary forms from ONE evaluation of every mask (img_w % 16 == 0): dense uint8 [N,img_h,img_w] (what
 * get_seg_masks returns) and the bit rows [N,img_h,ceil(img_w/64)] the mask NMS / contour kernels read. */
int nuhtc_paste_masks_dense_bits(const float *probs, const float *boxes, int N, int mh, int mw, int img_h, int img_w,
                                 float thr, uint8_t *dense, uint64_t *bits, int32_t *area, int32_t *bbox, void *stream);

/* ---- per-tile mask NMS -----------------------------------------------------------------------
 * Replaces `mask_nms(masks, pred_scores, thr)` of tools/infer_wsi.py:60-84 (pycocotools
 * rleEncode + rleIou + the greedy double loop), batched over tiles.
 *   nuhtc_pack_masks: dense uint8 masks [n,h,w] -> bit rows [n,h,ceil(w/64)] + area + bbox.
 *   nuhtc_mask_nms:   bits/area/bbox as above, scores [n] fp32, tile [n] int32 or NULL (tile id
 *                     per mask, < num_tiles; only masks of one tile interact).
 *                     IoU = |A&B| / |A|B| as double, suppressed when IoU > thr (double compare).
 *                     Order: score descending, ties higher index first (np.argsort(...)[::-1]).
 *   keep [n] int32 out, tile_start/tile_count [num_tiles] int32 out: tile t's kept ORIGINAL
 *   indices in score order are keep[tile_start[t] .. +tile_count[t]). */
int nuhtc_pack_masks(const uint8_t *masks, int n, int h, int w, uint64_t *bits, int32_t *area, int32_t *bbox,
                     void *stream);
size_t nuhtc_mask_nms_workspace_bytes(int n, int num_tiles, int max_tile_size);
int nuhtc_mask_nms(const uint64_t *bits, const int32_t *area, const int32_t *bbox, const float *scores,
                   const int32_t *tile, int n, int num_tiles, int max_tile_size, int h, int w, double thr,
                   int32_t *keep, int32_t *tile_start, int32_t *tile_count, int32_t *status, void *ws,
                   size_t ws_bytes, void *stream);

/* ---- cross-tile polygon merge ------------------------------------------------------------------
 * Replaces `merge_overlap(cells, overlap_threshold, merge_strategy)` of
 * tools/nuclei_merge.py:62-174 (shapely STRtree candidates + polygon IoU + greedy in score
 * order) on flat arrays.
 *   xy [sumV,2] fp64 ring vertices, voff [N+1] int64 ring offsets, score [N] fp64 (device).
 *   strategy 0 'probability', 1 'area'.
 *   keep_ids [N] int64 out: ORIGINAL indices of kept nuclei ordered by score rank
 *            (position r = nuclei_id r, nuclei_merge.py:201); num_keep [1] int64 out (device).
 *   status [1] int32 out: 0 ok, 1 candidate-pair capacity exceeded (retry with larger max_pairs).
 * This call SYNCHRONISES the stream internally between its phases (it sizes its pair list). */
size_t nuhtc_merge_workspace_bytes(int64_t N, int64_t sumV, int64_t max_pairs);
int nuhtc_merge(const double *xy, const int64_t *voff, const double *score, int64_t N, int64_t sumV,
                double thr, int strategy, int64_t max_pairs, int64_t *keep_ids, int64_t *num_keep,
                int32_t *status, void *ws, size_t ws_bytes, void *stream);

/* The two phases of the merge, exposed separately for the multi-GPU merge (nuhtc_b200/seam.py), where the
 * resolve rounds alternate with an exchange of seam-nucleus states between ranks:
 *   nuhtc_merge_graph : suppression graph of the N polygons as a CSR keyed by the suppressed nucleus:
 *                       in_list[in_off[b] .. in_off[b]+indeg[b]) = nuclei that outrank b (score desc, ties lower
 *                       index) and overlap it with IoU > thr.  indeg [N], in_off [N+1], in_list [max_pairs] int32
 *                       out (device); *num_pairs (HOST) = candidate pairs examined.  Synchronises the stream.
 *   nuhtc_merge_rounds: `rounds` sweeps of the greedy fixed-point rule over state [N] uint8
 *                       (0 undecided, 1 kept, 2 suppressed); nodes with frozen[i] != 0 are read but never written
 *                       (their state is owned by another rank).  remaining [1] int64 out (device): undecided,
 *                       non-frozen nodes after the last sweep.  No synchronisation. */
int nuhtc_merge_graph(const double *xy, const int64_t *voff, const double *score, int64_t N, int64_t sumV,
                      double thr, int64_t max_pairs, int32_t *indeg, int32_t *in_off, int32_t *in_list,
                      int64_t *num_pairs, int32_t *status, void *ws, size_t ws_bytes, void *stream);
/* y extent (min, max of the vertex y coordinates) of every ring: what `seam.merge_distributed` compares with the stripe
 * extents of the other ranks to find the nuclei that have to travel. */
int nuhtc_ring_yextent(const double *xy, const int64_t *voff, int64_t N, double *ymin, double *ymax, void *stream);
int nuhtc_merge_rounds(const int32_t *in_off, const int32_t *indeg, const int32_t *in_list, int64_t N,
                       const uint8_t *frozen, uint8_t *state, int64_t *remaining, int rounds, void *stream);

/* ---- mask -> contour (tile post-processing, SURVEY 8f-3) --------------------------------------
 * Replaces `mask2inst` (tools/infer_wsi.py:51-54): cv2.findContours(mask, cv2.RETR_TREE,
 * cv2.CHAIN_APPROX_SIMPLE)[0][0], called per nucleus at infer_wsi.py:528-529 after a device->host
 * copy of every dense mask.  Suzuki-Abe border following on the bit rows; contour [0] of the tree
 * is the last outer border in raster order whose parent is the frame.
 *   bits [n,h,ceil(w/64)] uint64 (nuhtc_paste_masks BITS kind / nuhtc_pack_masks), device.
 *   bbox [n,4] int32 or NULL: the tight boxes those calls return (saves a scan of every mask).
 *   select [n] uint8 or NULL: masks with select[m] == 0 are skipped (count 0); infer_wsi.py traces
 *   only the survivors of the mask NMS (nuhtc_keep_flags turns its keep lists into this array).
 *   out_xy [n,max_pts,2] int32 (x,y) in mask coordinates, out_count [n] int32: the contour's
 *   point count (0 for an empty mask).  A count above max_pts means the points were truncated.
 *   status [1] int32: 0 ok, 1 some contour longer than max_pts, 2 a mask wider/taller than 64 px
 *   whose frame does not fit shared memory (frames up to ~400x400 do).
 * nuhtc_contour_rings: closed rings for nuhtc_merge: for every mask m with voff[m+1]-voff[m] = k > 0
 *   writes k vertices (contour points, then its first point again: infer_wsi.py:53) + origin[m]
 *   (tile coordinate, infer_wsi.py:531; NULL = 0) as fp64 at out[voff[m]..); k = 0 skips the mask. */
int nuhtc_mask_contours(const uint64_t *bits, const int32_t *bbox, const uint8_t *select, int64_t n, int h, int w, int max_pts, int32_t *out_xy,
                        int32_t *out_count, int32_t *status, void *stream);
int nuhtc_contour_rings(const int32_t *xy, const int32_t *count, const int64_t *voff, const int32_t *origin,
                        int64_t n, int max_pts, double *out, void *stream);

/* ---- detection glue of the HTC test path ------------------------------------------------------
 * The element-wise steps between the heavy ops (dozens of small torch kernels per batch in the
 * reference), one launch each; every step is a separately rounded fp32 operation like the torch
 * chain it replaces.
 * nuhtc_delta2bbox: class-agnostic `delta2bbox` (mmdet/core/bbox/coder/delta_xywh_bbox_coder.py:
 *   163-260) as used by `regress_by_class` / `get_bboxes` (mmdet bbox_head.py:459-496, 330-380).
 *   rois [K,5] (with_batch=1; column 0 is copied to out) or [K,4]; deltas [K,4]; means/stds 4 HOST
 *   floats; max_h/max_w > 0 clamp to the frame (max_shape); divide_by != 0,1 divides the result
 *   (rescale=True, bbox_head.py:373-376).  out has the shape of rois.
 * nuhtc_multiclass_candidates: the candidate expansion of `multiclass_nms`
 *   (nuhtc/models/bbox_head.py:12-60): boxes [K,4] (row stride box_stride floats), scores [K,score_stride] (first num_classes
 *   columns), roi_tile = address of the batch-index column (stride tile_stride floats) ->
 *   cand_* [K*num_classes] (box, score, label, tile) and groups = tile if score > score_thr else -1.
 * nuhtc_detection_slots: `dets[:max_num]` (bbox_nms.py:98-100) without a host round trip: tile b's
 *   r-th kept candidate (nuhtc_nms keep/group_start/group_count) lands in slot b*max_per_img + r;
 *   empty slots get a box far outside the frame, score 0, tile -1, valid 0.  mask_rois [n,5] =
 *   (max(tile,0), box * scale_factor) (htc_roi_head.py:296-300).
 * nuhtc_tile_filter: margin / min_area filter of tools/infer_wsi.py:510-521 -> tile id or -1.
 * nuhtc_keep_flags: flags [n] uint8 = 1 for the indices listed in nuhtc_mask_nms's keep lists
 *   (keep[tile_start[t] .. +tile_count[t]) for every tile), 0 elsewhere: the `seg_mask[nms_idx]`
 *   selection of infer_wsi.py:527-531 without a host round trip. */
int nuhtc_delta2bbox(const float *rois, int with_batch, const float *deltas, int64_t K, const float *means,
                     const float *stds, int max_h, int max_w, double wh_ratio_clip, float divide_by, float *out,
                     void *stream);
int nuhtc_multiclass_candidates(const float *boxes, int box_stride, const float *scores, int score_stride, const float *roi_tile,
                                int tile_stride, int64_t K, int num_classes, float score_thr, float *cand_boxes,
                                float *cand_scores, int64_t *cand_labels, int32_t *cand_tile, int32_t *groups,
                                void *stream);
int nuhtc_detection_slots(const int64_t *keep, const int64_t *group_start, const int64_t *group_count, int num_tiles,
                          int max_per_img, const float *cand_boxes, const float *cand_scores, const int64_t *cand_labels,
                          const int32_t *cand_tile, float scale_factor, float *det_boxes, float *det_scores,
                          int64_t *det_labels, int32_t *det_tile, uint8_t *det_valid, int64_t *det_cand, float *mask_rois,
                          void *stream);
int nuhtc_tile_filter(const float *det_boxes, const int32_t *area, const int32_t *det_tile, int64_t D, int margin,
                      int img_h, int img_w, int min_area, int32_t *tile_ids, void *stream);
int nuhtc_keep_flags(const int32_t *keep, const int32_t *tile_start, const int32_t *tile_count, int num_tiles,
                     int max_tile_size, int64_t n, uint8_t *flags, void *stream);

/* ---- RPN proposal pre-selection (SURVEY 8f-2) ---------------------------------------------------
 * Replaces the per-level body of `RPNHead._get_bboxes_single` (mmdet/models/dense_heads/rpn_head.py:103-165:
 * permute, sigmoid, `scores.sort(descending=True)`, `[:nms_pre]`, index gathers) and the decode + min-size
 * test of `_bbox_post_process` (:167-236) for a whole batch in ONE launch.
 *   cls[l] [B,A,H_l,W_l] logits, reg[l] [B,4A,H_l,W_l], anchors[l] [H_l*W_l*A,4] in (h,w,a) order (device, fp32).
 *   Per image the output holds, level after level, k_l = min(nms_pre, n_l) candidates (nms_pre <= 0: all): the
 *   nms_pre best scores of the level in descending order, ties by ascending anchor index (levels with
 *   n_l <= nms_pre keep their natural order, as the reference does not sort them):
 *   boxes [B,sum k_l,4] decoded with means 0 / stds 1 and clamped to (max_h,max_w) when both > 0, scores
 *   (sigmoid applied when apply_sigmoid), labels [..] int64 = level, groups [..] int32 = image index, or -1
 *   when w or h <= min_bbox_size (min_bbox_size < 0: no test) -- the arrays nuhtc_nms reads.
 * nuhtc_rpn_topk_supported: 1 if every level that needs a selection fits the shared-memory select
 *   (H*W*A*4 + 24.3 KB <= 227 KB, nms_pre <= 2048); otherwise the caller uses a sort-based path. */
int nuhtc_rpn_topk_supported(const int *H, const int *W, int L, int A, int nms_pre);
int nuhtc_rpn_topk_decode(const float *const *cls, const float *const *reg, const float *const *anchors, const int *H,
                          const int *W, int L, int B, int A, int nms_pre, int apply_sigmoid, int max_h, int max_w,
                          double wh_ratio_clip, float min_bbox_size, float *boxes, float *scores, int64_t *labels,
                          int32_t *groups, void *stream);

/* ---- watershed proposals: instances of a semantic mask (SURVEY 8f-4) -----------------------------
 * Replaces the host tail of `HybridTaskCascadeRoIHead_Cus._watershed_proposal`
 * (nuhtc/models/htc_roi_head_cus.py:303-335: per image a device->host copy, ndi.binary_fill_holes,
 * ndi.distance_transform_edt, ndi.label(distance > 0.25), skimage watershed(-distance, markers, mask), a
 * relabel loop, a one-hot [n,H,W] tensor, areas and the `_inst_mask_to_bbox` loop :263-281).  With the
 * Euclidean distance as the landscape every mask pixel is a marker (distance >= 1 > 0.25), so the instances
 * are the 4-connected components of the hole-filled mask in raster order of their first pixel.
 *   mask [B,H,W] fp32 (0 = background, anything else = foreground; the reference's mask after binary_open).
 *   boxes [B,max_boxes,5] fp32 out: (x0, y0, x1+1, y1+1, 1.0) of the components with
 *   min_area < area < max_area, in label order; counts [B] int32 out: how many qualified (a count above
 *   max_boxes means the tail was dropped).  filled [B,H,W] uint8 out or NULL: the hole-filled mask. */
size_t nuhtc_mask_components_workspace_bytes(int B, int H, int W);
int nuhtc_mask_components(const float *mask, int B, int H, int W, int min_area, int max_area, int max_boxes,
                          float *boxes, int32_t *counts, uint8_t *filled, void *ws, size_t ws_bytes, void *stream);

/* ---- test-time image pipeline (SURVEY 8f-4, the tile loader) ---------------------------------
 * Replaces the per-tile CPU work of `inference_detector(model, [np.ndarray]*B)` (tools/infer_wsi.py:485 ->
 * mmdet/apis/inference.py:90-153) under the NuHTC test pipeline: Resize(keep_ratio=True) with cv2 INTER_LINEAR,
 * Normalize(mean, std, to_rgb), Pad(size_divisor), ImageToTensor and the batch collate, in ONE launch.
 *   tiles [B,h,w,3] uint8 HWC (device), out [B,3,pad_h,pad_w] fp32 (device, fully overwritten): the resized image in
 *   [0,new_h) x [0,new_w), 0 elsewhere.  mean3 / std3: 3 HOST floats per OUTPUT channel (Normalize's float32 arrays);
 *   to_rgb != 0 swaps channels 0 and 2.  Bit-exact with cv2.resize (uint8 fixed-point path) and with mmcv.imnormalize_
 *   (cv2.subtract / cv2.multiply with float64 scalars).  Upscaling and identity only: new_h >= h, new_w >= w,
 *   pad_h >= new_h, pad_w >= new_w.  B = 0 returns 0.  No allocation or synchronisation: CUDA-graph capturable. */
int nuhtc_preprocess_tiles(const uint8_t *tiles, int B, int h, int w, int new_h, int new_w, int pad_h, int pad_w, int to_rgb,
                           const float *mean3, const float *std3, float *out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NUHTC_B200_H */
