/*
 * unmore_b200 — C ABI of the B200-native multi-object reasoning path of unMORE.
 *
 * The reference (vLAR-group/unMORE) is pure Python and has no FFI: the boundary it offers is
 * the set of Python callables of object_reasoning.py / object_scoring.py / post_process.py.
 * Each entry point below replaces the arithmetic of one of those callables (cited per
 * function); unmore_b200/object_reasoning.py etc. keep the reference's Python signatures and
 * forward here through ctypes.  INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns all memory (inputs, outputs, workspaces); the library never allocates
 *     device memory and keeps no pointer after returning;
 *   - work is only enqueued on `stream` (a cudaStream_t); nothing synchronises the device;
 *   - return value 0 = ok, otherwise a negative UNMORE_E_* code or a positive cudaError_t;
 *     unmore_last_error() returns a thread-local description;
 *   - fields: [n_img, C, H, W] fp32 contiguous; channel indices are passed explicitly
 *     (the synthetic stacks use sdf=0, center_row=1, center_col=2, existence=3);
 *   - proposal lists are ragged with a fixed capacity: boxes [n_img, cap, 4] xyxy, fp32 or
 *     fp64 (boxes_f64 != 0; the reference hands fp64 anchors to round 0, object_reasoning.py
 *     :190-194), image i owning the first counts[i] rows; counts == NULL means all cap rows;
 *   - `ws` is a scheduling workspace of unmore_workspace_bytes(n_img) bytes (4-byte aligned): the work
 *     counter and the per-image row offsets, then, from the next 32-byte boundary, one window cache of
 *     unmore_boundary_refine per image (a fixed number of 32-byte slots each, 1 MB per image).  Every
 *     call re-initialises what it uses; nothing in it outlives a call.
 *   - resize semantics: bilinear, align_corners=False, NO antialias (torchvision 0.14.1, the
 *     version the reference pins), arithmetic bit-identical to ATen's CPU kernels.
 */
#ifndef UNMORE_B200_H_
#define UNMORE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UNMORE_E_INVALID (-1)   /* bad argument */
#define UNMORE_E_CAPACITY (-2)  /* a capacity / size limit of the kernels is exceeded */

typedef void* unmore_stream_t; /* cudaStream_t */

const char* unmore_last_error(void);
int unmore_version(void);
/* bytes of the scheduling workspace `ws` used by the list-driven kernels (grows by ~1 MB per image) */
size_t unmore_workspace_bytes(int n_img);

/* existence_checking — object_reasoning.py:491-523 (Binary_Classifier replaced by the mean of
 * the resized crop's existence channel).  scores_out: [n_img, cap] fp32. */
int unmore_existence_scores(const float* fields, int n_img, int C, int H, int W, int ch_exist,
                            const void* boxes, int boxes_f64, const int* counts, int cap,
                            float* scores_out, void* ws, unmore_stream_t stream);

/* The crop + Resize((128,128), BILINEAR) every stage starts with (object_reasoning.py:402-410,
 * 314-321, 500-508; object_scoring.py:126-134) and get_prediction_with_proposals (:301-337 /
 * object_scoring.py:112-157) as a stand-alone op: out [n_img, cap, n_channels, 128, 128] fp32 holds
 * the resized crop of channel channels_host[k] (a HOST array of 1..4 indices) for every proposal,
 * bit-identical to ATen's CPU bilinear kernel.  The fused kernels never materialise these tiles;
 * this entry point exists for signature parity and for testing the resampler directly. */
int unmore_crop_resize(const float* fields, int n_img, int C, int H, int W,
                       const int* channels_host, int n_channels, const void* boxes, int boxes_f64,
                       const int* counts, int cap, float* out, unmore_stream_t stream);

/* The same two stand-alone resize ops in the SECOND resize mode, antialias=True (ATen _upsample_bilinear2d_aa):
 * what torchvision >= 0.17 makes of the reference's transforms.Resize calls (object_reasoning.py:319,407,505;
 * object_scoring.py:131,206,222) when the pinned 0.14.1 is not what is installed.  Bit-exact against torch 2.11
 * CPU (weights with ATen's float/double mix, horizontal pass first, its accumulation order).  The fused
 * existence, center and refine kernels have antialiased forms (unmore_existence_scores_aa,
 * unmore_center_reasoning_aa, unmore_boundary_refine_aa); these produce the tiles for the scoring stage, for the
 * other *_from_tiles stages, for unmore_update_bbox_from_tiles and for inspection.  `scratch`: n_img*cap*n_channels*H*128 floats (crop) / B*128*out_w floats (mask). */
int unmore_crop_resize_aa(const float* fields, int n_img, int C, int H, int W, const int* channels_host,
                          int n_channels, const void* boxes, int boxes_f64, const int* counts, int cap,
                          float* out, void* scratch, size_t scratch_bytes, unmore_stream_t stream);
int unmore_mask_resize_aa(const unsigned char* masks, int B, int H, int W, int out_h, int out_w,
                          unsigned char* out, void* scratch, size_t scratch_bytes, unmore_stream_t stream);

/* The tile path of the second resize mode: the reasoning stages on PRE-RESAMPLED tiles (from unmore_crop_resize_aa,
 * or from anywhere else — e.g. the real per-crop nets of the reference, object_reasoning.py:311-333), so that
 * existence_checking, center_reasoning, one round of optimize_one_image_single_round and main_object_scoring run
 * with torchvision's antialias=True semantics.  Same arithmetic as the fused kernels after the resample.
 *   unmore_tile_means                      tiles [M] x [128,128] (tile_stride floats apart) -> mean per tile (a3)
 *   unmore_center_reasoning_from_tiles     tiles [n_img*cap, 3, 128,128] = (sdf, center_row, center_col) (a5-a8)
 *   unmore_boundary_round_from_tiles       tiles [M, 128,128] (sdf) + boxes [M,4] -> updated boxes fp32 / labels
 *                                          (a10-a12 of ONE round; deltas_ws [M,4] and max_ws [M] are scratch)
 *   unmore_score_and_rasterise_from_tiles  tiles [n_img*cap, 4, 128,128] = (sdf, center_row, center_col, existence);
 *                                          existence_scores (nullable) [n_img, cap]: per-crop classifier outputs used
 *                                          instead of the mean of the fourth tile; antialias selects the kernel that
 *                                          resizes the masks back to the box (a15) */
int unmore_tile_means(const float* tiles, long long tile_stride, int M, float* means_out, unmore_stream_t stream);
int unmore_center_reasoning_from_tiles(const float* tiles, int n_img, int H, int W, const void* boxes,
                                       int boxes_f64, const int* counts, int cap,
                                       double center_score_max_thres, double* max_values_out,
                                       int* argmax_out, double* splits_out, unsigned char* cc_counts_out,
                                       double* cc_boxes_out, int* cc_overflow, void* ws,
                                       unmore_stream_t stream);
int unmore_boundary_round_from_tiles(const float* tiles, int M, const void* boxes, int boxes_f64, int H, int W,
                                     float max_sdf_thres, float max_shrink_threshold, float delta_ratio,
                                     float* boxes_out, float* labels_out, float* deltas_ws, float* max_ws,
                                     unmore_stream_t stream);
int unmore_score_and_rasterise_from_tiles(const float* tiles, const float* existence_scores, int antialias,
                                          int n_img, int H, int W, const void* boxes, int boxes_f64,
                                          const int* counts, int cap, float* scores_out, float* tight_out,
                                          int* areas_out, uint32_t* masks_out, unmore_stream_t stream);

/* center_reasoning — object_reasoning.py:525-580 with batch_erode (utils/misc.py:10-20) and
 * center_field_to_anti_center_map (object_reasoning.py:360-377) fused.
 * max_values_out [n_img, cap] fp64: amax of the masked anti-center map;
 * argmax_out [n_img, cap] int32: -1 if the proposal passes (max <= thr), else yc*128+xc;
 * splits_out [n_img, cap, 4, 4] fp64 (nullable): left/right/top/bottom boxes of failing rows.
 * --analyze_cc (:561-572, separate_connected_components :207-256 + enlarge_proposals :259-291),
 * all three NULL when off: cc_counts_out [n_img, cap] u8 = number of component boxes emitted
 * for a PASSING proposal whose un-eroded union mask has >= 2 8-connected components (else 0);
 * cc_boxes_out [n_img, cap, unmore_cc_cap(), 4] fp64 the enlarged (x1.5, int-truncated, clipped
 * to W/H) component boxes in scipy label order; *cc_overflow is incremented for every proposal
 * with more components than unmore_cc_cap() (the extra ones are dropped — callers must check). */
int unmore_center_reasoning(const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                            int ch_center_row, int ch_center_col, const void* boxes, int boxes_f64,
                            const int* counts, int cap, double center_score_max_thres,
                            double* max_values_out, int* argmax_out, double* splits_out,
                            unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow,
                            void* ws, unmore_stream_t stream);
int unmore_cc_cap(void);

/* boundary_reasoning — object_reasoning.py:582-612: up to n_round rounds of
 * filter_small_proposal (:293-299) + optimize_one_image_single_round (:379-487), one warp per
 * proposal, box and label in registers, exit at the fixed point (label 1, box unchanged).
 * With n_round=1, apply_small_filter=0 it is exactly optimize_one_image_single_round.
 * boxes_out [n_img, cap, 4] fp32; labels_out [n_img, cap] fp32: 1 / 0 / -1 as the reference,
 * -2 = removed by filter_small_proposal (not in the reference's returned list);
 * rounds_out [n_img, cap] int32 (nullable): rounds actually evaluated.
 * Proposals of one image share the boundary terms of a crop window through the window cache in `ws`
 * (fields up to 32767 px per side); the results are bit-identical to evaluating every window. */
int unmore_boundary_refine(const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                           const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                           int apply_small_filter, int early_exit, float proposal_area_thres,
                           float max_sdf_thres, float max_shrink_threshold, float delta_ratio,
                           float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                           unmore_stream_t stream);

/* unmore_existence_scores, unmore_center_reasoning and unmore_boundary_refine in the SECOND resize mode
 * (antialias=True, see unmore_crop_resize_aa): same arguments, validation, workspace and outputs, with every crop
 * resampled by ATen's antialiased kernel inside the fused kernels instead of materialised as a tile; no scratch, one
 * kernel per call (plus the counts prefix).  Bit-identical to the tile path: the existence score equals
 * unmore_tile_means of the unmore_crop_resize_aa tile, center reasoning equals unmore_center_reasoning_from_tiles on
 * the (sdf, center_row, center_col) tiles (--analyze_cc included), and every refine round equals
 * unmore_boundary_round_from_tiles on the sdf tile (window cache, early exit and rounds_out as in the primary mode).
 * Callers detect these entry points by their symbols (unmore_version() is unchanged). */
int unmore_existence_scores_aa(const float* fields, int n_img, int C, int H, int W, int ch_exist,
                               const void* boxes, int boxes_f64, const int* counts, int cap,
                               float* scores_out, void* ws, unmore_stream_t stream);
int unmore_center_reasoning_aa(const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                               int ch_center_row, int ch_center_col, const void* boxes, int boxes_f64,
                               const int* counts, int cap, double center_score_max_thres,
                               double* max_values_out, int* argmax_out, double* splits_out,
                               unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow,
                               void* ws, unmore_stream_t stream);
int unmore_boundary_refine_aa(const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                              const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                              int apply_small_filter, int early_exit, float proposal_area_thres,
                              float max_sdf_thres, float max_shrink_threshold, float delta_ratio,
                              float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                              unmore_stream_t stream);

/* update_bbox_with_boundary_fields — object_reasoning.py:140-174 on pre-resampled tiles
 * [M, 128, 128] fp32.  deltas_out [M, 4] = (delta_x1, delta_y1, delta_x2, delta_y2);
 * max_out [M] (nullable) = amax of each tile. */
int unmore_update_bbox_from_tiles(const float* tiles, int M, float* deltas_out, float* max_out,
                                  unmore_stream_t stream);

/* Order-preserving selection (the boolean-mask indexing of the reference, e.g.
 * object_reasoning.py:422-426, 541-542, 630, 656).  For every image, entries e < count whose
 * predicate holds are copied in order to out [n_img, cap_out, 4]; each entry carries `group`
 * consecutive boxes (4 for the split lists), or group_counts[e] <= group of them when
 * group_counts (nullable, u8 [n_img, cap_in]) is given.  mode: 0 pred=u8 flags; 1 pred=fp32 >= thr;
 * 2 pred=fp32 == thr; 3 pred=int32 >= 0; 4 pred=int32 < 0; 5 pred=u8 != 0.  append != 0 appends
 * after the counts_out rows already present (torch.cat of two lists, :571, :644).  index_out
 * (nullable) [n_img, cap_out] receives the source entry index of each output row; *overflow
 * (nullable) is incremented for every image whose rows did not fit cap_out. */
int unmore_compact_boxes(const void* in, int in_f64, const int* counts_in, int cap_in, int group,
                         int mode, const void* pred, float thr, void* out, int out_f64, int cap_out,
                         int* counts_out, int append, int* index_out,
                         const unsigned char* group_counts, int* overflow, int n_img,
                         unmore_stream_t stream);

/* torchvision.ops.nms semantics — object_reasoning.py:661, object_scoring.py:238.
 * boxes [n_img, cap, 4] fp32; scores [n_img, cap] fp32 or NULL (all equal: index order);
 * keep_out [n_img, cap] int32 kept indices in descending-score order; keep_counts_out [n_img];
 * boxes_out (nullable) [n_img, cap, 4] kept boxes in that order.
 * order_ws: [n_img, cap] int32 scratch.  cap <= 32768. */
int unmore_box_nms(const float* boxes, const float* scores, const int* counts, int cap, int n_img,
                   float iou_threshold, int* keep_out, int* keep_counts_out, float* boxes_out,
                   int* order_ws, unmore_stream_t stream);

/* batch_erode — utils/misc.py:10-20 on [B, 128, 128] u8 masks (non-zero = set): num_round
 * erosions with a kernel_size x kernel_size ones kernel and zero border.  out: u8 {0,1}. */
int unmore_batch_erode(const unsigned char* masks, int B, int H, int W, int kernel_size, int num_round,
                       unsigned char* out, unmore_stream_t stream);

/* separate_connected_components — object_reasoning.py:207-256 on [B, 128, 128] u8 masks (non-zero
 * = set): 8-connected labelling in scipy.ndimage.label order.  counts_out [B] = number of
 * components; boxes_out [B, unmore_cc_cap(), 4] int32 = [x_start, y_start, x_stop, y_stop] of the
 * first unmore_cc_cap() components. */
int unmore_connected_components(const unsigned char* masks, int B, int H, int W, int* counts_out,
                                int* boxes_out, unmore_stream_t stream);

/* center_field_to_anti_center_map — object_reasoning.py:360-377: vote_maps [B, 2, H, W] fp32 ->
 * out [B, H, W] fp64 (5x5 normalised "points-at-me" correlation, zero padding, / 24). */
int unmore_anti_center_map(const float* vote_maps, int B, int H, int W, int kernel_size, double* out,
                           unmore_stream_t stream);

/* Large-K variant of unmore_box_nms for ONE list of K boxes (config "NMS sweep, 1k-16k"):
 * stable rank sort -> 64-wide suppression bit-matrix -> single-warp greedy scan.  Same results.
 * order_ws [K] int32; matrix_ws [K * ceil(K/64)] u64; keep_out [K]; keep_count_out [1]. */
int unmore_box_nms_matrix(const float* boxes, const float* scores, int K, float iou_threshold,
                          int* order_ws, void* matrix_ws, int* keep_out, int* keep_count_out,
                          unmore_stream_t stream);

/* main_object_scoring steps 1-6 — object_scoring.py:182-235: per box the existence / center /
 * boundary scores, the union of the two binary masks resized back to the box (bilinear +
 * round-half-even, :196-228), its tight box (pycocotools toBbox semantics, :160-164) and area.
 * scores_out [n_img, cap, 4] fp32 = (existence, center, boundary, 0);
 * tight_out [n_img, cap, 4] fp32 xyxy (zeros for an empty mask); areas_out [n_img, cap] int32;
 * masks_out (nullable) [n_img, cap, H, ceil(W/32)] u32, LSB = lowest x. */
int unmore_score_and_rasterise(const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                               int ch_center_row, int ch_center_col, int ch_exist, const void* boxes,
                               int boxes_f64, const int* counts, int cap, float* scores_out,
                               float* tight_out, int* areas_out, uint32_t* masks_out,
                               unmore_stream_t stream);

/* The mask resize of object_scoring.py:206-207 / 222-223 as a stand-alone op: masks [B, 128, 128] u8
 * (non-zero = set) -> Resize((out_h, out_w), BILINEAR) + round half to even -> out [B, out_h, out_w]
 * u8 {0,1}, in the exact arithmetic of the ATen CPU kernel that output size selects. */
int unmore_mask_resize(const unsigned char* masks, int B, int H, int W, int out_h, int out_w,
                       unsigned char* out, unmore_stream_t stream);

/* main_object_scoring steps 7b-8 (object_scoring.py:244-266) + the post_process predicate
 * (post_process.py:61-74) for the detections kept by the second NMS, in keep order:
 * out [n_img, cap, 5] fp64 = (score, existence_score, center_score, boundary_score, area_score);
 * bbox_xywh_out [n_img, cap, 4] fp32 COCO box; selected_out (nullable) [n_img, cap] u8 = 1 unless
 * existence < t_e or center < t_c or boundary < t_b — the thresholds are doubles and the fp32 scores are
 * compared in double, like the reference's Python floats (post_process.py:64-69), so a threshold that
 * is not representable in fp32 (0.7, ...) selects the same set. */
int unmore_final_scores(const float* scores, const float* tight, const int* areas, const int* keep,
                        const int* keep_counts, int cap, int n_img, double existence_score_thres,
                        double center_score_thres, double boundary_score_thres, double* out,
                        float* bbox_xywh_out, unsigned char* selected_out, unmore_stream_t stream);

/* Detection rows for the end-of-run collective (the image-sharded driver that formalises the reference's
 * --start_idx / --end_idx processes, datasets.py:432-435 + object_reasoning.py:662-665): appends the
 * detections of a batch to a fixed-capacity row buffer `rows` [max_rows + 1, 6] fp64 in image-major, NMS
 * keep order.  rows[0] = (row count so far, overflow flag, 0, 0, 0, 0) is the header and the append cursor
 * (zero it before the first batch); rows[1 + r] = (image_id, x, y, w, h, score).  image_ids [n_img] int64;
 * bbox_xywh [n_img, cap, 4] fp32 and out5 [n_img, cap, 5] fp64 as written by unmore_final_scores. */
int unmore_pack_detections(const long long* image_ids, const float* bbox_xywh, const double* out5,
                           const int* keep_counts, int cap, int n_img, double* rows, int max_rows,
                           unmore_stream_t stream);

/* Summed-area tables (north-star op (a); no reference counterpart, oracle = fp64 cumsum):
 * in [n_planes, H, W] fp32 -> out [n_planes, H+1, W+1] fp64, out[y][x] = sum in[:y, :x]. W <= 2048. */
int unmore_sat_build(const float* in, int n_planes, int H, int W, double* out, unmore_stream_t stream);

/* Same tables built in place from a field stack [n_img, C, H, W]: output plane (i, k) is channel
 * channels_host[k] of image i; out [n_img, n_channels, H+1, W+1] fp64.  channels_host is a HOST
 * array of 1..4 channel indices (north-star: existence and boundary-distance fields). */
int unmore_sat_build_fields(const float* fields, int n_img, int C, int H, int W,
                            const int* channels_host, int n_channels, double* out,
                            unmore_stream_t stream);

/* O(1) box sums from a table built over [n_img, planes_per_img, H, W]: the window is snapped
 * like the crops (floor x1,y1 / ceil x2,y2, object_reasoning.py:502).  sums_out / means_out
 * (nullable) [n_img, cap] fp64. */
int unmore_box_sums(const double* sat, int n_img, int planes_per_img, int plane, int H, int W,
                    const void* boxes, int boxes_f64, const int* counts, int cap, double* sums_out,
                    double* means_out, unmore_stream_t stream);

/* Bit-packing of dense masks: in [K, H, W] u8 (non-zero = set) -> out [K, H, ceil(W/32)] u32. */
int unmore_mask_pack(const unsigned char* in, size_t K, int H, int W, uint32_t* out, unmore_stream_t stream);

/* Area and tight box (half-open x1,y1,x2,y2; zeros if empty) of packed masks. */
int unmore_mask_stats(const uint32_t* masks, int K, int H, int W, int* areas_out, int* tight_out,
                      unmore_stream_t stream);

/* binary_mask_to_rle — object_scoring.py:167-170 (pycocotools maskApi.c rleEncode): column-major
 * run lengths of packed masks.  counts_out [K, max_runs] u32 (counts[0] = leading zeros, possibly
 * 0); n_runs_out [K] = number of runs; a mask with more than max_runs (or 8193) runs gets only its
 * run count written.  The compressed ASCII "counts" string is formed on the host from these
 * (unmore_b200/rle.py, rleToString). */
int unmore_mask_rle_counts(const uint32_t* masks, int K, int H, int W, int max_runs,
                           uint32_t* counts_out, int* n_runs_out, unmore_stream_t stream);

/* Mask-IoU NMS on packed masks (north-star op (c); no reference counterpart, oracle = dense
 * greedy restatement in torchvision's order): suppress j if popc(a&b)/(area_a+area_b-popc(a&b))
 * > thr (fp32 division of exact integers).  areas / tight from unmore_mask_stats.
 * order_ws [K] int32; matrix_ws [K * ceil(K/64)] u64; keep_out [K]; keep_count_out [1]. */
int unmore_mask_nms(const uint32_t* masks, int K, int H, int W, const float* scores, const int* areas,
                    const int* tight, float iou_threshold, int* order_ws, void* matrix_ws,
                    int* keep_out, int* keep_count_out, unmore_stream_t stream);

/* ---- Images of different sizes in one call ----------------------------------------------------------------------
 * A padded stack: fields [n_img, C, H, W] where (H, W) is the PITCH (the largest image), and image_hw [n_img, 2] int32
 * in DEVICE memory of the current device (8-byte aligned) holding (h_i, w_i), 1 <= h_i <= H, 1 <= w_i <= W.  Image i is
 * fields[i, :, :h_i, :w_i]; the padding may hold anything and no result depends on it.  Every address comes from the
 * pitch, every use of the image size (window snap, edge tests, clips) from (h_i, w_i); the kernels clamp the extents to
 * [1, pitch], so a bad table gives wrong numbers, never an out-of-range access.  Each call takes the arguments of its
 * uniform counterpart with image_hw after W, and gives every image exactly what the uniform call gives it alone.
 * Masks of unmore_score_and_rasterise_hw stay on the pitched canvas [n_img, cap, H, ceil(W/32)]: image i's are the
 * [:h_i, :ceil(w_i/32)] corner, every bit outside the image is 0.  unmore_sat_build_fields_hw reads the padding as
 * zeros, so entries [:h_i+1, :w_i+1] of image i's tables are those of the image alone; unmore_box_sums_hw takes such
 * tables.  A null, misaligned, host or other-device image_hw is rejected (UNMORE_E_INVALID) before anything runs.
 *
 * The second resize mode (antialias=True) has the same six forms: unmore_existence_scores_aa_hw,
 * unmore_center_reasoning_aa_hw, unmore_boundary_refine_aa_hw, unmore_crop_resize_aa_hw,
 * unmore_center_reasoning_from_tiles_hw and unmore_score_and_rasterise_from_tiles_hw, each with image_hw after W.  unmore_crop_resize_aa_hw snaps every window
 * to its image and sizes its scratch by the pitch (n_img*cap*n_channels*H*128 floats).  The two *_from_tiles_hw calls
 * take tiles cropped from the stack by unmore_crop_resize_aa_hw and the pitch as (H, W): the extents give the window
 * snap behind the split boxes, the --analyze_cc clip and the mask raster, whose canvas is the pitched one above. */
int unmore_existence_scores_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_exist,
                               const void* boxes, int boxes_f64, const int* counts, int cap, float* scores_out,
                               void* ws, unmore_stream_t stream);
int unmore_center_reasoning_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                               int ch_center_row, int ch_center_col, const void* boxes, int boxes_f64,
                               const int* counts, int cap, double center_score_max_thres, double* max_values_out,
                               int* argmax_out, double* splits_out, unsigned char* cc_counts_out,
                               double* cc_boxes_out, int* cc_overflow, void* ws, unmore_stream_t stream);
int unmore_boundary_refine_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                              const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                              int apply_small_filter, int early_exit, float proposal_area_thres,
                              float max_sdf_thres, float max_shrink_threshold, float delta_ratio,
                              float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                              unmore_stream_t stream);
int unmore_score_and_rasterise_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                                  int ch_sdf, int ch_center_row, int ch_center_col, int ch_exist,
                                  const void* boxes, int boxes_f64, const int* counts, int cap,
                                  float* scores_out, float* tight_out, int* areas_out, uint32_t* masks_out,
                                  unmore_stream_t stream);
int unmore_box_sums_hw(const double* sat, int n_img, int planes_per_img, int plane, int H, int W,
                       const int* image_hw, const void* boxes, int boxes_f64, const int* counts, int cap,
                       double* sums_out, double* means_out, unmore_stream_t stream);
int unmore_sat_build_fields_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                               const int* channels_host, int n_channels, double* out, unmore_stream_t stream);
int unmore_existence_scores_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                                  int ch_exist, const void* boxes, int boxes_f64, const int* counts, int cap,
                                  float* scores_out, void* ws, unmore_stream_t stream);
int unmore_boundary_refine_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                                 const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                                 int apply_small_filter, int early_exit, float proposal_area_thres,
                                 float max_sdf_thres, float max_shrink_threshold, float delta_ratio,
                                 float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                                 unmore_stream_t stream);
int unmore_center_reasoning_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                                  int ch_sdf, int ch_center_row, int ch_center_col, const void* boxes,
                                  int boxes_f64, const int* counts, int cap, double center_score_max_thres,
                                  double* max_values_out, int* argmax_out, double* splits_out,
                                  unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow, void* ws,
                                  unmore_stream_t stream);
int unmore_crop_resize_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                             const int* channels_host, int n_channels, const void* boxes, int boxes_f64,
                             const int* counts, int cap, float* out, void* scratch, size_t scratch_bytes,
                             unmore_stream_t stream);
int unmore_center_reasoning_from_tiles_hw(const float* tiles, int n_img, int H, int W, const int* image_hw,
                                          const void* boxes, int boxes_f64, const int* counts, int cap,
                                          double center_score_max_thres, double* max_values_out, int* argmax_out,
                                          double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out,
                                          int* cc_overflow, void* ws, unmore_stream_t stream);
int unmore_score_and_rasterise_from_tiles_hw(const float* tiles, const float* existence_scores, int antialias,
                                             int n_img, int H, int W, const int* image_hw, const void* boxes,
                                             int boxes_f64, const int* counts, int cap, float* scores_out,
                                             float* tight_out, int* areas_out, uint32_t* masks_out,
                                             unmore_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* UNMORE_B200_H_ */
