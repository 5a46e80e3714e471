// Internal launch interfaces between the C-ABI translation unit (capi.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace unmore {

// ---- refine.cu -----------------------------------------------------------------------
// Per-image window cache of the fused refine kernel: the boundary terms of a crop window depend only on the
// field plane and the snapped integer window, and proposals of one image converge onto the same windows.
// One open-addressed table of kWindowSlots 32-byte slots per image, in the workspace (make_worklist).
constexpr int kWindowSlots = 32768;   // ~15k distinct windows per benchmark image at most
static_assert((kWindowSlots & (kWindowSlots - 1)) == 0, "kWindowSlots must be a power of two");
constexpr int kWindowMaxSide = 32767;   // window corners are packed in 15 bits each; larger fields share nothing
struct alignas(32) WindowSlot {
  unsigned long long key;   // 0 = empty; packed window, bit 63 set once the terms below are published
  float max_sdf, pad;
  float4 d;                 // dx1, dy1, dx2, dy2
};
static_assert(sizeof(WindowSlot) == 32, "one sector per slot");

struct RefineParams {
  const float* fields;
  int C, H, W, ch_sdf;
  const void* boxes;  // [n_img, cap, 4] fp32 or fp64
  int boxes_f64;
  WorkList work;
  int n_round;
  int apply_small_filter;  // filter_small_proposal before every round (boundary_reasoning) or not (single round)
  int early_exit;
  float area_thres, max_sdf_thres, max_shrink_thres, delta_ratio;
  float4* boxes_out;   // [n_img, cap]
  float* labels_out;   // 1 / 0 / -1 as the reference; -2 = removed by filter_small_proposal
  int* rounds_out;     // rounds actually evaluated (nullable)
  WindowSlot* windows; // [n_img][kWindowSlots], zeroed before launch; nullptr: every round computes its terms
};
struct TileParams {
  const float* tiles;  // [M, 128, 128]
  int M;
  float4* deltas;      // [M] (dx1, dy1, dx2, dy2)
  float* max_sdf;      // [M] or nullptr
};
// image_hw: nullable [n_img, 2] (h, w) of each image inside the (H, W) pitch: the sized kernel variant
int launch_refine(const RefineParams& p, int num_sms, cudaStream_t stream, const int* image_hw = nullptr);
int launch_refine_aa(const RefineParams& p, int num_sms, cudaStream_t stream);   // antialiased crops
int launch_tiles(const TileParams& p, cudaStream_t stream);
int launch_round_update(const RefineParams& p, const float4* deltas, const float* max_sdf, int M, cudaStream_t stream);

// ---- exist.cu ------------------------------------------------------------------------
struct ExistParams {
  const float* fields;
  int C, H, W, ch_exist;
  const void* boxes;
  int boxes_f64;
  WorkList work;
  float* scores;  // [n_img, cap]
  const int* image_hw;  // nullable [n_img, 2] (h, w) of each image inside the (H, W) pitch: the sized kernel variant
};
int launch_existence(const ExistParams& p, int num_sms, cudaStream_t stream);
int launch_existence_aa(const ExistParams& p, int num_sms, cudaStream_t stream);   // antialiased crops
int launch_tile_means(const float* tiles, long long tile_stride, int M, float* out, cudaStream_t stream);
int launch_crop_resize(const float* fields, int n_img, int C, int H, int W, const int* channels, int n_ch,
                       const void* boxes, int boxes_f64, const int* counts, int cap, float* out, cudaStream_t stream);

int launch_crop_resize_aa(const float* fields, int n_img, int C, int H, int W, const int* channels, int n_ch,
                          const void* boxes, int boxes_f64, const int* counts, int cap, float* out, float* scratch,
                          cudaStream_t stream);
int launch_mask_resize_aa(const unsigned char* masks, int B, int oh, int ow, unsigned char* out, float* scratch, cudaStream_t stream);

// ---- center.cu -----------------------------------------------------------------------
constexpr int kCcCap = 16;   // connected-component boxes kept per proposal (--analyze_cc); overflow is counted
struct CenterParams {
  const float* tiles;   // nullable: pre-resampled [n_img * cap, 3, 128, 128] (sdf, center_row, center_col) instead of `fields`
  const float* fields;
  int C, H, W, ch_sdf, ch_crow, ch_ccol;
  const void* boxes;
  int boxes_f64;
  WorkList work;
  double thr;          // center_score_max_thres
  double* max_values;  // [n_img, cap] amax of the masked anti-center map (fp64)
  int* argmax;         // [n_img, cap] flat index yc*128+xc of the first maximum, -1 when the proposal passes
  double* splits;      // [n_img, cap, 4, 4] L/R/T/B boxes for failing proposals (nullable)
  // F.normalize(filter, dim=1) in fp32, then .double() (object_reasoning.py:372-373):
  // filt[i*5+j] = (2-i)/sqrt((2-i)^2+(2-j)^2); channel 1 uses the transposed entry
  double filt[25];
  // fp32 screening pass: (f[0][i][j], f[1][i][j]) as one aligned 64-bit pair per tap, so the packed FFMA2 reads
  // its filter operand straight from the constant bank (no per-use pair assembly in uniform registers)
  unsigned long long filt_pair[25];
  // --analyze_cc (object_reasoning.py:561-572); all three null when off
  unsigned char* cc_counts;  // [n_img, cap] component boxes emitted (0 unless the proposal passes with >= 2 components)
  double* cc_boxes;          // [n_img, cap, kCcCap, 4] enlarged component boxes
  int* cc_overflow;          // incremented once per proposal with more than kCcCap components
  const int* image_hw;       // nullable [n_img, 2] (h, w) of each image inside the (H, W) pitch: the sized kernel variant
};
int launch_center(const CenterParams& p, int num_sms, cudaStream_t stream);
int launch_components(const unsigned char* masks, int B, int* counts, int* boxes, cudaStream_t stream);
int launch_erode(const unsigned char* in, unsigned char* out, int B, int kernel_size, int num_round, cudaStream_t stream);
int launch_anti_center(const float* vote, double* out, int B, int H, int W, const double* filt25, cudaStream_t stream);

// ---- lists.cu ------------------------------------------------------------------------
int launch_prefix_counts(const int* counts, int n_img, int* offsets, cudaStream_t stream);

enum CompactMode { kFlagsU8 = 0, kScoreGE = 1, kLabelEQ = 2, kArgmaxGE0 = 3, kArgmaxLT0 = 4 };
struct CompactParams {
  const void* in;        // [n_img, cap_in, group, 4]
  int in_f64;
  const int* counts_in;  // nullable
  int cap_in;
  int group;             // boxes per entry (1, or 4 for split boxes); row stride of `in` when group_counts is set
  const unsigned char* group_counts;  // nullable [n_img, cap_in]: boxes actually carried by each entry (<= group)
  int* overflow;         // nullable: incremented per image whose output did not fit cap_out
  int mode;
  const void* pred;      // u8 flags / float scores / float labels / int argmax, [n_img, cap_in]
  float thr;
  void* out;             // [n_img, cap_out, 4]
  int out_f64;
  int cap_out;
  int* counts_out;       // [n_img]
  int append;            // 1: append after the counts_out[] rows already present
  int* index_out;        // nullable [n_img, cap_out]: source entry index of every output row
  int n_img;
};
int launch_compact(const CompactParams& p, cudaStream_t stream);
int launch_pack_detections(const long long* image_ids, const float4* bbox_xywh, const double* out5, const int* keep_counts,
                           int cap, int n_img, double* rows, int max_rows, cudaStream_t stream);

// ---- nms.cu --------------------------------------------------------------------------
struct NmsParams {
  const float4* boxes;   // [n_img, cap]
  const float* scores;   // [n_img, cap] or nullptr (all equal -> index order)
  const int* counts;     // nullable
  int cap, n_img;
  float iou_thr;
  int* keep;             // [n_img, cap] kept indices in descending-score order
  int* keep_counts;      // [n_img]
  float4* boxes_out;     // nullable [n_img, cap] kept boxes, same order
  int* order_ws;         // [n_img, cap] workspace
};
int launch_box_nms(const NmsParams& p, cudaStream_t stream);

// ---- score.cu ------------------------------------------------------------------------
struct ScoreParams {
  const float* tiles;  // nullable: pre-resampled [n_img * cap, 4, 128, 128] (sdf, center_row, center_col, existence)
  const float* exist_scores;  // nullable, tile path only: [n_img, cap] per-crop existence scores instead of the mean of tile 3
  int aa_raster;       // tile path only: resize the masks back to the box with the antialiased kernel
  const float* fields;
  int n_img, C, H, W, ch_sdf, ch_crow, ch_ccol, ch_exist;
  const void* boxes;   // [n_img, cap, 4]
  int boxes_f64;
  const int* counts;   // nullable
  int cap;
  float4* scores;      // [n_img, cap] (existence, center, boundary, 0)
  float4* tight;       // [n_img, cap] tight box xyxy of the union mask (zeros if empty)
  int* areas;          // [n_img, cap] set pixels
  uint32_t* masks;     // nullable [n_img, cap, H, ceil(W/32)] packed union masks
};
// The sized kernel variant's parameters (a struct of its own: a larger ScoreParams changes the code of score_kernel)
struct ScoreHwParams : ScoreParams {
  const int* image_hw; // [n_img, 2] (h, w) of each image inside the (H, W) pitch
};
int launch_score(const ScoreParams& p, cudaStream_t stream, const int* image_hw = nullptr);
int launch_mask_resize(const unsigned char* masks, int B, int oh, int ow, unsigned char* out, cudaStream_t stream);

struct FinalParams {
  const float4* scores;  // [n_img, cap]
  const float4* tight;   // [n_img, cap]
  const int* areas;      // [n_img, cap]
  const int* keep;       // [n_img, cap] indices kept by NMS, in order
  const int* keep_counts;
  int cap, n_img;
  double existence_thres, center_thres, boundary_thres;  // post_process.py:38-40 (Python floats: the fp32 scores are compared in double, :64-69)
  double* out;           // [n_img, cap, 5] (score, existence, center, boundary, area_score) in keep order
  float4* bbox_xywh;     // [n_img, cap] COCO-style box in keep order
  unsigned char* selected;  // nullable [n_img, cap] post_process predicate
};
int launch_final_scores(const FinalParams& p, cudaStream_t stream);

// ---- sat.cu, box_sums.cu --------------------------------------------------------------------------
int launch_sat(const float* in, double* out, int n_planes, int H, int W, int C, const int* channels, int n_ch,
               cudaStream_t stream);
// tables of a padded field stack: pixels outside each image's (h, w) enter the sums as zeros
int launch_sat_hw(const float* fields, double* out, int n_img, int H, int W, int C, const int* channels, int n_ch,
                  const int* image_hw, cudaStream_t stream);
int launch_box_sums(const double* sat, int planes_per_img, int plane, int H, int W, const void* boxes, int boxes_f64,
                    const int* counts, int cap, int n_img, double* sums, double* means, const int* image_hw,
                    cudaStream_t stream);
int launch_box_sums_hw(const double* sat, int planes_per_img, int plane, int H, int W, const void* boxes, int boxes_f64,
                       const int* counts, int cap, int n_img, double* sums, double* means, const int* image_hw,
                       cudaStream_t stream);

// ---- masks.cu ------------------------------------------------------------------------
int launch_mask_pack(const unsigned char* in, uint32_t* out, size_t n_masks, int H, int W, int num_sms, cudaStream_t stream);
int launch_rle_counts(const uint32_t* masks, int K, int H, int W, int max_runs, uint32_t* counts, int* n_runs,
                      cudaStream_t stream);
int launch_mask_stats(const uint32_t* masks, int K, int H, int Wp, int* areas, int4* tight, cudaStream_t stream);
int launch_matrix_nms(const uint32_t* masks, const float4* boxes, int K, int H, int Wp, const float* scores,
                      const int* areas, const int4* tight, float thr, int* order, unsigned long long* matrix,
                      int* keep, int* keep_count, cudaStream_t stream);

}  // namespace unmore
