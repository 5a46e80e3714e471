// C-ABI entry points (include/unmore_b200.h).  Argument checking, workspace carving and
// kernel launches only; no device allocation, no synchronisation, no global mutable state
// other than the thread-local error string.
#include <cstdio>
#include <cstdarg>
#include <cmath>
#include <cstring>

#include "../../include/unmore_b200.h"
#include "unmore_internal.h"

using namespace unmore;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int cuda_fail(int code, const char* what) {
  if (code == 0) return 0;
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString((cudaError_t)code));
  return code;
}

int num_sms() {  // of the current device; a plain attribute query, no cached state
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) == cudaSuccess &&
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
    return n;
  return 148;
}

// ws layout: [0] work counter, [1 .. n_img+1] exclusive prefix of counts (ints); then, at the first 32-byte
// aligned address after them, the window caches of unmore_boundary_refine: n_img tables of kWindowSlots
// WindowSlot entries, zeroed by that call (a table lives for one call; the other kernels leave it alone)
size_t worklist_bytes(int n_img) { return sizeof(int) * (size_t)(n_img + 2 > 2 ? n_img + 2 : 2); }

WindowSlot* window_tables(void* ws, int n_img) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(ws) + worklist_bytes(n_img);
  return reinterpret_cast<WindowSlot*>((a + alignof(WindowSlot) - 1) & ~(uintptr_t)(alignof(WindowSlot) - 1));
}

int make_worklist(WorkList& w, const int* counts, int n_img, int cap, void* ws, cudaStream_t s) {
  int* wsi = reinterpret_cast<int*>(ws);
  w.counter = wsi;
  w.n_img = n_img;
  w.cap = cap;
  w.total_dense = n_img * cap;
  w.offsets = nullptr;
  int e = (int)cudaMemsetAsync(wsi, 0, sizeof(int), s);
  if (e) return cuda_fail(e, "memset work counter");
  if (counts) {
    w.offsets = wsi + 1;
    e = launch_prefix_counts(counts, n_img, wsi + 1, s);
    if (e) return cuda_fail(e, "prefix_counts");
  }
  return 0;
}

// F.normalize(filter, dim=1) in fp32 then .double() (object_reasoning.py:372-373):
// filt[i*5+j] = (2-i)/max(sqrt((2-i)^2+(2-j)^2), 1e-12); channel 1 reads the transposed entry
void anti_center_filter(double* filt) {
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 5; ++j) {
      const int di = 2 - i, dj = 2 - j;
      const float n = std::sqrt((float)(di * di + dj * dj));
      filt[i * 5 + j] = (double)((float)di / (n > 1e-12f ? n : 1e-12f));
    }
}

// Both filter tables of the center kernel: fp64 for the exact pass, (channel 0, channel 1) fp32 pairs for the screening pass
void center_filters(CenterParams& p) {
  anti_center_filter(p.filt);
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 5; ++j) {   // exact casts: the table is fp32-valued
      const float f0 = (float)p.filt[i * 5 + j], f1 = (float)p.filt[j * 5 + i];
      unsigned lo, hi;
      memcpy(&lo, &f0, 4); memcpy(&hi, &f1, 4);
      p.filt_pair[i * 5 + j] = ((unsigned long long)hi << 32) | lo;
    }
}

int check_fields(const float* f, int n_img, int C, int H, int W) {
  if (!f || n_img <= 0 || C <= 0 || H <= 0 || W <= 0) return fail(UNMORE_E_INVALID, "bad field tensor");
  // the kernels are launched on the CURRENT device: a field stack that lives on another GPU would be read
  // through a foreign pointer (illegal address, or silent peer traffic) — refuse it instead
  cudaPointerAttributes attr;
  int dev = -1;
  if (cudaPointerGetAttributes(&attr, f) == cudaSuccess && attr.type == cudaMemoryTypeDevice &&
      cudaGetDevice(&dev) == cudaSuccess && attr.device != dev)
    return fail(UNMORE_E_INVALID, "field tensor lives on device %d but the current device is %d (set the device, or use the stream of the tensor's device)", attr.device, dev);
  (void)cudaGetLastError();
  return 0;
}

// The (h, w) table of a padded field stack (the *_hw entry points): the kernels read it, so it must be device memory
// of the current device, and 8-byte aligned (one int2 per image).  Host memory dereferenced in a kernel faults.
int check_extents(const char* name, const int* image_hw) {
  if (!image_hw) return fail(UNMORE_E_INVALID, "%s: image_hw is null", name);
  if (reinterpret_cast<uintptr_t>(image_hw) & 7) return fail(UNMORE_E_INVALID, "%s: image_hw must be 8-byte aligned", name);
  cudaPointerAttributes attr;
  int dev = -1;
  if (cudaPointerGetAttributes(&attr, image_hw) == cudaSuccess) {
    if (attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeUnregistered)
      return fail(UNMORE_E_INVALID, "%s: image_hw is host memory (it must be a device tensor)", name);
    if (attr.type == cudaMemoryTypeDevice && cudaGetDevice(&dev) == cudaSuccess && attr.device != dev)
      return fail(UNMORE_E_INVALID, "%s: image_hw lives on device %d but the current device is %d", name, attr.device, dev);
  }
  (void)cudaGetLastError();
  return 0;
}

// unmore_existence_scores / unmore_existence_scores_aa and their _hw forms: the same call in either resize mode, and
// on a padded stack (image_hw non-null)
int existence_scores(const char* name, bool aa, const float* fields, int n_img, int C, int H, int W, int ch_exist,
                     const void* boxes, int boxes_f64, const int* counts, int cap, float* scores_out, void* ws,
                     cudaStream_t s, const int* image_hw = nullptr) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !scores_out || !ws || cap < 0 || ch_exist < 0 || ch_exist >= C)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (cap == 0) return 0;
  ExistParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W; p.ch_exist = ch_exist;
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.scores = scores_out; p.image_hw = image_hw;
  if (int e = make_worklist(p.work, counts, n_img, cap, ws, s)) return e;
  if (aa) return cuda_fail(launch_existence_aa(p, num_sms(), s), "existence_aa_kernel");
  return cuda_fail(launch_existence(p, num_sms(), s), "existence_kernel");
}

// unmore_boundary_refine / unmore_boundary_refine_aa and their _hw forms
int boundary_refine(const char* name, bool aa, const float* fields, int n_img, int C, int H, int W, int ch_sdf,
                    const void* boxes, int boxes_f64, const int* counts, int cap, int n_round, int apply_small_filter,
                    int early_exit, float proposal_area_thres, float max_sdf_thres, float max_shrink_threshold,
                    float delta_ratio, float* boxes_out, float* labels_out, int* rounds_out, void* ws, cudaStream_t s,
                    const int* image_hw = nullptr) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !boxes_out || !labels_out || !ws || cap < 0 || n_round < 1 || ch_sdf < 0 || ch_sdf >= C)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (cap == 0) return 0;
  RefineParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W; p.ch_sdf = ch_sdf;
  p.boxes = boxes; p.boxes_f64 = boxes_f64;
  p.n_round = n_round; p.apply_small_filter = apply_small_filter; p.early_exit = early_exit;
  p.area_thres = proposal_area_thres; p.max_sdf_thres = max_sdf_thres;
  p.max_shrink_thres = max_shrink_threshold; p.delta_ratio = delta_ratio;
  p.boxes_out = reinterpret_cast<float4*>(boxes_out); p.labels_out = labels_out; p.rounds_out = rounds_out;
  p.image_hw = image_hw;
  if (int e = make_worklist(p.work, counts, n_img, cap, ws, s)) return e;
  if (W <= kWindowMaxSide && H <= kWindowMaxSide) {
    p.windows = window_tables(ws, n_img);
    const int e = (int)cudaMemsetAsync(p.windows, 0, sizeof(WindowSlot) * kWindowSlots * (size_t)n_img, s);
    if (e) return cuda_fail(e, "memset window tables");
  }
  if (aa) return cuda_fail(launch_refine_aa(p, num_sms(), s), "refine_aa_kernel");
  return cuda_fail(launch_refine(p, num_sms(), s), "refine_kernel");
}

// unmore_center_reasoning / unmore_center_reasoning_aa and their _hw forms
int center_reasoning(const char* name, bool aa, const float* fields, int n_img, int C, int H, int W, int ch_sdf, int ch_center_row,
                     int ch_center_col, const void* boxes, int boxes_f64, const int* counts, int cap,
                     double center_score_max_thres, double* max_values_out, int* argmax_out, double* splits_out,
                     unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow, void* ws, cudaStream_t s,
                     const int* image_hw = nullptr) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !max_values_out || !argmax_out || !ws || cap < 0 || ch_sdf < 0 || ch_sdf >= C || ch_center_row < 0 ||
      ch_center_row >= C || ch_center_col < 0 || ch_center_col >= C)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (cap == 0) return 0;
  CenterParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W;
  p.ch_sdf = ch_sdf; p.ch_crow = ch_center_row; p.ch_ccol = ch_center_col;
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.thr = center_score_max_thres;
  p.max_values = max_values_out; p.argmax = argmax_out; p.splits = splits_out;
  if ((cc_counts_out != nullptr) != (cc_boxes_out != nullptr) || (cc_counts_out != nullptr) != (cc_overflow != nullptr))
    return fail(UNMORE_E_INVALID, "%s: the three analyze_cc outputs go together", name);
  p.cc_counts = cc_counts_out; p.cc_boxes = cc_boxes_out; p.cc_overflow = cc_overflow;
  p.image_hw = image_hw;
  center_filters(p);
  if (int e = make_worklist(p.work, counts, n_img, cap, ws, s)) return e;
  if (aa) return cuda_fail(launch_center_aa(p, num_sms(), s), "center_aa_kernel");
  return cuda_fail(launch_center(p, num_sms(), s), "center_kernel");
}

// unmore_score_and_rasterise / unmore_score_and_rasterise_hw
int score_and_rasterise(const char* name, const float* fields, int n_img, int C, int H, int W, int ch_sdf, int ch_center_row,
                        int ch_center_col, int ch_exist, const void* boxes, int boxes_f64, const int* counts, int cap,
                        float* scores_out, float* tight_out, int* areas_out, uint32_t* masks_out, cudaStream_t s,
                        const int* image_hw = nullptr) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !scores_out || !tight_out || !areas_out || cap < 0 || ch_sdf < 0 || ch_sdf >= C || ch_center_row < 0 ||
      ch_center_row >= C || ch_center_col < 0 || ch_center_col >= C || ch_exist < 0 || ch_exist >= C)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (n_img > 65535) return fail(UNMORE_E_CAPACITY, "%s: n_img > 65535 per call", name);
  ScoreParams p{};
  p.fields = fields; p.n_img = n_img; p.C = C; p.H = H; p.W = W;
  p.ch_sdf = ch_sdf; p.ch_crow = ch_center_row; p.ch_ccol = ch_center_col; p.ch_exist = ch_exist;
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.counts = counts; p.cap = cap;
  p.scores = reinterpret_cast<float4*>(scores_out); p.tight = reinterpret_cast<float4*>(tight_out);
  p.areas = areas_out; p.masks = masks_out; p.image_hw = image_hw;
  return cuda_fail(launch_score(p, s), "score_kernel");
}

// unmore_box_sums / unmore_box_sums_hw
int box_sums(const char* name, const double* sat, int n_img, int planes_per_img, int plane, int H, int W, const void* boxes,
             int boxes_f64, const int* counts, int cap, double* sums_out, double* means_out, cudaStream_t s,
             const int* image_hw = nullptr) {
  if (!sat || !boxes || !sums_out || n_img < 0 || cap < 0 || plane < 0 || plane >= planes_per_img ||
      (image_hw && (H <= 0 || W <= 0)))
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  return cuda_fail(launch_box_sums(sat, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap, n_img, sums_out,
                                   means_out, image_hw, s),
                   "box_sums_kernel");
}

// unmore_crop_resize_aa / unmore_crop_resize_aa_hw
int crop_resize_aa(const char* name, const float* fields, int n_img, int C, int H, int W, const int* channels_host,
                   int n_channels, const void* boxes, int boxes_f64, const int* counts, int cap, float* out, void* scratch,
                   size_t scratch_bytes, cudaStream_t s, const int* image_hw = nullptr) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !out || !channels_host || cap < 0 || n_channels < 1 || n_channels > 4)
    return fail(UNMORE_E_INVALID, "%s: bad argument (1..4 channels)", name);
  for (int i = 0; i < n_channels; ++i)
    if (channels_host[i] < 0 || channels_host[i] >= C) return fail(UNMORE_E_INVALID, "%s: channel out of range", name);
  const size_t need = (size_t)n_img * cap * n_channels * H * 128 * sizeof(float);
  if (need && (!scratch || scratch_bytes < need))
    return fail(UNMORE_E_CAPACITY, "%s: scratch must hold n_img*cap*n_channels*H*128 floats (%zu bytes)", name, need);
  return cuda_fail(launch_crop_resize_aa(fields, n_img, C, H, W, channels_host, n_channels, boxes, boxes_f64, counts, cap, out,
                                         reinterpret_cast<float*>(scratch), s, image_hw),
                   "crop_resize_aa kernels");
}

// unmore_center_reasoning_from_tiles / unmore_center_reasoning_from_tiles_hw
int center_from_tiles(const char* name, const float* tiles, int n_img, int H, int W, const void* boxes, int boxes_f64,
                      const int* counts, int cap, double center_score_max_thres, double* max_values_out, int* argmax_out,
                      double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow, void* ws,
                      cudaStream_t s, const int* image_hw = nullptr) {
  if (!tiles || !boxes || !max_values_out || !argmax_out || !ws || cap < 0 || n_img <= 0 || H <= 0 || W <= 0)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (cap == 0) return 0;
  CenterParams p{};
  p.tiles = tiles; p.C = 3; p.H = H; p.W = W; p.ch_sdf = 0; p.ch_crow = 1; p.ch_ccol = 2;
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.thr = center_score_max_thres;
  p.max_values = max_values_out; p.argmax = argmax_out; p.splits = splits_out;
  if ((cc_counts_out != nullptr) != (cc_boxes_out != nullptr) || (cc_counts_out != nullptr) != (cc_overflow != nullptr))
    return fail(UNMORE_E_INVALID, "%s: the three analyze_cc outputs go together", name);
  p.cc_counts = cc_counts_out; p.cc_boxes = cc_boxes_out; p.cc_overflow = cc_overflow;
  p.image_hw = image_hw;
  center_filters(p);
  if (int e = make_worklist(p.work, counts, n_img, cap, ws, s)) return e;
  return cuda_fail(launch_center(p, num_sms(), s), "center_kernel (tiles)");
}

// unmore_score_and_rasterise_from_tiles / unmore_score_and_rasterise_from_tiles_hw
int score_from_tiles(const char* name, const float* tiles, const float* existence_scores, int antialias, int n_img, int H,
                     int W, const void* boxes, int boxes_f64, const int* counts, int cap, float* scores_out, float* tight_out,
                     int* areas_out, uint32_t* masks_out, cudaStream_t s, const int* image_hw = nullptr) {
  if (!tiles || !boxes || !scores_out || !tight_out || !areas_out || cap < 0 || n_img <= 0 || H <= 0 || W <= 0)
    return fail(UNMORE_E_INVALID, "%s: bad argument", name);
  if (n_img > 65535) return fail(UNMORE_E_CAPACITY, "%s: n_img > 65535 per call", name);
  ScoreParams p{};
  p.tiles = tiles; p.exist_scores = existence_scores; p.aa_raster = antialias; p.n_img = n_img; p.C = 4; p.H = H; p.W = W;
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.counts = counts; p.cap = cap;
  p.scores = reinterpret_cast<float4*>(scores_out); p.tight = reinterpret_cast<float4*>(tight_out);
  p.areas = areas_out; p.masks = masks_out; p.image_hw = image_hw;
  return cuda_fail(launch_score(p, s), "score_kernel (tiles)");
}

}  // namespace

extern "C" {

const char* unmore_last_error(void) { return g_err; }
int unmore_version(void) { return 102; }
size_t unmore_workspace_bytes(int n_img) {
  // the alignment slack lets `ws` be any 4-byte aligned pointer
  return worklist_bytes(n_img) + (n_img > 0 ? alignof(WindowSlot) - 1 + sizeof(WindowSlot) * kWindowSlots * (size_t)n_img : 0);
}

int unmore_existence_scores(const float* fields, int n_img, int C, int H, int W, int ch_exist, const void* boxes,
                            int boxes_f64, const int* counts, int cap, float* scores_out, void* ws,
                            unmore_stream_t stream) {
  return existence_scores("unmore_existence_scores", false, fields, n_img, C, H, W, ch_exist, boxes, boxes_f64, counts, cap,
                          scores_out, ws, (cudaStream_t)stream);
}

int unmore_existence_scores_aa(const float* fields, int n_img, int C, int H, int W, int ch_exist, const void* boxes,
                               int boxes_f64, const int* counts, int cap, float* scores_out, void* ws,
                               unmore_stream_t stream) {
  return existence_scores("unmore_existence_scores_aa", true, fields, n_img, C, H, W, ch_exist, boxes, boxes_f64, counts, cap,
                          scores_out, ws, (cudaStream_t)stream);
}

int unmore_crop_resize(const float* fields, int n_img, int C, int H, int W, const int* channels_host, int n_channels,
                       const void* boxes, int boxes_f64, const int* counts, int cap, float* out, unmore_stream_t stream) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!boxes || !out || !channels_host || cap < 0 || n_channels < 1 || n_channels > 4)
    return fail(UNMORE_E_INVALID, "unmore_crop_resize: bad argument (1..4 channels)");
  for (int i = 0; i < n_channels; ++i)
    if (channels_host[i] < 0 || channels_host[i] >= C) return fail(UNMORE_E_INVALID, "unmore_crop_resize: channel out of range");
  return cuda_fail(launch_crop_resize(fields, n_img, C, H, W, channels_host, n_channels, boxes, boxes_f64, counts, cap, out,
                                      (cudaStream_t)stream),
                   "crop_resize_kernel");
}

int unmore_crop_resize_aa(const float* fields, int n_img, int C, int H, int W, const int* channels_host, int n_channels,
                          const void* boxes, int boxes_f64, const int* counts, int cap, float* out, void* scratch,
                          size_t scratch_bytes, unmore_stream_t stream) {
  return crop_resize_aa("unmore_crop_resize_aa", fields, n_img, C, H, W, channels_host, n_channels, boxes, boxes_f64, counts,
                        cap, out, scratch, scratch_bytes, (cudaStream_t)stream);
}

int unmore_mask_resize_aa(const unsigned char* masks, int B, int H, int W, int out_h, int out_w, unsigned char* out,
                          void* scratch, size_t scratch_bytes, unmore_stream_t stream) {
  if (B < 0 || out_h < 0 || out_w < 0 || (B > 0 && (!masks || !out))) return fail(UNMORE_E_INVALID, "unmore_mask_resize_aa: bad argument");
  if (H != 128 || W != 128) return fail(UNMORE_E_INVALID, "unmore_mask_resize_aa: masks must be 128x128 (the crop side of the reference)");
  const size_t need = (size_t)B * 128 * out_w * sizeof(float);
  if (need && (!scratch || scratch_bytes < need))
    return fail(UNMORE_E_CAPACITY, "unmore_mask_resize_aa: scratch must hold B*128*out_w floats (%zu bytes)", need);
  return cuda_fail(launch_mask_resize_aa(masks, B, out_h, out_w, out, reinterpret_cast<float*>(scratch), (cudaStream_t)stream),
                   "mask_resize_aa kernels");
}

int unmore_center_reasoning(const float* fields, int n_img, int C, int H, int W, int ch_sdf, int ch_center_row,
                            int ch_center_col, const void* boxes, int boxes_f64, const int* counts, int cap,
                            double center_score_max_thres, double* max_values_out, int* argmax_out,
                            double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow,
                            void* ws, unmore_stream_t stream) {
  return center_reasoning("unmore_center_reasoning", false, fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col, boxes,
                          boxes_f64, counts, cap, center_score_max_thres, max_values_out, argmax_out, splits_out,
                          cc_counts_out, cc_boxes_out, cc_overflow, ws, (cudaStream_t)stream);
}

int unmore_center_reasoning_aa(const float* fields, int n_img, int C, int H, int W, int ch_sdf, int ch_center_row,
                               int ch_center_col, const void* boxes, int boxes_f64, const int* counts, int cap,
                               double center_score_max_thres, double* max_values_out, int* argmax_out,
                               double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow,
                               void* ws, unmore_stream_t stream) {
  return center_reasoning("unmore_center_reasoning_aa", true, fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col,
                          boxes, boxes_f64, counts, cap, center_score_max_thres, max_values_out, argmax_out, splits_out,
                          cc_counts_out, cc_boxes_out, cc_overflow, ws, (cudaStream_t)stream);
}

int unmore_boundary_refine(const float* fields, int n_img, int C, int H, int W, int ch_sdf, const void* boxes,
                           int boxes_f64, const int* counts, int cap, int n_round, int apply_small_filter,
                           int early_exit, float proposal_area_thres, float max_sdf_thres, float max_shrink_threshold,
                           float delta_ratio, float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                           unmore_stream_t stream) {
  return boundary_refine("unmore_boundary_refine", false, fields, n_img, C, H, W, ch_sdf, boxes, boxes_f64, counts, cap, n_round,
                         apply_small_filter, early_exit, proposal_area_thres, max_sdf_thres, max_shrink_threshold,
                         delta_ratio, boxes_out, labels_out, rounds_out, ws, (cudaStream_t)stream);
}

int unmore_boundary_refine_aa(const float* fields, int n_img, int C, int H, int W, int ch_sdf, const void* boxes,
                              int boxes_f64, const int* counts, int cap, int n_round, int apply_small_filter,
                              int early_exit, float proposal_area_thres, float max_sdf_thres, float max_shrink_threshold,
                              float delta_ratio, float* boxes_out, float* labels_out, int* rounds_out, void* ws,
                              unmore_stream_t stream) {
  return boundary_refine("unmore_boundary_refine_aa", true, fields, n_img, C, H, W, ch_sdf, boxes, boxes_f64, counts, cap,
                         n_round, apply_small_filter, early_exit, proposal_area_thres, max_sdf_thres, max_shrink_threshold,
                         delta_ratio, boxes_out, labels_out, rounds_out, ws, (cudaStream_t)stream);
}

int unmore_update_bbox_from_tiles(const float* tiles, int M, float* deltas_out, float* max_out,
                                  unmore_stream_t stream) {
  if (M < 0 || (M > 0 && (!tiles || !deltas_out))) return fail(UNMORE_E_INVALID, "unmore_update_bbox_from_tiles: bad argument");
  TileParams p{tiles, M, reinterpret_cast<float4*>(deltas_out), max_out};
  return cuda_fail(launch_tiles(p, (cudaStream_t)stream), "tiles_kernel");
}

// ---- tile path (second resize mode, antialias=True): the same stages on PRE-RESAMPLED tiles -------------------------
int unmore_tile_means(const float* tiles, long long tile_stride, int M, float* means_out, unmore_stream_t stream) {
  if (M < 0 || tile_stride < 128 * 128 || (M > 0 && (!tiles || !means_out))) return fail(UNMORE_E_INVALID, "unmore_tile_means: bad argument");
  return cuda_fail(launch_tile_means(tiles, tile_stride, M, means_out, (cudaStream_t)stream), "tile_means_kernel");
}

int unmore_center_reasoning_from_tiles(const float* tiles, int n_img, int H, int W, const void* boxes, int boxes_f64,
                                       const int* counts, int cap, double center_score_max_thres, double* max_values_out,
                                       int* argmax_out, double* splits_out, unsigned char* cc_counts_out,
                                       double* cc_boxes_out, int* cc_overflow, void* ws, unmore_stream_t stream) {
  return center_from_tiles("unmore_center_reasoning_from_tiles", tiles, n_img, H, W, boxes, boxes_f64, counts, cap,
                           center_score_max_thres, max_values_out, argmax_out, splits_out, cc_counts_out, cc_boxes_out,
                           cc_overflow, ws, (cudaStream_t)stream);
}

int unmore_boundary_round_from_tiles(const float* tiles, int M, const void* boxes, int boxes_f64, int H, int W,
                                     float max_sdf_thres, float max_shrink_threshold, float delta_ratio, float* boxes_out,
                                     float* labels_out, float* deltas_ws, float* max_ws, unmore_stream_t stream) {
  if (M < 0 || H <= 0 || W <= 0 || (M > 0 && (!tiles || !boxes || !boxes_out || !labels_out || !deltas_ws || !max_ws)))
    return fail(UNMORE_E_INVALID, "unmore_boundary_round_from_tiles: bad argument");
  if (M == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  TileParams t{tiles, M, reinterpret_cast<float4*>(deltas_ws), max_ws};
  if (int e = cuda_fail(launch_tiles(t, s), "tiles_kernel")) return e;
  RefineParams p{};
  p.H = H; p.W = W; p.boxes = boxes; p.boxes_f64 = boxes_f64;
  p.max_sdf_thres = max_sdf_thres; p.max_shrink_thres = max_shrink_threshold; p.delta_ratio = delta_ratio;
  p.boxes_out = reinterpret_cast<float4*>(boxes_out); p.labels_out = labels_out;
  return cuda_fail(launch_round_update(p, reinterpret_cast<const float4*>(deltas_ws), max_ws, M, s), "round_update_kernel");
}

int unmore_score_and_rasterise_from_tiles(const float* tiles, const float* existence_scores, int antialias, int n_img, int H,
                                          int W, const void* boxes, int boxes_f64, const int* counts, int cap,
                                          float* scores_out, float* tight_out, int* areas_out, uint32_t* masks_out,
                                          unmore_stream_t stream) {
  return score_from_tiles("unmore_score_and_rasterise_from_tiles", tiles, existence_scores, antialias, n_img, H, W, boxes,
                          boxes_f64, counts, cap, scores_out, tight_out, areas_out, masks_out, (cudaStream_t)stream);
}

int unmore_cc_cap(void) { return kCcCap; }

int unmore_compact_boxes(const void* in, int in_f64, const int* counts_in, int cap_in, int group, int mode,
                         const void* pred, float thr, void* out, int out_f64, int cap_out, int* counts_out,
                         int append, int* index_out, const unsigned char* group_counts, int* overflow, int n_img,
                         unmore_stream_t stream) {
  if (!in || !pred || !out || !counts_out || cap_in < 0 || cap_out < 0 || group < 1 || mode < 0 || mode > 5 || n_img < 0)
    return fail(UNMORE_E_INVALID, "unmore_compact_boxes: bad argument");
  CompactParams p{};
  p.in = in; p.in_f64 = in_f64; p.counts_in = counts_in; p.cap_in = cap_in; p.group = group; p.mode = mode;
  p.pred = pred; p.thr = thr; p.out = out; p.out_f64 = out_f64; p.cap_out = cap_out; p.counts_out = counts_out;
  p.append = append; p.index_out = index_out; p.n_img = n_img;
  p.group_counts = group_counts; p.overflow = overflow;
  return cuda_fail(launch_compact(p, (cudaStream_t)stream), "compact_kernel");
}

int unmore_box_nms(const float* boxes, const float* scores, const int* counts, int cap, int n_img, float iou_threshold,
                   int* keep_out, int* keep_counts_out, float* boxes_out, int* order_ws, unmore_stream_t stream) {
  if (cap < 0 || n_img < 0 || (n_img > 0 && !keep_counts_out)) return fail(UNMORE_E_INVALID, "unmore_box_nms: bad argument");
  if (n_img == 0) return 0;
  if (cap == 0) return cuda_fail((int)cudaMemsetAsync(keep_counts_out, 0, sizeof(int) * n_img, (cudaStream_t)stream), "memset");
  if (!boxes || !keep_out || !order_ws) return fail(UNMORE_E_INVALID, "unmore_box_nms: bad argument");
  if (cap > 32768) return fail(UNMORE_E_CAPACITY, "unmore_box_nms: cap %d > 32768", cap);
  NmsParams p{};
  p.boxes = reinterpret_cast<const float4*>(boxes); p.scores = scores; p.counts = counts; p.cap = cap; p.n_img = n_img;
  p.iou_thr = iou_threshold; p.keep = keep_out; p.keep_counts = keep_counts_out;
  p.boxes_out = reinterpret_cast<float4*>(boxes_out); p.order_ws = order_ws;
  return cuda_fail(launch_box_nms(p, (cudaStream_t)stream), "box_nms_kernel");
}

int unmore_batch_erode(const unsigned char* masks, int B, int H, int W, int kernel_size, int num_round,
                       unsigned char* out, unmore_stream_t stream) {
  if (B < 0 || kernel_size < 1 || !(kernel_size & 1) || num_round < 0 || (B > 0 && (!masks || !out)))
    return fail(UNMORE_E_INVALID, "unmore_batch_erode: bad argument");
  if (H != kCrop || W != kCrop) return fail(UNMORE_E_CAPACITY, "unmore_batch_erode: only 128x128 crops (got %dx%d)", H, W);
  return cuda_fail(launch_erode(masks, out, B, kernel_size, num_round, (cudaStream_t)stream), "erode_kernel");
}

int unmore_connected_components(const unsigned char* masks, int B, int H, int W, int* counts_out, int* boxes_out,
                                unmore_stream_t stream) {
  if (B < 0 || (B > 0 && (!masks || !counts_out || !boxes_out)))
    return fail(UNMORE_E_INVALID, "unmore_connected_components: bad argument");
  if (H != kCrop || W != kCrop) return fail(UNMORE_E_CAPACITY, "unmore_connected_components: only 128x128 crops (got %dx%d)", H, W);
  return cuda_fail(launch_components(masks, B, counts_out, boxes_out, (cudaStream_t)stream), "components_kernel");
}

int unmore_anti_center_map(const float* vote_maps, int B, int H, int W, int kernel_size, double* out,
                           unmore_stream_t stream) {
  if (B < 0 || H <= 0 || W <= 0 || (B > 0 && (!vote_maps || !out)))
    return fail(UNMORE_E_INVALID, "unmore_anti_center_map: bad argument");
  if (kernel_size != 5) return fail(UNMORE_E_CAPACITY, "unmore_anti_center_map: kernel_size must be 5 (reference call site)");
  double filt[25];
  anti_center_filter(filt);
  return cuda_fail(launch_anti_center(vote_maps, out, B, H, W, filt, (cudaStream_t)stream), "anti_center_kernel");
}

int unmore_box_nms_matrix(const float* boxes, const float* scores, int K, float iou_threshold, int* order_ws,
                          void* matrix_ws, int* keep_out, int* keep_count_out, unmore_stream_t stream) {
  if (K < 0 || !keep_count_out || (K > 0 && (!boxes || !order_ws || !matrix_ws || !keep_out)))
    return fail(UNMORE_E_INVALID, "unmore_box_nms_matrix: bad argument");
  return cuda_fail(launch_matrix_nms(nullptr, reinterpret_cast<const float4*>(boxes), K, 0, 0, scores, nullptr, nullptr,
                                     iou_threshold, order_ws, reinterpret_cast<unsigned long long*>(matrix_ws), keep_out,
                                     keep_count_out, (cudaStream_t)stream),
                   "box matrix nms");
}

int unmore_score_and_rasterise(const float* fields, int n_img, int C, int H, int W, int ch_sdf, int ch_center_row,
                               int ch_center_col, int ch_exist, const void* boxes, int boxes_f64, const int* counts,
                               int cap, float* scores_out, float* tight_out, int* areas_out, uint32_t* masks_out,
                               unmore_stream_t stream) {
  return score_and_rasterise("unmore_score_and_rasterise", fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col,
                             ch_exist, boxes, boxes_f64, counts, cap, scores_out, tight_out, areas_out, masks_out,
                             (cudaStream_t)stream);
}

int unmore_mask_resize(const unsigned char* masks, int B, int H, int W, int out_h, int out_w, unsigned char* out,
                       unmore_stream_t stream) {
  if (B < 0 || out_h < 0 || out_w < 0 || (B > 0 && out_h > 0 && out_w > 0 && (!masks || !out)))
    return fail(UNMORE_E_INVALID, "unmore_mask_resize: bad argument");
  if (H != kCrop || W != kCrop) return fail(UNMORE_E_CAPACITY, "unmore_mask_resize: only 128x128 crops (got %dx%d)", H, W);
  return cuda_fail(launch_mask_resize(masks, B, out_h, out_w, out, (cudaStream_t)stream), "mask_resize_kernel");
}

int unmore_final_scores(const float* scores, const float* tight, const int* areas, const int* keep,
                        const int* keep_counts, int cap, int n_img, double existence_score_thres, double center_score_thres,
                        double boundary_score_thres, double* out, float* bbox_xywh_out, unsigned char* selected_out,
                        unmore_stream_t stream) {
  if (!scores || !tight || !areas || !keep || !keep_counts || !out || !bbox_xywh_out || cap < 0 || n_img < 0)
    return fail(UNMORE_E_INVALID, "unmore_final_scores: bad argument");
  FinalParams p{};
  p.scores = reinterpret_cast<const float4*>(scores); p.tight = reinterpret_cast<const float4*>(tight);
  p.areas = areas; p.keep = keep; p.keep_counts = keep_counts; p.cap = cap; p.n_img = n_img;
  p.existence_thres = existence_score_thres; p.center_thres = center_score_thres; p.boundary_thres = boundary_score_thres;
  p.out = out; p.bbox_xywh = reinterpret_cast<float4*>(bbox_xywh_out); p.selected = selected_out;
  return cuda_fail(launch_final_scores(p, (cudaStream_t)stream), "final_scores_kernel");
}

int unmore_pack_detections(const long long* image_ids, const float* bbox_xywh, const double* out5, const int* keep_counts,
                           int cap, int n_img, double* rows, int max_rows, unmore_stream_t stream) {
  if (!image_ids || !bbox_xywh || !out5 || !keep_counts || !rows || cap < 0 || n_img < 0 || max_rows < 0)
    return fail(UNMORE_E_INVALID, "unmore_pack_detections: bad argument");
  return cuda_fail(launch_pack_detections(image_ids, reinterpret_cast<const float4*>(bbox_xywh), out5, keep_counts, cap, n_img,
                                          rows, max_rows, (cudaStream_t)stream),
                   "pack_detections_kernel");
}

int unmore_sat_build(const float* in, int n_planes, int H, int W, double* out, unmore_stream_t stream) {
  if (n_planes < 0 || H <= 0 || W <= 0 || (n_planes > 0 && (!in || !out)))
    return fail(UNMORE_E_INVALID, "unmore_sat_build: bad argument");
  if (W > 2048) return fail(UNMORE_E_CAPACITY, "unmore_sat_build: W %d > 2048", W);
  return cuda_fail(launch_sat(in, out, n_planes, H, W, 0, nullptr, 0, nullptr, (cudaStream_t)stream), "sat_kernel");
}

int unmore_sat_build_fields(const float* fields, int n_img, int C, int H, int W, const int* channels_host, int n_channels,
                            double* out, unmore_stream_t stream) {
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (!out || !channels_host || n_channels < 1 || n_channels > 4)
    return fail(UNMORE_E_INVALID, "unmore_sat_build_fields: bad argument (1..4 channels)");
  for (int i = 0; i < n_channels; ++i)
    if (channels_host[i] < 0 || channels_host[i] >= C) return fail(UNMORE_E_INVALID, "unmore_sat_build_fields: channel out of range");
  if (W > 2048) return fail(UNMORE_E_CAPACITY, "unmore_sat_build_fields: W %d > 2048", W);
  return cuda_fail(launch_sat(fields, out, n_img * n_channels, H, W, C, channels_host, n_channels, nullptr, (cudaStream_t)stream),
                   "sat_kernel");
}

int unmore_box_sums(const double* sat, int n_img, int planes_per_img, int plane, int H, int W, const void* boxes,
                    int boxes_f64, const int* counts, int cap, double* sums_out, double* means_out,
                    unmore_stream_t stream) {
  return box_sums("unmore_box_sums", sat, n_img, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap, sums_out,
                  means_out, (cudaStream_t)stream);
}

int unmore_mask_pack(const unsigned char* in, size_t K, int H, int W, uint32_t* out, unmore_stream_t stream) {
  if (H <= 0 || W <= 0 || (K > 0 && (!in || !out))) return fail(UNMORE_E_INVALID, "unmore_mask_pack: bad argument");
  return cuda_fail(launch_mask_pack(in, out, K, H, W, num_sms(), (cudaStream_t)stream), "pack_kernel");
}

int unmore_mask_stats(const uint32_t* masks, int K, int H, int W, int* areas_out, int* tight_out,
                      unmore_stream_t stream) {
  if (K < 0 || H <= 0 || W <= 0 || (K > 0 && (!masks || !areas_out || !tight_out)))
    return fail(UNMORE_E_INVALID, "unmore_mask_stats: bad argument");
  return cuda_fail(launch_mask_stats(masks, K, H, (W + 31) >> 5, areas_out, reinterpret_cast<int4*>(tight_out),
                                     (cudaStream_t)stream),
                   "mask_stats_kernel");
}

int unmore_mask_rle_counts(const uint32_t* masks, int K, int H, int W, int max_runs, uint32_t* counts_out,
                           int* n_runs_out, unmore_stream_t stream) {
  if (K < 0 || H <= 0 || W <= 0 || max_runs < 1 || (K > 0 && (!masks || !counts_out || !n_runs_out)))
    return fail(UNMORE_E_INVALID, "unmore_mask_rle_counts: bad argument");
  return cuda_fail(launch_rle_counts(masks, K, H, W, max_runs, counts_out, n_runs_out, (cudaStream_t)stream),
                   "rle_counts_kernel");
}

int unmore_mask_nms(const uint32_t* masks, int K, int H, int W, const float* scores, const int* areas, const int* tight,
                    float iou_threshold, int* order_ws, void* matrix_ws, int* keep_out, int* keep_count_out,
                    unmore_stream_t stream) {
  if (K < 0 || !keep_count_out || (K > 0 && (!masks || !areas || !tight || !order_ws || !matrix_ws || !keep_out)))
    return fail(UNMORE_E_INVALID, "unmore_mask_nms: bad argument");
  return cuda_fail(launch_matrix_nms(masks, nullptr, K, H, (W + 31) >> 5, scores, areas, reinterpret_cast<const int4*>(tight),
                                     iou_threshold, order_ws, reinterpret_cast<unsigned long long*>(matrix_ws), keep_out,
                                     keep_count_out, (cudaStream_t)stream),
                   "mask matrix nms");
}

// ---- padded stacks of images of different sizes: H, W are the pitch, image_hw [n_img, 2] int32 (device) the extents --
int unmore_existence_scores_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_exist,
                               const void* boxes, int boxes_f64, const int* counts, int cap, float* scores_out, void* ws,
                               unmore_stream_t stream) {
  const char* name = "unmore_existence_scores_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return existence_scores(name, false, fields, n_img, C, H, W, ch_exist, boxes, boxes_f64, counts, cap, scores_out, ws,
                          (cudaStream_t)stream, image_hw);
}

int unmore_center_reasoning_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                               int ch_center_row, int ch_center_col, const void* boxes, int boxes_f64, const int* counts,
                               int cap, double center_score_max_thres, double* max_values_out, int* argmax_out,
                               double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out, int* cc_overflow,
                               void* ws, unmore_stream_t stream) {
  const char* name = "unmore_center_reasoning_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return center_reasoning(name, false, fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col, boxes, boxes_f64, counts, cap,
                          center_score_max_thres, max_values_out, argmax_out, splits_out, cc_counts_out, cc_boxes_out,
                          cc_overflow, ws, (cudaStream_t)stream, image_hw);
}

int unmore_boundary_refine_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                              const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                              int apply_small_filter, int early_exit, float proposal_area_thres, float max_sdf_thres,
                              float max_shrink_threshold, float delta_ratio, float* boxes_out, float* labels_out,
                              int* rounds_out, void* ws, unmore_stream_t stream) {
  const char* name = "unmore_boundary_refine_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return boundary_refine(name, false, fields, n_img, C, H, W, ch_sdf, boxes, boxes_f64, counts, cap, n_round,
                         apply_small_filter, early_exit, proposal_area_thres, max_sdf_thres, max_shrink_threshold,
                         delta_ratio, boxes_out, labels_out, rounds_out, ws, (cudaStream_t)stream, image_hw);
}

int unmore_score_and_rasterise_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                                  int ch_center_row, int ch_center_col, int ch_exist, const void* boxes, int boxes_f64,
                                  const int* counts, int cap, float* scores_out, float* tight_out, int* areas_out,
                                  uint32_t* masks_out, unmore_stream_t stream) {
  const char* name = "unmore_score_and_rasterise_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return score_and_rasterise(name, fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col, ch_exist, boxes, boxes_f64,
                             counts, cap, scores_out, tight_out, areas_out, masks_out, (cudaStream_t)stream, image_hw);
}

int unmore_box_sums_hw(const double* sat, int n_img, int planes_per_img, int plane, int H, int W, const int* image_hw,
                       const void* boxes, int boxes_f64, const int* counts, int cap, double* sums_out, double* means_out,
                       unmore_stream_t stream) {
  const char* name = "unmore_box_sums_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return box_sums(name, sat, n_img, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap, sums_out, means_out,
                  (cudaStream_t)stream, image_hw);
}

int unmore_sat_build_fields_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                               const int* channels_host, int n_channels, double* out, unmore_stream_t stream) {
  const char* name = "unmore_sat_build_fields_hw";
  if (int e = check_fields(fields, n_img, C, H, W)) return e;
  if (int e = check_extents(name, image_hw)) return e;
  if (!out || !channels_host || n_channels < 1 || n_channels > 4)
    return fail(UNMORE_E_INVALID, "%s: bad argument (1..4 channels)", name);
  for (int i = 0; i < n_channels; ++i)
    if (channels_host[i] < 0 || channels_host[i] >= C) return fail(UNMORE_E_INVALID, "%s: channel out of range", name);
  if (W > 2048) return fail(UNMORE_E_CAPACITY, "%s: W %d > 2048", name, W);
  return cuda_fail(launch_sat(fields, out, n_img * n_channels, H, W, C, channels_host, n_channels, image_hw, (cudaStream_t)stream),
                   "sat_kernel");
}

// the second resize mode (antialias=True) on a padded stack
int unmore_existence_scores_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_exist,
                                  const void* boxes, int boxes_f64, const int* counts, int cap, float* scores_out, void* ws,
                                  unmore_stream_t stream) {
  const char* name = "unmore_existence_scores_aa_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return existence_scores(name, true, fields, n_img, C, H, W, ch_exist, boxes, boxes_f64, counts, cap, scores_out, ws,
                          (cudaStream_t)stream, image_hw);
}

int unmore_boundary_refine_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                                 const void* boxes, int boxes_f64, const int* counts, int cap, int n_round,
                                 int apply_small_filter, int early_exit, float proposal_area_thres, float max_sdf_thres,
                                 float max_shrink_threshold, float delta_ratio, float* boxes_out, float* labels_out,
                                 int* rounds_out, void* ws, unmore_stream_t stream) {
  const char* name = "unmore_boundary_refine_aa_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return boundary_refine(name, true, fields, n_img, C, H, W, ch_sdf, boxes, boxes_f64, counts, cap, n_round,
                         apply_small_filter, early_exit, proposal_area_thres, max_sdf_thres, max_shrink_threshold,
                         delta_ratio, boxes_out, labels_out, rounds_out, ws, (cudaStream_t)stream, image_hw);
}

int unmore_center_reasoning_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw, int ch_sdf,
                                  int ch_center_row, int ch_center_col, const void* boxes, int boxes_f64,
                                  const int* counts, int cap, double center_score_max_thres, double* max_values_out,
                                  int* argmax_out, double* splits_out, unsigned char* cc_counts_out,
                                  double* cc_boxes_out, int* cc_overflow, void* ws, unmore_stream_t stream) {
  const char* name = "unmore_center_reasoning_aa_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return center_reasoning(name, true, fields, n_img, C, H, W, ch_sdf, ch_center_row, ch_center_col, boxes, boxes_f64, counts,
                          cap, center_score_max_thres, max_values_out, argmax_out, splits_out, cc_counts_out, cc_boxes_out,
                          cc_overflow, ws, (cudaStream_t)stream, image_hw);
}

int unmore_crop_resize_aa_hw(const float* fields, int n_img, int C, int H, int W, const int* image_hw,
                             const int* channels_host, int n_channels, const void* boxes, int boxes_f64, const int* counts,
                             int cap, float* out, void* scratch, size_t scratch_bytes, unmore_stream_t stream) {
  const char* name = "unmore_crop_resize_aa_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return crop_resize_aa(name, fields, n_img, C, H, W, channels_host, n_channels, boxes, boxes_f64, counts, cap, out, scratch,
                        scratch_bytes, (cudaStream_t)stream, image_hw);
}

int unmore_center_reasoning_from_tiles_hw(const float* tiles, int n_img, int H, int W, const int* image_hw,
                                          const void* boxes, int boxes_f64, const int* counts, int cap,
                                          double center_score_max_thres, double* max_values_out, int* argmax_out,
                                          double* splits_out, unsigned char* cc_counts_out, double* cc_boxes_out,
                                          int* cc_overflow, void* ws, unmore_stream_t stream) {
  const char* name = "unmore_center_reasoning_from_tiles_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return center_from_tiles(name, tiles, n_img, H, W, boxes, boxes_f64, counts, cap, center_score_max_thres, max_values_out,
                           argmax_out, splits_out, cc_counts_out, cc_boxes_out, cc_overflow, ws, (cudaStream_t)stream,
                           image_hw);
}

int unmore_score_and_rasterise_from_tiles_hw(const float* tiles, const float* existence_scores, int antialias, int n_img,
                                             int H, int W, const int* image_hw, const void* boxes, int boxes_f64,
                                             const int* counts, int cap, float* scores_out, float* tight_out,
                                             int* areas_out, uint32_t* masks_out, unmore_stream_t stream) {
  const char* name = "unmore_score_and_rasterise_from_tiles_hw";
  if (int e = check_extents(name, image_hw)) return e;
  return score_from_tiles(name, tiles, existence_scores, antialias, n_img, H, W, boxes, boxes_f64, counts, cap, scores_out,
                          tight_out, areas_out, masks_out, (cudaStream_t)stream, image_hw);
}

}  // extern "C"
