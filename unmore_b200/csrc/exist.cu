// existence_checking (object_reasoning.py:491-523) under the field-stub bridge: the
// Binary_Classifier stand-in is the mean of the resized crop's existence channel, so the
// score of a proposal is mean_{128x128} bilinear(existence[y1:y2, x1:x2]).
//
// One warp per proposal, lane owns 4 output columns; the horizontally interpolated source
// rows are cached across output rows (resample.cuh), so small crops cost ~in_h row fetches.
#include "aa_rows.cuh"
#include "resample.cuh"
#include "unmore_internal.h"

namespace unmore {

constexpr int kExistWarps = 8;

// SIZED: the fields are a padded stack and p.image_hw holds each image's (h, w) inside the (H, W) pitch; addresses
// come from the pitch, the window snap from the image's own extent.
template <bool SIZED>
__device__ __forceinline__ void existence_items(const ExistParams& p) {
  __shared__ int2 tapy_all[kExistWarps][kCrop];   // vertical taps of the warp's current window: (i0, bits of l1)
  const int lane = threadIdx.x & 31;
  int2* const tapy = tapy_all[threadIdx.x >> 5];
  const unsigned tapy_addr = smem_addr(tapy);
  const int total = worklist_total(p.work);
  int img = 0;   // image of the previous work item: the locate hint
  for (;;) {
    const int id = worklist_next_warp(p.work);
    if (id >= total) break;
    int k;
    worklist_locate(p.work, id, img, k);
    const size_t row = (size_t)img * p.work.cap + k;
    double x1, y1, x2, y2;
    load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
    Window win;
    if constexpr (SIZED) {
      const int2 e = image_extent(p.image_hw, img, p.H, p.W);
      win = snap_window<double>(x1, y1, x2, y2, e.y, e.x);
    } else {
      win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
    }
    float score = 0.f;  // zero-size crop: the reference raises; defined as "nothing there"
    if (!win.empty()) {
      ColTaps taps;
      taps.init<kStrided>(lane, win.w());
      PlaneRows plane;
      plane.init(p.fields + ((size_t)img * p.C + p.ch_exist) * p.H * p.W, p.W, win);
      const float scale_y = __fdiv_rn((float)win.h(), (float)kCrop);
      const int in_h = win.h();
      // the 128 vertical taps once per proposal, four per lane; one broadcast 8-byte load per row afterwards
      __syncwarp();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const AxisTap t = axis_tap(scale_y, lane + 32 * q, in_h);
        tapy[lane + 32 * q] = make_int2(t.i0, __float_as_int(t.l1));
      }
      __syncwarp();
      double acc = 0.0;
      f32x2 part = pk2(0.f, 0.f);   // two fp32 partial sums per lane, flushed to fp64 every 8 rows
      for (int i = 0; i < kCrop; ++i) {
        f32x2 v[2];
        int i0, l1b;
        asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(i0), "=r"(l1b) : "r"(tapy_addr + 8u * (unsigned)i) : "memory");
        AxisTap vt;
        vt.i0 = i0; vt.i1 = min(i0 + 1, in_h - 1);
        vt.l1 = __int_as_float(l1b); vt.l0 = __fsub_rn(1.f, vt.l1);
        plane.row2(taps, vt, v);
        part = add2(part, add2(v[0], v[1]));
        if ((i & 7) == 7) {
          float lo, hi;
          upk2(part, lo, hi);
          acc += (double)(lo + hi);
          part = pk2(0.f, 0.f);
        }
      }
      acc = warp_sum(acc);
      score = (float)(acc * (1.0 / (kCrop * kCrop)));
    }
    if (lane == 0) p.scores[row] = score;
  }
}

__global__ void __launch_bounds__(kExistWarps * 32) existence_kernel(const ExistParams p) { existence_items<false>(p); }
__global__ void __launch_bounds__(kExistWarps * 32) existence_hw_kernel(const ExistParams p) { existence_items<true>(p); }

// The second resize mode (antialias=True): the mean of the antialiased crop (aa_rows.cuh), summed in exactly the order
// above, so the score equals tile_means_kernel on the tile of unmore_crop_resize_aa bit for bit.
constexpr int kAaExistWarps = 2;   // 15 KB of shared memory per warp
constexpr int kAaExistMinBlocks = 7;
__global__ void __launch_bounds__(kAaExistWarps * 32, kAaExistMinBlocks) existence_aa_kernel(const ExistParams p) {
  __shared__ AaRowsSmem rows_all[kAaExistWarps];
  const int lane = threadIdx.x & 31;
  AaRowsSmem& rows = rows_all[threadIdx.x >> 5];
  const int total = worklist_total(p.work);
  int img = 0;
  for (;;) {
    const int id = worklist_next_warp(p.work);
    if (id >= total) break;
    int k;
    worklist_locate(p.work, id, img, k);
    const size_t row = (size_t)img * p.work.cap + k;
    double x1, y1, x2, y2;
    load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
    const Window win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
    float score = 0.f;
    if (!win.empty()) {
      AaCropRows src;
      src.init(lane, rows, p.fields + ((size_t)img * p.C + p.ch_exist) * p.H * p.W, p.W, win);
      double acc = 0.0;
      f32x2 part = pk2(0.f, 0.f);
      for (int i = 0; i < kCrop; ++i) {
        f32x2 v[2];
        src.issue(lane, i);
        src.finish(v);
        part = add2(part, add2(v[0], v[1]));
        if ((i & 7) == 7) {
          float lo, hi;
          upk2(part, lo, hi);
          acc += (double)(lo + hi);
          part = pk2(0.f, 0.f);
        }
      }
      acc = warp_sum(acc);
      score = (float)(acc * (1.0 / (kCrop * kCrop)));
    }
    if (lane == 0) p.scores[row] = score;
  }
}

// ---- a2 / a4 as a stand-alone op: the resized crops themselves --------------------------------
// crop + Resize((128,128), BILINEAR) of object_reasoning.py:402-410 / get_prediction_with_proposals
// (:301-337, object_scoring.py:112-157) for every (proposal, selected channel): out[row][k] is the
// 128x128 tile of channel ch[k].  One warp per (proposal, channel); lane owns columns lane + 32c so
// every output row is written as four coalesced 128-byte segments.
struct CropParams {
  const float* fields;
  int C, H, W;
  int n_ch, ch[4];
  const void* boxes;
  int boxes_f64;
  const int* counts;
  int cap, n_img;
  float* out;   // [n_img, cap, n_ch, 128, 128]
};

__global__ void __launch_bounds__(kExistWarps * 32) crop_resize_kernel(const CropParams p) {
  const int lane = threadIdx.x & 31;
  const long long gw = (long long)blockIdx.x * kExistWarps + (threadIdx.x >> 5);
  const long long total = (long long)p.n_img * p.cap * p.n_ch;
  if (gw >= total) return;
  const int k = (int)(gw % p.n_ch);
  const size_t row = (size_t)(gw / p.n_ch);
  const int img = (int)(row / p.cap), e = (int)(row % p.cap);
  if (p.counts && e >= p.counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
  const Window win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
  float* o = p.out + ((size_t)row * p.n_ch + k) * kCrop * kCrop;
  if (win.empty()) {
    for (int q = lane; q < kCrop * kCrop; q += 32) o[q] = 0.f;
    return;
  }
  ColTaps taps;
  taps.init<kStrided>(lane, win.w());
  PlaneRows plane;
  plane.init(p.fields + ((size_t)img * p.C + p.ch[k]) * p.H * p.W, p.W, win);
  const float scale_y = __fdiv_rn((float)win.h(), (float)kCrop);
  for (int i = 0; i < kCrop; ++i) {
    float v[4];
    plane.row(taps, axis_tap(scale_y, i, win.h()), v);
#pragma unroll
    for (int c = 0; c < 4; ++c) o[i * kCrop + lane + 32 * c] = v[c];
  }
}

int launch_crop_resize(const float* fields, int n_img, int C, int H, int W, const int* channels, int n_ch,
                       const void* boxes, int boxes_f64, const int* counts, int cap, float* out, cudaStream_t stream) {
  const long long total = (long long)n_img * cap * n_ch;
  if (total <= 0) return 0;
  CropParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W; p.n_ch = n_ch;
  for (int i = 0; i < n_ch; ++i) p.ch[i] = channels[i];
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.counts = counts; p.cap = cap; p.n_img = n_img; p.out = out;
  crop_resize_kernel<<<(unsigned)((total + kExistWarps - 1) / kExistWarps), kExistWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

// existence_checking on PRE-RESAMPLED tiles (the tile path of the second resize mode, antialias=True: the tiles come
// from unmore_crop_resize_aa): score = mean of the [128,128] existence tile, summed in the same order as
// existence_kernel (lane = columns l, l+32, l+64, l+96; fp32 partials flushed to fp64 every 8 rows).
__global__ void __launch_bounds__(kExistWarps * 32) tile_means_kernel(const float* __restrict__ tiles, long long tile_stride,
                                                                      int M, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int m = blockIdx.x * kExistWarps + (threadIdx.x >> 5);
  if (m >= M) return;
  const float* t = tiles + (size_t)m * tile_stride;
  double acc = 0.0;
  f32x2 part = pk2(0.f, 0.f);
  for (int i = 0; i < kCrop; ++i) {
    const float* r = t + i * kCrop + lane;
    const f32x2 v0 = pk2(__ldg(r), __ldg(r + 32)), v1 = pk2(__ldg(r + 64), __ldg(r + 96));
    part = add2(part, add2(v0, v1));
    if ((i & 7) == 7) {
      float lo, hi;
      upk2(part, lo, hi);
      acc += (double)(lo + hi);
      part = pk2(0.f, 0.f);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) out[m] = (float)(acc * (1.0 / (kCrop * kCrop)));
}

int launch_tile_means(const float* tiles, long long tile_stride, int M, float* out, cudaStream_t stream) {
  if (M <= 0) return 0;
  tile_means_kernel<<<(M + kExistWarps - 1) / kExistWarps, kExistWarps * 32, 0, stream>>>(tiles, tile_stride, M, out);
  return (int)cudaGetLastError();
}

int launch_existence(const ExistParams& p, int num_sms, cudaStream_t stream) {
  if (p.image_hw) existence_hw_kernel<<<num_sms * 4, kExistWarps * 32, 0, stream>>>(p);
  else existence_kernel<<<num_sms * 4, kExistWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

int launch_existence_aa(const ExistParams& p, int num_sms, cudaStream_t stream) {
  existence_aa_kernel<<<num_sms * kAaExistMinBlocks, kAaExistWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

}  // namespace unmore
