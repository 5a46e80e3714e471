// Antialiased crop rows for the fused kernels of the second resize mode (antialias=True): the 128x128 crop of one
// plane, produced one output row at a time with the same `issue(lane, i)` / `finish(out[2])` interface as CropRows
// (refine.cu), so the refine round loop and the existence sum run on it unchanged.
//
// Every value equals, bit for bit, what aa_crop_h_kernel followed by aa_crop_v_kernel (resample_aa.cu) writes: the
// same weights (aa_weights: sequential fp32 sum, then r / total), the horizontal pass first, the aa_accumulate order,
// and aa_dot directly for windows with more taps than the tables hold.
//
// Per warp (AaRowsSmem): the horizontal spans and weights of the 128 output columns, built once per window, and a
// ring of horizontally filtered source rows, filled as the output rows advance (the vertical spans only move down).
// Lane l owns columns l, l+32, l+64, l+96 in both tables and both passes, so no lane reads what another lane wrote
// and the passes need no __syncwarp.  The vertical weights of an output row are computed once per warp, tap q in
// lane q, and handed out by shuffles, which also form their fp32 total in tap order.
#pragma once
#include "resample_aa.cuh"

namespace unmore {

// A window scale s needs at most 2s + 1 taps: the tables cover windows up to 704 px wide and 960 px high, and 480x640
// fields need at most 11 horizontal and 9 vertical taps.  Columns with more taps take aa_dot
// (weights recomputed per tap); output rows with more taps than the ring holds filter their source rows on the fly.
constexpr int kAaRowTaps = 12;
constexpr int kAaRingRows = 16;
static_assert((kAaRingRows & (kAaRingRows - 1)) == 0, "kAaRingRows must be a power of two");
static_assert(kAaRingRows <= 32, "the vertical weights of a ring row are spread over the lanes of a warp");

struct AaRowsSmem {
  float wh[kAaRowTaps][kCrop];     // normalised horizontal weights, [tap][column]
  int2 hspan[kCrop];               // (xmin, taps) of each column
  float ring[kAaRingRows][kCrop];  // horizontally filtered source row y in slot y % kAaRingRows
};

struct AaCropRows {
  AaRowsSmem* s;
  const float* origin;   // &plane[win.y1 * W + win.x1]
  int stride;            // W
  AaAxis ax, ay;
  int filled;            // the ring holds every row of [ymin, filled) that the current output row needs
  float pend[4];

  __device__ __forceinline__ void init(int lane, AaRowsSmem& sm, const float* plane, int W, const Window& win) {
    s = &sm;
    origin = plane + (size_t)win.y1 * W + win.x1;
    stride = W;
    ax.init(win.w(), kCrop);
    ay.init(win.h(), kCrop);
    filled = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = lane + 32 * c;
      int xmin, n;
      aa_weights(ax, j, xmin, n, &s->wh[0][j], kCrop, kAaRowTaps);
      s->hspan[j] = make_int2(xmin, n);
    }
  }
  // the horizontal pass at source row y, column j: aa_crop_h_kernel's T[y][j]
  __device__ __forceinline__ float hval(int y, int j) const {
    const float* srow = origin + (size_t)y * stride;
    const int2 sp = s->hspan[j];
    if (sp.y <= 0) return 0.f;
    if (sp.y > kAaRowTaps) return aa_dot(ax, j, [&](int x) { return __ldg(srow + x); });
    return aa_accumulate(sp.y, [&](int q) { return __ldg(srow + sp.x + q); }, [&](int q) { return s->wh[q][j]; });
  }
  __device__ __forceinline__ void issue(int lane, int i) {
    float center;
    int ymin, n;
    ay.span(i, center, ymin, n);
    if (n <= 0) {
#pragma unroll
      for (int c = 0; c < 4; ++c) pend[c] = 0.f;
      return;
    }
    if (n > kAaRingRows) {
#pragma unroll
      for (int c = 0; c < 4; ++c) pend[c] = aa_dot(ay, i, [&](int y) { return hval(y, lane + 32 * c); });
      return;
    }
    // rows below `filled` are in the ring already; writing row y evicts row y - kAaRingRows < ymin
    for (int y = max(filled, ymin); y < ymin + n; ++y) {
      float* slot = s->ring[y & (kAaRingRows - 1)];
#pragma unroll
      for (int c = 0; c < 4; ++c) slot[lane + 32 * c] = hval(y, lane + 32 * c);
    }
    filled = max(filled, ymin + n);
    const float r = lane < n ? ay.raw_weight(ymin + lane, center) : 0.f;
    float total = 0.f;
    for (int q = 0; q < n; ++q) total = __fadd_rn(total, __shfl_sync(kFullMask, r, q));
    const float w = total != 0.f ? __fdiv_rn(r, total) : r;
    // aa_accumulate's order for the lane's four columns at once
    auto row = [&](int q) { return s->ring[(ymin + q) & (kAaRingRows - 1)]; };
    {
      const float w0 = __shfl_sync(kFullMask, w, 0);
      const float* t = row(0);
#pragma unroll
      for (int c = 0; c < 4; ++c) pend[c] = __fmul_rn(t[lane + 32 * c], w0);
    }
    const int main_taps = ((n - 1) / 4) * 4;
    int q = 1;
    for (; q <= main_taps; ++q) {
      const float wq = __shfl_sync(kFullMask, w, q);
      const float* t = row(q);
#pragma unroll
      for (int c = 0; c < 4; ++c) pend[c] = __fadd_rn(pend[c], __fmul_rn(t[lane + 32 * c], wq));
    }
    for (; q < n; ++q) {
      const float wq = __shfl_sync(kFullMask, w, q);
      const float* t = row(q);
#pragma unroll
      for (int c = 0; c < 4; ++c) pend[c] = __fmaf_rn(t[lane + 32 * c], wq, pend[c]);
    }
  }
  __device__ __forceinline__ void finish(f32x2 out[2]) { out[0] = pk2(pend[0], pend[1]); out[1] = pk2(pend[2], pend[3]); }
};

}  // namespace unmore
