// The two passes of the stand-alone antialiased crop (unmore_crop_resize_aa, arithmetic contract in resample_aa.cu) as
// kernel templates.  SIZED = false is instantiated in resample_aa.cu, SIZED = true (a padded stack of images of
// different sizes) in resample_aa_hw.cu: compiled beside the sized variant, the uniform kernels' code changes.
#pragma once
#include "resample_aa.cuh"

namespace unmore {

struct AaCropParams {
  const float* fields;
  int C, H, W;
  int n_ch, ch[4];
  const void* boxes;
  int boxes_f64;
  const int* counts;
  int cap, n_img;
  float* out;      // [n_img, cap, n_ch, 128, 128]
  float* scratch;  // [n_img * cap * n_ch, H, 128]
};
// The sized variants' parameters (a struct of its own, as ScoreHwParams: the uniform kernels keep their code).
// SIZED: a padded stack; the window snaps to the image's extent, addresses and the scratch rows go by the pitch.
struct AaCropHwParams : AaCropParams {
  const int* image_hw;  // [n_img, 2] (h, w) of each image inside the (H, W) pitch
};
template <bool SIZED> struct AaCropArgs { using type = AaCropParams; };
template <> struct AaCropArgs<true> { using type = AaCropHwParams; };

// Two passes with the intermediate in the caller's scratch buffer, grid = (tile, 8 row slices): the weight tables of
// a block (the fp64 / division part: ~90% of the instructions of a dot) are built once in shared memory — thread j
// the horizontal weights of column j, the first threads the vertical weights of the block's output rows.  Windows
// more than ~11x the tile size in a dimension (more than kAaMaxTaps taps) take aa_dot directly, the same arithmetic.
// (A single fused kernel with the intermediate in a per-column shared ring, one thread per column, was measured
// slower: 92.7 vs 79.9 ms on the profile workload — too little parallelism per tile to hide the tap loads.)
constexpr int kAaMaxTaps = 24, kAaSlices = 8;

// pass 1: T[tile][y][j] = sum_x window[y][x] * wx_j[x] for every row y of the crop window
template <bool SIZED>
__global__ void __launch_bounds__(kCrop) aa_crop_h_kernel(const typename AaCropArgs<SIZED>::type p) {
  __shared__ float wh[kAaMaxTaps][kCrop];   // [tap][column]: thread j reads its own column
  const long long tile = blockIdx.x;             // (row, channel)
  const int k = (int)(tile % p.n_ch);
  const size_t row = (size_t)(tile / p.n_ch);
  const int img = (int)(row / p.cap), e = (int)(row % p.cap);
  if (p.counts && e >= p.counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
  Window win;
  if constexpr (SIZED) {   // both passes read the same entry, clamped the same way: they agree on the window
    const int2 ext = image_extent(p.image_hw, img, p.H, p.W);
    win = snap_window<double>(x1, y1, x2, y2, ext.y, ext.x);
  } else {
    win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
  }
  if (win.empty()) return;
  AaAxis ax;
  ax.init(win.w(), kCrop);
  const float* plane = p.fields + ((size_t)img * p.C + p.ch[k]) * p.H * p.W + (size_t)win.y1 * p.W + win.x1;
  float* T = p.scratch + (size_t)tile * p.H * kCrop;
  const int j = threadIdx.x;
  int xmin, nx;
  aa_weights(ax, j, xmin, nx, &wh[0][j], kCrop, kAaMaxTaps);   // column-private: no barrier needed
  for (int y = blockIdx.y; y < win.h(); y += gridDim.y) {
    const float* srow = plane + (size_t)y * p.W;
    float t;
    if (nx <= 0) t = 0.f;
    else if (nx > kAaMaxTaps) t = aa_dot(ax, j, [&](int x) { return __ldg(srow + x); });
    else t = aa_accumulate(nx, [&](int q) { return __ldg(srow + xmin + q); }, [&](int q) { return wh[q][j]; });
    T[(size_t)y * kCrop + j] = t;
  }
}

// pass 2: out[tile][i][j] = sum_y T[tile][y][j] * wy_i[y]
template <bool SIZED>
__global__ void __launch_bounds__(kCrop) aa_crop_v_kernel(const typename AaCropArgs<SIZED>::type p) {
  constexpr int kRows = kCrop / kAaSlices;   // output rows of one block: blockIdx.y + kAaSlices * r
  __shared__ float wv[kRows][kAaMaxTaps];
  __shared__ int vmin[kRows], vn[kRows];
  const long long tile = blockIdx.x;
  const int k = (int)(tile % p.n_ch);
  const size_t row = (size_t)(tile / p.n_ch);
  const int img = (int)(row / p.cap), e = (int)(row % p.cap);
  if (p.counts && e >= p.counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
  Window win;
  if constexpr (SIZED) {   // both passes read the same entry, clamped the same way: they agree on the window
    const int2 ext = image_extent(p.image_hw, img, p.H, p.W);
    win = snap_window<double>(x1, y1, x2, y2, ext.y, ext.x);
  } else {
    win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
  }
  float* o = p.out + ((size_t)row * p.n_ch + k) * kCrop * kCrop;
  const int j = threadIdx.x;
  if (win.empty()) {
    for (int i = blockIdx.y; i < kCrop; i += gridDim.y) o[i * kCrop + j] = 0.f;
    return;
  }
  AaAxis ay;
  ay.init(win.h(), kCrop);
  if (j < kRows) {
    int ymin, ny;
    aa_weights(ay, blockIdx.y + kAaSlices * j, ymin, ny, &wv[j][0], 1, kAaMaxTaps);
    vmin[j] = ymin; vn[j] = ny;
  }
  __syncthreads();
  const float* T = p.scratch + (size_t)tile * p.H * kCrop;
  for (int r = 0; r < kRows; ++r) {
    const int i = blockIdx.y + kAaSlices * r, ymin = vmin[r], n = vn[r];
    float t;
    if (n <= 0) t = 0.f;
    else if (n > kAaMaxTaps) t = aa_dot(ay, i, [&](int y) { return T[(size_t)y * kCrop + j]; });
    else t = aa_accumulate(n, [&](int q) { return T[(size_t)(ymin + q) * kCrop + j]; }, [&](int q) { return wv[r][q]; });
    o[i * kCrop + j] = t;
  }
}

template <bool SIZED>
static int launch_crop_aa_t(const typename AaCropArgs<SIZED>::type& p, long long tiles, cudaStream_t stream) {
  dim3 grid((unsigned)tiles, kAaSlices);
  aa_crop_h_kernel<SIZED><<<grid, kCrop, 0, stream>>>(p);
  int e = (int)cudaGetLastError();
  if (e) return e;
  aa_crop_v_kernel<SIZED><<<grid, kCrop, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

// resample_aa_hw.cu
int launch_crop_resize_aa_hw(const AaCropParams& p, long long tiles, const int* image_hw, cudaStream_t stream);

}  // namespace unmore
