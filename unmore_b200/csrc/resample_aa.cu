// The second resize mode: antialias=True, i.e. ATen's _upsample_bilinear2d_aa — what torchvision >= 0.17 gives
// transforms.Resize by default at object_reasoning.py:319,407,505 and object_scoring.py:131,206,222 (the reference
// pins torchvision 0.14.1, where tensors are never antialiased; antialias=False is this repo's primary mode and the
// mode of most fused kernels).  Provided for the stand-alone ops a2 (crop + resize to 128x128) and N2 (mask
// resize back to the box + round half to even), bit-exact against torch 2.11 CPU:
//
//   * weights (HelperInterpBase::_compute_indices_min_size_weights_aa, opmath = float, double literals):
//       scale = float(in)/float(out); support = max(scale, 1); invscale = scale >= 1 ? float(1.0/scale) : 1
//       center = float(double(scale) * (i + 0.5))
//       xmin = max(int64(double(center - support) + 0.5), 0); xmax = min(int64(double(center + support) + 0.5), in)
//       w_j = tri(float((double(float(j + xmin) - center) + 0.5) * double(invscale))), normalised by their fp32 sum
//   * separable, HORIZONTAL pass over every source row first, then the vertical pass on the fp32 intermediate;
//   * accumulation order of the compiled interpolate_aa_single_dim loop (pinned by experiment,
//     oracle/oracle.py::_aa_pass): t = s0*w0; then groups of four taps with separate multiply and add; the
//     remaining (n-1) mod 4 taps with a fused multiply-add.
//
// Two kernels with the intermediate in a caller-provided scratch buffer: tiles for the *_from_tiles stages.  The fused
// existence and refine kernels compute the same values row by row (aa_rows.cuh).
#include "resample_aa.cuh"
#include "unmore_internal.h"

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

// Two passes with the intermediate in the caller's scratch buffer, grid = (tile, 8 row slices): the weight tables of
// a block (the fp64 / division part: ~90% of the instructions of a dot) are built once in shared memory — thread j
// the horizontal weights of column j, the first threads the vertical weights of the block's output rows.  Windows
// more than ~11x the tile size in a dimension (more than kAaMaxTaps taps) take aa_dot directly, the same arithmetic.
// (A single fused kernel with the intermediate in a per-column shared ring, one thread per column, was measured
// slower: 92.7 vs 79.9 ms on the profile workload — too little parallelism per tile to hide the tap loads.)
constexpr int kAaMaxTaps = 24, kAaSlices = 8;

// pass 1: T[tile][y][j] = sum_x window[y][x] * wx_j[x] for every row y of the crop window
__global__ void __launch_bounds__(kCrop) aa_crop_h_kernel(const AaCropParams p) {
  __shared__ float wh[kAaMaxTaps][kCrop];   // [tap][column]: thread j reads its own column
  const long long tile = blockIdx.x;             // (row, channel)
  const int k = (int)(tile % p.n_ch);
  const size_t row = (size_t)(tile / p.n_ch);
  const int img = (int)(row / p.cap), e = (int)(row % p.cap);
  if (p.counts && e >= p.counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
  const Window win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
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
__global__ void __launch_bounds__(kCrop) aa_crop_v_kernel(const AaCropParams p) {
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
  const Window win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
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

int launch_crop_resize_aa(const float* fields, int n_img, int C, int H, int W, const int* channels, int n_ch,
                          const void* boxes, int boxes_f64, const int* counts, int cap, float* out, float* scratch,
                          cudaStream_t stream) {
  const long long tiles = (long long)n_img * cap * n_ch;
  if (tiles <= 0) return 0;
  AaCropParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W; p.n_ch = n_ch;
  for (int i = 0; i < n_ch; ++i) p.ch[i] = channels[i];
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.counts = counts; p.cap = cap; p.n_img = n_img; p.out = out; p.scratch = scratch;
  dim3 grid((unsigned)tiles, kAaSlices);
  aa_crop_h_kernel<<<grid, kCrop, 0, stream>>>(p);
  int e = (int)cudaGetLastError();
  if (e) return e;
  aa_crop_v_kernel<<<grid, kCrop, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

// ---- N2 with antialias: masks [B,128,128] u8 -> [B,oh,ow] u8, value = round-half-even(resize(float(mask))) ----
__global__ void __launch_bounds__(256) aa_mask_h_kernel(const unsigned char* __restrict__ masks, int B, int ow, float* __restrict__ T) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // (b, y, j)
  if (id >= (size_t)B * kCrop * ow) return;
  const int j = (int)(id % ow);
  const int y = (int)((id / ow) % kCrop);
  const size_t b = id / ((size_t)ow * kCrop);
  AaAxis ax;
  ax.init(kCrop, ow);
  const unsigned char* srow = masks + (b * kCrop + y) * kCrop;
  T[id] = aa_dot(ax, j, [&](int x) { return srow[x] ? 1.f : 0.f; });
}
__global__ void __launch_bounds__(256) aa_mask_v_kernel(const float* __restrict__ T, int B, int oh, int ow, unsigned char* __restrict__ out) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // (b, i, j)
  if (id >= (size_t)B * oh * ow) return;
  const int j = (int)(id % ow);
  const int i = (int)((id / ow) % oh);
  const size_t b = id / ((size_t)ow * oh);
  AaAxis ay;
  ay.init(kCrop, oh);
  const float* Tb = T + b * kCrop * ow;
  const float v = aa_dot(ay, i, [&](int y) { return Tb[(size_t)y * ow + j]; });
  out[id] = rintf(v) != 0.f ? 1 : 0;   // torch.round (half to even) then the cast back to the integer mask
}

int launch_mask_resize_aa(const unsigned char* masks, int B, int oh, int ow, unsigned char* out, float* scratch, cudaStream_t stream) {
  const size_t n1 = (size_t)B * kCrop * ow, n2 = (size_t)B * oh * ow;
  if (n1 == 0 || n2 == 0) return 0;
  aa_mask_h_kernel<<<(unsigned)((n1 + 255) / 256), 256, 0, stream>>>(masks, B, ow, scratch);
  int e = (int)cudaGetLastError();
  if (e) return e;
  aa_mask_v_kernel<<<(unsigned)((n2 + 255) / 256), 256, 0, stream>>>(scratch, B, oh, ow, out);
  return (int)cudaGetLastError();
}

}  // namespace unmore
