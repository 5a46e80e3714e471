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
// Two kernels (aa_crop.cuh) with the intermediate in a caller-provided scratch buffer: tiles for the *_from_tiles stages.  The fused
// existence and refine kernels compute the same values row by row (aa_rows.cuh), so does the center kernel (center.cuh).
#include "aa_crop.cuh"
#include "unmore_internal.h"

namespace unmore {

int launch_crop_resize_aa(const float* fields, int n_img, int C, int H, int W, const int* channels, int n_ch,
                          const void* boxes, int boxes_f64, const int* counts, int cap, float* out, float* scratch,
                          cudaStream_t stream, const int* image_hw) {
  const long long tiles = (long long)n_img * cap * n_ch;
  if (tiles <= 0) return 0;
  AaCropParams p{};
  p.fields = fields; p.C = C; p.H = H; p.W = W; p.n_ch = n_ch;
  for (int i = 0; i < n_ch; ++i) p.ch[i] = channels[i];
  p.boxes = boxes; p.boxes_f64 = boxes_f64; p.counts = counts; p.cap = cap; p.n_img = n_img; p.out = out; p.scratch = scratch;
  return image_hw ? launch_crop_resize_aa_hw(p, tiles, image_hw, stream) : launch_crop_aa_t<false>(p, tiles, stream);
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
