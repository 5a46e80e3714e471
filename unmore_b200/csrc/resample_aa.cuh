// Weights and accumulation order of ATen's antialiased bilinear kernel (_upsample_bilinear2d_aa), shared by the
// stand-alone antialias ops (resample_aa.cu), the antialiased mask rasteriser of the scoring kernel (score.cu) and the
// antialiased row source of the fused existence and refine kernels (aa_rows.cuh).
// See resample_aa.cu for the arithmetic contract; pinned by oracle/oracle.py::aa_index_weights / _aa_pass.
#pragma once
#include "common.cuh"

namespace unmore {

struct AaAxis {
  int in_size, out_size;
  float scale, support, invscale;
  __device__ __forceinline__ void init(int in, int out) {
    in_size = in; out_size = out;
    scale = __fdiv_rn((float)in, (float)out);
    support = scale >= 1.f ? scale : 1.f;
    invscale = scale >= 1.f ? (float)(1.0 / (double)scale) : 1.f;
  }
  __device__ __forceinline__ void span(int i, float& center, int& xmin, int& n) const {
    center = (float)((double)scale * ((double)i + 0.5));
    const long long lo = (long long)((double)__fsub_rn(center, support) + 0.5);
    const long long hi = (long long)((double)__fadd_rn(center, support) + 0.5);
    xmin = (int)max(lo, 0ll);
    n = (int)min(hi, (long long)in_size) - xmin;
  }
  __device__ __forceinline__ float raw_weight(int x, float center) const {
    float v = (float)(((double)__fsub_rn((float)x, center) + 0.5) * (double)invscale);
    v = fabsf(v);
    return v < 1.f ? (float)(1.0 - (double)v) : 0.f;
  }
};

// sum_j src(j) * w_j with ATen's weights and accumulation order; `src(j)` yields tap xmin + j
template <class Src>
__device__ __forceinline__ float aa_dot(const AaAxis& a, int i, Src src) {
  float center;
  int xmin, n;
  a.span(i, center, xmin, n);
  if (n <= 0) return 0.f;
  float total = 0.f;
  for (int j = 0; j < n; ++j) total = __fadd_rn(total, a.raw_weight(xmin + j, center));
  auto w = [&](int j) {
    const float r = a.raw_weight(xmin + j, center);
    return total != 0.f ? __fdiv_rn(r, total) : r;
  };
  float t = __fmul_rn(src(xmin), w(0));
  const int main_taps = ((n - 1) / 4) * 4;
  int j = 1;
  for (; j <= main_taps; ++j) t = __fadd_rn(t, __fmul_rn(src(xmin + j), w(j)));
  for (; j < n; ++j) t = __fmaf_rn(src(xmin + j), w(j), t);
  return t;
}

// Weights of one output index, normalised exactly as aa_dot does (sequential fp32 sum, then r / total).
__device__ __forceinline__ void aa_weights(const AaAxis& a, int i, int& xmin, int& n, float* w, int stride, int max_taps) {
  float center;
  a.span(i, center, xmin, n);
  if (n <= 0 || n > max_taps) return;
  float total = 0.f;
  for (int k = 0; k < n; ++k) total = __fadd_rn(total, a.raw_weight(xmin + k, center));
  for (int k = 0; k < n; ++k) {
    const float r = a.raw_weight(xmin + k, center);
    w[k * stride] = total != 0.f ? __fdiv_rn(r, total) : r;
  }
}
// aa_dot's accumulation order over a weight table: first tap a product, groups of four with separate multiply and
// add, the remaining (n-1) mod 4 fused
template <class Src, class Wt>
__device__ __forceinline__ float aa_accumulate(int n, Src src, Wt w) {
  float t = __fmul_rn(src(0), w(0));
  const int main_taps = ((n - 1) / 4) * 4;
  int k = 1;
  for (; k <= main_taps; ++k) t = __fadd_rn(t, __fmul_rn(src(k), w(k)));
  for (; k < n; ++k) t = __fmaf_rn(src(k), w(k), t);
  return t;
}

}  // namespace unmore
