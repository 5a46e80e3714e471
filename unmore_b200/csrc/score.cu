// main_object_scoring steps 1-6 (object_scoring.py:182-235) for a list of discovered boxes:
//   existence / center / boundary scores from the resized 128x128 crop (:189-193),
//   the two binary masks (||center|| > 0.5, sigmoid(sdf) > 0.5) resized back to the box with
//   bilinear + round-half-even (:196-225), their union pasted on the image canvas (:228),
//   the tight box of the union (pycocotools rleToBbox semantics, :160-164) and its area.
// Masks leave the kernel bit-packed: [H, ceil(W/32)] words per mask, LSB = lowest x.
//
// One CTA per box.  round(v) == 1  <=>  v > 0.5 for v in [0,1] (half-to-even sends exactly 0.5
// to 0), so the rasteriser only needs the comparison; the interpolation itself follows ATen's
// two CPU kernels bit for bit (generic kernel for h+w > 128, small-output kernel otherwise —
// see common.cuh) because near-tie values decide mask bits.
#include "resample.cuh"
#include "resample_aa.cuh"
#include "unmore_internal.h"

namespace unmore {

constexpr int kScoreThreads = 256;
constexpr int kScoreWarps = kScoreThreads / 32;
constexpr int kMaxBoxSide = 2048;  // x-tap table in shared memory

struct ScoreSmem {
  uint32_t cmask[kCrop][4];
  uint32_t bmask[kCrop][4];
  unsigned char tx0[kMaxBoxSide], tx1[kMaxBoxSide];
  float tw0[kMaxBoxSide], tw1[kMaxBoxSide];
  double red_sum[kScoreWarps];
  float red_c[kScoreWarps], red_b[kScoreWarps];
  int xmin, xmax, ymin, ymax, area;
};

__device__ __forceinline__ float bit_at(const uint32_t m[kCrop][4], int y, int x) {
  return (float)((m[y][x >> 5] >> (x & 31)) & 1u);
}

// One output pixel of Resize((oh, ow), BILINEAR) applied to a 128x128 {0,1} mask followed by
// round-half-even (object_scoring.py:206-207): the bit is interp > 0.5, with the interpolation in the
// exact arithmetic of whichever ATen CPU kernel the output size selects (common.cuh).
__device__ __forceinline__ bool resized_mask_bit(const uint32_t m[kCrop][4], const AxisTap& ty, int x0, int x1, float w0,
                                                 float w1, bool small_path) {
  const float v00 = bit_at(m, ty.i0, x0), v01 = bit_at(m, ty.i0, x1);
  const float v10 = bit_at(m, ty.i1, x0), v11 = bit_at(m, ty.i1, x1);
  float val;
  if (!small_path) {
    val = lerp_v(lerp_h(v00, v01, w0, w1), lerp_h(v10, v11, w0, w1), ty.l0, ty.l1);
  } else {
    const float p00 = __fmul_rn(ty.l0, w0), p01 = __fmul_rn(ty.l0, w1);
    const float p10 = __fmul_rn(ty.l1, w0), p11 = __fmul_rn(ty.l1, w1);
    val = __fmaf_rn(p11, v11, __fmaf_rn(p10, v10, __fmaf_rn(p00, v00, __fmul_rn(p01, v01))));
  }
  return val > 0.5f;
}

// The same pixel in the second resize mode (antialias=True): ATen's separable antialiased kernel on the {0,1} mask,
// horizontal pass first — T[yy][x] = sum_xx wx * bit(yy, xx) — then the vertical pass over T; every T value is
// recomputed where it is needed (same arithmetic, same rounding as the two-pass form of resample_aa.cu).
__device__ __forceinline__ bool resized_mask_bit_aa(const uint32_t m[kCrop][4], const AaAxis& ay, const AaAxis& ax, int y, int x) {
  const float v = aa_dot(ay, y, [&](int yy) { return aa_dot(ax, x, [&](int xx) { return bit_at(m, yy, xx); }); });
  return v > 0.5f;   // round half to even: exactly 0.5 -> 0
}

// TILES_AA = false: the fused primary path (crop + plain bilinear resample inside the kernel, antialias=False).
// TILES_AA = true: the tile path — the four channels come PRE-RESAMPLED from p.tiles ([n_img * cap, 4, 128, 128] = sdf,
// center_row, center_col, existence: from unmore_crop_resize_aa in the second resize mode, or from the per-crop nets
// of the reference's original mode); the masks are rasterised back to the box with the antialiased kernel when
// p.aa_raster is set and with the plain one otherwise; p.exist_scores, when given, replaces the mean of the fourth
// tile (the reference's classifier puts out one scalar per crop, object_scoring.py:140-150).
// The window snaps to the image's extent (image_extent; on the tile path, that of the image the tiles were cropped
// from); the mask canvas stays H x ceil(W/32) words of the pitch (bits outside the image stay 0).
template <bool TILES_AA>
__global__ void __launch_bounds__(kScoreThreads) score_kernel(const ScoreParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  ScoreSmem& sm = *reinterpret_cast<ScoreSmem*>(smem_raw);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int img = blockIdx.y, k = blockIdx.x;
  const int n = p.counts ? p.counts[img] : p.cap;
  if (k >= n) return;
  const size_t row = (size_t)img * p.cap + k;
  double bx1, by1, bx2, by2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, row, bx1, by1, bx2, by2);
  const int2 e = image_extent(p.image_hw, img, p.H, p.W);
  const Window win = snap_window<double>(bx1, by1, bx2, by2, e.y, e.x);
  const int Wp = (p.W + 31) >> 5;
  uint32_t* mask_out = p.masks ? p.masks + row * (size_t)p.H * Wp : nullptr;
  if (tid == 0) { sm.xmin = 1 << 30; sm.ymin = 1 << 30; sm.xmax = -1; sm.ymax = -1; sm.area = 0; }
  if (win.empty() || win.w() > kMaxBoxSide) {  // the reference raises on a zero-size crop
    if (mask_out)
      for (int q = tid; q < p.H * Wp; q += kScoreThreads) mask_out[q] = 0u;
    if (tid == 0) {
      p.scores[row] = make_float4(0.f, 0.f, 0.f, 0.f);
      p.tight[row] = make_float4(0.f, 0.f, 0.f, 0.f);
      p.areas[row] = 0;
    }
    return;
  }
  // ---- 1. resample the four channels; warp w owns rows 16w .. 16w+15
  {
    ColTaps taps;
    if constexpr (!TILES_AA) taps.init<kStrided>(lane, win.w());
    const size_t plane_sz = (size_t)p.H * p.W;
    const float* base = p.fields + (size_t)img * p.C * plane_sz;
    const float* const planes[4] = {base + p.ch_sdf * plane_sz, base + p.ch_crow * plane_sz,
                                    base + p.ch_ccol * plane_sz, base + p.ch_exist * plane_sz};
    MultiPlaneRows<4> rows;
    if constexpr (!TILES_AA) rows.init(planes, p.W, win);
    const float* tile = TILES_AA ? p.tiles + row * (size_t)(4 * kCrop * kCrop) : nullptr;
    const float scale_y = __fdiv_rn((float)win.h(), (float)kCrop);
    const int in_h = win.h();
    double esum = 0.0;
    float cmax = 0.f, bmax = -INFINITY;
    constexpr int kRows = kCrop / kScoreWarps;
    for (int ii = 0; ii < kRows; ++ii) {
      const int i = warp * kRows + ii;
      const AxisTap v = axis_tap(scale_y, i, in_h);
      float sabe[4][4];
      if constexpr (TILES_AA) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int c = 0; c < 4; ++c) sabe[q][c] = __ldg(tile + (q * kCrop + i) * kCrop + lane + 32 * c);
      } else {
        rows.row(taps, v, sabe);
      }
      const float (&s)[4] = sabe[0];
      const float (&a)[4] = sabe[1];
      const float (&b)[4] = sabe[2];
      const float (&e)[4] = sabe[3];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float sq = __fadd_rn(__fmul_rn(a[c], a[c]), __fmul_rn(b[c], b[c]));  // torch.norm order
        cmax = fmaxf(cmax, sq);
        bmax = fmaxf(bmax, s[c]);
        // columns 32c .. 32c+31 of row i, LSB = lowest column
        const uint32_t wc = __ballot_sync(kFullMask, sq > UNMORE_NORM_HALF_SQ_THRESHOLD);
        const uint32_t wb = __ballot_sync(kFullMask, s[c] > UNMORE_SIGMOID_HALF_THRESHOLD);
        if (lane == 0) { sm.cmask[i][c] = wc; sm.bmask[i][c] = wb; }
      }
      esum += (double)((e[0] + e[1]) + (e[2] + e[3]));
    }
    esum = warp_sum(esum);
    cmax = warp_max(cmax);
    bmax = warp_max(bmax);
    if (lane == 0) { sm.red_sum[warp] = esum; sm.red_c[warp] = cmax; sm.red_b[warp] = bmax; }
  }
  // ---- 2. x taps of the resize back to the box (128 -> ow), shared by both masks
  const int ow = win.w(), oh = win.h();
  const float sx = __fdiv_rn((float)kCrop, (float)ow), sy = __fdiv_rn((float)kCrop, (float)oh);
  const bool aa_raster = TILES_AA && p.aa_raster;
  for (int x = tid; x < ow && !aa_raster; x += kScoreThreads) {
    const AxisTap t = axis_tap(sx, x, kCrop);
    sm.tx0[x] = (unsigned char)t.i0; sm.tx1[x] = (unsigned char)t.i1; sm.tw0[x] = t.l0; sm.tw1[x] = t.l1;
  }
  __syncthreads();
  if (tid == 0) {
    double es = 0.0;
    float cm = 0.f, bm = -INFINITY;
    for (int w = 0; w < kScoreWarps; ++w) { es += sm.red_sum[w]; cm = fmaxf(cm, sm.red_c[w]); bm = fmaxf(bm, sm.red_b[w]); }
    // (existence, center, boundary, unused)
    const float ex = (TILES_AA && p.exist_scores) ? p.exist_scores[row] : (float)(es * (1.0 / (kCrop * kCrop)));
    p.scores[row] = make_float4(ex, __fsqrt_rn(cm), bm, 0.f);
  }
  // ---- 3. rasterise the union on the image canvas, one 32-pixel word per thread step
  const bool small_path = (oh + ow) <= 128;
  AaAxis aax, aay;
  if (aa_raster) { aax.init(kCrop, ow); aay.init(kCrop, oh); }
  int xmin = 1 << 30, xmax = -1, ymin = 1 << 30, ymax = -1, area = 0;
  for (int q = tid; q < p.H * Wp; q += kScoreThreads) {
    const int y = q / Wp, wx = q - y * Wp;
    uint32_t word = 0u;
    const int xb = wx << 5;
    if (y >= win.y1 && y < win.y2 && xb < win.x2 && xb + 32 > win.x1) {
      const AxisTap ty = axis_tap(sy, y - win.y1, kCrop);
      const int lo = max(xb, win.x1), hi = min(xb + 32, win.x2);
      for (int x = lo; x < hi; ++x) {
        const int ox = x - win.x1;
        bool on = false;
        if (aa_raster) {
          on = resized_mask_bit_aa(sm.cmask, aay, aax, y - win.y1, ox) || resized_mask_bit_aa(sm.bmask, aay, aax, y - win.y1, ox);
        } else {
          const int x0 = sm.tx0[ox], x1 = sm.tx1[ox];
          const float w0 = sm.tw0[ox], w1 = sm.tw1[ox];
#pragma unroll
          for (int mm = 0; mm < 2; ++mm) {
            const uint32_t (*m)[4] = mm == 0 ? sm.cmask : sm.bmask;
            on = on || resized_mask_bit(m, ty, x0, x1, w0, w1, small_path);
          }
        }
        word |= (on ? 1u : 0u) << (x - xb);
      }
    }
    if (mask_out) mask_out[q] = word;
    if (word) {
      area += __popc(word);
      xmin = min(xmin, xb + __ffs(word) - 1);
      xmax = max(xmax, xb + 31 - __clz(word));
      ymin = min(ymin, y);
      ymax = max(ymax, y);
    }
  }
  // ---- 4. tight box + area
  area = warp_sum(area);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    xmin = min(xmin, __shfl_xor_sync(kFullMask, xmin, o));
    ymin = min(ymin, __shfl_xor_sync(kFullMask, ymin, o));
    xmax = max(xmax, __shfl_xor_sync(kFullMask, xmax, o));
    ymax = max(ymax, __shfl_xor_sync(kFullMask, ymax, o));
  }
  if (lane == 0) {
    atomicAdd(&sm.area, area);
    atomicMin(&sm.xmin, xmin); atomicMin(&sm.ymin, ymin);
    atomicMax(&sm.xmax, xmax); atomicMax(&sm.ymax, ymax);
  }
  __syncthreads();
  if (tid == 0) {
    // rleToBbox: [xmin, ymin, xmax-xmin+1, ymax-ymin+1] -> xyxy = [xmin, ymin, xmax+1, ymax+1]; zeros if empty
    if (sm.area > 0) p.tight[row] = make_float4((float)sm.xmin, (float)sm.ymin, (float)(sm.xmax + 1), (float)(sm.ymax + 1));
    else p.tight[row] = make_float4(0.f, 0.f, 0.f, 0.f);
    p.areas[row] = sm.area;
  }
}

// Stand-alone form of the mask resize (unit parity with the reference's Resize on int64 masks):
// masks [B,128,128] u8 -> out [B, oh, ow] u8.  One CTA per mask.
__global__ void __launch_bounds__(256) mask_resize_kernel(const unsigned char* __restrict__ masks, int B, int oh, int ow,
                                                          unsigned char* __restrict__ out) {
  __shared__ uint32_t m[kCrop][4];
  const int b = blockIdx.x, tid = threadIdx.x;
  const unsigned char* src = masks + (size_t)b * kCrop * kCrop;
  for (int w = tid; w < kCrop * 4; w += 256) {
    uint32_t word = 0;
    for (int k = 0; k < 32; ++k) word |= (src[w * 32 + k] ? 1u : 0u) << k;
    m[w >> 2][w & 3] = word;
  }
  __syncthreads();
  const float sx = __fdiv_rn((float)kCrop, (float)ow), sy = __fdiv_rn((float)kCrop, (float)oh);
  const bool small_path = (oh + ow) <= 128;
  unsigned char* o = out + (size_t)b * oh * ow;
  for (int q = tid; q < oh * ow; q += 256) {
    const int y = q / ow, x = q - y * ow;
    const AxisTap ty = axis_tap(sy, y, kCrop), tx = axis_tap(sx, x, kCrop);
    o[q] = resized_mask_bit(m, ty, tx.i0, tx.i1, tx.l0, tx.l1, small_path) ? 1 : 0;
  }
}

int launch_mask_resize(const unsigned char* masks, int B, int oh, int ow, unsigned char* out, cudaStream_t stream) {
  if (B <= 0 || oh <= 0 || ow <= 0) return 0;
  mask_resize_kernel<<<B, 256, 0, stream>>>(masks, B, oh, ow, out);
  return (int)cudaGetLastError();
}

template <bool TILES_AA>
static int launch_score_t(const ScoreParams& p, cudaStream_t stream) {
  cudaError_t e = cudaFuncSetAttribute(score_kernel<TILES_AA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ScoreSmem));
  if (e != cudaSuccess) return (int)e;
  score_kernel<TILES_AA><<<dim3(p.cap, p.n_img), kScoreThreads, sizeof(ScoreSmem), stream>>>(p);
  return (int)cudaGetLastError();
}

int launch_score(const ScoreParams& p, cudaStream_t stream) {
  if (p.n_img <= 0 || p.cap <= 0) return 0;
  return p.tiles ? launch_score_t<true>(p, stream) : launch_score_t<false>(p, stream);
}

// area_score, final score, COCO xywh box and the post_process predicate (object_scoring.py:244-266,
// post_process.py:61-74) for the detections kept by the second NMS.  One CTA per image.
__global__ void __launch_bounds__(256) final_scores_kernel(const FinalParams p) {
  __shared__ int smax;
  const int b = blockIdx.x;
  const int n = min(p.keep_counts[b], p.cap);
  const int* keep = p.keep + (size_t)b * p.cap;
  if (threadIdx.x == 0) smax = 0;
  __syncthreads();
  int m = 0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) m = max(m, p.areas[(size_t)b * p.cap + keep[i]]);
  m = max(m, __shfl_xor_sync(kFullMask, m, 16)); m = max(m, __shfl_xor_sync(kFullMask, m, 8));
  m = max(m, __shfl_xor_sync(kFullMask, m, 4));  m = max(m, __shfl_xor_sync(kFullMask, m, 2));
  m = max(m, __shfl_xor_sync(kFullMask, m, 1));
  if ((threadIdx.x & 31) == 0) atomicMax(&smax, m);
  __syncthreads();
  const double max_area = (double)smax;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const size_t src = (size_t)b * p.cap + keep[i], dst = (size_t)b * p.cap + i;
    const float4 s = p.scores[src];
    const float4 t = p.tight[src];
    const double mask_score = (double)p.areas[src] / max_area;   // int64 / int64 -> float64 (:245)
    const double area_score = pow(mask_score, 0.25);             // (:255)
    // numpy float32 scalars multiply in fp32, the float64 area score promotes the last product
    const float ecb = __fmul_rn(__fmul_rn(s.x, s.y), s.z);
    double* o = p.out + dst * 5;
    o[0] = (double)ecb * area_score;  // score
    o[1] = (double)s.x;               // existence_score
    o[2] = (double)s.y;               // center_score
    o[3] = (double)s.z;               // boundary_score
    o[4] = area_score;                // area_score
    p.bbox_xywh[dst] = make_float4(t.x, t.y, __fsub_rn(t.z, t.x), __fsub_rn(t.w, t.y));
    if (p.selected)
      p.selected[dst] = !((double)s.x < p.existence_thres || (double)s.y < p.center_thres || (double)s.z < p.boundary_thres) ? 1 : 0;
  }
}

int launch_final_scores(const FinalParams& p, cudaStream_t stream) {
  if (p.n_img <= 0) return 0;
  final_scores_kernel<<<p.n_img, 256, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

}  // namespace unmore
