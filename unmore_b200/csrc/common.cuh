// Shared device helpers for the unMORE reasoning kernels (sm_100a).
//
// Arithmetic contract: the resampling helpers reproduce, bit for bit, the fp32
// arithmetic of ATen's CPU bilinear kernels (torch 2.11, aten/src/ATen/native/cpu/
// UpSampleKernel.cpp) that torchvision.transforms.Resize dispatches to at
// object_reasoning.py:319,407,505 and object_scoring.py:131,206,222 — found by
// experiment and pinned in tests/test_oracle_golden.py (oracle.resize_bilinear_np):
//   scale = float(in) / float(out)
//   src   = max(fma(scale, i + 0.5, -0.5), 0);  i0 = min(int(src), in-1);  i1 = i0 + (i0 < in-1)
//   l1    = clamp(src - i0, 0, 1);  l0 = 1 - l1
//   generic kernel (out_h + out_w > 128):
//       t0 = fma(v00, w0, v01*w1); t1 = fma(v10, w0, v11*w1); out = fma(t0, h0, t1*h1)
//   small-output kernel (out_h + out_w <= 128):
//       out = fma(h1*w1, v11, fma(h1*w0, v10, fma(h0*w0, v00, (h0*w1)*v01)))
// Explicit __fmul_rn/__fmaf_rn keep nvcc from re-associating or contracting differently.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace unmore {

constexpr int kCrop = 128;                 // crop side hard-coded by the reference
constexpr unsigned kFullMask = 0xffffffffu;
// sigmoid(x) > 0.5 on the reference's CPU path  <=>  x > 1.5 * 2^-24 (0x33c00000); pinned in
// tests/test_oracle_golden.py::test_sigmoid_threshold_constant
#define UNMORE_SIGMOID_HALF_THRESHOLD 8.94069671630859375e-08f
// ||c|| > 0.5 with ||c|| = sqrt_rn(s), s = round(a*a) + round(b*b)  <=>  s > 0.25 * (1 + 2^-23)
// (0x3e800001): the first float whose correctly rounded square root exceeds 0.5 is 0x3e800002.
// Lets the mask kernels skip the IEEE square root; pinned in tests/test_oracle_golden.py.
#define UNMORE_NORM_HALF_SQ_THRESHOLD 0.2500000298023223876953125f

struct AxisTap {
  int i0, i1;
  float l0, l1;
};

__device__ __forceinline__ AxisTap axis_tap(float scale, int i, int in_size) {
  // ATen clamps lambda to [0, 1]; that clamp can never bind here: src >= 0 after the max, i0 is
  // either floor(src) (lambda in [0,1)) or the clamped last index, and src < in - 0.5 keeps
  // src - (in-1) < 0.5.  Dropping it removes three instructions from every output row.
  const float src = fmaxf(__fmaf_rn(scale, (float)i + 0.5f, -0.5f), 0.f);
  const int i0 = min((int)src, in_size - 1);
  AxisTap t;
  t.i0 = i0;
  t.i1 = min(i0 + 1, in_size - 1);
  t.l1 = __fsub_rn(src, (float)i0);
  t.l0 = __fsub_rn(1.f, t.l1);
  return t;
}

// horizontal stage of the generic kernel: fma(v0, w0, v1*w1)
__device__ __forceinline__ float lerp_h(float v0, float v1, float w0, float w1) {
  return __fmaf_rn(v0, w0, __fmul_rn(v1, w1));
}
// vertical stage: fma(t0, h0, t1*h1)
__device__ __forceinline__ float lerp_v(float t0, float t1, float h0, float h1) {
  return __fmaf_rn(t0, h0, __fmul_rn(t1, h1));
}

// ---- packed fp32 pairs (sm_100a FFMA2 / FMUL2 / FADD2): two IEEE round-to-nearest fp32 operations per
// issue slot, bit-identical per element to the scalar __fmaf_rn / __fmul_rn / __fadd_rn forms.  ptxas folds a
// pair built from one scalar twice into a broadcast operand (R.F32) and constants into immediates.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// the two lerp stages of the generic ATen kernel on a pair of pixels
__device__ __forceinline__ f32x2 lerp_h2(f32x2 v0, f32x2 v1, f32x2 w0, f32x2 w1) { return fma2(v0, w0, mul2(v1, w1)); }
__device__ __forceinline__ f32x2 lerp_v2(f32x2 t0, f32x2 t1, float h0, float h1) {
  return fma2(t0, pk2(h0, h0), mul2(t1, pk2(h1, h1)));
}

// Predicated shared-memory stores on a 32-bit shared address with an immediate byte offset: one instruction
// each.  (`if (pred) smem[i] = v` makes the compiler wrap the store in reconvergence bookkeeping and
// re-derive the address per store: ~6 instructions in a row loop.)
__device__ __forceinline__ unsigned smem_addr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
template <int OFF>
__device__ __forceinline__ void st_shared_b32_if(bool pred, unsigned addr, unsigned v) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.b32 [%1+%3], %2; }" ::"r"((unsigned)pred), "r"(addr), "r"(v), "n"(OFF) : "memory");
}
template <int OFF>
__device__ __forceinline__ void st_shared_b64_if(bool pred, unsigned addr, unsigned long long v) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %0, 0; @q st.shared.b64 [%1+%3], %2; }" ::"r"((unsigned)pred), "r"(addr), "l"(v), "n"(OFF) : "memory");
}

// ---- bulk-copy engine (TMA, cp.async.bulk) + mbarrier primitives, shared by the SAT scan and the TMA-fed
// existence kernel: one elected lane issues whole-row copies into shared memory, completion is tracked by the
// transaction count of an mbarrier, consumers spin on its phase parity.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                 : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}


// a predicate that is the same in every lane, stated in a form the compiler can see (vote result)
__device__ __forceinline__ bool warp_uniform(bool b) { return __any_sync(kFullMask, b) != 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFullMask, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
  return v;
}

// ---------------------------------------------------------------------------------------
// Ragged work lists.  Boxes live in [n_img, cap, 4]; image i owns the first counts[i]
// rows (counts == nullptr: all cap rows).  `offsets` (n_img+1 ints, exclusive prefix of
// counts) is built by prefix_counts_kernel; warps pull flat item ids from an atomic
// counter so long-running proposals (refine: 1..50 rounds) do not strand a CTA.
// ---------------------------------------------------------------------------------------
struct WorkList {
  const int* offsets;  // n_img + 1, or nullptr when dense
  int* counter;        // zeroed before launch
  int n_img;
  int cap;
  int total_dense;     // n_img * cap when offsets == nullptr
};

__device__ __forceinline__ int worklist_total(const WorkList& w) {
  return w.offsets ? __ldg(w.offsets + w.n_img) : w.total_dense;
}

// One lane fetches, all lanes get the id.
__device__ __forceinline__ int worklist_next_warp(const WorkList& w) {
  int id = 0;
  if ((threadIdx.x & 31) == 0) id = atomicAdd(w.counter, 1);
  return __shfl_sync(kFullMask, id, 0);
}

// `img` holds the image of the PREVIOUS item this warp / CTA pulled (0 before the first): ids only grow, so
// the owner is found by walking forward from there — usually zero or one step — and the 8-probe binary
// search (a chain of dependent loads with the CTA idle behind it) is only the fallback for long jumps.
__device__ __forceinline__ void worklist_locate(const WorkList& w, int id, int& img, int& k) {
  if (!w.offsets) {
    img = id / w.cap;
    k = id - img * w.cap;
    return;
  }
  {
    int cur = min(max(img, 0), w.n_img - 1);
    int base = __ldg(w.offsets + cur);
    if (base <= id) {
      int steps = 0;
      int next = __ldg(w.offsets + cur + 1);
      while (next <= id && steps < 4) { ++cur; base = next; next = __ldg(w.offsets + cur + 1); ++steps; }
      if (next > id) { img = cur; k = id - base; return; }
    }
  }
  int lo = 0, hi = w.n_img;  // find img with offsets[img] <= id < offsets[img+1]
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (__ldg(w.offsets + mid) <= id) lo = mid; else hi = mid;
  }
  img = lo;
  k = id - __ldg(w.offsets + lo);
}

template <typename T>
__device__ __forceinline__ void load_box(const void* boxes, bool f64, size_t row, T& x1, T& y1, T& x2, T& y2);

template <>
__device__ __forceinline__ void load_box<double>(const void* boxes, bool f64, size_t row, double& x1, double& y1,
                                                 double& x2, double& y2) {
  if (f64) {
    const double4 b = reinterpret_cast<const double4*>(boxes)[row];
    x1 = b.x; y1 = b.y; x2 = b.z; y2 = b.w;
  } else {
    const float4 b = reinterpret_cast<const float4*>(boxes)[row];
    x1 = b.x; y1 = b.y; x2 = b.z; y2 = b.w;
  }
}

// Crop window of a proposal: floor(x1), floor(y1), ceil(x2), ceil(y2)  (object_reasoning.py:404),
// clamped to the image (the reference never produces out-of-range boxes: every producer clips).
struct Window {
  int x1, y1, x2, y2;
  __device__ __forceinline__ int w() const { return x2 - x1; }
  __device__ __forceinline__ int h() const { return y2 - y1; }
  __device__ __forceinline__ bool empty() const { return x2 <= x1 || y2 <= y1; }
};

// Extent (h, w) of image `img` of a padded field stack, from its [n_img, 2] int32 table (one 8-byte read-only load;
// the table is 8-byte aligned, checked by the C ABI).  Clamped to [1, pitch]: a bad entry gives wrong numbers, never
// an address outside the pitched planes.  The load is volatile so that a kernel which reads the extent again after a
// long stretch of work (refine) really re-reads it (an L1 hit) instead of holding it in two registers meanwhile.
__device__ __forceinline__ int2 image_extent(const int* image_hw, int img, int H, int W) {
  int2 e;
  asm volatile("ld.global.nc.v2.s32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "l"(image_hw + 2 * (size_t)img));
  return make_int2(min(max(e.x, 1), H), min(max(e.y, 1), W));
}

template <typename T>
__device__ __forceinline__ Window snap_window(T x1, T y1, T x2, T y2, int W, int H) {
  Window w;
  w.x1 = max(0, min(W, (int)floor(x1)));
  w.y1 = max(0, min(H, (int)floor(y1)));
  w.x2 = max(0, min(W, (int)ceil(x2)));
  w.y2 = max(0, min(H, (int)ceil(y2)));
  return w;
}

}  // namespace unmore
