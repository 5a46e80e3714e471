// Summed-area tables of per-image fields and O(1) box sums (north-star op (a); the reference
// has no counterpart — SURVEY.md §8a row A — so the oracle is a float64 cumsum restatement).
//
//   S[y][x] = sum_{v<y, u<x} f[v][u]   stored as fp64 [H+1, W+1] (first row / column zero)
//   boxsum  = S[y2][x2] - S[y1][x2] - S[y2][x1] + S[y1][x1]   on the snapped window
//
// fp64 because an fp32 table of a 480x640 field reaches ~3e5 and differencing then loses
// ~2e-2 absolute.  HBM-bound: 4 B read + 8 B written per pixel.  One warp sweeps one plane top
// to bottom: each lane owns 4 consecutive columns of every 128-column step (one coalesced
// float4 load), does a 3-add serial prefix, a 5-step warp-shuffle scan of the lane totals,
// and keeps the running column sums (the vertical scan) in registers, so no shared-memory
// exchange or barrier is needed.  Results are restaged through a 1 KB per-warp shared buffer
// so every global store instruction writes 32 consecutive doubles.
#include "unmore_internal.h"

namespace unmore {

constexpr int kSatWarps = 4;

__device__ __forceinline__ double shfl_up_d(double v, int o) { return __shfl_up_sync(kFullMask, v, o); }

// Plane p of the output is channel sel.ch[p % sel.n] of image p / sel.n of a [n_img, C, H, W] stack
// (sel.n == 0: `in` is a dense [n_planes, H, W] tensor), so the tables are built in place from
// the field stack without a gather copy.
struct PlaneSel { int n, C, ch[4]; };

// On a padded field stack (sel.n > 0, image_hw non-null) the pixels outside each image's (h, w) are read as zeros, so
// every entry S[y][x] with y <= h, x <= w is, bit for bit, that of the image built alone (a padded value would
// otherwise reach the lane's scan total, and through it the columns left of it).  PADDED = false compiles the kernel
// without the table and the mask (image_hw is null): with them, a uniform 642-px-wide stack took 2% longer (168
// instead of 128 registers at STEPS = 8; one B200 at 1000 W).
template <int STEPS, bool PADDED>
__global__ void __launch_bounds__(kSatWarps * 32) sat_kernel(const float* __restrict__ in, double* __restrict__ out,
                                                              int n_planes, int H, int W, const PlaneSel sel,
                                                              const int* __restrict__ image_hw) {
  __shared__ double stage[kSatWarps][128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int plane = blockIdx.x * kSatWarps + warp;
  if (plane >= n_planes) return;
  const int img = sel.n ? plane / sel.n : 0;   // sel.n == 0 (a dense stack of planes) comes without a table
  const int2 ext = image_extent(PADDED ? image_hw : nullptr, img, H, W);
  const size_t src_plane = sel.n ? (size_t)img * sel.C + sel.ch[plane % sel.n] : (size_t)plane;
  const float* src = in + src_plane * H * W;
  double* dst = out + (size_t)plane * (H + 1) * (W + 1);
  const int OW = W + 1;
  for (int x = lane; x < OW; x += 32) dst[x] = 0.0;  // row 0
  double vacc[STEPS][4];
#pragma unroll
  for (int s = 0; s < STEPS; ++s) vacc[s][0] = vacc[s][1] = vacc[s][2] = vacc[s][3] = 0.0;
  const bool vec_ok = (W & 3) == 0;
  for (int y = 0; y < H; ++y) {
    const float* rowp = src + (size_t)y * W;
    double* orow = dst + (size_t)(y + 1) * OW;
    float4 v[STEPS];
#pragma unroll
    for (int s = 0; s < STEPS; ++s) {
      const int x = s * 128 + 4 * lane;
      if (vec_ok && x + 3 < W) {
        v[s] = __ldcs(reinterpret_cast<const float4*>(rowp + x));  // streamed once: evict-first
      } else {
        v[s].x = x < W ? rowp[x] : 0.f;
        v[s].y = x + 1 < W ? rowp[x + 1] : 0.f;
        v[s].z = x + 2 < W ? rowp[x + 2] : 0.f;
        v[s].w = x + 3 < W ? rowp[x + 3] : 0.f;
      }
      if constexpr (PADDED) {   // padding was read (inside the pitch); it enters the sums as zeros
        const int rw = y < ext.x ? ext.y : 0;
        v[s].x = x < rw ? v[s].x : 0.f;
        v[s].y = x + 1 < rw ? v[s].y : 0.f;
        v[s].z = x + 2 < rw ? v[s].z : 0.f;
        v[s].w = x + 3 < rw ? v[s].w : 0.f;
      }
    }
    if (lane == 0) orow[0] = 0.0;  // column 0
    double carry = 0.0;            // row prefix of everything left of this step
#pragma unroll
    for (int s = 0; s < STEPS; ++s) {
      if (s * 128 >= W) break;
      const double a0 = (double)v[s].x, a1 = a0 + (double)v[s].y, a2 = a1 + (double)v[s].z, a3 = a2 + (double)v[s].w;
      double incl = a3;  // inclusive scan of lane totals
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = shfl_up_d(incl, o);
        if (lane >= o) incl += t;
      }
      const double base = carry + (incl - a3);
      carry += __shfl_sync(kFullMask, incl, 31);
      vacc[s][0] += base + a0; vacc[s][1] += base + a1; vacc[s][2] += base + a2; vacc[s][3] += base + a3;
      // restage: lane l holds columns 4l..4l+3; store instruction j writes columns 32j + lane
      __syncwarp();
      *reinterpret_cast<double2*>(&stage[warp][4 * lane]) = make_double2(vacc[s][0], vacc[s][1]);
      *reinterpret_cast<double2*>(&stage[warp][4 * lane + 2]) = make_double2(vacc[s][2], vacc[s][3]);
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = s * 128 + 32 * j + lane;
        if (x < W) __stcs(orow + 1 + x, stage[warp][32 * j + lane]);
      }
    }
  }
}

// ---- TMA-fed variant ----------------------------------------------------------------------
// Same arithmetic, but the input rows arrive through the bulk-copy engine: lane 0 of each warp keeps
// kSatStages whole rows (W*4 bytes each) in flight with cp.async.bulk into a per-warp shared-memory
// ring, completion tracked by one mbarrier per slot.  The rows wait in shared memory instead of in
// registers, so a warp has 6 rows (15 KB at W=640) outstanding instead of one
// (ring depth 3 / 4 / 6 / 8 measured: 4720 / 4699 / 5433 / 4387 GB/s at 3000 planes; 5-7 tie at 5950 GB/s at 8000).
// Needs W % 4 == 0 (16-byte rows) and a stack without padding; launch_sat takes the register-fed kernel otherwise.
constexpr int kSatStages = 6;

template <int STEPS>
__global__ void __launch_bounds__(kSatWarps * 32) sat_kernel_tma(const float* __restrict__ in, double* __restrict__ out,
                                                                  int n_planes, int H, int W, const PlaneSel sel) {
  extern __shared__ __align__(128) unsigned char sat_smem[];
  __shared__ double stage[kSatWarps][128];
  __shared__ __align__(8) uint64_t bars[kSatWarps][kSatStages];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int plane = blockIdx.x * kSatWarps + warp;
  if (plane >= n_planes) return;
  const uint32_t row_bytes = (uint32_t)W * 4u;
  float* ring = reinterpret_cast<float*>(sat_smem) + (size_t)warp * kSatStages * W;
  const size_t src_plane = sel.n ? (size_t)(plane / sel.n) * sel.C + sel.ch[plane % sel.n] : (size_t)plane;
  const float* src = in + src_plane * H * W;
  double* dst = out + (size_t)plane * (H + 1) * (W + 1);
  const int OW = W + 1;
  if (lane == 0) {
    for (int k = 0; k < kSatStages; ++k) mbar_init(&bars[warp][k], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    for (int k = 0; k < kSatStages && k < H; ++k) {
      mbar_expect_tx(&bars[warp][k], row_bytes);
      bulk_g2s(ring + (size_t)k * W, src + (size_t)k * W, row_bytes, &bars[warp][k]);
    }
  }
  __syncwarp();
  for (int x = lane; x < OW; x += 32) dst[x] = 0.0;  // row 0
  double vacc[STEPS][4];
#pragma unroll
  for (int s = 0; s < STEPS; ++s) vacc[s][0] = vacc[s][1] = vacc[s][2] = vacc[s][3] = 0.0;
  for (int y = 0; y < H; ++y) {
    const int slot = y % kSatStages;
    mbar_wait(&bars[warp][slot], (uint32_t)((y / kSatStages) & 1));
    const float* rowp = ring + (size_t)slot * W;
    double* orow = dst + (size_t)(y + 1) * OW;
    float4 v[STEPS];
#pragma unroll
    for (int s = 0; s < STEPS; ++s) {
      const int x = s * 128 + 4 * lane;
      v[s] = x + 3 < W ? *reinterpret_cast<const float4*>(rowp + x) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();  // every lane has its copy of the row: the slot may be refilled
    if (lane == 0 && y + kSatStages < H) {
      mbar_expect_tx(&bars[warp][slot], row_bytes);
      bulk_g2s(ring + (size_t)slot * W, src + (size_t)(y + kSatStages) * W, row_bytes, &bars[warp][slot]);
    }
    if (lane == 0) orow[0] = 0.0;  // column 0
    double carry = 0.0;
#pragma unroll
    for (int s = 0; s < STEPS; ++s) {
      if (s * 128 >= W) break;
      const double a0 = (double)v[s].x, a1 = a0 + (double)v[s].y, a2 = a1 + (double)v[s].z, a3 = a2 + (double)v[s].w;
      double incl = a3;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double t = shfl_up_d(incl, o);
        if (lane >= o) incl += t;
      }
      const double base = carry + (incl - a3);
      carry += __shfl_sync(kFullMask, incl, 31);
      vacc[s][0] += base + a0; vacc[s][1] += base + a1; vacc[s][2] += base + a2; vacc[s][3] += base + a3;
      __syncwarp();
      *reinterpret_cast<double2*>(&stage[warp][4 * lane]) = make_double2(vacc[s][0], vacc[s][1]);
      *reinterpret_cast<double2*>(&stage[warp][4 * lane + 2]) = make_double2(vacc[s][2], vacc[s][3]);
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int x = s * 128 + 32 * j + lane;
        if (x < W) __stcs(orow + 1 + x, stage[warp][32 * j + lane]);
      }
    }
  }
}

template <int STEPS>
static int launch_sat_tma(const float* in, double* out, int n_planes, int H, int W, const PlaneSel& sel, int grid,
                          cudaStream_t stream) {
  const size_t smem = (size_t)kSatWarps * kSatStages * W * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(sat_kernel_tma<STEPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  sat_kernel_tma<STEPS><<<grid, kSatWarps * 32, smem, stream>>>(in, out, n_planes, H, W, sel);
  return (int)cudaGetLastError();
}

template <bool PADDED>
static int launch_sat_regs(const float* in, double* out, int n_planes, int H, int W, const PlaneSel& sel,
                           const int* image_hw, int grid, int steps, cudaStream_t stream) {
  if (steps <= 5) sat_kernel<5, PADDED><<<grid, kSatWarps * 32, 0, stream>>>(in, out, n_planes, H, W, sel, image_hw);
  else if (steps <= 8) sat_kernel<8, PADDED><<<grid, kSatWarps * 32, 0, stream>>>(in, out, n_planes, H, W, sel, image_hw);
  else sat_kernel<16, PADDED><<<grid, kSatWarps * 32, 0, stream>>>(in, out, n_planes, H, W, sel, image_hw);
  return (int)cudaGetLastError();
}

int launch_sat(const float* in, double* out, int n_planes, int H, int W, int C, const int* channels, int n_ch,
               const int* image_hw, cudaStream_t stream) {
  if (n_planes <= 0) return 0;
  PlaneSel sel{};
  sel.n = n_ch; sel.C = C;
  for (int i = 0; i < n_ch && i < 4; ++i) sel.ch[i] = channels[i];
  const int grid = (n_planes + kSatWarps - 1) / kSatWarps;
  const int steps = (W + 127) / 128;
  // bulk-copy path: 16-byte aligned rows (W % 4 == 0; planes of a 16-byte aligned tensor then are too)
  if (!image_hw && (W & 3) == 0 && ((size_t)H * W & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && steps <= 8) {
    if (steps <= 5) return launch_sat_tma<5>(in, out, n_planes, H, W, sel, grid, stream);
    return launch_sat_tma<8>(in, out, n_planes, H, W, sel, grid, stream);
  }
  if (steps > 16) return -2;
  if (image_hw) return launch_sat_regs<true>(in, out, n_planes, H, W, sel, image_hw, grid, steps, stream);
  return launch_sat_regs<false>(in, out, n_planes, H, W, sel, nullptr, grid, steps, stream);
}

// boxsum (top of the file): the tables are indexed on the pitch, the window snaps to the image's own extent.
__global__ void box_sums_kernel(const double* __restrict__ sat, int planes_per_img, int plane, int H, int W,
                                const void* __restrict__ boxes, int boxes_f64, const int* __restrict__ counts, int cap,
                                int n_img, double* __restrict__ sums, double* __restrict__ means,
                                const int* __restrict__ image_hw) {
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n_img * cap) return;
  const int img = id / cap, k = id - img * cap;
  if (counts && k >= counts[img]) return;
  double x1, y1, x2, y2;
  load_box<double>(boxes, boxes_f64 != 0, (size_t)id, x1, y1, x2, y2);
  const int2 e = image_extent(image_hw, img, H, W);
  const Window w = snap_window<double>(x1, y1, x2, y2, e.y, e.x);
  const double* S = sat + ((size_t)img * planes_per_img + plane) * (H + 1) * (W + 1);
  const int OW = W + 1;
  double s = 0.0;
  if (!w.empty())
    s = S[(size_t)w.y2 * OW + w.x2] - S[(size_t)w.y1 * OW + w.x2] - S[(size_t)w.y2 * OW + w.x1] + S[(size_t)w.y1 * OW + w.x1];
  sums[id] = s;
  if (means) means[id] = w.empty() ? 0.0 : s / ((double)w.w() * (double)w.h());
}

int launch_box_sums(const double* sat, int planes_per_img, int plane, int H, int W, const void* boxes, int boxes_f64,
                    const int* counts, int cap, int n_img, double* sums, double* means, const int* image_hw,
                    cudaStream_t stream) {
  const int total = n_img * cap;
  if (total <= 0) return 0;
  box_sums_kernel<<<(total + 255) / 256, 256, 0, stream>>>(sat, planes_per_img, plane, H, W, boxes, boxes_f64, counts, cap,
                                                            n_img, sums, means, image_hw);
  return (int)cudaGetLastError();
}

}  // namespace unmore
