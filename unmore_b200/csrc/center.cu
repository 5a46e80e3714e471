// center_reasoning in the primary resize mode and on tiles (the kernel: center.cuh), and the stand-alone unit ops.
#include "center.cuh"

namespace unmore {

// variable-distance shifts spelled out on 64-bit halves (the compiler-generated variable
// __int128 shift produced wrong rows on sm_100a; constant shifts are fine)
__device__ __forceinline__ u128 shr128(u128 v, int s) {
  const unsigned long long lo = (unsigned long long)v, hi = (unsigned long long)(v >> 64);
  if (s <= 0) return v;
  if (s >= 128) return 0;
  if (s >= 64) return (u128)(hi >> (s - 64));
  return ((u128)(hi >> s) << 64) | (u128)((lo >> s) | (hi << (64 - s)));
}
__device__ __forceinline__ u128 shl128(u128 v, int s) {
  const unsigned long long lo = (unsigned long long)v, hi = (unsigned long long)(v >> 64);
  if (s <= 0) return v;
  if (s >= 128) return 0;
  if (s >= 64) return (u128)(lo << (s - 64)) << 64;
  return ((u128)((hi << s) | (lo >> (64 - s))) << 64) | (u128)(lo << s);
}

// ---- stand-alone unit ops (signature parity with utils/misc.py:10-20 and object_reasoning.py:360-377)

// batch_erode on 128x128 masks: num_round erosions with a k x k ones kernel and zero border
// == one erosion with side (k-1)*num_round+1 and zero border.  One warp per mask row set.
__global__ void __launch_bounds__(kCrop) erode_kernel(const unsigned char* __restrict__ in, unsigned char* __restrict__ out,
                                                      int B, int radius) {
  __shared__ uint32_t hrun[kCrop][4];
  const int b = blockIdx.x, r = threadIdx.x;
  const unsigned char* m = in + (size_t)b * kCrop * kCrop;
  uint32_t w4[4] = {0u, 0u, 0u, 0u};
  for (int c = 0; c < kCrop; ++c) w4[c >> 5] |= (m[r * kCrop + c] ? 1u : 0u) << (c & 31);
  const u128 v = load_row(w4);
  // run of (2*radius+1) set bits starting at bit j, by shift-AND doubling
  const int len = 2 * radius + 1;
  u128 run = v;
  int have = 1;
  while (have * 2 <= len) { run &= shr128(run, have); have *= 2; }
  if (have < len) run &= shr128(run, len - have);
  store_row(hrun[r], shl128(run, radius));
  __syncthreads();
  u128 e = 0;
  if (r >= radius && r < kCrop - radius) {
    e = ~(u128)0;
    for (int d = -radius; d <= radius; ++d) e &= load_row(hrun[r + d]);
  }
  unsigned char* o = out + (size_t)b * kCrop * kCrop;
  store_row(w4, e);
  for (int c = 0; c < kCrop; ++c) o[r * kCrop + c] = (unsigned char)((w4[c >> 5] >> (c & 31)) & 1u);
}

int launch_erode(const unsigned char* in, unsigned char* out, int B, int kernel_size, int num_round, cudaStream_t stream) {
  if (B <= 0) return 0;
  const int radius = ((kernel_size - 1) / 2) * num_round;
  erode_kernel<<<B, kCrop, 0, stream>>>(in, out, B, radius);
  return (int)cudaGetLastError();
}

// center_field_to_anti_center_map: 5x5 cross-correlation, zero padding 2, fp64, divided by 24.
struct AntiFilt { double f[25]; };
__global__ void __launch_bounds__(256) anti_center_kernel(const float* __restrict__ vote, double* __restrict__ out, int B,
                                                          int H, int W, const AntiFilt filt) {
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (size_t)B * H * W) return;
  const int x = (int)(id % W), y = (int)((id / W) % H);
  const size_t b = id / ((size_t)H * W);
  const float* c0 = vote + (b * 2) * (size_t)H * W;
  const float* c1 = c0 + (size_t)H * W;
  double acc = 0.0;
#pragma unroll
  for (int di = 0; di < 5; ++di)
#pragma unroll
    for (int dj = 0; dj < 5; ++dj) {
      const int yy = y + di - 2, xx = x + dj - 2;
      if ((di == 2 && dj == 2) || yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
      acc = fma(filt.f[di * 5 + dj], (double)c0[(size_t)yy * W + xx], acc);
      acc = fma(filt.f[dj * 5 + di], (double)c1[(size_t)yy * W + xx], acc);
    }
  out[id] = __ddiv_rn(acc, 24.0);
}

int launch_anti_center(const float* vote, double* out, int B, int H, int W, const double* filt25, cudaStream_t stream) {
  const size_t total = (size_t)B * H * W;
  if (total == 0) return 0;
  AntiFilt f;
  for (int i = 0; i < 25; ++i) f.f[i] = filt25[i];
  anti_center_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(vote, out, B, H, W, f);
  return (int)cudaGetLastError();
}

// stand-alone separate_connected_components on [B,128,128] u8 masks: counts + raw slice boxes
struct CcSmem {
  uint32_t mask[kCrop][4];
  uint16_t lab[kCrop * kCrop];
  uint16_t rank[kCrop * kCrop];
  int scan[kCenterWarps];
  int box[4][kCcCap];
};
__global__ void __launch_bounds__(kCenterThreads) components_kernel(const unsigned char* __restrict__ masks, int B,
                                                                    int* __restrict__ counts, int* __restrict__ boxes) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CcSmem& sm = *reinterpret_cast<CcSmem*>(smem_raw);
  const int b = blockIdx.x, tid = threadIdx.x;
  const unsigned char* m = masks + (size_t)b * kCrop * kCrop;
  for (int w = tid; w < kCrop * 4; w += kCenterThreads) {
    uint32_t word = 0;
    for (int k = 0; k < 32; ++k) word |= (m[w * 32 + k] ? 1u : 0u) << k;
    sm.mask[w >> 2][w & 3] = word;
  }
  __syncthreads();
  const int n = label_components(sm.mask, sm.lab, sm.rank, sm.scan, sm.box);
  if (tid == 0) counts[b] = n;
  if (tid < min(n, kCcCap)) {
    int* o = boxes + ((size_t)b * kCcCap + tid) * 4;   // [x_start, y_start, x_stop, y_stop]
    o[0] = sm.box[0][tid]; o[1] = sm.box[1][tid]; o[2] = sm.box[2][tid] + 1; o[3] = sm.box[3][tid] + 1;
  }
}

int launch_components(const unsigned char* masks, int B, int* counts, int* boxes, cudaStream_t stream) {
  if (B <= 0) return 0;
  // function attributes are per device: set on every launch (microseconds), no cached state
  cudaError_t e = cudaFuncSetAttribute(components_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CcSmem));
  if (e != cudaSuccess) return (int)e;
  components_kernel<<<B, kCenterThreads, sizeof(CcSmem), stream>>>(masks, B, counts, boxes);
  return (int)cudaGetLastError();
}

int launch_center(const CenterParams& p, int num_sms, cudaStream_t stream) {
  if (p.tiles) return p.cc_counts ? launch_center_t<true, -1>(p, num_sms, stream) : launch_center_t<false, -1>(p, num_sms, stream);
  const bool spec = p.H * p.W == kSpecPlaneElems && p.ch_crow == p.ch_sdf + 1 && p.ch_ccol == p.ch_sdf + 2;
  if (p.cc_counts) return spec ? launch_center_t<true, kSpecPlaneElems>(p, num_sms, stream) : launch_center_t<true, 0>(p, num_sms, stream);
  // row skipping (the lattice pre-pass) pays on the loose proposals of the first pass — the one that asks for split boxes
  if (p.splits)
    return spec ? launch_center_t<false, kSpecPlaneElems, true>(p, num_sms, stream) : launch_center_t<false, 0, true>(p, num_sms, stream);
  return spec ? launch_center_t<false, kSpecPlaneElems>(p, num_sms, stream) : launch_center_t<false, 0>(p, num_sms, stream);
}

}  // namespace unmore
