// Bit-packed masks and mask-IoU NMS (north-star op (c); no reference counterpart — SURVEY.md
// §8a row C — the oracle is a dense greedy restatement with the order / tie-break of
// torchvision.ops.nms).
//
//   pack:   dense u8 [K, H, W] (non-zero = set) -> u32 [K, H, ceil(W/32)], LSB = lowest x
//   stats:  area (popcount) and tight box of every packed mask
//   nms:    stable descending rank sort -> 64-wide suppression bit-matrix with exact integer
//           IoU (popc(a & b) over the intersection of the tight boxes only, skipped when the
//           box-overlap / area bound already proves IoU <= thr) -> single-warp greedy scan
#include "unmore_internal.h"

namespace unmore {

// ---- pack --------------------------------------------------------------------------------
// 4 bytes -> 4 bits (byte != 0), 5 instructions: bit 7 of every byte := "byte is non-zero" (mask the top bits so the
// add cannot carry across bytes, add 0x7f, OR the original top bit back in), then one multiply gathers bits
// 7 / 15 / 23 / 31 into bits 28..31 (0x00204081 = 2^21 + 2^14 + 2^7 + 1; the ten partial-product bits land on distinct
// positions, so nothing carries).  The SIMD-video form (__vcmpne4 + four shift/mask pairs) is emulated on sm_100a and
// cost ~18 ALU instructions per word: the kernel sat on the ALU pipe (91%) at 0.66-0.81 of HBM (profiles/r01_pack_kernel.md);
// the multiply runs on the otherwise idle FMA pipe.
__device__ __forceinline__ uint32_t nz4(uint32_t w) {
  const uint32_t m = (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) & 0x80808080u;
  uint32_t g;
  asm("mul.lo.u32 %0, %1, 0x00204081;" : "=r"(g) : "r"(m));
  return g >> 28;
}

// fast path: W % 32 == 0.  A lane loads 16 pixels (one uint4), pairs of lanes form a word.  Persistent grid-stride loop:
// every thread keeps kPackUnroll independent 16-byte loads in flight and requests the NEXT batch before it packs the
// current one, so the HBM pipe never drains between batches and there is no per-CTA launch / drain overhead (the
// one-shot form reached 0.57 / 0.74 / 0.80 of the measured copy bandwidth at 1k / 4k / 16k masks; this form with 4
// resident CTAs per SM: 0.79 / 0.88 / 0.94, where a plain device copy of the same bytes reaches 0.84 / 0.96 / 0.99).
constexpr int kPackUnroll = 4;
constexpr int kPackCtasPerSm = 4;   // measured: 2 / 3 / 4 / 5 / 8 CTAs per SM -> 0.82 / 0.92 / 0.94 / 0.91 / 0.87 of the copy bandwidth at 16k masks
__global__ void __launch_bounds__(256) pack_kernel_vec(const uint4* __restrict__ in, uint32_t* __restrict__ out,
                                                       size_t n_vec) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;   // even: lane pairs stay together in every batch
  size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint4 v[kPackUnroll], nxt[kPackUnroll];
#pragma unroll
  for (int u = 0; u < kPackUnroll; ++u) {
    const size_t i = i0 + u * stride;
    v[u] = i < n_vec ? __ldcs(in + i) : make_uint4(0u, 0u, 0u, 0u);
  }
  for (; i0 < n_vec; i0 += kPackUnroll * stride) {
    const size_t j0 = i0 + kPackUnroll * stride;
#pragma unroll
    for (int u = 0; u < kPackUnroll; ++u) {
      const size_t i = j0 + u * stride;
      nxt[u] = i < n_vec ? __ldcs(in + i) : make_uint4(0u, 0u, 0u, 0u);
    }
#pragma unroll
    for (int u = 0; u < kPackUnroll; ++u) {
      const size_t i = i0 + u * stride;
      const uint32_t bits = nz4(v[u].x) | (nz4(v[u].y) << 4) | (nz4(v[u].z) << 8) | (nz4(v[u].w) << 12);
      const uint32_t hi = __shfl_down_sync(kFullMask, bits, 1);
      if (!(threadIdx.x & 1) && i < n_vec) __stcs(out + (i >> 1), bits | (hi << 16));
      v[u] = nxt[u];
    }
  }
}

__global__ void __launch_bounds__(256) pack_kernel_generic(const unsigned char* __restrict__ in,
                                                           uint32_t* __restrict__ out, size_t n_rows, int W, int Wp) {
  const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n_rows * Wp) return;
  const size_t r = q / Wp;
  const int wx = (int)(q - r * Wp);
  const unsigned char* p = in + r * W + (size_t)wx * 32;
  const int n = min(32, W - wx * 32);
  uint32_t word = 0;
  for (int b = 0; b < n; ++b) word |= (p[b] ? 1u : 0u) << b;
  out[q] = word;
}

int launch_mask_pack(const unsigned char* in, uint32_t* out, size_t n_masks, int H, int W, int num_sms, cudaStream_t stream) {
  if (n_masks == 0) return 0;
  const int Wp = (W + 31) >> 5;
  if ((W & 31) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
    const size_t n_vec = n_masks * H * (size_t)W / 16;
    const size_t per_block = 256 * (size_t)kPackUnroll;   // n_vec is even (W % 32 == 0), so lane pairs never straddle strides
    const size_t want = (n_vec + per_block - 1) / per_block;
    const size_t resident = (size_t)num_sms * kPackCtasPerSm;
    pack_kernel_vec<<<(unsigned)(want < resident ? want : resident), 256, 0, stream>>>(reinterpret_cast<const uint4*>(in), out, n_vec);
  } else {
    const size_t total = n_masks * H * (size_t)Wp;
    pack_kernel_generic<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(in, out, n_masks * (size_t)H, W, Wp);
  }
  return (int)cudaGetLastError();
}

// ---- stats -------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) mask_stats_kernel(const uint32_t* __restrict__ masks, int K, int H, int Wp,
                                                         int* __restrict__ areas, int4* __restrict__ tight) {
  __shared__ int s_area, s_x1, s_y1, s_x2, s_y2;
  const int k = blockIdx.x;
  if (threadIdx.x == 0) { s_area = 0; s_x1 = 1 << 30; s_y1 = 1 << 30; s_x2 = -1; s_y2 = -1; }
  __syncthreads();
  const uint32_t* m = masks + (size_t)k * H * Wp;
  int area = 0, x1 = 1 << 30, y1 = 1 << 30, x2 = -1, y2 = -1;
  for (int q = threadIdx.x; q < H * Wp; q += blockDim.x) {
    const uint32_t w = __ldg(m + q);
    if (w) {
      const int y = q / Wp, xb = (q - y * Wp) << 5;
      area += __popc(w);
      x1 = min(x1, xb + __ffs(w) - 1); x2 = max(x2, xb + 31 - __clz(w));
      y1 = min(y1, y); y2 = max(y2, y);
    }
  }
  area = warp_sum(area);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    x1 = min(x1, __shfl_xor_sync(kFullMask, x1, o)); y1 = min(y1, __shfl_xor_sync(kFullMask, y1, o));
    x2 = max(x2, __shfl_xor_sync(kFullMask, x2, o)); y2 = max(y2, __shfl_xor_sync(kFullMask, y2, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&s_area, area);
    atomicMin(&s_x1, x1); atomicMin(&s_y1, y1); atomicMax(&s_x2, x2); atomicMax(&s_y2, y2);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    areas[k] = s_area;
    tight[k] = s_area > 0 ? make_int4(s_x1, s_y1, s_x2 + 1, s_y2 + 1) : make_int4(0, 0, 0, 0);  // half-open
  }
}

// ---- stable descending rank sort ---------------------------------------------------------
__global__ void __launch_bounds__(256) rank_sort_kernel(const float* __restrict__ scores, int K, int* __restrict__ order) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= K) return;
  if (!scores) { order[i] = i; return; }
  const float si = scores[i];
  int rank = 0;
  for (int j = 0; j < K; ++j) {
    const float sj = __ldg(scores + j);
    rank += (sj > si || (sj == si && j < i)) ? 1 : 0;
  }
  order[rank] = i;
}

// ---- suppression bit-matrix --------------------------------------------------------------
// grid (cb, rb) with cb >= rb: one CTA owns the 64 x 64 tile of sorted rows rb*64.. against sorted
// columns cb*64...  matrix[r][cb] bit c  <=>  IoU(sorted r, sorted cb*64+c) > thr, c later than r.
//  1. one thread per pair: tight-box overlap and the area / overlap bound decide most pairs
//     without touching the masks (IoU is monotone in the intersection, so if even
//     min(area_i, area_j, box overlap) cannot exceed thr the pair is clean);
//  2. the undecided pairs are queued in shared memory and the 8 warps drain the queue, each
//     pair's popc(a & b) over the intersection window spread across the 32 lanes — a pair costs
//     (rows x words) / 32 steps instead of serialising in one thread next to idle neighbours.
constexpr int kIouThreads = 256;

__global__ void __launch_bounds__(kIouThreads) mask_iou_matrix_kernel(const uint32_t* __restrict__ masks, int K, int H, int Wp,
                                                                      const int* __restrict__ order, const int* __restrict__ areas,
                                                                      const int4* __restrict__ tight, float thr,
                                                                      unsigned long long* __restrict__ matrix) {
  const int rb = blockIdx.y, cb = blockIdx.x;
  if (cb < rb) return;
  __shared__ int r_idx[64], r_area[64], c_idx[64], c_area[64];
  __shared__ int4 r_box[64], c_box[64];
  __shared__ unsigned long long bits[64];
  __shared__ unsigned short queue[64 * 64];
  __shared__ int n_queue;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int rows = min(64, K - rb * 64), cols = min(64, K - cb * 64);
  if (tid < 64) {
    bits[tid] = 0ull;
    if (tid < rows) { const int i = order[rb * 64 + tid]; r_idx[tid] = i; r_area[tid] = areas[i]; r_box[tid] = tight[i]; }
    if (tid < cols) { const int j = order[cb * 64 + tid]; c_idx[tid] = j; c_area[tid] = areas[j]; c_box[tid] = tight[j]; }
  }
  if (tid == 0) n_queue = 0;
  __syncthreads();
  for (int q = tid; q < 64 * 64; q += kIouThreads) {
    const int r = q >> 6, c = q & 63;
    if (r >= rows || c >= cols || (rb == cb && c <= r)) continue;
    const int4 bi = r_box[r], bj = c_box[c];
    const int ix1 = max(bi.x, bj.x), iy1 = max(bi.y, bj.y), ix2 = min(bi.z, bj.z), iy2 = min(bi.w, bj.w);
    if (ix2 <= ix1 || iy2 <= iy1) continue;
    const int ai = r_area[r], aj = c_area[c];
    const int ub = min(min(ai, aj), (ix2 - ix1) * (iy2 - iy1));
    if (!(__fdiv_rn((float)ub, (float)(ai + aj - ub)) > thr)) continue;
    queue[atomicAdd(&n_queue, 1)] = (unsigned short)q;
  }
  __syncthreads();
  const int nq = n_queue;
  for (int e = warp; e < nq; e += kIouThreads / 32) {
    const int q = queue[e], r = q >> 6, c = q & 63;
    const int4 bi = r_box[r], bj = c_box[c];
    const int ix1 = max(bi.x, bj.x), iy1 = max(bi.y, bj.y), ix2 = min(bi.z, bj.z), iy2 = min(bi.w, bj.w);
    const int w1 = ix1 >> 5, nw = ((ix2 + 31) >> 5) - w1, nwin = nw * (iy2 - iy1);
    const uint32_t* mi = masks + (size_t)r_idx[r] * H * Wp + (size_t)iy1 * Wp + w1;
    const uint32_t* mj = masks + (size_t)c_idx[c] * H * Wp + (size_t)iy1 * Wp + w1;
    int inter = 0;
    for (int t = lane; t < nwin; t += 32) {
      const int y = t / nw, w = t - y * nw;
      inter += __popc(__ldg(mi + (size_t)y * Wp + w) & __ldg(mj + (size_t)y * Wp + w));
    }
    inter = warp_sum(inter);
    if (lane == 0 && __fdiv_rn((float)inter, (float)(r_area[r] + c_area[c] - inter)) > thr)
      atomicOr(&bits[r], 1ull << c);
  }
  __syncthreads();
  const int nblk = (K + 63) >> 6;
  if (tid < rows) matrix[(size_t)(rb * 64 + tid) * nblk + cb] = bits[tid];
}

// Box-IoU variant of the matrix (torchvision arithmetic), for large-K box NMS.
__global__ void __launch_bounds__(64) box_iou_matrix_kernel(const float4* __restrict__ boxes, int K,
                                                            const int* __restrict__ order, float thr,
                                                            unsigned long long* __restrict__ matrix) {
  const int rb = blockIdx.y, cb = blockIdx.x;
  if (cb < rb) return;
  __shared__ float4 s_box[64];
  const int cols = min(64, K - cb * 64);
  if ((int)threadIdx.x < cols) s_box[threadIdx.x] = boxes[order[cb * 64 + threadIdx.x]];
  __syncthreads();
  const int r = rb * 64 + threadIdx.x;
  if (r >= K) return;
  const float4 bi = boxes[order[r]];
  const float iarea = __fmul_rn(__fsub_rn(bi.z, bi.x), __fsub_rn(bi.w, bi.y));
  const int nblk = (K + 63) >> 6;
  unsigned long long bits = 0ull;
  const int c0 = (rb == cb) ? (int)threadIdx.x + 1 : 0;
  for (int c = c0; c < cols; ++c) {
    const float4 bj = s_box[c];
    const float xx1 = fmaxf(bi.x, bj.x), yy1 = fmaxf(bi.y, bj.y), xx2 = fminf(bi.z, bj.z), yy2 = fminf(bi.w, bj.w);
    const float w = fmaxf(0.f, __fsub_rn(xx2, xx1)), h = fmaxf(0.f, __fsub_rn(yy2, yy1));
    const float inter = __fmul_rn(w, h);
    const float jarea = __fmul_rn(__fsub_rn(bj.z, bj.x), __fsub_rn(bj.w, bj.y));
    if (__fdiv_rn(inter, __fsub_rn(__fadd_rn(iarea, jarea), inter)) > thr) bits |= 1ull << c;
  }
  matrix[(size_t)r * nblk + cb] = bits;
}

// ---- greedy scan over the matrix (one warp) -----------------------------------------------
__global__ void __launch_bounds__(32) greedy_scan_kernel(const unsigned long long* __restrict__ matrix, int K,
                                                         const int* __restrict__ order, int* __restrict__ keep,
                                                         int* __restrict__ keep_count) {
  extern __shared__ unsigned long long removed[];  // ceil(K/64) words
  const int nblk = (K + 63) >> 6;
  const int lane = threadIdx.x;
  for (int w = lane; w < nblk; w += 32) removed[w] = 0ull;
  __syncwarp();
  int nk = 0;
  for (int i = 0; i < K; ++i) {
    if ((removed[i >> 6] >> (i & 63)) & 1ull) continue;  // uniform
    if (lane == 0) keep[nk] = order[i];
    ++nk;
    const unsigned long long* row = matrix + (size_t)i * nblk;
    for (int w = (i >> 6) + lane; w < nblk; w += 32) removed[w] |= row[w];
    __syncwarp();
  }
  if (lane == 0) *keep_count = nk;
}

// ---- COCO run-length counts (pycocotools maskApi.c rleEncode semantics) ----------------------
// Column-major scan (t = x*H + y); counts[0] is the length of the leading run of zeros (possibly 0),
// then alternating one / zero runs.  n_runs_out reports the true number of runs even when it exceeds
// max_runs (then nothing is written for that mask and the caller falls back to a larger buffer).
//
// One CTA per mask, word-parallel: the bit-packed rows are staged in shared memory (coalesced, odd row
// stride), transposed in 32x32 bit blocks with warp ballots into column-major words T[x][j] (bit b = row
// 32j + b of column x), and the run boundaries are the set bits of T ^ (T << 1 | last bit of the previous
// word of the column-major stream).  Each thread owns a contiguous range of stream words: a block scan of
// the change counts and of the last change position gives every thread its output slot and the position
// its first run starts from; the counts are then written straight to global memory.  ~30 k warp
// instructions per 480x640 mask; the bit-serial form below (one divide + one load per bit, twice) needs
// ~290 k and is kept for masks whose two shared arrays do not fit.
constexpr int kRleThreads = 256;
constexpr int kRleMaxRuns = 8192;   // bit-serial fallback only: change positions staged in 32 KB of shared memory
constexpr int kRleMaxDynSmem = 200 * 1024;

// STAGE_ROWS = false: the rows are read from global memory by the transpose itself (strided, one sector per lane) —
// for masks whose rows + transposed words do not fit the shared memory together (1024x1024: 135 + 131 KB)
template <bool STAGE_ROWS>
__global__ void __launch_bounds__(kRleThreads) rle_counts_kernel(const uint32_t* __restrict__ masks, int K, int H, int W,
                                                                  int Wp, int max_runs, uint32_t* __restrict__ counts,
                                                                  int* __restrict__ n_runs) {
  extern __shared__ uint32_t rle_smem[];
  __shared__ int wsum[kRleThreads / 32], wlast[kRleThreads / 32];
  const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Hw = (H + 31) >> 5, stride = Wp | 1;
  uint32_t* rows = rle_smem;                                            // [H][stride]
  uint32_t* T = rle_smem + (STAGE_ROWS ? (size_t)H * stride : 0);       // [W][Hw]
  const uint32_t* m = masks + (size_t)k * H * Wp;
  if constexpr (STAGE_ROWS) {
    for (int idx = tid; idx < H * Wp; idx += kRleThreads) {
      const int y = idx / Wp, w = idx - y * Wp;
      rows[y * stride + w] = __ldg(m + idx);
    }
    __syncthreads();
  }
  for (int q = warp; q < Hw * Wp; q += kRleThreads / 32) {   // 32 rows x 32 columns per step
    const int j = q / Wp, w = q - j * Wp, y = 32 * j + lane;
    const uint32_t word = y < H ? (STAGE_ROWS ? rows[y * stride + w] : __ldg(m + (size_t)y * Wp + w)) : 0u;
    uint32_t mine = 0;
#pragma unroll
    for (int b = 0; b < 32; ++b) {
      const uint32_t bal = __ballot_sync(kFullMask, (word >> b) & 1u);
      if (lane == b) mine = bal;
    }
    const int x = 32 * w + lane;
    if (x < W) T[x * Hw + j] = mine;
  }
  __syncthreads();
  const int G = W * Hw, N = H * W;
  const int per = (G + kRleThreads - 1) / kRleThreads;
  const int g0 = min(tid * per, G), g1 = min(g0 + per, G);
  const uint32_t tail_mask = (H & 31) ? ((1u << (H & 31)) - 1u) : ~0u;   // valid rows of the last word of a column
  // boundaries inside stream word g = (x, j): bit b set <=> pixel (x, 32j + b) differs from its predecessor in the scan
  auto changes = [&](int g, int x, int j) -> uint32_t {
    const uint32_t t = T[g];
    uint32_t carry;
    if (j > 0) carry = T[g - 1] >> 31;
    else carry = x > 0 ? (T[g - 1] >> ((H - 1) & 31)) & 1u : 0u;     // last row of the previous column; 0 before t = 0
    return (t ^ ((t << 1) | carry)) & (j == Hw - 1 ? tail_mask : ~0u);
  };
  int mine = 0, last = -1;
  {
    int x = g0 / Hw, j = g0 - x * Hw;
    for (int g = g0; g < g1; ++g) {
      const uint32_t c = changes(g, x, j);
      if (c) { mine += __popc(c); last = x * H + 32 * j + (31 - __clz(c)); }
      if (++j == Hw) { j = 0; ++x; }
    }
  }
  int incl = mine, lmax = last;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(kFullMask, incl, o);
    const int z = __shfl_up_sync(kFullMask, lmax, o);
    if (lane >= o) { incl += y; lmax = max(lmax, z); }
  }
  int prev = __shfl_up_sync(kFullMask, lmax, 1);   // last change before this thread inside the warp
  if (lane == 0) prev = -1;
  if (lane == 31) { wsum[warp] = incl; wlast[warp] = lmax; }
  __syncthreads();
  int base = 0, total = 0, glast = -1;
  for (int w = 0; w < kRleThreads / 32; ++w) {
    if (w < warp) { base += wsum[w]; prev = max(prev, wlast[w]); }
    total += wsum[w];
    glast = max(glast, wlast[w]);
  }
  const int runs = total + 1;
  if (tid == 0) n_runs[k] = runs;
  if (runs > max_runs) return;   // uniform
  uint32_t* out = counts + (size_t)k * max_runs;
  int r = base + incl - mine;
  int pp = prev < 0 ? 0 : prev;   // the first run starts at t = 0
  {
    int x = g0 / Hw, j = g0 - x * Hw;
    for (int g = g0; g < g1; ++g) {
      uint32_t c = changes(g, x, j);
      while (c) {
        const int t = x * H + 32 * j + __ffs((int)c) - 1;
        c &= c - 1;
        out[r++] = (uint32_t)(t - pp);
        pp = t;
      }
      if (++j == Hw) { j = 0; ++x; }
    }
  }
  if (tid == 0) out[total] = (uint32_t)(N - (glast < 0 ? 0 : glast));
}

// bit-serial form: each thread scans a contiguous range of t, change positions are ranked with a block scan and
// staged in shared memory, counts are their differences
__global__ void __launch_bounds__(kRleThreads) rle_counts_kernel_serial(const uint32_t* __restrict__ masks, int K, int H, int W,
                                                                         int Wp, int max_runs, uint32_t* __restrict__ counts,
                                                                         int* __restrict__ n_runs) {
  __shared__ uint32_t pos[kRleMaxRuns];
  __shared__ int wsum[kRleThreads / 32];
  const int k = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t* m = masks + (size_t)k * H * Wp;
  const int N = H * W;
  const int per = (N + kRleThreads - 1) / kRleThreads;
  const int t0 = min(tid * per, N), t1 = min(t0 + per, N);
  auto bit = [&](int t) -> uint32_t {
    const int x = t / H, y = t - x * H;
    return (__ldg(m + (size_t)y * Wp + (x >> 5)) >> (x & 31)) & 1u;
  };
  // pass 1: count the changes in [t0, t1)
  uint32_t prev = t0 > 0 ? bit(t0 - 1) : 0u;
  int mine = 0;
  {
    uint32_t p = prev;
    for (int t = t0; t < t1; ++t) { const uint32_t b = bit(t); mine += (b != p); p = b; }
  }
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(kFullMask, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  int base = 0, total = 0;
  for (int w = 0; w < kRleThreads / 32; ++w) { if (w < warp) base += wsum[w]; total += wsum[w]; }
  const int runs = total + 1;
  if (tid == 0) n_runs[k] = runs;
  if (runs > max_runs || total > kRleMaxRuns) return;   // uniform
  // pass 2: record the change positions
  int r = base + incl - mine;
  {
    uint32_t p = prev;
    for (int t = t0; t < t1; ++t) { const uint32_t b = bit(t); if (b != p) pos[r++] = (uint32_t)t; p = b; }
  }
  __syncthreads();
  uint32_t* out = counts + (size_t)k * max_runs;
  for (int j = tid; j < runs; j += kRleThreads) {
    const uint32_t lo = j == 0 ? 0u : pos[j - 1];
    const uint32_t hi = j == total ? (uint32_t)N : pos[j];
    out[j] = hi - lo;
  }
}

int launch_rle_counts(const uint32_t* masks, int K, int H, int W, int max_runs, uint32_t* counts, int* n_runs,
                      cudaStream_t stream) {
  if (K <= 0) return 0;
  const int Wp = (W + 31) >> 5, Hw = (H + 31) >> 5;
  const size_t smem_t = (size_t)W * Hw * sizeof(uint32_t), smem = smem_t + (size_t)H * (Wp | 1) * sizeof(uint32_t);
  // function attributes are per device: set on every launch (microseconds), no cached state
  if (smem <= (size_t)kRleMaxDynSmem) {
    cudaError_t e = cudaFuncSetAttribute(rle_counts_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    rle_counts_kernel<true><<<K, kRleThreads, smem, stream>>>(masks, K, H, W, Wp, max_runs, counts, n_runs);
    return (int)cudaGetLastError();
  }
  if (smem_t <= (size_t)kRleMaxDynSmem) {
    cudaError_t e = cudaFuncSetAttribute(rle_counts_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_t);
    if (e != cudaSuccess) return (int)e;
    rle_counts_kernel<false><<<K, kRleThreads, smem_t, stream>>>(masks, K, H, W, Wp, max_runs, counts, n_runs);
    return (int)cudaGetLastError();
  }
  rle_counts_kernel_serial<<<K, kRleThreads, 0, stream>>>(masks, K, H, W, Wp, max_runs, counts, n_runs);
  return (int)cudaGetLastError();
}

int launch_mask_stats(const uint32_t* masks, int K, int H, int Wp, int* areas, int4* tight, cudaStream_t stream) {
  if (K <= 0) return 0;
  mask_stats_kernel<<<K, 256, 0, stream>>>(masks, K, H, Wp, areas, tight);
  return (int)cudaGetLastError();
}

int launch_matrix_nms(const uint32_t* masks, const float4* boxes, int K, int H, int Wp, const float* scores,
                      const int* areas, const int4* tight, float thr, int* order, unsigned long long* matrix,
                      int* keep, int* keep_count, cudaStream_t stream) {
  if (K <= 0) return (int)cudaMemsetAsync(keep_count, 0, sizeof(int), stream);
  rank_sort_kernel<<<(K + 255) / 256, 256, 0, stream>>>(scores, K, order);
  const int nblk = (K + 63) >> 6;
  dim3 grid(nblk, nblk);
  if (masks) mask_iou_matrix_kernel<<<grid, kIouThreads, 0, stream>>>(masks, K, H, Wp, order, areas, tight, thr, matrix);
  else box_iou_matrix_kernel<<<grid, 64, 0, stream>>>(boxes, K, order, thr, matrix);
  greedy_scan_kernel<<<1, 32, nblk * sizeof(unsigned long long), stream>>>(matrix, K, order, keep, keep_count);
  return (int)cudaGetLastError();
}

}  // namespace unmore
