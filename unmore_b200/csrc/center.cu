// center_reasoning (object_reasoning.py:525-580, analyze_cc off): per proposal, resample the
// boundary-distance and the two center-field channels to 128x128, threshold them into a
// union mask (sigmoid(sdf) > 0.5  OR  ||center|| > 0.5), erode it 3 x (9x9, zero border)
// (utils/misc.py:10-20), evaluate the anti-center map (5x5 fp64 correlation, :360-377) on the
// surviving pixels, and either pass the proposal (max <= thr) or split it at the arg-max.
//
// One CTA (256 threads, two CTAs per SM) per proposal.  The mask lives as 128-bit rows; three 9x9 zero-border
// erosions compose to a single 25x25 zero-border erosion, done with shift-AND doubling on
// the packed rows and a 25-row AND.  Everything within 12 px of the crop border is eroded
// away, which subsumes the reference's 10-px frame zeroing (:535-538), so only the central
// 108x108 window of the center field (rows/cols 10..117) is ever read by the correlation:
// that window is what is staged in shared memory (93,312 B, channels interleaved -> two CTAs per SM).
#include "resample.cuh"
#include "unmore_internal.h"

namespace unmore {

constexpr int kCenterThreads = 256;
constexpr int kCenterWarps = kCenterThreads / 32;
constexpr int kWinLo = 10, kWinHi = 118, kWin = kWinHi - kWinLo;  // staged window of the center field
constexpr int kWinStride = 110;   // pixels per staged row: 880 B, so 8 lanes on consecutive rows hit 8 distinct 16-B bank groups
constexpr int kErode = 12;                                         // 3 rounds x radius 4
constexpr int kCandCap = 1024;                                     // queue of pixels for the exact fp64 pass

struct CenterSmem {
  float2 c[kWin * kWinStride];     // staged center field, (row, col) channels interleaved: one aligned pair per pixel
  uint32_t mask[kCrop][4];   // union mask, bit j of row i = column j (LSB = lowest column)
  uint32_t hrun[kCrop][4];   // horizontally eroded rows
  uint32_t ero[kCrop][4];    // fully eroded mask
  double red_val[kCenterWarps];
  int red_idx[kCenterWarps];
  float red_f[kCenterWarps];
  float red_m[kCenterWarps];
  int bcast_i[2];
  int cc_scan[kCenterWarps];
  int cand_n;                // candidate pixels of the exact pass (b1 -> b2)
  uint16_t cand[kCandCap];
  int cc_box[4][kCcCap];   // x_min, y_min, x_max, y_max per component (first kCcCap components)
};

typedef unsigned __int128 u128;

__device__ __forceinline__ u128 load_row(const uint32_t r[4]) {
  return ((u128)r[3] << 96) | ((u128)r[2] << 64) | ((u128)r[1] << 32) | (u128)r[0];
}
__device__ __forceinline__ void store_row(uint32_t r[4], u128 v) {
  r[0] = (uint32_t)v; r[1] = (uint32_t)(v >> 32); r[2] = (uint32_t)(v >> 64); r[3] = (uint32_t)(v >> 96);
}

// 8-connected components of a 128x128 bit mask (scipy.ndimage.label with a 3x3 structure, as
// separate_connected_components object_reasoning.py:207-256 calls it).  Labels are the smallest flat
// index of the component (min-propagation over the 8-neighbourhood + pointer jumping), so ranking
// the roots in raster order reproduces scipy's numbering.  All kCenterThreads threads must call.
// lab / rank: 16384 x u16 scratch each.  Returns the component count; box[0..3][k] receives
// x_min, y_min, x_max, y_max of the first kCcCap components (when there are >= 1).
__device__ int label_components(const uint32_t (*mask)[4], uint16_t* lab, uint16_t* rank, int* scan,
                                int (*box)[kCcCap]) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kPix = kCrop * kCrop, kPer = (kPix + kCenterThreads - 1) / kCenterThreads;
  auto bit = [&](int q) { return (mask[q >> 7][(q >> 5) & 3] >> (q & 31)) & 1u; };
  for (int q = tid; q < kPix; q += kCenterThreads) lab[q] = bit(q) ? (uint16_t)q : (uint16_t)0xFFFF;
  __syncthreads();
  for (;;) {
    int changed = 0;
    for (int q = tid; q < kPix; q += kCenterThreads) {
      const uint16_t l = lab[q];
      if (l == 0xFFFF) continue;
      const int r = q >> 7, c = q & 127;
      uint16_t m = l;
#pragma unroll
      for (int dr = -1; dr <= 1; ++dr) {
        const int rr = r + dr;
        if (rr < 0 || rr >= kCrop) continue;
#pragma unroll
        for (int dc = -1; dc <= 1; ++dc) {
          const int cc = c + dc;
          if (cc < 0 || cc >= kCrop) continue;
          const uint16_t o = lab[rr * kCrop + cc];
          m = o < m ? o : m;            // 0xFFFF (background) never wins
        }
      }
      if (m < l) { lab[q] = m; changed = 1; }
    }
    __syncthreads();
    for (int q = tid; q < kPix; q += kCenterThreads) {   // pointer jumping to the current root
      uint16_t l = lab[q];
      if (l == 0xFFFF) continue;
      uint16_t ll = lab[l];
      while (ll < l) { l = ll; ll = lab[l]; }
      lab[q] = l;
    }
    if (!__syncthreads_or(changed)) break;
  }
  // rank the roots in raster order: thread t owns pixels [t*kPer, (t+1)*kPer)
  int mine = 0;
  for (int q = tid * kPer; q < min((tid + 1) * kPer, kPix); ++q) mine += (lab[q] == (uint16_t)q) ? 1 : 0;
  int incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(kFullMask, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) scan[warp] = incl;
  if (tid < 4 * kCcCap) box[tid / kCcCap][tid % kCcCap] = (tid / kCcCap < 2) ? (1 << 30) : -1;
  __syncthreads();
  int base = 0, total = 0;
  for (int w = 0; w < kCenterWarps; ++w) { if (w < warp) base += scan[w]; total += scan[w]; }
  int rk = base + incl - mine;
  for (int q = tid * kPer; q < min((tid + 1) * kPer, kPix); ++q)
    if (lab[q] == (uint16_t)q) rank[q] = (uint16_t)min(rk++, 0xFFFF);
  __syncthreads();
  for (int q = tid; q < kPix; q += kCenterThreads) {
    const uint16_t l = lab[q];
    if (l == 0xFFFF) continue;
    const int k2 = rank[l];
    if (k2 >= kCcCap) continue;
    atomicMin(&box[0][k2], q & 127); atomicMin(&box[1][k2], q >> 7);
    atomicMax(&box[2][k2], q & 127); atomicMax(&box[3][k2], q >> 7);
  }
  __syncthreads();
  return total;
}

// Row source of stage 1: the boundary-distance plane with the lane's columns paired (like PlaneRows) and the
// two center-field planes paired PER COLUMN, (row, col) in one 64-bit register pair.  The packed lerps then
// produce exactly the (c_row, c_col) pairs the staging store, the squared norm and the strip correlation
// want, with no re-pairing moves.  Arithmetic per element is the same ATen bilinear as everywhere else.
template <int PLANE_ELEMS>
struct CenterRows {
  const float* origin[3];
  int stride;
  int cy0, cy1;
  f32x2 sa[2], sb[2];   // sdf: rows i0 / i1, element h = columns 2h, 2h+1 of the lane
  f32x2 ca[4], cb[4];   // center field: rows i0 / i1, element c = (row, col) channels of column c

  __device__ __forceinline__ void init(const float* const planes[3], int W, const Window& win) {
#pragma unroll
    for (int p = 0; p < 3; ++p) origin[p] = planes[p] + (size_t)win.y1 * W + win.x1;
    stride = W;
    cy0 = cy1 = -1;
  }
  // the 24 taps of one source row (3 planes x 4 columns x left / right) ...
  __device__ __forceinline__ void load_taps(const ColTaps& t, int y, float v0[3][4], float v1[3][4]) const {
    const int ro = y * stride;
    if constexpr (PLANE_ELEMS > 0) {
      const float* rowp = elem_ptr(origin[0], ro);   // warp-uniform
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float* a0 = byte_ptr(rowp, t.x0[c]);
        const float* a1 = byte_ptr(rowp, t.x1[c]);
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          v0[p][c] = __ldg(a0 + p * PLANE_ELEMS);
          v1[p][c] = __ldg(a1 + p * PLANE_ELEMS);
        }
      }
    } else {
#pragma unroll
      for (int p = 0; p < 3; ++p) {
        const float* rowp = elem_ptr(origin[p], ro);   // warp-uniform
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            v0[p][c] = __ldg(byte_ptr(rowp, t.x0[c]));
          v1[p][c] = __ldg(byte_ptr(rowp, t.x1[c]));
        }
      }
    }
  }
  // ... and their horizontal interpolation
  __device__ __forceinline__ void lerp_taps(const ColTaps& t, const float v0[3][4], const float v1[3][4], f32x2 s[2], f32x2 cc[4]) const {
    float w0[4], w1[4];
    upk2(t.w0[0], w0[0], w0[1]); upk2(t.w0[1], w0[2], w0[3]);
    upk2(t.w1[0], w1[0], w1[1]); upk2(t.w1[1], w1[2], w1[3]);
#pragma unroll
    for (int h = 0; h < 2; ++h)
      s[h] = lerp_h2(pk2(v0[0][2 * h], v0[0][2 * h + 1]), pk2(v1[0][2 * h], v1[0][2 * h + 1]), t.w0[h], t.w1[h]);
#pragma unroll
    for (int c = 0; c < 4; ++c)
      cc[c] = lerp_h2(pk2(v0[1][c], v0[2][c]), pk2(v1[1][c], v1[2][c]), pk2(w0[c], w0[c]), pk2(w1[c], w1[c]));
  }
  __device__ __forceinline__ void hrows(const ColTaps& t, int y, f32x2 s[2], f32x2 cc[4]) const {
    float v0[3][4], v1[3][4];
    load_taps(t, y, v0, v1);
    lerp_taps(t, v0, v1, s, cc);
  }
  // s[c] = sdf of column lane + 32c; ab[c] = (c_row, c_col) of that column
  __device__ __forceinline__ void row(const ColTaps& t, const AxisTap& v, float s[4], f32x2 ab[4]) {
    if (v.i0 != cy0 || v.i1 != cy1) {          // warp-uniform
      if (v.i0 == cy1) {
        sa[0] = sb[0]; sa[1] = sb[1];
#pragma unroll
        for (int c = 0; c < 4; ++c) ca[c] = cb[c];
      } else {
        hrows(t, v.i0, sa, ca);
      }
      if (v.i1 == v.i0) {
        sb[0] = sa[0]; sb[1] = sa[1];
#pragma unroll
        for (int c = 0; c < 4; ++c) cb[c] = ca[c];
      } else {
        hrows(t, v.i1, sb, cb);
      }
      cy0 = v.i0; cy1 = v.i1;
    }
    upk2(lerp_v2(sa[0], sb[0], v.l0, v.l1), s[0], s[1]);
    upk2(lerp_v2(sa[1], sb[1], v.l0, v.l1), s[2], s[3]);
#pragma unroll
    for (int c = 0; c < 4; ++c) ab[c] = lerp_v2(ca[c], cb[c], v.l0, v.l1);
  }
};

// Row source over PRE-RESAMPLED tiles (PLANE_ELEMS = -1): [3, 128, 128] per proposal = (sdf, center_row, center_col),
// e.g. from unmore_crop_resize_aa — the tile path of the second resize mode.  Same output contract as CenterRows::row.
struct CenterTileRows {
  const float* tile;
  __device__ __forceinline__ void row(int lane, int i, float s[4], f32x2 ab[4]) const {
    const float* r = tile + i * kCrop + lane;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      s[c] = __ldg(r + 32 * c);
      ab[c] = pk2(__ldg(r + kCrop * kCrop + 32 * c), __ldg(r + 2 * kCrop * kCrop + 32 * c));
    }
  }
};

// PLANE_ELEMS: 0 = any field size / channel order; H*W = the three channels are consecutive planes of a field
// of exactly that size (the COCO-val shape the batch path runs on), see MultiPlaneRows.
// SIZED: a padded stack, p.image_hw holds each image's (h, w) inside the (H, W) pitch.  The window snap and the
// --analyze_cc clip use the image's extent; plane addressing and PLANE_ELEMS go by the pitch.
constexpr int kSpecPlaneElems = 480 * 640;
template <bool ANALYZE_CC, int PLANE_ELEMS, bool ROW_SKIP, bool SIZED = false>
__global__ void __launch_bounds__(kCenterThreads, 2) center_kernel(const CenterParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  CenterSmem& sm = *reinterpret_cast<CenterSmem*>(smem_raw);
  // Work items are fetched one proposal ahead by thread 0: the id is requested at the top of a proposal, the
  // owner image is located after stage 1 (the atomic has long returned), the box is copied into shared memory
  // by cp.async (no registers, nothing waits on it) and everything is published by the barrier that ends the
  // proposal — so a new proposal starts from shared memory instead of a chain of dependent global accesses.
  struct WorkItem { int id, img, k, pad; double box[4]; };
  __shared__ __align__(16) WorkItem s_item[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int total = worklist_total(p.work);
  auto fetch_box = [&](int slot, int fimg, int fk) {   // thread 0 only
    const size_t frow = (size_t)fimg * p.work.cap + fk;
    const unsigned dst = smem_addr(&s_item[slot].box[0]);
    if (p.boxes_f64) {
      const char* src = reinterpret_cast<const char*>(p.boxes) + frow * 32;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + 16), "l"(src + 16) : "memory");
    } else {
      const char* src = reinterpret_cast<const char*>(p.boxes) + frow * 16;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    }
  };
  if (tid == 0) {
    const int id0 = atomicAdd(p.work.counter, 1);
    int img0 = 0, k0 = 0;
    if (id0 < total) {
      worklist_locate(p.work, id0, img0, k0);
      fetch_box(0, img0, k0);
    }
    s_item[0].id = id0; s_item[0].img = img0; s_item[0].k = k0;
    asm volatile("cp.async.wait_all;" ::: "memory");
  }
  __syncthreads();
  for (int it = 0;; ++it) {
    const int cur = it & 1;
    const int id = s_item[cur].id;
    if (id >= total) break;
    const int img = s_item[cur].img, k = s_item[cur].k;
    const size_t row = (size_t)img * p.work.cap + k;
    double x1, y1, x2, y2;
    if (p.boxes_f64) {
      x1 = s_item[cur].box[0]; y1 = s_item[cur].box[1]; x2 = s_item[cur].box[2]; y2 = s_item[cur].box[3];
    } else {
      const float* bf = reinterpret_cast<const float*>(&s_item[cur].box[0]);
      x1 = bf[0]; y1 = bf[1]; x2 = bf[2]; y2 = bf[3];
    }
    int next_id = total, next_img = img, next_k = 0;
    if (tid == 0) next_id = atomicAdd(p.work.counter, 1);
    bool next_located = false;
    auto locate_next = [&]() {   // thread 0, once per proposal, well after the atomic was issued
      if (tid == 0 && !next_located) {
        if (next_id < total) {
          worklist_locate(p.work, next_id, next_img, next_k);
          fetch_box(cur ^ 1, next_img, next_k);
        }
        next_located = true;
      }
    };
    Window win;
    if constexpr (SIZED) {
      const int2 e = image_extent(p.image_hw, img, p.H, p.W);
      win = snap_window<double>(x1, y1, x2, y2, e.y, e.x);
    } else {
      win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
    }
    double best = 0.0;
    int best_idx = -1;
    if (!win.empty()) {
      // ---- 1. resample 3 channels; warp w owns kRowsPerWarp consecutive output rows
      ColTaps taps;
      taps.init<kStrided>(lane, win.w());
      const size_t plane_sz = (size_t)p.H * p.W;
      const float* base = p.fields + (size_t)img * p.C * plane_sz;
      const float* const planes[3] = {base + p.ch_sdf * plane_sz, base + p.ch_crow * plane_sz,
                                      base + p.ch_ccol * plane_sz};
      CenterRows<(PLANE_ELEMS > 0 ? PLANE_ELEMS : 0)> rows;
      CenterTileRows trows{PLANE_ELEMS < 0 ? p.tiles + row * (size_t)(3 * kCrop * kCrop) : nullptr};
      if constexpr (PLANE_ELEMS >= 0) rows.init(planes, p.W, win);
      const float scale_y = __fdiv_rn((float)win.h(), (float)kCrop);
      const int in_h = win.h();
      float cabs = 0.f;  // max |center field| over the tile (>= the staged window's): scales the fp32 screening margin
      // staging predicates of this lane's four columns lane + 32c: columns 32..95 are always inside the window
      const bool col_in[4] = {lane >= kWinLo, true, true, lane + 96 < kWinHi};   // [1], [2] unused: always inside
      // Rows are resampled in two phases (kLattice).  Phase 0: the eight LATTICE rows 8, 24, ..., 120, one per warp.
      // A pixel survives the 25x25 erosion only if every row within 12 of it carries a run of 25 set columns
      // around it, and every window of 25 rows contains a lattice row: a lattice row WITHOUT any such run rules out
      // all survivors within 12 rows of it.  That leaves a row range [rmin, rmax] that can hold survivors (often
      // none: the proposal passes with max 0), and only rows rmin-12 .. rmax+12 are resampled in phase 1 — the
      // erosion of [rmin, rmax] reads nothing else, and the correlation reads the staged field within 2 rows of a
      // survivor.  Exact: every value that is computed is computed by the same arithmetic, the rest is never read.
      // --analyze_cc needs the whole union mask (components of passing proposals) and keeps the single full pass;
      // so does the second pass over the split halves (launch_center): they are cut through their object, few of
      // their rows can be skipped and the extra phase costs more than it saves there (+5% measured).
      constexpr bool kLattice = ROW_SKIP && !ANALYZE_CC && PLANE_ELEMS >= 0;
      constexpr int kLatFirst = 8, kLatStride = 16, kLatRows = kCrop / kLatStride;
      constexpr int kRowsPerWarp = (kCrop + kCenterWarps - 1) / kCenterWarps;
      int i_begin, i_end, i_step;
      if constexpr (kLattice) { i_begin = kLatFirst + kLatStride * warp; i_end = kCrop; i_step = kLatStride * kCenterWarps; }
      else { i_begin = warp * kRowsPerWarp; i_end = min(kCrop, i_begin + kRowsPerWarp); i_step = 1; }
      int rmin = kErode, rmax = kCrop - kErode - 1;   // rows that can hold survivors
      bool no_survivors = false;
      // shared addresses of row 0: staging slot of column `lane`, mask words of the row
      const unsigned stage_base = smem_addr(&sm.c[0]) + (unsigned)(((0 - kWinLo) * kWinStride + (lane - kWinLo)) * 8);
      const unsigned mask_base = smem_addr(&sm.mask[0][0]);
      const bool lane0 = lane == 0;
#pragma unroll 1
      for (int phase = 0; phase < (kLattice ? 2 : 1); ++phase) {
        // the vertical taps of the warp's rows are computed ONCE, one row per lane, and handed out by shuffle: the
        // I2F / FFMA / F2I / I2F chain of axis_tap no longer sits in front of every row's loads
        const AxisTap my_tap = axis_tap(scale_y, min(i_begin + lane * i_step, kCrop - 1), in_h);
        int j = 0;
        for (int i = i_begin; i < i_end; i += i_step, ++j) {
          if (kLattice && phase == 1 && (i & (kLatStride - 1)) == kLatFirst) continue;   // done in phase 0
          const bool row_in = i >= kWinLo && i < kWinHi;   // warp-uniform
          const unsigned stage_addr = stage_base + (unsigned)(i * (kWinStride * 8));
          const unsigned mask_addr = mask_base + 16u * (unsigned)i;
          AxisTap v;
          v.i0 = __shfl_sync(kFullMask, my_tap.i0, j);
          v.l1 = __shfl_sync(kFullMask, my_tap.l1, j);
          v.i1 = min(v.i0 + 1, in_h - 1);
          v.l0 = __fsub_rn(1.f, v.l1);
          float s[4];
          f32x2 ab[4];
          if constexpr (PLANE_ELEMS < 0) trows.row(lane, i, s, ab);
          else rows.row(taps, v, s, ab);
          uint32_t word[4];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            // ||c|| > 0.5 exactly as torch.norm (round(a*a) + round(b*b), IEEE sqrt), via the
            // equivalent threshold on the squared norm
            float a2, b2;
            upk2(mul2(ab[c], ab[c]), a2, b2);
            const float sq = __fadd_rn(a2, b2);
            const bool on = (s[c] > UNMORE_SIGMOID_HALF_THRESHOLD) || (sq > UNMORE_NORM_HALF_SQ_THRESHOLD);
            word[c] = __ballot_sync(kFullMask, on);  // columns 32c .. 32c+31, LSB = lowest
            cabs = fmaxf(cabs, sq);   // max of the squared norms: sqrt of it bounds max(|a|, |b|) (one instruction instead of three)
          }
          st_shared_b32_if<0>(lane0, mask_addr, word[0]);
          st_shared_b32_if<4>(lane0, mask_addr, word[1]);
          st_shared_b32_if<8>(lane0, mask_addr, word[2]);
          st_shared_b32_if<12>(lane0, mask_addr, word[3]);
          st_shared_b64_if<0>(row_in && col_in[0], stage_addr, ab[0]);
          st_shared_b64_if<256>(row_in, stage_addr, ab[1]);
          st_shared_b64_if<512>(row_in, stage_addr, ab[2]);
          st_shared_b64_if<768>(row_in && col_in[3], stage_addr, ab[3]);
        }
        if (kLattice && phase == 0) {
          __syncthreads();
          // every warp derives the same row range from the lattice rows (no second barrier, no broadcast)
          bool alive_row = false;
          if (lane < kLatRows) {
            u128 m = load_row(sm.mask[kLatFirst + kLatStride * lane]);
            m &= m >> 1; m &= m >> 2; m &= m >> 4; m &= m >> 8; m &= m >> 9;   // bit j: columns j .. j+24 set
            alive_row = m != 0;
          }
          const unsigned alive = __ballot_sync(kFullMask, alive_row);
          unsigned long long klo = 0, khi = 0;   // rows within kErode of a dead lattice row
#pragma unroll
          for (int k = 0; k < kLatRows; ++k) {
            const int l = kLatFirst + kLatStride * k, a = l - kErode < 0 ? 0 : l - kErode, b = l + kErode > kCrop - 1 ? kCrop - 1 : l + kErode;
            unsigned long long lo = 0, hi = 0;
            for (int r = a; r <= b; ++r) { if (r < 64) lo |= 1ull << r; else hi |= 1ull << (r - 64); }   // folds to constants
            if (!((alive >> k) & 1u)) { klo |= lo; khi |= hi; }
          }
          const unsigned long long clo = ~klo & (~0ull << kErode), chi = ~khi & (~0ull >> kErode);   // rows 12..63, 64..115
          if (!(clo | chi)) { no_survivors = true; break; }
          rmin = clo ? __ffsll((long long)clo) - 1 : 63 + __ffsll((long long)chi);
          rmax = chi ? 127 - __clzll((long long)chi) : 63 - __clzll((long long)clo);
          const int rlo = rmin - kErode, n = rmax + kErode + 1 - rlo, per = (n + kCenterWarps - 1) / kCenterWarps;
          i_begin = rlo + warp * per; i_end = min(rlo + n, i_begin + per); i_step = 1;
        }
      }
      if (!no_survivors) {
      cabs = warp_max(cabs);
      cabs = __fmul_rn(__fsqrt_ru(cabs), 1.000001f);   // an upper bound of max |center field| is all the margin needs
      if (lane == 0) sm.red_f[warp] = cabs;
      __syncthreads();
      locate_next();
      // ---- 2. erosion: 25-runs along rows, then AND of 25 rows
      if (tid == kCrop) sm.cand_n = 0;   // an idle thread of this phase; ordered by the barriers around it
      if (tid < kCrop) {
        u128 m = load_row(sm.mask[tid]);
        m &= m >> 1; m &= m >> 2; m &= m >> 4; m &= m >> 8;  // bit j: columns j..j+15 set
        m &= m >> 9;                                          // bit j: columns j..j+24 set
        store_row(sm.hrun[tid], m << kErode);                 // centre the run
      }
      __syncthreads();
      if (tid < kCrop) {
        u128 e = 0;
        if (tid >= rmin && tid <= rmax) {   // rows outside cannot hold survivors (and their neighbours may not have been resampled)
          e = ~(u128)0;
#pragma unroll 5
          for (int d = -kErode; d <= kErode; ++d) e &= load_row(sm.hrun[tid + d]);
        }
        store_row(sm.ero[tid], e);
      }
      __syncthreads();
      // ---- 3. anti-center map on surviving pixels, then masked max / first arg-max.
      // The map is needed in fp64 only where it can decide the result (the maximum).  So: (a) an
      // fp32 register-tiled 5x5x2 correlation over 1x8 pixel strips that contain surviving pixels
      // gives a screening maximum M32; (b) every surviving pixel whose fp32 value is within a
      // rigorous rounding margin of M32 is re-evaluated exactly as the reference does (fp64
      // products of the fp32-normalised filter, / 24) and competes for (max, first index).
      constexpr int kInner = kCrop - 2 * kErode;   // 104: only rows/cols 12..115 can survive
      constexpr int kStrips = kInner / 8;          // 13 strips of 8 columns per row
      constexpr int kMaxOwn = (kInner * kStrips + kCenterThreads - 1) / kCenterThreads;  // 3
      float own_max[kMaxOwn];
      auto strip_bits = [&](int r, int k) -> uint32_t {
        const int c = kErode + 8 * k;              // first column of the strip
        const uint32_t lo = sm.ero[r][c >> 5], hi = sm.ero[r][min((c >> 5) + 1, 3)];
        return (__funnelshift_r(lo, hi, c & 31)) & 0xffu;
      };
      // acc[x] = sum over the 24 taps of f0*c0 + f1*c1 for the 8 pixels of the strip.  With the channels
      // interleaved in shared memory every tap of every pixel is one aligned (c0, c1) pair, so a tap costs one
      // FFMA2 against the (f0, f1) filter pair: the two channels accumulate in the two halves and are added
      // at the end (the rounding differs from a single chain, which the screening margin covers).
      auto strip_scores = [&](int r, int k, float acc[8]) {
        f32x2 acc2[8];
#pragma unroll
        for (int x = 0; x < 8; ++x) acc2[x] = pk2(0.f, 0.f);
        const int c = kErode + 8 * k;
#pragma unroll
        for (int di = 0; di < 5; ++di) {
          const int o = (r + di - 2 - kWinLo) * kWinStride + (c - 2 - kWinLo);  // multiple of 4 pixels = 32 bytes
          f32x2 v[12];
#pragma unroll
          for (int q2 = 0; q2 < 6; ++q2) {
            const ulonglong2 t = *reinterpret_cast<const ulonglong2*>(&sm.c[o + 2 * q2]);
            v[2 * q2] = t.x; v[2 * q2 + 1] = t.y;
          }
#pragma unroll
          for (int dj = 0; dj < 5; ++dj) {
            if (di == 2 && dj == 2) continue;
            const f32x2 f = p.filt_pair[di * 5 + dj];
#pragma unroll
            for (int x = 0; x < 8; ++x) acc2[x] = fma2(f, v[x + dj], acc2[x]);
          }
        }
#pragma unroll
        for (int x = 0; x < 8; ++x) {
          float lo, hi;
          upk2(acc2[x], lo, hi);
          acc[x] = lo + hi;
        }
      };
      float m32 = -INFINITY;
#pragma unroll
      for (int m = 0; m < kMaxOwn; ++m) {
        own_max[m] = -INFINITY;
        const int q = tid + m * kCenterThreads;
        if (q < kInner * kStrips) {
          const int r = kErode + q % kInner, k = q / kInner;   // consecutive lanes -> consecutive rows: conflict-free LDS.128
          const uint32_t bits = strip_bits(r, k);
          if (bits) {
            float acc[8];
            strip_scores(r, k, acc);
#pragma unroll
            for (int x = 0; x < 8; ++x)
              if ((bits >> x) & 1u) own_max[m] = fmaxf(own_max[m], acc[x]);
            m32 = fmaxf(m32, own_max[m]);
          }
        }
      }
      m32 = warp_max(m32);
      float cmax = 0.f;
      if (lane == 0) sm.red_m[warp] = m32;
      __syncthreads();
      {  // every thread folds the per-warp partials itself (broadcast reads): no serial section, one barrier less
        float mm = -INFINITY, cm = 0.f;
#pragma unroll
        for (int w = 0; w < kCenterWarps; ++w) { mm = fmaxf(mm, sm.red_m[w]); cm = fmaxf(cm, sm.red_f[w]); }
        m32 = mm;
        cmax = cm;
      }
      // |fp32 sum - exact sum| <= 48 ops * 2^-24 * sum|f||c| <= 48 * 2^-24 * 31 * cmax (before the / 24);
      // a tie of the true maximum can sit at most twice that below M32.  Padded x4.
      const float margin = 8.0f * 48.0f * 5.9604645e-08f * 31.0f * cmax;
      // (b1) every pixel that can still be the maximum goes into a shared queue ...
      const float cand_thr = m32 - margin;
      const bool any_cand = m32 != -INFINITY;
#pragma unroll
      for (int m = 0; m < kMaxOwn; ++m) {
        if (!any_cand || !(own_max[m] >= cand_thr)) continue;
        const int q = tid + m * kCenterThreads;
        const int r = kErode + q % kInner, k = q / kInner;
        const uint32_t bits = strip_bits(r, k);
        float acc[8];
        strip_scores(r, k, acc);
#pragma unroll
        for (int x = 0; x < 8; ++x) {
          if (((bits >> x) & 1u) && acc[x] >= cand_thr) {
            const int slot = atomicAdd(&sm.cand_n, 1);
            if (slot < kCandCap) sm.cand[slot] = (uint16_t)(r * kCrop + kErode + 8 * k + x);
          }
        }
      }
      __syncthreads();
      // (b2) ... and is re-evaluated exactly as the reference does, one pixel per thread: the 96-term fp64
      // chains of all candidates run side by side instead of one after the other in whichever thread owns them
      auto exact = [&](int r, int c) -> double {
        double e = 0.0;
#pragma unroll
        for (int di = 0; di < 5; ++di) {
#pragma unroll
          for (int dj = 0; dj < 5; ++dj) {
            if (di == 2 && dj == 2) continue;
            const float2 cc = sm.c[(r + di - 2 - kWinLo) * kWinStride + (c + dj - 2 - kWinLo)];
            e = fma(p.filt[di * 5 + dj], (double)cc.x, e);   // f[0][i][j] = (2-i)/n
            e = fma(p.filt[dj * 5 + di], (double)cc.y, e);   // f[1][i][j] = (2-j)/n
          }
        }
        return __ddiv_rn(e, 24.0);
      };
      double tbest = 0.0;
      int tidx = -1;
      const int n_cand = sm.cand_n;
      if (n_cand <= kCandCap) {
        for (int q = tid; q < n_cand; q += kCenterThreads) {
          const int flat = sm.cand[q];
          const double e = exact(flat >> 7, flat & (kCrop - 1));
          if (tidx < 0 || e > tbest || (e == tbest && flat < tidx)) { tbest = e; tidx = flat; }
        }
      } else {
        // a plateau (e.g. a constant field): more candidates than the queue holds; each thread walks its own strips
#pragma unroll 1
        for (int m = 0; m < kMaxOwn; ++m) {
          if (!(own_max[m] >= cand_thr)) continue;
          const int q = tid + m * kCenterThreads;
          const int r = kErode + q % kInner, k = q / kInner;
          const uint32_t bits = strip_bits(r, k);
          float acc[8];
          strip_scores(r, k, acc);
#pragma unroll 1
          for (int x = 0; x < 8; ++x) {
            if (!((bits >> x) & 1u) || !(acc[x] >= cand_thr)) continue;
            const int c = kErode + 8 * k + x;
            const double e = exact(r, c);
            const int flat = r * kCrop + c;
            if (tidx < 0 || e > tbest || (e == tbest && flat < tidx)) { tbest = e; tidx = flat; }
          }
        }
      }
      // block arg-max, ties -> smallest flat index (torch.argmax returns the first maximum)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(kFullMask, tbest, o);
        const int oi = __shfl_xor_sync(kFullMask, tidx, o);
        if (oi >= 0 && (tidx < 0 || ov > tbest || (ov == tbest && oi < tidx))) { tbest = ov; tidx = oi; }
      }
      if (lane == 0) { sm.red_val[warp] = tbest; sm.red_idx[warp] = tidx; }
      __syncthreads();
      if (warp == 0) {   // the first warp folds the per-warp results with shuffles
        double ov = lane < kCenterWarps ? sm.red_val[lane] : 0.0;
        int oi = lane < kCenterWarps ? sm.red_idx[lane] : -1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double pv = __shfl_xor_sync(kFullMask, ov, o);
          const int pi = __shfl_xor_sync(kFullMask, oi, o);
          if (pi >= 0 && (oi < 0 || pv > ov || (pv == ov && pi < oi))) { ov = pv; oi = pi; }
        }
        best = ov; best_idx = oi;
      }
      }   // !no_survivors
    }
    if (tid == 0) {
      // amax over the whole map: pixels outside the eroded mask contribute 0
      const double maxv = (best_idx >= 0 && best > 0.0) ? best : 0.0;
      const bool pass = maxv <= p.thr;
      sm.bcast_i[0] = pass ? 1 : 0;
      p.max_values[row] = maxv;
      p.argmax[row] = pass ? -1 : best_idx;
      if (!pass && p.splits) {
        const int yc = best_idx / kCrop, xc = best_idx % kCrop;
        const double xr = (double)((float)xc / (float)kCrop), yr = (double)((float)yc / (float)kCrop);
        const double xs = __dadd_rn(x1, __dmul_rn(__dsub_rn(x2, x1), xr));
        const double ys = __dadd_rn(y1, __dmul_rn(__dsub_rn(y2, y1), yr));
        double* o = p.splits + row * 16;
        o[0] = x1; o[1] = y1; o[2] = xs; o[3] = y2;    // left   (:553)
        o[4] = xs; o[5] = y1; o[6] = x2; o[7] = y2;    // right  (:554)
        o[8] = x1; o[9] = y1; o[10] = x2; o[11] = ys;  // top    (:555)
        o[12] = x1; o[13] = ys; o[14] = x2; o[15] = y2;  // bottom (:556)
      }
    }
    // ---- 4. --analyze_cc (:561-572): 8-connected components of the un-eroded union mask of a
    // PASSING proposal (separate_connected_components :207-256); if there are several, each
    // component's bbox, enlarged x1.5 about its centre with int() truncation and clipped against the
    // image size (enlarge_proposals :259-291 — the reference feeds crop coordinates there), becomes a
    // new proposal.  Labels are the smallest flat index of the component (min-propagation over the
    // 8-neighbourhood + pointer jumping), so component order == scipy's raster first-pixel order.
    if constexpr (ANALYZE_CC) {
      __syncthreads();
      int n_comp = 0;
      if (sm.bcast_i[0] && !win.empty()) {
        n_comp = label_components(sm.mask, reinterpret_cast<uint16_t*>(sm.c), reinterpret_cast<uint16_t*>(sm.c) + kCrop * kCrop,
                                  sm.cc_scan, sm.cc_box);   // the staged fields are dead now: reuse their storage
        if (n_comp >= 2) {
          if (tid < min(n_comp, kCcCap)) {
            // bbox = [x_start, y_start, x_stop, y_stop] (slice bounds); enlarge in Python float arithmetic
            const double bx1 = sm.cc_box[0][tid], by1 = sm.cc_box[1][tid];
            const double bx2 = sm.cc_box[2][tid] + 1, by2 = sm.cc_box[3][tid] + 1;
            const double cx = (bx1 + bx2) / 2, cy = (by1 + by2) / 2;
            const double nw = (bx2 - bx1) * 1.5, nh = (by2 - by1) * 1.5;
            double* o = p.cc_boxes + (row * kCcCap + tid) * 4;
            o[0] = (double)(int)fmax(cx - nw / 2, 0.0);
            o[1] = (double)(int)fmax(cy - nh / 2, 0.0);
            if constexpr (SIZED) {
              const int2 e = image_extent(p.image_hw, img, p.H, p.W);
              o[2] = (double)(int)fmin(cx + nw / 2, (double)e.y);
              o[3] = (double)(int)fmin(cy + nh / 2, (double)e.x);
            } else {
              o[2] = (double)(int)fmin(cx + nw / 2, (double)p.W);
              o[3] = (double)(int)fmin(cy + nh / 2, (double)p.H);
            }
          }
          if (tid == 0 && n_comp > kCcCap) atomicAdd(p.cc_overflow, 1);
        }
      }
      if (tid == 0) p.cc_counts[row] = (unsigned char)(n_comp >= 2 ? min(n_comp, kCcCap) : 0);
    }
    locate_next();   // zero-size crops skip the stages above
    if (tid == 0) {
      s_item[cur ^ 1].id = next_id; s_item[cur ^ 1].img = next_img; s_item[cur ^ 1].k = next_k;
      asm volatile("cp.async.wait_all;" ::: "memory");
    }
    __syncthreads();  // publishes the next work item; shared tiles are reused by the next proposal
  }
}

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

template <bool CC, int PE, bool RS = false>
static int launch_center_t(const CenterParams& p, int num_sms, cudaStream_t stream) {
  // function attributes are per device: set on every launch (microseconds), no cached state
  if constexpr (PE >= 0) {
    if (p.image_hw) {   // a padded stack: the sized variant
      cudaError_t e = cudaFuncSetAttribute(center_kernel<CC, PE, RS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CenterSmem));
      if (e != cudaSuccess) return (int)e;
      center_kernel<CC, PE, RS, true><<<num_sms * 2, kCenterThreads, sizeof(CenterSmem), stream>>>(p);
      return (int)cudaGetLastError();
    }
  }
  cudaError_t e = cudaFuncSetAttribute(center_kernel<CC, PE, RS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(CenterSmem));
  if (e != cudaSuccess) return (int)e;
  center_kernel<CC, PE, RS><<<num_sms * 2, kCenterThreads, sizeof(CenterSmem), stream>>>(p);
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
