// Boundary reasoning: update_bbox_with_boundary_fields (object_reasoning.py:140-174),
// optimize_one_image_single_round (:379-487) and the round loop of boundary_reasoning
// (:582-612), fused into one persistent kernel.
//
// One warp owns one proposal for its whole life (<= n_round rounds): the box and label
// stay in registers, each round re-snaps the crop window, resamples the boundary-distance
// channel straight from the (L2-resident) field, reduces the soft-foreground/background
// gradient averages, takes the four border maxima and applies the box update.  Proposals
// are independent in the reference (no cross-proposal term anywhere in the loop), so the
// per-round filter_small_proposal / boolean-mask compactions become per-proposal exits.
#include "aa_rows.cuh"
#include "resample.cuh"
#include "unmore_internal.h"

namespace unmore {

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// sigmoid as the soft foreground mask (object_reasoning.py:153); 2 MUFU + 2 FP32 ops
__device__ __forceinline__ float soft_fg(float s) {
  return rcp_approx(1.f + ex2_approx(-1.4426950408889634f * s));
}

// one predicated store instead of a divergent branch around it (common.cuh)
__device__ __forceinline__ void st_shared_if(bool pred, float* smem_ptr, float v) {
  st_shared_b32_if<0>(pred, smem_addr(smem_ptr), __float_as_uint(v));
}

struct TileRows {  // pre-resampled [128,128] tile (unit op a10): lane reads its four columns lane + 32c
  const float* tile;
  float pend[4];
  __device__ __forceinline__ void issue(int lane, int i) {
#pragma unroll
    for (int c = 0; c < 4; ++c) pend[c] = __ldg(tile + i * kCrop + lane + 32 * c);
  }
  __device__ __forceinline__ void finish(f32x2 out[2]) { out[0] = pk2(pend[0], pend[1]); out[1] = pk2(pend[2], pend[3]); }
};

template <int ROW_ELEMS>
struct CropRows {  // crop window of the boundary-distance channel, resampled on the fly
  ColTaps taps;
  PlaneRows plane;
  PlaneRows::Fetch pend;
  unsigned tapy_addr;   // shared address of this warp's vertical-tap table (BorderCols::tapy)
  int in_h;
  // The 128 vertical taps of the window are computed once per round, four per lane, and read back as one
  // broadcast 8-byte load per row (instead of ten instructions of tap arithmetic per row).
  __device__ __forceinline__ void init_rows(int lane, int2* tapy, int h) {
    in_h = h;
    const float scale_y = __fdiv_rn((float)h, (float)kCrop);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const AxisTap t = axis_tap(scale_y, lane + 32 * k, h);
      tapy[lane + 32 * k] = make_int2(t.i0, __float_as_int(t.l1));
    }
    tapy_addr = smem_addr(tapy);
    __syncwarp();
  }
  __device__ __forceinline__ void issue(int /*lane*/, int i) {
    int i0, l1b;
    asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(i0), "=r"(l1b) : "r"(tapy_addr + 8u * (unsigned)i) : "memory");
    AxisTap v;
    v.i0 = i0;
    v.i1 = min(i0 + 1, in_h - 1);
    v.l1 = __int_as_float(l1b);
    v.l0 = __fsub_rn(1.f, v.l1);
    plane.issue<ROW_ELEMS>(taps, v, pend);
  }
  __device__ __forceinline__ void finish(f32x2 out[2]) { plane.finish(taps, pend, out); }
};

// Per-warp scratch (4 KB): the four borders of the resampled tile — S[i][0], S[i][126] for i in [0,127),
// S[0][j], S[126][j] — so the border pass needs no resample, and the fp64 running sums of each lane.
// Keeping these out of registers is what lets the split-phase row fetch fit the register budget.
struct BorderCols {
  float left[kCrop];
  float right[kCrop];
  float top[kCrop];
  float bot[kCrop];
  double acc[4][32];   // sum A, sum A*g, sum B, sum B*g per lane
  int2 tapy[kCrop];    // vertical taps of the current window: (i0, bits of l1) per output row
  int pub;             // lane 0: window-cache slot to publish this round's terms into, or -1 (in shared memory: a
                       // register live across boundary_terms costs spills around its row loop)
};

struct Deltas {
  float max_sdf;
  float dx1, dy1, dx2, dy2;
};

// a10 on one proposal.  `src.issue(lane, i)` / `src.finish(out)` yield S[i][lane + 32c], c = 0..3, as two packed pairs.
// The per-pixel formula runs on pairs (FFMA2 / FMUL2 / FADD2): one issue slot per two pixels for
// everything but the three MUFU evaluations and the horizontal difference.
template <class RowSrc>
__device__ __forceinline__ Deltas boundary_terms(RowSrc& src, BorderCols& cols, int lane) {
  f32x2 ra[2], rb[2];
  src.issue(lane, 0);
  src.finish(ra);
  src.issue(lane, 1);
  float mx;
  {
    float t0, t1, t2, t3;
    upk2(ra[0], t0, t1);
    upk2(ra[1], t2, t3);
    mx = fmaxf(fmaxf(t0, t1), fmaxf(t2, t3));
    cols.top[lane] = t0; cols.top[lane + 32] = t1; cols.top[lane + 64] = t2; cols.top[lane + 96] = t3;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) cols.acc[k][lane] = 0.0;
  const f32x2 kZero2 = pk2(0.f, 0.f), kOne2 = pk2(1.f, 1.f);
  f32x2 fA = kZero2, fAg = kZero2, fB = kZero2, fBg = kZero2;
  const bool first_lane = lane == 0, last_lane = lane == 31;
  const int next_lane = (lane + 1) & 31;
  // One output row of the 127x127 region: cur = S[i][.], nxt = S[i+1][.].
  auto process = [&](const f32x2 (&cur)[2], const f32x2 (&nxt)[2], int i) {
    float c0, c1, c2, c3, n0, n1, n2, n3;
    upk2(cur[0], c0, c1); upk2(cur[1], c2, c3);
    upk2(nxt[0], n0, n1); upk2(nxt[1], n2, n3);
    // Lane l holds columns l, l+32, l+64, l+96 (a tap request of the warp then covers 32 consecutive output
    // columns, ~5 L1 sectors instead of ~26 with four adjacent columns per lane — the L1 data pipe was the
    // busiest unit of this kernel).  The right neighbour of column l+32c is the next lane's same element, or
    // lane 0's NEXT element for lane 31; lane 0 therefore hands out its elements shifted by one.
    const float r0 = __shfl_sync(kFullMask, first_lane ? c1 : c0, next_lane);
    const float r1 = __shfl_sync(kFullMask, first_lane ? c2 : c1, next_lane);
    const float r2 = __shfl_sync(kFullMask, first_lane ? c3 : c2, next_lane);
    const float r3 = __shfl_sync(kFullMask, c3, next_lane);   // lane 31: column 128 does not exist (pixel excluded below)
    st_shared_if(first_lane, &cols.left[i], c0);        // column 0
    st_shared_if(lane == 30, &cols.right[i], c3);       // column 126 = 30 + 96
    const f32x2 dx[2] = {pk2(r0 - c0, r1 - c1), pk2(r2 - c2, r3 - c3)};
    // the pixels of a lane are independent dependency chains (ex2 -> +1 -> rcp -> 1-a); stage them so the
    // MUFU latencies overlap instead of serialising pixel after pixel
    f32x2 t[2], u[2], g[2], a[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const f32x2 dy = sub2(nxt[h], cur[h]);
      t[h] = fma2(dy, dy, mul2(dx[h], dx[h]));
      u[h] = mul2(cur[h], pk2(-1.4426950408889634f, -1.4426950408889634f));
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {   // ||grad|| only feeds the averaged sums
      float tl, th, ul, uh;
      upk2(t[h], tl, th); upk2(u[h], ul, uh);
      u[h] = pk2(ex2_approx(ul), ex2_approx(uh));
      g[h] = pk2(sqrt_approx(tl), sqrt_approx(th));
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) u[h] = add2(u[h], kOne2);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float ul, uh;
      upk2(u[h], ul, uh);
      a[h] = pk2(rcp_approx(ul), rcp_approx(uh));
    }
    {
      const f32x2 b = sub2(kOne2, a[0]);
      fA = add2(fA, a[0]); fAg = fma2(a[0], g[0], fAg);
      fB = add2(fB, b);    fBg = fma2(b, g[0], fBg);
    }
    {
      // column 127 (lane 31's fourth column = second pixel of its upper pair) is outside the 127x127 region: its
      // foreground and background weights are forced to zero
      float al, ah, bl, bh;
      upk2(a[1], al, ah);
      upk2(sub2(kOne2, a[1]), bl, bh);
      const f32x2 am = pk2(al, last_lane ? 0.f : ah), b = pk2(bl, last_lane ? 0.f : bh);
      fA = add2(fA, am); fAg = fma2(am, g[1], fAg);
      fB = add2(fB, b);  fBg = fma2(b, g[1], fBg);
    }
    mx = fmaxf(fmaxf(mx, fmaxf(n0, n1)), fmaxf(n2, n3));
  };
  // fp32 partial sums (two per lane) are flushed into the lane's fp64 sums every 8 rows (16 px per partial):
  // keeps the 16129-term sums within ~1e-7 of exact without paying an F2F+DADD per pixel
  auto flush = [&]() {
    float lo, hi;
    upk2(fA, lo, hi); cols.acc[0][lane] += (double)(lo + hi);
    upk2(fAg, lo, hi); cols.acc[1][lane] += (double)(lo + hi);
    upk2(fB, lo, hi); cols.acc[2][lane] += (double)(lo + hi);
    upk2(fBg, lo, hi); cols.acc[3][lane] += (double)(lo + hi);
    fA = fAg = fB = fBg = kZero2;
  };
  // rows ping-pong between ra / rb so no register copies are needed; the taps of row i+2 are requested
  // before row i is processed and collected after it
  for (int i = 0; i < kCrop - 2; i += 2) {
    src.finish(rb);            // row i+1
    src.issue(lane, i + 2);
    process(ra, rb, i);
    src.finish(ra);            // row i+2
    src.issue(lane, i + 3);    // i + 3 <= 127
    process(rb, ra, i + 1);
    if ((i & 7) == 6) flush();
  }
  // i = 126: ra holds row 126, row 127 is in flight
  {
    float t0, t1, t2, t3;
    upk2(ra[0], t0, t1);
    upk2(ra[1], t2, t3);
    cols.bot[lane] = t0; cols.bot[lane + 32] = t1; cols.bot[lane + 64] = t2; cols.bot[lane + 96] = t3;
  }
  src.finish(rb);
  process(ra, rb, kCrop - 2);
  flush();
  const double dA = cols.acc[0][lane], dAg = cols.acc[1][lane], dB = cols.acc[2][lane], dBg = cols.acc[3][lane];
  Deltas d;
  d.max_sdf = warp_max(mx);
  const float sumA = (float)warp_sum(dA);
  const float sumAg = (float)warp_sum(dAg);
  const float sumB = (float)warp_sum(dB);
  const float sumBg = (float)warp_sum(dBg);
  // avg gradient norms and step sizes, fp32 like the reference (:155-158)
  const float avg_fg = __fdiv_rn(sumAg, __fadd_rn(sumA, 1e-8f));
  const float avg_bg = __fdiv_rn(sumBg, __fadd_rn(sumB, 1e-8f));
  const float step_fg = __fdiv_rn(1.f, __fadd_rn(avg_fg, 1e-10f));
  const float step_bg = __fdiv_rn(1.f, __fadd_rn(avg_bg, 1e-10f));
  auto movement = [&](float s) {
    const float a = soft_fg(s);
    const float b = 1.f - a;
    return __fmul_rn(__fadd_rn(__fmul_rn(step_fg, a), __fmul_rn(step_bg, b)), s);
  };
  __syncwarp();
  float m_top = -INFINITY, m_bot = -INFINITY, m_left = -INFINITY, m_right = -INFINITY;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int i = lane + 32 * c;   // position along the border; 127 is outside the region
    if (i < kCrop - 1) {
      m_top = fmaxf(m_top, movement(cols.top[i]));
      m_bot = fmaxf(m_bot, movement(cols.bot[i]));
      m_left = fmaxf(m_left, movement(cols.left[i]));
      m_right = fmaxf(m_right, movement(cols.right[i]));
    }
  }
  __syncwarp();
  d.dx1 = -warp_max(m_left);
  d.dy1 = -warp_max(m_top);
  d.dx2 = warp_max(m_right);
  d.dy2 = warp_max(m_bot);
  return d;
}

// ---- window cache (WindowSlot, unmore_internal.h) ----------------------------------------------------------
// Deltas are a function of the field plane and the snapped window only, and boundary_terms gives the same bits
// whichever warp runs it, so a round may take them from the warp that computed its window first.  Only lane 0
// touches the table, once per round.  A slot goes 0 -> key (claimed: the claimer is computing) -> key | ready
// (published with a release store after the terms).  A warp that finds its window claimed waits a bounded
// number of polls (sleeping, so the other warps of the SM get its issue slots), then computes the terms itself
// without publishing; so does a warp whose probe path is full.  No warp waits on another without a limit.
constexpr int kWindowProbes = 16;
constexpr int kWindowWaitPolls = 160;   // 64 ns doubling to 1 us per poll: at most ~160 us of sleep
constexpr unsigned long long kWindowReady = 1ull << 63;

__device__ __forceinline__ unsigned long long window_key(const Window& w) {
  return (unsigned long long)w.x1 | (unsigned long long)w.y1 << 15 | (unsigned long long)w.x2 << 30 |
         (unsigned long long)w.y2 << 45;
}
__device__ __forceinline__ unsigned long long ld_acquire_key(const WindowSlot* s) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(&s->key) : "memory");
  return v;
}

// Lane 0.  true: `d` holds the published terms of the window.  false: the caller computes them, and publishes
// them into slot `pub` when pub >= 0 (this warp claimed it).
__device__ __forceinline__ bool window_lookup(WindowSlot* table, const Window& win, Deltas& d, int& pub) {
  const unsigned long long key = window_key(win);
  const unsigned h = (unsigned)((key * 0x9E3779B97F4A7C15ull) >> 32);
  pub = -1;
  for (int probe = 0; probe < kWindowProbes; ++probe) {
    const int i = (int)((h + probe) & (kWindowSlots - 1));
    WindowSlot* s = table + i;
    unsigned long long k = ld_acquire_key(s);
    if (k == 0) {
      if (atomicCAS(&s->key, 0ull, key) == 0ull) { pub = i; return false; }
      k = ld_acquire_key(s);   // lost the race: the slot now holds some window, claimed or published
    }
    if ((k & ~kWindowReady) != key) continue;
    for (int poll = 0, ns = 64; !(k & kWindowReady); ++poll) {
      if (poll == kWindowWaitPolls) return false;
      __nanosleep(ns);
      ns = min(2 * ns, 1024);
      k = ld_acquire_key(s);
    }
    asm volatile("ld.relaxed.gpu.global.f32 %0, [%1];" : "=f"(d.max_sdf) : "l"(&s->max_sdf) : "memory");
    asm volatile("ld.relaxed.gpu.global.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(d.dx1), "=f"(d.dy1), "=f"(d.dx2), "=f"(d.dy2) : "l"(&s->d) : "memory");
    return true;
  }
  return false;
}

__device__ __forceinline__ void window_publish(WindowSlot* s, const Window& win, const Deltas& d) {
  s->max_sdf = d.max_sdf;
  s->d = make_float4(d.dx1, d.dy1, d.dx2, d.dy2);
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(&s->key), "l"(window_key(win) | kWindowReady) : "memory");
}

template <typename T>
struct BoxT { T x1, y1, x2, y2; };

// The box update of one round for one proposal, arithmetic in T (double on round 0 when the caller hands in
// fp64 proposals — promotion at object_reasoning.py:190-194 — float afterwards).
// Returns the label of this round and the updated box (fp32, :479).
// (W, H): the image's size (its own extent in a padded stack).
template <typename T>
__device__ __forceinline__ int apply_update(const RefineParams& p, int W, int H, const Window& win, const Deltas& d, BoxT<T> b,
                                            float4& out) {
  // signed deltas: >0 expands, <0 shrinks; expansion is ignored on sides glued to the image edge (:444-447)
  float sg[4] = {-d.dx1, -d.dy1, d.dx2, d.dy2};
  const bool edge[4] = {win.x1 == 0, win.y1 == 0, win.x2 == W, win.y2 == H};
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (sg[k] > 0.f && edge[k]) sg[k] = 0.f;
  const float max_exp = fmaxf(fmaxf(sg[0], sg[1]), fmaxf(sg[2], sg[3]));
  const float max_shr = fminf(fminf(sg[0], sg[1]), fminf(sg[2], sg[3]));
  const int label = (max_exp <= 0.f && max_shr >= -p.max_shrink_thres) ? 1 : 0;
  // asymmetric step (:457-460): expansions x(1+ratio), shrinks x(1-ratio)
  float dl[4];
  dl[0] = __fsub_rn(d.dx1, __fmul_rn(fabsf(d.dx1), p.delta_ratio));
  dl[1] = __fsub_rn(d.dy1, __fmul_rn(fabsf(d.dy1), p.delta_ratio));
  dl[2] = __fadd_rn(d.dx2, __fmul_rn(fabsf(d.dx2), p.delta_ratio));
  dl[3] = __fadd_rn(d.dy2, __fmul_rn(fabsf(d.dy2), p.delta_ratio));
  if (label == 1) dl[0] = dl[1] = dl[2] = dl[3] = 0.f;
  // post_process_bbox_update (:177-196): separate multiply and add, no contraction
  T nx1, ny1, nx2, ny2;
  if constexpr (sizeof(T) == 8) {
    const double xr = __ddiv_rn(__dsub_rn(b.x2, b.x1), 128.0), yr = __ddiv_rn(__dsub_rn(b.y2, b.y1), 128.0);
    nx1 = __dadd_rn(b.x1, __dmul_rn((double)dl[0], xr));
    ny1 = __dadd_rn(b.y1, __dmul_rn((double)dl[1], yr));
    nx2 = __dadd_rn(b.x2, __dmul_rn((double)dl[2], xr));
    ny2 = __dadd_rn(b.y2, __dmul_rn((double)dl[3], yr));
  } else {
    const float xr = __fdiv_rn(__fsub_rn(b.x2, b.x1), 128.f), yr = __fdiv_rn(__fsub_rn(b.y2, b.y1), 128.f);
    nx1 = __fadd_rn(b.x1, __fmul_rn(dl[0], xr));
    ny1 = __fadd_rn(b.y1, __fmul_rn(dl[1], yr));
    nx2 = __fadd_rn(b.x2, __fmul_rn(dl[2], xr));
    ny2 = __fadd_rn(b.y2, __fmul_rn(dl[3], yr));
  }
  if (nx1 < (T)0) nx1 = (T)0;
  if (ny1 < (T)0) ny1 = (T)0;
  if (nx2 > (T)W) nx2 = (T)W;
  if (ny2 > (T)H) ny2 = (T)H;
  out = make_float4((float)nx1, (float)ny1, (float)nx2, (float)ny2);
  return label;
}

constexpr int kRefineWarps = 6;
constexpr int kRefineMinBlocks = 3;   // resident CTAs per SM, in __launch_bounds__ and in the grid of launch_refine
constexpr int kSpecRowElems = 640;   // row pitch of the COCO-val-shaped fields the batch path runs on
// The persistent round loop: warps pull proposals from the worklist until it is empty.  `terms(plane, win)` computes
// the boundary terms of a window from its resampled rows; the resize mode only changes where those rows come from.
// SIZED: a padded stack, p.image_hw holds each image's (h, w) inside the (H, W) pitch.  The extent is read where the
// window is snapped and again where the box is updated, so it is not live across the terms (registers are tight).
template <bool SIZED, class Terms>
__device__ __forceinline__ void refine_proposals(const RefineParams& p, BorderCols& cols, int lane, Terms terms,
                                                 const int* image_hw = nullptr) {
  const int total = worklist_total(p.work);
  int img = 0;   // image of the previous work item: the locate hint
  for (;;) {
    const int id = worklist_next_warp(p.work);
    if (id >= total) break;
    int k;
    worklist_locate(p.work, id, img, k);
    const size_t row = (size_t)img * p.work.cap + k;
    const float* plane = p.fields + ((size_t)img * p.C + p.ch_sdf) * p.H * p.W;
    BoxT<float> bf;
    {
      double x1, y1, x2, y2;
      load_box<double>(p.boxes, p.boxes_f64 != 0, row, x1, y1, x2, y2);
      bf = {(float)x1, (float)y1, (float)x2, (float)y2};
    }
    float4 cur = make_float4(bf.x1, bf.y1, bf.x2, bf.y2);
    float label = 0.f;
    int rounds = 0;
    for (int r = 0; r < p.n_round; ++r) {
      // round 0 of fp64 proposals runs its window snap, area filter and box update in double; the fp64 box is
      // re-read from memory where it is needed instead of living in registers through the resampling loop
      const bool dbl = (r == 0) && p.boxes_f64;
      Window win;
      bool keep;
      int ih = p.H, iw = p.W;
      if constexpr (SIZED) {
        const int2 e = image_extent(image_hw, img, p.H, p.W);
        ih = e.x; iw = e.y;
      }
      if (dbl) {
        BoxT<double> bd;
        load_box<double>(p.boxes, true, row, bd.x1, bd.y1, bd.x2, bd.y2);
        keep = __dmul_rn(__dsub_rn(bd.x2, bd.x1), __dsub_rn(bd.y2, bd.y1)) > (double)p.area_thres;
        win = snap_window<double>(bd.x1, bd.y1, bd.x2, bd.y2, iw, ih);
      } else {
        keep = __fmul_rn(__fsub_rn(bf.x2, bf.x1), __fsub_rn(bf.y2, bf.y1)) > p.area_thres;
        win = snap_window<float>(bf.x1, bf.y1, bf.x2, bf.y2, iw, ih);
      }
      if (p.apply_small_filter && !keep) { label = -2.f; break; }  // filter_small_proposal (:293-299), strict '>'
      float4 nb = make_float4(0.f, 0.f, 0.f, 0.f);
      int lab = -1;   // a zero-size crop (the reference would raise) is defined as "no object"
      bool fixed = false;
      // boundary_terms stays at the nesting depth it had without the cache: one more level of divergent control
      // flow around it costs registers and instructions in its row loop
      Deltas d;
      int hit = 0;
      if (p.windows && lane == 0 && !win.empty()) hit = window_lookup(p.windows + (size_t)img * kWindowSlots, win, d, cols.pub);
      hit = __shfl_sync(kFullMask, hit, 0);
      if (!win.empty() && !hit) {
        d = terms(plane, win);
        if (p.windows && lane == 0 && cols.pub >= 0) window_publish(p.windows + (size_t)img * kWindowSlots + cols.pub, win, d);
      }
      if (hit) {
        d.max_sdf = __shfl_sync(kFullMask, d.max_sdf, 0);
        d.dx1 = __shfl_sync(kFullMask, d.dx1, 0);
        d.dy1 = __shfl_sync(kFullMask, d.dy1, 0);
        d.dx2 = __shfl_sync(kFullMask, d.dx2, 0);
        d.dy2 = __shfl_sync(kFullMask, d.dy2, 0);
      }
      if (!win.empty()) {
        if (d.max_sdf > p.max_sdf_thres) {
          if constexpr (SIZED) {
            const int2 e = image_extent(image_hw, img, p.H, p.W);
            ih = e.x; iw = e.y;
          } else {
            ih = p.H; iw = p.W;
          }
          if (dbl) {
            BoxT<double> bd;
            load_box<double>(p.boxes, true, row, bd.x1, bd.y1, bd.x2, bd.y2);
            lab = apply_update<double>(p, iw, ih, win, d, bd, nb);
            // fp64 round 0: the fp32 cast must be exact and the fp32 area test of round 1 must agree
            fixed = (double)nb.x == bd.x1 && (double)nb.y == bd.y1 && (double)nb.z == bd.x2 && (double)nb.w == bd.y2 &&
                    (!p.apply_small_filter || __fmul_rn(__fsub_rn(nb.z, nb.x), __fsub_rn(nb.w, nb.y)) > p.area_thres);
          } else {
            lab = apply_update<float>(p, iw, ih, win, d, bf, nb);
            fixed = true;
          }
        }
      }
      rounds = r + 1;
      label = (float)lab;
      fixed = fixed && lab == 1 && nb.x == cur.x && nb.y == cur.y && nb.z == cur.z && nb.w == cur.w;
      cur = nb;
      bf.x1 = nb.x; bf.y1 = nb.y; bf.x2 = nb.z; bf.y2 = nb.w;
      // label 1 with an unchanged box is an exact fixed point of the remaining rounds
      // (same window, same field, same arithmetic); label -1 leaves a zero box that the
      // next round's area filter removes
      if (p.early_exit && fixed) break;
      if (lab < 0 && p.apply_small_filter && p.area_thres >= 0.f) {
        if (r + 1 < p.n_round) label = -2.f;
        break;
      }
    }
    if (lane == 0) {
      p.boxes_out[row] = cur;
      p.labels_out[row] = label;
      if (p.rounds_out) p.rounds_out[row] = rounds;
    }
  }
}

template <int ROW_ELEMS, bool SIZED>
__device__ __forceinline__ void refine_crops(const RefineParams& p, const int* image_hw) {
  __shared__ BorderCols cols_all[kRefineWarps];
  const int lane = threadIdx.x & 31;
  BorderCols& cols = cols_all[threadIdx.x >> 5];
  refine_proposals<SIZED>(p, cols, lane, [&](const float* plane, const Window& win) {
    CropRows<ROW_ELEMS> src;
    src.taps.template init<kStrided>(lane, win.w());
    src.plane.init(plane, p.W, win);
    src.init_rows(lane, cols.tapy, win.h());
    return boundary_terms(src, cols, lane);
  }, image_hw);
}

template <int ROW_ELEMS>
__global__ void __launch_bounds__(kRefineWarps * 32, kRefineMinBlocks) refine_kernel(const RefineParams p) {
  refine_crops<ROW_ELEMS, false>(p, nullptr);
}
// the same on a padded stack: image_hw [n_img, 2] holds each image's (h, w) inside the (H, W) pitch
template <int ROW_ELEMS>
__global__ void __launch_bounds__(kRefineWarps * 32, kRefineMinBlocks) refine_hw_kernel(const RefineParams p,
                                                                                        const int* __restrict__ image_hw) {
  refine_crops<ROW_ELEMS, true>(p, image_hw);
}

// The second resize mode: the same round loop on antialiased rows (aa_rows.cuh).  A warp needs 15 KB more shared
// memory for the weight table and the row ring, so fewer warps fit an SM.
constexpr int kAaRefineWarps = 2;
constexpr int kAaRefineMinBlocks = 5;
__global__ void __launch_bounds__(kAaRefineWarps * 32, kAaRefineMinBlocks) refine_aa_kernel(const RefineParams p) {
  __shared__ BorderCols cols_all[kAaRefineWarps];
  __shared__ AaRowsSmem rows_all[kAaRefineWarps];
  const int lane = threadIdx.x & 31;
  BorderCols& cols = cols_all[threadIdx.x >> 5];
  AaRowsSmem& rows = rows_all[threadIdx.x >> 5];
  refine_proposals<false>(p, cols, lane, [&](const float* plane, const Window& win) {
    AaCropRows src;
    src.init(lane, rows, plane, p.W, win);
    return boundary_terms(src, cols, lane);
  });
}

__global__ void __launch_bounds__(kRefineWarps * 32) tiles_kernel(const TileParams p) {
  __shared__ BorderCols cols_all[kRefineWarps];
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * kRefineWarps + (threadIdx.x >> 5);
  if (warp >= p.M) return;
  TileRows src{p.tiles + (size_t)warp * kCrop * kCrop};
  const Deltas d = boundary_terms(src, cols_all[threadIdx.x >> 5], lane);
  if (lane == 0) {
    p.deltas[warp] = make_float4(d.dx1, d.dy1, d.dx2, d.dy2);
    if (p.max_sdf) p.max_sdf[warp] = d.max_sdf;
  }
}

// One round of optimize_one_image_single_round (object_reasoning.py:421-479) AFTER the tile reductions: max_sdf
// filter, label, asymmetric step, post_process_bbox_update and clip for M proposals whose deltas / max_sdf came from
// tiles_kernel.  The tile path of the second resize mode (antialias=True): crop (unmore_crop_resize_aa) -> tiles ->
// tiles_kernel -> this.  Same arithmetic as the fused kernel (apply_update), one thread per proposal.
__global__ void __launch_bounds__(128) round_update_kernel(const RefineParams p, const float4* __restrict__ deltas,
                                                           const float* __restrict__ max_sdf, int M) {
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  double x1, y1, x2, y2;
  load_box<double>(p.boxes, p.boxes_f64 != 0, (size_t)m, x1, y1, x2, y2);
  const Window win = snap_window<double>(x1, y1, x2, y2, p.W, p.H);
  float4 nb = make_float4(0.f, 0.f, 0.f, 0.f);
  int lab = -1;
  if (!win.empty() && max_sdf[m] > p.max_sdf_thres) {
    const float4 dl = deltas[m];
    Deltas d;
    d.max_sdf = max_sdf[m]; d.dx1 = dl.x; d.dy1 = dl.y; d.dx2 = dl.z; d.dy2 = dl.w;
    if (p.boxes_f64) {
      lab = apply_update<double>(p, p.W, p.H, win, d, BoxT<double>{x1, y1, x2, y2}, nb);
    } else {
      lab = apply_update<float>(p, p.W, p.H, win, d, BoxT<float>{(float)x1, (float)y1, (float)x2, (float)y2}, nb);
    }
  }
  p.boxes_out[m] = nb;
  p.labels_out[m] = (float)lab;
}

int launch_round_update(const RefineParams& p, const float4* deltas, const float* max_sdf, int M, cudaStream_t stream) {
  if (M <= 0) return 0;
  round_update_kernel<<<(M + 127) / 128, 128, 0, stream>>>(p, deltas, max_sdf, M);
  return (int)cudaGetLastError();
}

int launch_refine(const RefineParams& p, int num_sms, cudaStream_t stream, const int* image_hw) {
  const int ctas = num_sms * kRefineMinBlocks;  // warps pull proposals dynamically
  if (image_hw) {   // the row-pitch specialisation goes by the pitch
    if (p.W == kSpecRowElems) refine_hw_kernel<kSpecRowElems><<<ctas, kRefineWarps * 32, 0, stream>>>(p, image_hw);
    else refine_hw_kernel<0><<<ctas, kRefineWarps * 32, 0, stream>>>(p, image_hw);
  } else if (p.W == kSpecRowElems) refine_kernel<kSpecRowElems><<<ctas, kRefineWarps * 32, 0, stream>>>(p);
  else refine_kernel<0><<<ctas, kRefineWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

int launch_refine_aa(const RefineParams& p, int num_sms, cudaStream_t stream) {
  refine_aa_kernel<<<num_sms * kAaRefineMinBlocks, kAaRefineWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

int launch_tiles(const TileParams& p, cudaStream_t stream) {
  if (p.M <= 0) return 0;
  tiles_kernel<<<(p.M + kRefineWarps - 1) / kRefineWarps, kRefineWarps * 32, 0, stream>>>(p);
  return (int)cudaGetLastError();
}

}  // namespace unmore
