// Per-column cost tables ("table build").
//
//   frame_tables_kernel  : per frame, the vB-only parts of the pairwise
//                          transition priors (StixelsKernels.cu:40-42, 98-144,
//                          173-187) -- they depend on the road model only.
//   column_tables_kernel : per (frame, column): per-row data costs
//                          (:371-446), the prefix sums the reference computes
//                          with in-kernel Blelloch scans (:452-469,
//                          StixelsKernels.h:73-103) and the object-cost LUT of
//                          ComputeObjectLUT (:236-296, 959-978).
//
// Float prefix sums are order-sensitive; both scan orders of the reference are
// reproduced exactly (see blelloch_prefix_warp / object_lut_rows below).
#include <cstdlib>
#include "kernels.h"

namespace isx {

namespace {

// ---------------------------------------------------------------------------
// Static transition record S[vB], vB in [1, H):   (p = vB - 1)
//  0 pc      = ln(H - vB)                       GetPriorCost            (:40-42)
//  1 t1_hi   = max(gf[p],0) + eps               ObjectFromGround cases  (:120-144)
//  2 t1_lo   = max(gf[p],0) - eps
//  3 tr1_hi  4 tr1_mid  5 tr1_lo                its three finite values
//  6 sky_fg  = gf[p] < 1 ? pc : inf             SkyFromGround           (:98-106)
//  7 oo_base = pc + (p < vhor ? -ln .7 : ln 2)  ObjectFromObject prefix (:151-152)
//  8 tr3     = pc + ln(D - eps)                 ObjectFromSky           (:173-183)
//  9 g_prev  = -ln .3 + pc                      GetPriorCostGround      (:185-187)
// 10 sky_fo  = ln 2 + pc                        SkyFromObject           (:88-96)
// ---------------------------------------------------------------------------
__global__ void frame_tables_kernel(const float *__restrict__ ground, const int *__restrict__ vhor_arr,
                                    float *__restrict__ stat, KParams p) {
  const int f = blockIdx.y;
  const int vB = blockIdx.x * blockDim.x + threadIdx.x;
  const int H = p.rows;
  if (vB >= H) return;
  float *S = stat + ((size_t)f * H + vB) * kStatWords;
  if (vB == 0) {
    for (int i = 0; i < kStatWords; i++) S[i] = 0.0f;
    return;
  }
  const float *gf = ground + (size_t)f * 3 * H;
  const int vhor = vhor_arr[f];
  const int pv = vB - 1;
  const float eps = p.epsilon;

  // FFMA(lg2(H-vB), ln2, -0): the -__logf(1.0f) term folds to -0.
  const float pc = ffma(lg2_approx((float)(H - vB)), kLn2, -0.0f);
  const float fnp = clamp_neg(gf[pv]);
  const float t1_hi = fadd(fnp, eps);
  const float t1_lo = fsub(fnp, eps);
  const float og_base = fadd(pc, kNegLog07);
  const float tr1_hi = fadd(neg_log_div(p.pgrav, fsub(fadd(-fnp, p.max_disf), eps)), og_base);
  const float tr1_mid = fadd(neg_log_div(fsub(fadd(-p.pgrav, 1.0f), p.pblg), fadd(eps, eps)), og_base);
  const float tr1_lo = fadd(neg_log_div(p.pblg, t1_lo), og_base);
  const float sky_fg = (gf[pv] < 1.0f) ? pc : inf_f();
  const float oo_base = fadd(pc, (pv < vhor) ? kNegLog07 : kLn2);
  const float tr3 = fadd(pc, ffma(lg2_approx(fsub(p.max_disf, eps)), kLn2, -0.0f));
  const float g_prev = ffma(-kLn2, kLg2_03, pc);
  const float sky_fo = ffma(kLn2, 1.0f, pc);
  S[0] = pc;  S[1] = t1_hi;  S[2] = t1_lo;  S[3] = tr1_hi;  S[4] = tr1_mid;  S[5] = tr1_lo;
  S[6] = sky_fg;  S[7] = oo_base;  S[8] = tr3;  S[9] = g_prev;  S[10] = sky_fo;  S[11] = 0.0f;
}

// ---------------------------------------------------------------------------
// Blelloch-order exclusive prefix sum of e[0..H) (H <= 1024, TALL: H <= 2047), one warp.
//
// The reference scans in place with the classic work-efficient tree
// (StixelsKernels.h:73-103): block sums are pairwise trees U(.), and ps[i]
// folds, from the most to the least significant set bit of i,
//      prefix = prefix + U(aligned block that bit selects).
// A butterfly (shfl_xor) reproduces U(.) of every aligned block; the value a
// lane receives at level b while its bit b is set is exactly the U(left
// sibling) the down-sweep adds.  Levels 0-4 live inside a 32-row chunk,
// levels 5-9 across the (<= 32) chunk totals.  A taller tree only adds top
// levels that pass 0 to the left, so ps[i] does not depend on the padded size:
// TALL frames have a second group of 32 chunk totals (chunks 32-63), whose
// prefixes start from level 10, 0 + U(rows 0..1023).
// ---------------------------------------------------------------------------
template <bool TALL>
__device__ void blelloch_prefix_warp(const float *e, int H, float *ps) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const int nchunks = (H + 31) >> 5;
  float total_k = 0.0f;  // lane k: U(chunk k)
  float total2_k = 0.0f;  // TALL, lane k: U(chunk 32 + k)
  for (int k = 0; k < nchunks; k++) {
    const int v = (k << 5) + lane;
    float x = v < H ? e[v] : 0.0f;
#pragma unroll
    for (int b = 0; b < 5; b++) x = fadd(x, __shfl_xor_sync(full, x, 1 << b));
    if constexpr (TALL) {
      if (lane == (k & 31)) {
        if (k < 32) total_k = x;
        else total2_k = x;
      }
    } else {
      if (lane == k) total_k = x;
    }
  }
  float y = total_k, left[5];
#pragma unroll
  for (int b = 0; b < 5; b++) {
    const float o = __shfl_xor_sync(full, y, 1 << b);
    left[b] = o;
    y = fadd(y, o);
  }
  float hi = 0.0f;  // lane k: prefix of chunk k's first row
#pragma unroll
  for (int b = 4; b >= 0; b--)
    if ((lane >> b) & 1) hi = fadd(hi, left[b]);
  float hi2 = 0.0f;  // TALL, lane k: prefix of chunk 32 + k's first row
  if constexpr (TALL) {
    float y2 = total2_k, left2[5];
#pragma unroll
    for (int b = 0; b < 5; b++) {
      const float o = __shfl_xor_sync(full, y2, 1 << b);
      left2[b] = o;
      y2 = fadd(y2, o);
    }
    hi2 = fadd(0.0f, y);  // level 10: the root of the first 1024 rows
#pragma unroll
    for (int b = 4; b >= 0; b--)
      if ((lane >> b) & 1) hi2 = fadd(hi2, left2[b]);
  }
  const int kmax = H >> 5;  // chunk index of row H itself
  for (int k = 0; k <= kmax; k++) {
    const int v = (k << 5) + lane;
    float x = v < H ? e[v] : 0.0f;
    float lo[5];
#pragma unroll
    for (int b = 0; b < 5; b++) {
      const float o = __shfl_xor_sync(full, x, 1 << b);
      lo[b] = o;
      x = fadd(x, o);
    }
    float pre;
    if constexpr (TALL) {
      // H <= 2047: row H lies in chunk 63 or below, there is no root total to store
      pre = __shfl_sync(full, k < 32 ? hi : hi2, k & 31);
    } else {
      // k == 32 only for H == 1024, lane 0: the root total.
      pre = (k < 32) ? __shfl_sync(full, hi, k & 31) : y;
    }
#pragma unroll
    for (int b = 4; b >= 0; b--)
      if ((lane >> b) & 1) pre = fadd(pre, lo[b]);
    if (v <= H) ps[v] = pre;
  }
}

// Exact integer exclusive prefix sums (any order is bit-identical).
template <typename T>
__device__ void exact_prefix_warp(const T *e, int n, T *ps) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  T carry = 0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    T x = i < n ? e[i] : (T)0;
    T incl = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const T o = __shfl_up_sync(full, incl, d);
      if (lane >= d) incl += o;
    }
    if (i < n) ps[i] = carry + incl - x;
    carry += __shfl_sync(full, incl, 31);
  }
  if (lane == 0) ps[n] = carry;
}

constexpr int kTabThreads = 256;

// Dynamic shared memory carve-up (bytes), Hp = H + 1 rounded up to 4.
// Every array is scanned in place (a scan reads e[v] and writes ps[v] from the same lane; a 1/8-resolution channel
// value is recovered as ps[q + 1] - ps[q], exact in integers), and the sums of the instance means themselves are
// 32-bit (only their squares need 64): 50 KB per CTA at 1024 rows, so that FOUR CTAs share an SM (r1/r2a: 71 KB, three).
// Frames taller than 1024 rows need up to 100 KB (2047 rows): two CTAs per SM.
struct TabSmem {
  int Hp, nq;
  size_t off_e[4], off_seg, off_i64, off_i32, total;
  __host__ __device__ TabSmem(int H, int hs2) {
    Hp = (H + 1 + 3) & ~3;
    nq = H / 8 + 1;  // prefix entries per 1/8-res channel (index v>>3 for v <= H)
    size_t o = 0;
    off_i64 = o; o += (size_t)Hp * 8 * 2;
    off_i32 = o; o += (size_t)Hp * 4 * 2;
    for (int i = 0; i < 4; i++) { off_e[i] = o; o += (size_t)Hp * 4; }
    off_seg = o; o += (size_t)20 * (nq + 1) * 4;
    total = (o + 15) & ~(size_t)15;
    (void)hs2;
  }
};

// Integer guards of the table build, so that no int32 prefix sum can wrap (TALL: up to 2047 rows, 256 entries of a
// 1/8-resolution channel):
//   kMeanRowLimit: |instance mean of a row|; 1024 rows (TALL: 2047) of them stay below 2^30;
//   kClassLimit:   a class value; P_c(v) = 8 * ps[q] + seg[q] * r over <= 129 (TALL: 256) entries stays below 2^31;
//   kSqOffLimit:   each squared offset; their sum per entry is <= 2 * kSqOffLimit = kClassLimit.
template <bool TALL> struct TabLimits {
  static constexpr int kMeanRowLimit = TALL ? 1 << 19 : 1 << 20;
  static constexpr int kClassLimit = TALL ? 1 << 19 : 1 << 20;
  static constexpr int kSqOffLimit = TALL ? 1 << 18 : 1 << 19;
};

template <bool TALL>
__global__ void __launch_bounds__(kTabThreads, 4)
column_tables_kernel(const float *__restrict__ joined, const int32_t *__restrict__ segmentation,
                     const float *__restrict__ ground, const int *__restrict__ vhor_arr,
                     uint32_t *__restrict__ records_b, int *__restrict__ error_flag, int *__restrict__ col_flags,
                     KParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int H = p.rows, C = p.realcols;
  const int col = blockIdx.x, f = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const TabSmem L(H, p.hs2);
  float *e_disp = reinterpret_cast<float *>(smem + L.off_e[0]);
  float *e_valid = reinterpret_cast<float *>(smem + L.off_e[1]);
  float *e_ground = reinterpret_cast<float *>(smem + L.off_e[2]);
  float *e_sky = reinterpret_cast<float *>(smem + L.off_e[3]);
  // the four float arrays are contiguous and scanned in place: array i = e_disp + i * Hp
  long long *ps_i64 = reinterpret_cast<long long *>(smem + L.off_i64);    // [2][Hp]: sum mx^2, sum my^2
  int *ps_i32 = reinterpret_cast<int *>(smem + L.off_i32);                // [2][Hp]: sum mx, sum my
  int *seg_ps = reinterpret_cast<int *>(smem + L.off_seg);                // [20][nq+1]
  const int nq = L.nq, segld = nq + 1;

  const float *d_col = joined + ((size_t)f * C + col) * H;
  const int32_t *seg_col = segmentation + ((size_t)f * C + col) * p.n_channels * p.hs2;
  const float *gf = ground + (size_t)f * 3 * H;
  const float *norm_g = gf + H, *inv_g = gf + 2 * H;
  const int vhor = vhor_arr[f];
  const float invalid = p.invalid_disparity;
  const int K = p.n_classes;  // 19; channel K = y offsets, K+1 = x offsets
  const bool has_oy = K < p.n_channels, has_ox = K + 1 < p.n_channels;
  constexpr int kMeanRowLimit = TabLimits<TALL>::kMeanRowLimit;

  // ---- 1/8-resolution channels: the 19 classes, and as a 20th the sum of the two squared offsets (:411-416; the
  //      DP only ever uses the sum, ComputeNonInstanceOffsetCost :62-70).  Warp = channel, lane = entry: the loads of
  //      a thread are independent of each other (the first version waited for every load in turn). ----
  bool negative_class_value = false;
#pragma unroll
  for (int c = warp; c < 20; c += kTabThreads / 32) {
#pragma unroll 5
    for (int q = lane; q < nq; q += 32) {
      int v = 0;
      if (c < K) {
        if (c < p.n_channels && q < p.hs2) v = __ldg(seg_col + (size_t)c * p.hs2 + q);
        negative_class_value |= v < 0 || v > TabLimits<TALL>::kClassLimit;   // the int32 prefix sums cannot wrap
      } else {
        int oy = 0, ox = 0;
        if (q < p.hs2 && has_oy) oy = __ldg(seg_col + (size_t)K * p.hs2 + q);
        if (q < p.hs2 && has_ox) ox = __ldg(seg_col + (size_t)(K + 1) * p.hs2 + q);
        oy = oy * oy;
        ox = ox * ox;
        negative_class_value |= oy < 0 || oy > TabLimits<TALL>::kSqOffLimit || ox < 0 ||
                                ox > TabLimits<TALL>::kSqOffLimit;   // their sum: likewise
        v = oy + ox;
      }
      seg_ps[c * segld + q] = v;
    }
  }
  // ---- per-row terms (:371-446): four rows per thread, their loads first ----
  bool out_of_range = false;
  for (int v0 = tid; v0 < H; v0 += 4 * kTabThreads) {
    float d4[4], g0[4], gi[4], gn[4];
    int oy4[4], ox4[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int v = v0 + j * kTabThreads;
      const bool ok = v < H;
      const int q = v / kDownsample;
      d4[j] = ok ? __ldg(d_col + v) : 0.0f;
      oy4[j] = (ok && q < p.hs2 && has_oy) ? __ldg(seg_col + (size_t)K * p.hs2 + q) : 0;
      ox4[j] = (ok && q < p.hs2 && has_ox) ? __ldg(seg_col + (size_t)(K + 1) * p.hs2 + q) : 0;
      const bool gr = ok && v < vhor;
      g0[j] = gr ? __ldg(gf + v) : 0.0f;
      gi[j] = gr ? __ldg(inv_g + v) : 0.0f;
      gn[j] = gr ? __ldg(norm_g + v) : 0.0f;
    }
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int v = v0 + j * kTabThreads;
      if (v >= H) break;
      const float d = d4[j];
      if (invalid >= 0.0f) {
        const int va = d != invalid;
        e_valid[v] = (float)va;
        e_disp[v] = fmul((float)va, d);
      } else {
        e_valid[v] = 1.0f;  // unused by the reference in this mode (ComputeMean divides by the height)
        e_disp[v] = d;
      }
      // sky_lut: GetDataCostSky (:201-215), zero below the horizon (:424-433)
      float sky = 0.0f;
      if (v >= vhor) {
        sky = p.pnexists_given_sky_log;
        if (d != invalid) {
          const float g = ffma(fmul(d, d), p.inv_sigma2_sky, p.normalization_sky);
          sky = fadd(fmin_(g, p.puniform_sky), p.nopnexists_given_sky_log);
        }
      }
      e_sky[v] = sky;
      // ground_lut: GetDataCostGround (:217-234), +inf at/above the horizon (:437-446)
      float grd = inf_f();
      if (v < vhor) {
        grd = p.pnexists_given_ground_log;
        if (d != invalid) {
          const float diff = fsub(d, g0[j]);
          const float g = ffma(fmul(diff, diff), gi[j], gn[j]);
          grd = fadd(fmin_(g, p.puniform), p.nopnexists_given_ground_log);
        }
      }
      e_ground[v] = grd;
      // instance means (:400-409): C++ double arithmetic truncated toward zero
      const long long mx = (long long)((p.column_step * col + 0.5 * (p.column_step - 1.0)) + ox4[j] + 0.5);
      const long long my = (long long)(v - oy4[j] + 0.5);
      out_of_range |= mx <= -kMeanRowLimit || mx >= kMeanRowLimit || my <= -kMeanRowLimit || my >= kMeanRowLimit;
      ps_i32[0 * L.Hp + v] = (int)mx;
      ps_i32[1 * L.Hp + v] = (int)my;
      ps_i64[0 * L.Hp + v] = mx * mx;
      ps_i64[1 * L.Hp + v] = my * my;
    }
  }
  // The pruning DP kernels bound a segment's class sums from below by those of a shorter one, which needs
  // non-negative values whose int32 prefix sums do not wrap (they are trunc(8 * -log softmax) and squared pixel
  // offsets, wrappers.py:50-61); a column that breaks this is flagged and walked exhaustively.
  const int any_negative = __syncthreads_or(negative_class_value ? 1 : 0);
  if (tid == 0) col_flags[(size_t)f * C + col] = any_negative;

  // ---- prefix sums, in place: warps 0-3 float (Blelloch order), 4-5 int64, 6-7 int32; then all: 1/8-res ints ----
  if (warp < 4) {
    blelloch_prefix_warp<TALL>(e_disp + warp * L.Hp, H, e_disp + warp * L.Hp);
  } else if (warp < 6) {
    exact_prefix_warp<long long>(ps_i64 + (warp - 4) * L.Hp, H, ps_i64 + (warp - 4) * L.Hp);
  } else {
    exact_prefix_warp<int>(ps_i32 + (warp - 6) * L.Hp, H, ps_i32 + (warp - 6) * L.Hp);
  }
  // 20 channels over 8 warps: the integer warps (done first) take three each, the float warps two
  for (int c = 19 - ((warp + 4) & 7); c >= 0; c -= kTabThreads / 32)
    exact_prefix_warp<int>(seg_ps + c * segld, nq, seg_ps + c * segld);
  __syncthreads();

  // ---- records, v in [0, H]: one 128-byte row per v (common.cuh).  Eight lanes share a row, lane g writes words
  //      4g .. 4g+3 as one 16-byte store, so a warp instruction stores 512 contiguous bytes (four full lines).
  //      Groups 0-4 are the 20 integer words (one formula, evaluated by every lane: no branch), 5-7 the float words
  //      (one more branch for those three lanes, which select their words). ----
  uint4 *recb_col = reinterpret_cast<uint4 *>(records_b + ((size_t)f * C + col) * (size_t)p.rec_stride * kRecBWords);
  const long long lim2 = 1ll << (24 + kSqSplitBits);
  const int lim1 = 1 << 24;
  const long long lomask = (1ll << kSqSplitBits) - 1;
  // A thread keeps its lane group g and its row phase r = v & 7 for the whole loop (v advances by 32 rows), so what
  // depends on them is chosen once: the channel group of the integer words, the 64-bit sum a float lane splits, the
  // float arrays it copies.
  const int g = tid & 7, r = (tid >> 3) & 7;
  const int *ps_grp = seg_ps + (4 * (g < 5 ? g : 4)) * segld;
  const long long *ps_sq = ps_i64 + (g == 5 ? 0 : L.Hp);          // g == 5: sum mx^2, g == 6: sum my^2
  const float *pf_a = g == 6 ? e_disp : e_ground, *pf_b = g == 6 ? e_valid : e_sky;
#pragma unroll 2
  for (int v = tid >> 3; v <= H; v += kTabThreads / 8) {
    uint4 w;
    {
      // P_c(v) = 8*ps[q] + seg[q]*r  (Cityscapes.h:28-42), seg[q] = ps[q+1] - ps[q]; word 19 = the same for the
      // summed squared offsets
      const int *ps = ps_grp + (v >> 3);
      const int a0 = ps[0], a1 = ps[segld], a2 = ps[2 * segld], a3 = ps[3 * segld];
      w.x = (uint32_t)(a0 * kDownsample + (ps[1] - a0) * r);
      w.y = (uint32_t)(a1 * kDownsample + (ps[segld + 1] - a1) * r);
      w.z = (uint32_t)(a2 * kDownsample + (ps[2 * segld + 1] - a2) * r);
      w.w = (uint32_t)(a3 * kDownsample + (ps[3 * segld + 1] - a3) * r);
    }
    if (g >= 5) {
      // instance-mean sums as exactly representable floats (see common.cuh): words 20 .. 25; float sums: 26 .. 29
      const int smx = ps_i32[0 * L.Hp + v], smy = ps_i32[1 * L.Hp + v];
      const long long sq = ps_sq[v];
      out_of_range |= (g == 5 && (smx <= -lim1 || smx >= lim1 || smy <= -lim1 || smy >= lim1)) || (g != 7 && sq >= lim2);
      const float hi = (float)(sq & ~lomask), lo = (float)(sq & lomask);
      const float fa = pf_a[v], fb = pf_b[v];
      w.x = __float_as_uint(g == 5 ? (float)smx : g == 6 ? hi : fa);
      w.y = __float_as_uint(g == 5 ? (float)smy : g == 6 ? lo : fb);
      w.z = g == 7 ? 0u : __float_as_uint(g == 5 ? hi : fa);
      w.w = g == 7 ? 0u : __float_as_uint(g == 5 ? lo : fb);
    }
    recb_col[v * (kRecBWords / 4) + g] = w;
  }
  if (out_of_range) atomicOr(error_flag + f, kErrOffsetRange);
}

// ---------------------------------------------------------------------------
// Object-cost LUT (ComputeObjectLUT, StixelsKernels.cu:236-296, 959-978):
//   LUT[fn][v+1] = sum_{r<=v} obj_cost_lut[fn][(int)d[r]]
// in the reference's summation order (warp_prefix_sum / ComputePrefixSumWarp2): 32-row chunks, the
// running total joins row 0 of the chunk BEFORE a Kogge-Stone scan (lane L: x += x[L-j], j = 1,2,4,8,16).
//
// The reference runs that scan across the lanes of a warp (5 shuffles per chunk and fn row), which made
// the first version of this kernel LSU-bound.  Here one THREAD owns a whole chunk of one fn row: its 32
// values sit in registers, the Kogge-Stone network is 129 FADDs in exactly the reference's association,
// and the chunk carry is a register.  A warp covers 32 consecutive fn rows (lane = fn), reads the
// transposed cost table [dis][fn] (one 128-byte line per row of the chunk) and transposes its 32 x 32
// result tile through shared memory so that every store is a full 128-byte line of one fn row.
// ---------------------------------------------------------------------------
constexpr int kLutWarps = 4;
constexpr int kLutThreads = kLutWarps * 32;

// 32-bit address arithmetic for the two address streams of the kernel (the same trick as the DP's LUT gathers,
// dp.cu): the transposed cost table (64 KB) and one column of the object LUT (< 4 GB, never straddling a multiple of
// 4 GB: lut_column_address) each keep ONE upper address word, so an address costs one IMAD / IADD instead of the
// five instructions of a 64-bit multiply-add (the first version spent 8 instructions per gather, 5 per store).
__device__ __forceinline__ float ldg_lo_hi(unsigned lo, unsigned hi) {
  float r;
  asm("{\n\t.reg .b64 a;\n\tmov.b64 a, {%1, %2};\n\tld.global.nc.f32 %0, [a];\n\t}" : "=f"(r) : "r"(lo), "r"(hi));
  return r;
}
__device__ __forceinline__ void stg_lo_hi(unsigned lo, unsigned hi, float v) {
  asm volatile("{\n\t.reg .b64 a;\n\tmov.b64 a, {%0, %1};\n\tst.global.f32 [a], %2;\n\t}" ::"r"(lo), "r"(hi), "f"(v)
               : "memory");
}

// MAXH: the largest frame height of the instantiation (1024, or 2048 for frames of up to 2047 rows: up to 64 chunk
// carries per LUT row)
template <int MAXH>
__global__ void __launch_bounds__(kLutThreads)
object_lut_kernel(const float *__restrict__ joined, const float *__restrict__ cost_t,
                  float *__restrict__ object_lut, KParams p) {
  __shared__ __align__(16) uint8_t dis_s[MAXH + 32];
  __shared__ float tile[kLutWarps][32][33];
  const int H = p.rows, C = p.realcols, D = p.max_dis;
  const int Dp = (D + 31) & ~31;
  const int col = blockIdx.x, f = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float *d_col = joined + ((size_t)f * C + col) * H;
  const int Hc = (H + 31) & ~31;
  for (int v = threadIdx.x; v < Hc; v += kLutThreads) {
    int di = 0;  // rows past H count as disparity 0, like the reference's padded loop (:262-272)
    if (v < H) {
      di = (int)d_col[v];  // (int) d as LUT index (:246-248)
      di = di < 0 ? 0 : (di >= D ? D - 1 : di);
    }
    dis_s[v] = (uint8_t)di;
  }
  __syncthreads();
  const int fn0 = (blockIdx.y * kLutWarps + warp) * 32;
  if (fn0 >= D) return;
  const unsigned long long lut_addr = lut_column_address((unsigned long long)object_lut, (size_t)f * C + col,
                                                         p.lut_cols, (size_t)D * p.lut_stride * 4);
  const unsigned lut_hi = (unsigned)(lut_addr >> 32);
  const unsigned stride4 = (unsigned)p.lut_stride * 4u;
  // column fn of the transposed table (padded to 32 columns, always in range); the table does not straddle 4 GB
  // (isx_initialize checks), so its upper address word is that of its first byte
  const unsigned long long cost_addr = (unsigned long long)(cost_t + fn0 + lane);
  const unsigned cost_lo = (unsigned)cost_addr, cost_hi = (unsigned)(cost_addr >> 32);
  const unsigned row4 = (unsigned)Dp * 4u;   // bytes per disparity row of the transposed table
  float(*tl)[33] = tile[warp];
  const bool full = fn0 + 32 <= D;           // every row of the 32 x 32 tile exists (D is a multiple of 32)
  float carry = 0.0f;
  for (int i = 0; i < Hc; i += 32) {
    float x[32];
    const uint4 *dq = reinterpret_cast<const uint4 *>(dis_s + i);
    const uint4 d0 = dq[0], d1 = dq[1];
    const uint32_t dw[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
    for (int r = 0; r < 32; r++) {
      const unsigned dis = __byte_perm(dw[r >> 2], 0u, 0x4440u | (unsigned)(r & 3));   // byte r & 3, zero-extended
      x[r] = ldg_lo_hi(dis * row4 + cost_lo, cost_hi);
    }
    x[0] = fadd(x[0], carry);
#pragma unroll
    for (int j = 1; j < 32; j <<= 1) {
#pragma unroll
      for (int L = 31; L >= j; L--) x[L] = fadd(x[L], x[L - j]);
    }
    carry = x[31];
    __syncwarp();
#pragma unroll
    for (int r = 0; r < 32; r++) tl[lane][r] = x[r];
    __syncwarp();
    const int v = i + lane;
    if (v < H) {
      unsigned lo = (unsigned)lut_addr + (unsigned)fn0 * stride4 + 4u * (unsigned)v;   // out[v] = LUT[fn][v + 1]
      if (full) {
#pragma unroll
        for (int r = 0; r < 32; r++) {
          stg_lo_hi(lo, lut_hi, tl[r][lane]);
          lo += stride4;
        }
      } else {
#pragma unroll
        for (int r = 0; r < 32; r++) {
          if (fn0 + r < D) stg_lo_hi(lo, lut_hi, tl[r][lane]);
          lo += stride4;
        }
      }
    }
  }
}

}  // namespace

void launch_frame_tables(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s) {
  dim3 grid((p.rows + 255) / 256, nframes);
  frame_tables_kernel<<<grid, 256, 0, s>>>(b.ground, b.vhor, b.stat, p);
  g_launch_count++;
}

static size_t tab_smem_bytes(const KParams &p) { return TabSmem(p.rows, p.hs2).total; }

// ISX_TAB_CTAS_PER_SM=n (experiments): pads the dynamic shared memory of the table kernels so that at most n of their
// CTAs are resident per SM -- with the table stream above the DP's priority (ISX_TABLES_PRIO=1) the HBM-bound table
// CTAs then sit BESIDE the issue-bound DP CTAs instead of replacing them.
static size_t padded_smem(size_t need, size_t static_bytes) {
  static const int n = [] {
    const char *e = std::getenv("ISX_TAB_CTAS_PER_SM");
    return e ? std::atoi(e) : 0;
  }();
  if (n <= 0) return need;
  const size_t per_cta = (size_t)(227 * 1024) / (size_t)(n + 1) + 1024;  // n fit, n + 1 do not
  const size_t want = per_cta > static_bytes + 1024 ? per_cta - static_bytes - 1024 : 0;   // 1 KB reserved per CTA
  return want > need ? want : need;
}

template <bool TALL>
static void launch_column_tables_rows(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s) {
  constexpr int kLutMaxH = TALL ? 2048 : 1024;
  dim3 grid(p.realcols, nframes);
  const size_t smem = padded_smem(tab_smem_bytes(p), 0);
  static SmemOptIn optin, optin_lut;
  opt_in_smem(column_tables_kernel<TALL>, optin);
  opt_in_smem(object_lut_kernel<kLutMaxH>, optin_lut);
  column_tables_kernel<TALL><<<grid, kTabThreads, smem, s>>>(b.joined, b.segmentation, b.ground, b.vhor, b.records_b,
                                                              b.error_flag, b.col_flags, p);
  dim3 lgrid(p.realcols, (p.max_dis + 32 * kLutWarps - 1) / (32 * kLutWarps), nframes);
  object_lut_kernel<kLutMaxH><<<lgrid, kLutThreads, padded_smem(0, sizeof(float) * kLutWarps * 32 * 33 + kLutMaxH + 32), s>>>(
      b.joined, b.obj_cost_lut_t, b.object_lut, p);
  g_launch_count += 2;
}

void launch_column_tables(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s) {
  if (p.rows > kShortRows) launch_column_tables_rows<true>(p, b, nframes, s);
  else launch_column_tables_rows<false>(p, b, nframes, s);
}

}  // namespace isx
