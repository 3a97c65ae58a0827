// The ground/object/sky dynamic program over one stixel column.
// Replaces the first-segment block and the vB loop of StixelsKernel<PAIRWISE>
// (InstanceStixels/src/StixelsKernels.cu:477-839).
//
// The column's rows are cut into tiles of 32 top rows (lane l of a warp owns vT = a + l) and into chunks of 32
// candidate bottom rows vB.  A (tile, chunk) pair with tile >= chunk is one unit of work: 32 x 32 DP cells,
// evaluated by one warp with the records R[vT+1] of its rows in 30 registers ("A side", each lane reads its own
// 128-byte row) and the records R[vB] of the chunk in shared memory ("B side", the same rows as one 4 KB bulk
// async copy per chunk: cp.async.bulk + mbarrier).  Because one of GROUND/SKY is +inf for every row (ground only
// exists below the horizon, sky only at/above it) the cost table keeps two slots per row: "gs" (ground if
// vT < vhor else sky) and "object".  No tensor cores: the recurrence is min-plus, not a dense contraction.
//
// Three kernels share the cell arithmetic below (cell_base / cell_finish / dp_steps):
//
//  dp_kernel<PAIRWISE>        chunk-major, every unit.  One CTA (4 or 8 warps) per column; the chunk's B records sit
//                             in a ring of shared-memory slots, units are drawn from shared-memory counters chunk by
//                             chunk (lowest tile first), a tile's running (cost, vB) minima are handed from unit
//                             (t, j-1) to (t, j) through the output array; in pairwise mode the diagonal units
//                             (tile == chunk) form the serial chain of the column (row vB-1 final -> transition
//                             scalars Q[vB] -> row vB) and are taken the moment their tile is complete.  Strict '<'
//                             in ascending vB order is the reference's tie rule (lowest vB wins).
//                             Used for small pairwise launches, and as the exhaustive reference of the other two.
//  dp_unary_pruned_kernel     unary mode: a warp owns a tile and walks its chunks downwards from the diagonal until
//                             a lower bound proves that nothing below can win (exact branch and bound).
//  dp_pairwise_walk_kernel    pairwise mode: one warp per column, tile by tile behind the diagonal chain, each
//                             off-diagonal unit only if its lower bound does not exceed the carried minima.
// Both pruning kernels return the same bytes as dp_kernel (tests/test_gpu_parity.py); their headers derive the bounds.
#include <cstdlib>

#include "dp_common.cuh"
#include "kernels.h"

namespace isx {

std::atomic<unsigned long long> g_launch_count{0};

namespace {

// Warps per column CTA: 4 for throughput (4-5 CTAs per SM); 8 when a launch has fewer columns than
// two per SM (single frames), where the latency of one column is what the caller waits for.
constexpr int kDpWarps = 4;
constexpr int kDpWarpsLatency = 8;
constexpr int kSstBufs = 2;    // staged static transition records: diagonal j uses buffer j & 1
constexpr int kChunk = 32;
constexpr int kStages = 4;     // ring slots of 4 KB
constexpr int kPrefetch = 2;   // chunks the producer runs ahead (< kStages)
// steps per iteration of the inner loop (2 or 4) and resident CTAs per SM the register budget aims at
#ifndef ISX_UNARY_UNROLL
#define ISX_UNARY_UNROLL 2
#endif
#ifndef ISX_UNARY_CTAS
#define ISX_UNARY_CTAS 5
#endif
// whether the dead-ground-slot variant of the inner loop is instantiated
#ifndef ISX_DEAD_SLOT
#define ISX_DEAD_SLOT(pairwise) true
#endif
#ifndef ISX_PAIRWISE_UNROLL_DEAD
#define ISX_PAIRWISE_UNROLL_DEAD 4
#endif
#ifndef ISX_PAIRWISE_CTAS
#define ISX_PAIRWISE_CTAS 4
#endif
// pairwise (128 registers): the dead-slot loop (45 % of the units) is unrolled by four, the others by two
#ifndef ISX_PAIRWISE_UNROLL
#define ISX_PAIRWISE_UNROLL 2
#endif
constexpr int kSlotWords = kChunk * kRecBWords;
constexpr int kSlotBytes = kSlotWords * 4;
constexpr int kSstWords = ((kChunk + 1) * kStatWords + 3) & ~3;  // staged static transition records of a chunk

struct DpConsts {
  float pw, dw, sw, iw;
  float dm1f;            // max_dis - 1 as float (LUT row clamp)
  unsigned lut_stride4;  // bytes per fn row of the object LUT
  unsigned lut_hi;       // upper 32 address bits of this column's LUT (it never straddles 4 GB, common.cuh)
  float epsilon;
};

// LUT gather with a 32-bit computed low address word: {lo, hi} + OFF.  The immediate is added by
// the load unit in 64 bits, so it may carry; lo itself is exact modulo 2^32 inside the column.
template <int OFF>
__device__ __forceinline__ float ldg_lut(unsigned lo, unsigned hi) {
  float r;
  asm("{\n\t.reg .b64 a;\n\tmov.b64 a, {%1, %2};\n\tld.global.nc.f32 %0, [a+%3];\n\t}"
      : "=f"(r)
      : "r"(lo), "r"(hi), "n"(OFF));
  return r;
}

__device__ __forceinline__ float f_(uint32_t u) { return __uint_as_float(u); }

// A side of a unit: the record of this lane's row vT + 1, one 128-byte row of the row-major records (eight 16-byte
// loads per lane; a warp touches 32 consecutive lines).  A pruning kernel loads it once per TILE, not per unit.
__device__ __forceinline__ void load_a_side(uint32_t (&A)[kRecWords], const uint32_t *__restrict__ recb, int row) {
  const uint4 *r4 = reinterpret_cast<const uint4 *>(recb + (size_t)row * kRecBWords);
#pragma unroll
  for (int g = 0; g < (kRecWords + 3) / 4; g++) {
    const uint4 t = __ldg(r4 + g);
    A[4 * g] = t.x;
    A[4 * g + 1] = t.y;
    if (4 * g + 2 < kRecWords) A[4 * g + 2] = t.z;
    if (4 * g + 3 < kRecWords) A[4 * g + 3] = t.w;
  }
}
// one word of one row of the row-major records
__device__ __forceinline__ uint32_t rec_word(const uint32_t *__restrict__ recb, int row, int word) {
  return __ldg(recb + (size_t)row * kRecBWords + word);
}

// ---- mbarrier / bulk-copy primitives (PTX; SASS: SYNCS.*, UBLKCP) ----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, 0x989680;\n\t"
      "@P1 bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- one DP cell per lane: segment (vB .. vT) of this lane's row vT ----
// The chain-independent part: everything that does not need the costs of row vB - 1.
struct CellBase {
  float seg_gs, data_gs, seg_o, data_o, fn;
};

//   A : R[vT+1] in registers,  brow: R[vB] in shared memory (warp-uniform address)
//   nf: segment height as float;  ca / cb: biased low address words of LUT[0][vT] / LUT[0][vB-1]
//   (cb + BOFF addresses row vB - 1; BOFF is the compile-time part of the unrolled step)
// GROUND: 1 = ground side, 0 = sky side, 2 = decided at run time by `ground_rt` (diagonal units),
//         3 = ground side of a tile that lies entirely at/above the horizon: the ground prefix of every row
//             of the tile is +inf (ground_lut, StixelsKernels.cu:437-446), so the ground slot can never win
//             and its terms are not evaluated
// The object-LUT gather of one cell: segment mean -> LUT row -> the two gathered prefix values.  It comes first in
// the cell so that the two L2 gathers are in flight while the rest of the cell is evaluated (pairwise 37.2 -> 35.6 ms
// per 64 frames against the order "semantic terms first"; issuing them a whole iteration ahead cost more in extra
// moves and loads than it hid).
struct LutFetch {
  float fn, hi, lo;
};

//   a_disp / a_valid: words kRecDisp / kRecValid of R[vT+1];  brow: R[vB] in shared memory
template <bool FIRST, bool HAS_INVALID, int BOFF>
__device__ __forceinline__ LutFetch lut_fetch(uint32_t a_disp, uint32_t a_valid, const uint32_t *__restrict__ brow,
                                              unsigned ca, unsigned cb, float nf, const DpConsts &c) {
  // ---- disparity terms: ComputeMean (:47-60) + clamp (:651-653) ----
  const float sd = fsub(f_(a_disp), f_(brow[kRecDisp]));
  float mean;
  if constexpr (HAS_INVALID) {
    const float vd = fsub(f_(a_valid), f_(brow[kRecValid]));
    const float m = fmul(sd, rcp_approx(vd));
    mean = (vd != 0.0f) ? m : 0.0f;
  } else {
    mean = fmul(sd, rcp_approx(nf));
  }
  LutFetch F;
  F.fn = fmaxf(mean, 0.0f);  // == clamp_neg for every comparison downstream (mean is never NaN)
  // floor(fn) as LUT row: add.rz of 2^23 leaves floor(fn) in the mantissa; ca / cb are the low
  // address words of LUT[0][vT] / LUT[0][vB-1] minus 0x4B000000 rows (mod 2^32), so one 32-bit
  // multiply-add (IMAD) forms each address; the upper word is constant per column.
  const float fbias = __fadd_rz(fminf(F.fn, c.dm1f), 8388608.0f);
  const unsigned roff = (unsigned)__float_as_int(fbias) * c.lut_stride4;
  F.hi = ldg_lut<0>(roff + ca, c.lut_hi);
  F.lo = FIRST ? 0.0f : ldg_lut<BOFF>(roff + cb, c.lut_hi);
  return F;
}

template <bool FIRST, int GROUND, bool HAS_INVALID, int BOFF = 0>
__device__ __forceinline__ CellBase cell_base(const uint32_t (&A)[kRecWords], const uint32_t *__restrict__ brow,
                                              unsigned ca, unsigned cb, float nf, const DpConsts &c,
                                              bool ground_rt = true) {
  const bool ground = GROUND == 2 ? ground_rt : GROUND != 0;
  constexpr bool kGsDead = GROUND == 3;
  const LutFetch F = lut_fetch<FIRST, HAS_INVALID, BOFF>(A[kRecDisp], A[kRecValid], brow, ca, cb, nf, c);
  uint32_t Bw[32];
  {
    const uint4 *b4 = reinterpret_cast<const uint4 *>(brow);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const uint4 t = b4[k];
      Bw[4 * k] = t.x; Bw[4 * k + 1] = t.y; Bw[4 * k + 2] = t.z; Bw[4 * k + 3] = t.w;
    }
  }
  // ---- semantic sums (Cityscapes.h:28-123), exact ints; min commutes with the
  //      monotone int->float conversion and the float add of the offset term ----
  int s_ni = (int)(A[2] - Bw[2]);
#pragma unroll
  for (int k = 3; k < 10; k++) s_ni = min(s_ni, (int)(A[k] - Bw[k]));
  int s_in = (int)(A[11] - Bw[11]);
#pragma unroll
  for (int k = 12; k < 19; k++) s_in = min(s_in, (int)(A[k] - Bw[k]));
  const int s_off = (int)(A[kRecOff] - Bw[kRecOff]);
  const int s_gs = kGsDead ? 0 : ground ? min((int)(A[0] - Bw[0]), (int)(A[1] - Bw[1])) : (int)(A[kSkyClass] - Bw[kSkyClass]);
  const float f_off = (float)s_off;
  const float nic = fmul(f_off, c.iw);  // ComputeNonInstanceOffsetCost * weight (:618-621)

  // ---- instance variance term (:72-86, 611-616); float prefixes reproduce I2F.S64(diff) ----
  const float rn = rcp_approx(nf);
  const float fmx = fsub(f_(A[kRecMx]), f_(Bw[kRecMx]));
  const float fmy = fsub(f_(A[kRecMy]), f_(Bw[kRecMy]));
  const float fmx2 = fadd(fsub(f_(A[kRecMx2Hi]), f_(Bw[kRecMx2Hi])), fsub(f_(A[kRecMx2Lo]), f_(Bw[kRecMx2Lo])));
  const float fmy2 = fadd(fsub(f_(A[kRecMy2Hi]), f_(Bw[kRecMy2Hi])), fsub(f_(A[kRecMy2Lo]), f_(Bw[kRecMy2Lo])));
  const float var = ffma(-fmul(fmy, fmy), rn, fadd(fmy2, ffma(-fmul(fmx, fmx), rn, fmx2)));
  const float ic = fmul(var, c.iw);
  CellBase b;
  b.seg_o = fmin_(fadd(nic, (float)s_ni), fadd(ic, (float)s_in));
  // In the first-segment block nvcc contracted `min(road, sidewalk) + weight * offsets` into one
  // FFMA (reference SASS of StixelsKernels.cu:502-506); everywhere else it is FMUL + FADD.
  b.seg_gs = kGsDead ? 0.0f : FIRST ? ffma(f_off, c.iw, (float)s_gs) : fadd(nic, (float)s_gs);
  b.fn = F.fn;
  b.data_o = fsub(F.hi, F.lo);
  b.data_gs = kGsDead ? 0.0f : ground ? fsub(f_(A[kRecGround]), f_(Bw[kRecGround])) : fsub(f_(A[kRecSky]), f_(Bw[kRecSky]));
  return b;
}

// Prior + combine (:548-560, 575-584, 700-720, 740-766, 788-824).
template <bool PAIRWISE, bool FIRST, int GROUND>
__device__ __forceinline__ void cell_finish(const CellBase &b, float ih, const RowInfo &q, float first_k_gs,
                                            float first_k_o, const DpConsts &c, float &cost_gs, float &cost_o,
                                            bool ground_rt = true) {
  const bool ground = GROUND == 2 ? ground_rt : GROUND != 0;
  if constexpr (GROUND == 3) {
    // the ground slot is dead (see cell_base): only the object slot
    float k_o = 0.0f;
    if constexpr (PAIRWISE) {
      float p1, p2, p3;
      object_priors(q, true, b.fn, c.epsilon, p1, p2, p3);
      k_o = fmul(fmin_(p3, fmin_(p1, p2)), c.pw);
      cost_o = ffma(b.seg_o, c.sw, ffma(b.data_o, c.dw, k_o));
    } else {
      cost_o = ffma(b.seg_o, c.sw, ffma(ih, c.pw, fmul(b.data_o, c.dw)));
    }
    cost_gs = inf_f();
    return;
  }
  if constexpr (PAIRWISE) {
    float k_gs, k_o;
    if constexpr (FIRST) {
      k_gs = first_k_gs;
      k_o = first_k_o;
    } else {
      float p1, p2, p3;
      object_priors(q, ground, b.fn, c.epsilon, p1, p2, p3);
      k_gs = q.gs_k;
      k_o = fmul(fmin_(p3, fmin_(p1, p2)), c.pw);
    }
    cost_gs = ffma(b.seg_gs, c.sw, ffma(b.data_gs, c.dw, k_gs));
    cost_o = ffma(b.seg_o, c.sw, ffma(b.data_o, c.dw, k_o));
  } else {
    cost_gs = ffma(b.seg_gs, c.sw, ffma(ih, c.pw, fmul(b.data_gs, c.dw)));
    cost_o = ffma(b.seg_o, c.sw, ffma(ih, c.pw, fmul(b.data_o, c.dw)));
  }
}

__device__ __forceinline__ RowInfo load_row_info(const float *__restrict__ qrow) {
  const float4 *qd = reinterpret_cast<const float4 *>(qrow);
  const float4 q0 = qd[0], q1 = qd[1], q2 = qd[2];
  RowInfo q;
  q.gs_k = q0.x; q.a1 = q0.y; q.a2 = q0.z; q.a3 = q0.w;
  q.a4 = q1.x; q.a5 = q1.y; q.p2_hi = q1.z; q.p2_lo = q1.w;
  q.p2_mid = q2.x; q.t2_hi = q2.y; q.t2_lo = q2.z; q.pm = q2.w;
  return q;
}

__device__ __forceinline__ void store_row_info(float *qrow, const RowInfo &q) {
  float4 *qd = reinterpret_cast<float4 *>(qrow);
  qd[0] = make_float4(q.gs_k, q.a1, q.a2, q.a3);
  qd[1] = make_float4(q.a4, q.a5, q.p2_hi, q.p2_lo);
  qd[2] = make_float4(q.p2_mid, q.t2_hi, q.t2_lo, q.pm);
}

struct Best {
  float gs, o;
  int vb_gs, vb_o;
};

// Steps [k0, k1) of one unit; the whole range lies on one side of the horizon.
//   DIAG (unary only): tile == chunk, lane l is live for k <= l only (vT >= vB).
// One step: U = position inside the manually unrolled pair (compile-time LUT / record offsets).
template <bool PAIRWISE, int GROUND, bool DIAG, bool HAS_INVALID, int U>
__device__ __forceinline__ void dp_step(const uint32_t (&A)[kRecWords], const uint32_t *__restrict__ brow,
                                        unsigned ca, unsigned cb, const float *__restrict__ ihs,
                                        const float *__restrict__ ihp, int nk, const float *__restrict__ qrow,
                                        int vB, int k, int lane, float nf, const DpConsts &c, Best &best) {
  // dead lanes of the diagonal unit (vT < vB) evaluate a harmless dummy cell of height >= 1
  const float nfc = DIAG ? fmaxf(nf, 1.0f) : nf;
  RowInfo q{};
  float ih = 0.0f;
  if constexpr (PAIRWISE) q = load_row_info(qrow + U * kDynWords);
  else ih = DIAG ? ihs[max(nk - U, 1)] : ihp[-U];  // ihp = ihs + nk, nk = vT + 1 - vB of step U = 0
  const CellBase b = cell_base<false, GROUND, HAS_INVALID, 4 * U>(A, brow + U * kRecBWords, ca, cb, nfc, c);
  float cost_gs, cost_o;
  cell_finish<PAIRWISE, false, GROUND>(b, ih, q, 0.0f, 0.0f, c, cost_gs, cost_o);
  const bool live = !DIAG || lane >= k;
  if (GROUND != 3 && live && cost_gs < best.gs) { best.gs = cost_gs; best.vb_gs = vB; }
  if (live && cost_o < best.o) { best.o = cost_o; best.vb_o = vB; }
}

template <bool PAIRWISE, int GROUND, bool DIAG, bool HAS_INVALID>
__device__ __forceinline__ void dp_steps(const uint32_t (&A)[kRecWords], const uint32_t *__restrict__ bchunk,
                                         unsigned cb0, unsigned ca, const float *__restrict__ ihs,
                                         const float *__restrict__ qs, int vb0, int k0, int k1, int n0, int lane,
                                         const DpConsts &c, Best &best) {
  float nf = (float)(n0 - k0);  // segment height vT + 1 - vB, kept as a float counter
  const float *ihp = ihs + (n0 - k0);
  unsigned cb = cb0 + 4u * (unsigned)k0;
  const uint32_t *brow = bchunk + k0 * kRecBWords;
  const float *qrow = qs + k0 * kDynWords;
  constexpr int kDpUnroll = PAIRWISE ? (GROUND == 3 ? ISX_PAIRWISE_UNROLL_DEAD : ISX_PAIRWISE_UNROLL) : ISX_UNARY_UNROLL;
  int k = k0;
#define ISX_DP_STEP(U)                                                                                          \
  dp_step<PAIRWISE, GROUND, DIAG, HAS_INVALID, U>(A, brow, ca, cb, ihs, ihp, n0 - k, qrow, vb0 + k + U, k + U, lane, \
                                                  U == 0 ? nf : fadd(nf, -(float)U), c, best)
  for (; k + kDpUnroll <= k1; k += kDpUnroll) {
    ISX_DP_STEP(0);
    ISX_DP_STEP(1);
    if constexpr (kDpUnroll == 4) {
      ISX_DP_STEP(2);
      ISX_DP_STEP(3);
    }
    nf = fadd(nf, -(float)kDpUnroll);
    ihp -= kDpUnroll;
    cb += 4u * kDpUnroll;
    brow += kDpUnroll * kRecBWords;
    qrow += kDpUnroll * kDynWords;
  }
  for (; k < k1; k++) {
    ISX_DP_STEP(0);
    nf = fadd(nf, -1.0f);
    ihp -= 1;
    cb += 4u;
    brow += kRecBWords;
    qrow += kDynWords;
  }
#undef ISX_DP_STEP
}

// Shared-memory carve-up (bytes).  Kept small on purpose: shared memory and L1 share one 228 KB array,
// and the object-LUT gathers of four resident column CTAs live in what is left.
struct DpLayout {
  int nt;
  size_t off_ring, off_bars, off_cnt, off_ih, off_qs, off_qnext, off_sst, off_odr, total;
  __host__ __device__ DpLayout(int H, int D, bool pairwise) {
    nt = (H + kChunk - 1) / kChunk;
    size_t o = 0;
    off_ring = o; o += (size_t)kStages * kSlotBytes;
    off_bars = o; o += (size_t)2 * kStages * 8;            // full[kStages] | qfull[kStages]
    off_cnt = o; o += (size_t)(3 * nt + 1) * 4;            // per chunk: units handed out | finished; per tile: chunks done; next diagonal
    o = (o + 15) & ~(size_t)15;
    off_ih = off_qs = off_qnext = off_sst = off_odr = o;
    if (!pairwise) {
      off_ih = o; o += (size_t)(H + 1) * 4;
    } else {
      off_qs = o; o += (size_t)kStages * kChunk * kDynWords * 4;
      off_qnext = o; o += (size_t)2 * kDynWords * 4;
      off_sst = o; o += (size_t)kSstBufs * kSstWords * 4;    // one diagonal runs at a time; the next may already stage
      off_odr = o; o += (size_t)((D + 3) & ~3) * 4;
    }
    total = (o + 15) & ~(size_t)15;
  }
};

__device__ __forceinline__ Best load_best(const float4 *p) {
  const float4 v = __ldcg(p);  // L2: written by another warp of this CTA (st.cg + fence + flag)
  return Best{v.x, v.y, __float_as_int(v.z), __float_as_int(v.w)};
}
__device__ __forceinline__ void store_best(float4 *p, const Best &b) {
  __stcg(p, make_float4(b.gs, b.o, __int_as_float(b.vb_gs), __int_as_float(b.vb_o)));
}

template <bool PAIRWISE, bool HAS_INVALID, int WARPS, int HP>
__global__ void __launch_bounds__(WARPS * 32, WARPS == kDpWarps ? (PAIRWISE ? ISX_PAIRWISE_CTAS : ISX_UNARY_CTAS) : 2)
dp_kernel(const uint32_t *__restrict__ records_b,
          const float *__restrict__ object_lut, const float *__restrict__ stat, float *__restrict__ pm_out,
          const int *__restrict__ vhor_arr, const float *__restrict__ object_disparity_range,
          const float *__restrict__ inverse_height, float4 *dp_out, KParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int kDpThreads = WARPS * 32;
  const unsigned full_mask = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31;
  const int gcol = blockIdx.x;  // frame * C + column
  const int H = p.rows, C = p.realcols;
  constexpr int Hp = HP;  // == p.rec_stride; a constant so that the A-side word offsets are immediates
  const int f = gcol / C;
  const int vhor = vhor_arr[f];
  const float inf = inf_f();
  const DpLayout L(H, p.max_dis, PAIRWISE);
  const int nt = L.nt;

  uint32_t *ring = reinterpret_cast<uint32_t *>(smem_raw + L.off_ring);
  uint64_t *bar_full = reinterpret_cast<uint64_t *>(smem_raw + L.off_bars);
  uint64_t *bar_q = bar_full + kStages;
  int *cnt_out = reinterpret_cast<int *>(smem_raw + L.off_cnt);  // [nt] units handed out, per chunk
  int *cnt_fin = cnt_out + nt;                                    // [nt] units finished, per chunk
  int *tile_done = cnt_fin + nt;                                  // [nt] chunks finished, per tile
  int *diag_next = tile_done + nt;                                // next diagonal unit to run (pairwise)
  float *ihs = reinterpret_cast<float *>(smem_raw + L.off_ih);
  float *qs = reinterpret_cast<float *>(smem_raw + L.off_qs);
  float *qnext = reinterpret_cast<float *>(smem_raw + L.off_qnext);
  float *sst = reinterpret_cast<float *>(smem_raw + L.off_sst);
  float *odr = reinterpret_cast<float *>(smem_raw + L.off_odr);

  DpConsts c;
  c.pw = p.prior_weight; c.dw = p.disparity_weight; c.sw = p.segmentation_weight; c.iw = p.instance_weight;
  c.dm1f = (float)(p.max_dis - 1);
  c.lut_stride4 = (unsigned)p.lut_stride * 4u;
  c.epsilon = p.epsilon;

  const uint32_t *recb = records_b + (size_t)gcol * Hp * kRecBWords;
  // low / high address words of LUT[0][0] of this column; the low word carries the -2^23-rows bias of
  // the float -> row trick in cell_base (all modulo 2^32)
  const unsigned long long lut_addr = lut_column_address((unsigned long long)object_lut, (size_t)gcol, p.lut_cols,
                                                         (size_t)p.max_dis * p.lut_stride * 4);
  c.lut_hi = (unsigned)(lut_addr >> 32);
  const unsigned lutb = (unsigned)lut_addr - 0x4B000000u * c.lut_stride4;
  const float *S = stat + (size_t)f * H * kStatWords;
  float *pm_col = pm_out + (size_t)gcol * H;
  // The running (cost, vB) minima of a row live in the output array itself between the units of its
  // tile (L2-resident; one 16-byte load and store per lane and unit).
  float4 *out = dp_out + (size_t)gcol * H;

  // ---- one-time setup ----
  if (tid == 0) {
    for (int s = 0; s < kStages; s++) {
      mbar_init(&bar_full[s], 1);
      mbar_init(&bar_q[s], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < 3 * nt + 1; i += kDpThreads) cnt_out[i] = 0;
  if constexpr (!PAIRWISE) {
    for (int i = tid; i <= H; i += kDpThreads) ihs[i] = __ldg(inverse_height + i);
  } else {
    for (int i = tid; i < p.max_dis; i += kDpThreads) odr[i] = __ldg(object_disparity_range + i);
  }
  __syncthreads();

  // ---- producer: chunk ch -> ring slot ch % kStages (one elected lane).  The slot is free once
  //      every unit of the chunk that used it before has finished. ----
  auto produce = [&](int ch) {
    if (ch >= nt) return;
    const int s = ch % kStages;
    if (ch >= kStages) {
      const int old = ch - kStages;
      while (*reinterpret_cast<volatile int *>(cnt_fin + old) < nt - old) __nanosleep(64);
      __threadfence_block();
    }
    mbar_arrive_expect_tx(&bar_full[s], kSlotBytes);
    bulk_g2s(ring + (size_t)s * kSlotWords, recb + (size_t)ch * kSlotWords, kSlotBytes, &bar_full[s]);
  };
  if (tid == 0)
    for (int ch = 0; ch < kPrefetch; ch++) produce(ch);

  // first-segment priors (:189-199)
  const float first_k_gs = fmul(ffma(1.0f, kLn2, p.rows_log), c.pw);

  int jcur = 0;  // chunk this warp currently draws units from (warp-uniform, only grows)
  while (true) {
    // ---- draw the next unit ----
    int idx = 0, jsel = nt, tsel = 0;
    if (lane == 0) {
      if constexpr (PAIRWISE) {
        // The diagonal units form the serial chain of the column (diag j -> unit (j+1, j) -> diag j+1), so a
        // diagonal is taken the moment its tile has finished all earlier chunks; otherwise the next
        // off-diagonal unit, chunk-major, lowest tile first.  A warp that finds neither retires: the warp
        // that finishes unit (d, d-1) re-enters here and finds diagonal d ready.
        volatile int *vdiag = diag_next;
        while (true) {
          const int d = *vdiag;
          if (d < nt && *reinterpret_cast<volatile int *>(tile_done + d) >= d) {
            if (atomicCAS(diag_next, d, d + 1) == d) {
              jsel = tsel = d;
              idx = -1;
              break;
            }
            continue;
          }
          while (jcur < nt) {
            idx = atomicAdd(&cnt_out[jcur], 1);
            if (jcur + 1 + idx < nt) break;
            jcur++;
          }
          if (jcur < nt) {
            jsel = jcur;
            tsel = jcur + 1 + idx;
          }
          break;
        }
      } else {
        // chunk-major, lowest tile first (the diagonal unit is index 0 of its chunk)
        while (jcur < nt) {
          idx = atomicAdd(&cnt_out[jcur], 1);
          if (jcur + idx < nt) break;
          jcur++;
        }
        jsel = jcur;
        tsel = jcur + idx;
      }
    }
    jcur = __shfl_sync(full_mask, jcur, 0);
    idx = __shfl_sync(full_mask, idx, 0);
    jsel = __shfl_sync(full_mask, jsel, 0);
    tsel = __shfl_sync(full_mask, tsel, 0);
    if (jsel >= nt) break;
    const int j = jsel, t = tsel;
    if (idx == 0 && lane == 0) produce(j + kPrefetch);  // the first unit of a chunk keeps the ring filled
    __syncwarp();
    const int slot = j % kStages;
    const unsigned parity = (unsigned)(j / kStages) & 1u;
    const int vb0 = j * kChunk;
    const int nsteps = min(kChunk, H - vb0);
    // steps with vB <= vhor are on the ground side (predecessor row vB-1 below the horizon)
    const int kg = max(0, min(nsteps, vhor + 1 - vb0));
    const uint32_t *bchunk = ring + (size_t)slot * kSlotWords;
    float *qs_slot = qs + (size_t)slot * kChunk * kDynWords;
    const int vT = t * kChunk + lane;
    const bool row_ok = vT < H;
    const int vTc = row_ok ? vT : H - 1;

    // A side of the unit (independent of every wait below)
    uint32_t A[kRecWords];
    load_a_side(A, recb, vTc + 1);
    const unsigned ca = lutb + 4u * (unsigned)vTc;
    const unsigned cb0 = lutb + 4u * (unsigned)(vb0 - 1);  // row vB - 1 of step k: cb0 + 4k

    if constexpr (PAIRWISE) {
      if (t == j) {
        // stage the static transition records of vB = vb0 .. vb0 + 32 for the wavefront
        float *sst_j = sst + (j % kSstBufs) * kSstWords;
        for (int i = lane; i < (kChunk + 1) * kStatWords; i += 32)
          sst_j[i] = (vb0 + i / kStatWords) < H ? __ldg(S + (size_t)vb0 * kStatWords + i) : 0.0f;
      }
    }

    mbar_wait(&bar_full[slot], parity);
    // minima of this tile over the earlier chunks: written by the warp that did (t, j-1).  A counter,
    // not an mbarrier: units (t, j-2), (t, j-1), (t, j) can be in flight at once, and a parity wait
    // must not run more than one phase ahead.
    Best best{inf, inf, 0, 0};
    if (j > 0) {
      while (*reinterpret_cast<volatile int *>(tile_done + t) < j) __nanosleep(32);
      __threadfence_block();
      best = load_best(out + vTc);
    }

    if constexpr (PAIRWISE) {
      if (t == j) {
        // ================= diagonal unit: the wavefront =================
        // One pass, software-pipelined: the chain-independent part of step k+1 (cell_base) is issued
        // before the chain of step k (row vB-1 final -> Q[vB] -> cell -> row vB) so that it fills the
        // chain's latency.
        const float *sst_j = sst + (j % kSstBufs) * kSstWords;
        // prefix values at the start row of the best object segment so far (previous_mean needs them)
        float lo_d = f_(rec_word(recb, best.vb_o, kRecDisp));
        float lo_v = f_(rec_word(recb, best.vb_o, kRecValid));
        // Q[vb0] comes from the previous diagonal
        if (j > 0) {
          mbar_wait(&bar_q[(j - 1) % kStages], (unsigned)((j - 1) / kStages) & 1u);
          if (lane < kDynWords) qs_slot[lane] = qnext[(j & 1) * kDynWords + lane];
          __syncwarp();
        }
        auto finish_row = [&](int vB, int src_lane, float hi_d, float hi_v) {
          // row vB-1 (lane src_lane) is final: previous_mean of its best object segment (:674-685)
          const float c_gs = __shfl_sync(full_mask, best.gs, src_lane), c_o = __shfl_sync(full_mask, best.o, src_lane);
          const int o_vb = __shfl_sync(full_mask, best.vb_o, src_lane);
          const float l_d = __shfl_sync(full_mask, lo_d, src_lane), l_v = __shfl_sync(full_mask, lo_v, src_lane);
          const bool ground_side = vB - 1 < vhor;
          const float pm = segment_mean(hi_d, l_d, hi_v, l_v, vB - o_vb, HAS_INVALID);
          RowPriors rp;
          return make_row_info(sst_j + (vB - vb0) * kStatWords, ground_side, ground_side ? c_gs : inf, c_o,
                               ground_side ? inf : c_gs, pm, odr, p, &rp);
        };
        auto base_of = [&](int k) {
          const int vB = vb0 + k;
          return cell_base<false, 2, HAS_INVALID>(A, bchunk + k * kRecBWords, ca, lutb + 4u * (unsigned)(vB - 1),
                                                  (float)max(vTc + 1 - vB, 1), c, k < kg);
        };
        CellBase b_cur = (j == 0) ? cell_base<true, 1, HAS_INVALID>(A, bchunk, ca, lutb, (float)(vTc + 1), c)
                                  : base_of(0);
        for (int k = 0; k < nsteps; k++) {
          const int vB = vb0 + k;
          // prefix sums at row vB: "hi" of the finished row vB-1 and "lo" of segments starting at vB
          const float ps_d = f_(bchunk[k * kRecBWords + kRecDisp]), ps_v = f_(bchunk[k * kRecBWords + kRecValid]);
          CellBase b_next = b_cur;
          if (k + 1 < nsteps) b_next = base_of(k + 1);
          RowInfo q{};
          if (k > 0) {
            q = finish_row(vB, k - 1, ps_d, ps_v);
            if (lane == 0) {
              store_row_info(qs_slot + k * kDynWords, q);
              pm_col[vB] = q.pm;
            }
          } else if (vB > 0) {
            q = load_row_info(qs_slot);
          }
          float cost_gs, cost_o;
          if (vB == 0) {
            const float first_k_o = fmul(fadd(fadd((vT <= vhor) ? kLn2 : 0.0f, p.rows_log), p.max_dis_log), c.pw);
            cell_finish<true, true, 1>(b_cur, 0.0f, q, first_k_gs, first_k_o, c, cost_gs, cost_o);
          } else {
            cell_finish<true, false, 2>(b_cur, 0.0f, q, 0.0f, 0.0f, c, cost_gs, cost_o, k < kg);
          }
          const bool live = row_ok && lane >= k;
          if (live && cost_gs < best.gs) { best.gs = cost_gs; best.vb_gs = vB; }
          if (live && cost_o < best.o) { best.o = cost_o; best.vb_o = vB; lo_d = ps_d; lo_v = ps_v; }
          b_cur = b_next;
        }
        // Q[vb0 + 32] for the next diagonal (row vb0 + 31 is final now)
        if (vb0 + kChunk < H) {
          const int vB = vb0 + kChunk;
          const RowInfo q = finish_row(vB, 31, f_(rec_word(recb, vB, kRecDisp)),
                                       f_(rec_word(recb, vB, kRecValid)));
          if (lane == 0) {
            store_row_info(qnext + ((j + 1) & 1) * kDynWords, q);
            pm_col[vB] = q.pm;
          }
        }
        // the diagonal unit is the last one of its tile: the rows are final
        if (row_ok) store_best(out + vT, best);
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(&bar_q[slot]);
          atomicAdd(&cnt_fin[j], 1);
        }
        continue;
      }
      mbar_wait(&bar_q[slot], parity);
    }

    {
      const int n0 = vTc + 1 - vb0;
      int k0 = 0;
      if (j == 0) {
        // first segment, vB = 0 (:481-594)
        const CellBase b = cell_base<true, 1, HAS_INVALID>(A, bchunk, ca, lutb, (float)n0, c);
        RowInfo q{};
        const float first_k_o =
            PAIRWISE ? fmul(fadd(fadd((vT <= vhor) ? kLn2 : 0.0f, p.rows_log), p.max_dis_log), c.pw) : 0.0f;
        float cost_gs, cost_o;
        cell_finish<PAIRWISE, true, 1>(b, PAIRWISE ? 0.0f : ihs[n0], q, first_k_gs, first_k_o, c, cost_gs, cost_o);
        if (cost_gs < best.gs) { best.gs = cost_gs; best.vb_gs = 0; }
        if (cost_o < best.o) { best.o = cost_o; best.vb_o = 0; }
        k0 = 1;
      }
      if (!PAIRWISE && t == j) {
        // unary diagonal unit: vT >= vB predicate; afterwards the rows are final
        dp_steps<PAIRWISE, 1, true, HAS_INVALID>(A, bchunk, cb0, ca, ihs, qs_slot, vb0, k0, max(k0, kg), n0, lane, c,
                                                 best);
        dp_steps<PAIRWISE, 0, true, HAS_INVALID>(A, bchunk, cb0, ca, ihs, qs_slot, vb0, max(k0, kg), nsteps, n0, lane,
                                                 c, best);
      } else {
        // ground-side steps of a tile that lies entirely at/above the horizon cannot yield a ground stixel
        if (ISX_DEAD_SLOT(PAIRWISE) && t * kChunk >= vhor)
          dp_steps<PAIRWISE, 3, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, qs_slot, vb0, k0, max(k0, kg), n0, lane,
                                                    c, best);
        else
          dp_steps<PAIRWISE, 1, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, qs_slot, vb0, k0, max(k0, kg), n0, lane,
                                                    c, best);
        dp_steps<PAIRWISE, 0, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, qs_slot, vb0, max(k0, kg), nsteps, n0, lane,
                                                  c, best);
      }
      if (row_ok) store_best(out + vT, best);
    }
    // hand the tile's minima to the next chunk's unit; the chunk's slot has one reader less
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      if (t > j) *reinterpret_cast<volatile int *>(tile_done + t) = j + 1;
      atomicAdd(&cnt_fin[j], 1);
    }
  }
}


// ---------------------------------------------------------------------------
// Unary mode with exact pruning (branch and bound over the vB chunks of a tile).
//
// In unary mode a cell's cost is a function of its own segment only (previous costs are not accumulated,
// StixelsKernels.cu:713-720, 758-766, 815-824): cost = sw*seg + pw/n + dw*data, where seg is a sum of
// non-negative integers over the rows of the segment.  So every cell of a far unit is bounded from below
// by what its shortest segment must cost at least, and once the rows of a tile have found a cheap
// segment in the chunks next to the diagonal, the chunks further down cannot win any more -- with the
// tuned weights (pw = 1e4) the best segment of a row is a few dozen rows long.
//
// One warp owns a tile and walks its chunks DOWNWARDS from the diagonal (j = t, t-1, ...):
//   * inside a unit the steps ascend with strict '<' as before; a unit's minima replace the carried ones
//     when they are '<=', so that among equal costs the lowest vB still wins (the reference's tie rule);
//   * before chunk j-1 every lane evaluates a lower bound of all its cells still to come (vB <= last row of
//     chunk j-1, its own vT):
//         seg_c(vB, vT) >= P_c(vT + 1) - P_c(last row of chunk j-1)                          (prefixes are monotone)
//         instance term >= -2^-19 * iw * (sum of squared means up to the tile)               (float error of the variance)
//         data terms    >= rows * min(0, smallest per-row cost)                              (over the longest segment)
//     combined with the same monotone float operations as the cell itself, minus the slack prune_bound() derives
//     from the magnitudes involved; the bound only grows further down, so the walk stops as soon as
//     it exceeds the carried cost of both slots in every row of the tile.
// The result is bit-identical to the exhaustive scan (same cells win, same ties); tests run both.
// B records travel global -> shared memory per warp (two 4 KB buffers, cp.async.bulk + mbarrier), the next
// chunk speculatively while the current one is evaluated.
// ---------------------------------------------------------------------------
#ifndef ISX_UNARY_PRUNE
#define ISX_UNARY_PRUNE 1
#endif

// ---- how far a computed cell cost can lie below the bound's exact value (derivation: DESIGN.md section 4) ----
// A bound X = sw * seg_lb + (dw * data_lb + prior_lb) is evaluated with the cell's own operations on lower bounds
// of its inputs, and float rounding is monotone, so the only places where the cell can come out BELOW X are
//  (a) the data term: it is the difference of two float prefix sums (object LUT rows, ground / sky prefixes), each
//      the result of at most 37 additions (32 chunk carries + 5 Kogge-Stone / Blelloch levels) of partial sums whose
//      magnitude is at most rows * cmax (cmax = largest |per-row cost| of the model): |error| <= 2 * 37 * 2^-24 *
//      rows * cmax, plus one rounding each for the bound's own rows * lb product and its scaling by dw.
//      kDataErr = 2^-17 = 128 * 2^-24 covers 2 * 37 + 6 roundings.  Frames of up to 2047 rows have up to 64 chunk
//      carries, 69 additions: kDataErrTall = 2^-16 = 256 * 2^-24 covers 2 * 69 + 6 = 144 roundings;
//  (b) the order of the final operations (the cell: one FFMA on the data term and the prior, then one on the class
//      sum; the bound: FMUL, FADD, FFMA): each rounding is relative 2^-24 of a value no larger than
//      |X| + |dw * data_lb| + |prior_lb|; kRelErr = 2^-20 leaves a factor 16 over the <= 4 roundings involved.
// Nothing else is hand-picked: with the data slack of its record stride, the bound holds for any rows up to
// kMaxRows, any max_dis and non-negative weights.
constexpr float kDataErr = 7.62939453125e-06f;     // 2^-17
constexpr float kDataErrTall = 1.52587890625e-05f; // 2^-16
constexpr float kRelErr = 9.5367431640625e-07f;    // 2^-20
template <int HP>
__device__ __forceinline__ constexpr float data_err() { return HP > kRecStride ? kDataErrTall : kDataErr; }
__device__ __forceinline__ float prune_bound(float x, float dneg, float prior, float data_slack) {
  if (!(x < inf_f())) return x;   // +inf (no finite candidate in the chunk) stays +inf; NaN never prunes
  const float mag = fadd(fadd(fabsf(x), fabsf(dneg)), fabsf(prior));
  return fsub(x, ffma(mag, kRelErr, data_slack));
}
#ifndef ISX_PRUNED_CTAS
#define ISX_PRUNED_CTAS 4  // 128 registers: carried + local minima and the bound ingredients beside the 30 A words
#endif

struct PruneLayout {
  size_t off_stage, off_bars, off_ih, off_misc, total;
  __host__ __device__ PruneLayout(int H, int warps) {
    size_t o = 0;
    off_stage = o; o += (size_t)warps * 2 * kSlotBytes;
    off_bars = o; o += (size_t)warps * 2 * 8;
    off_ih = o; o += (size_t)(H + 1) * 4;
    o = (o + 15) & ~(size_t)15;
    off_misc = o; o += 16;
    total = (o + 15) & ~(size_t)15;
  }
};

template <bool HAS_INVALID, int WARPS, int HP>
__global__ void __launch_bounds__(WARPS * 32, WARPS == kDpWarps ? ISX_PRUNED_CTAS : 2)
dp_unary_pruned_kernel(const uint32_t *__restrict__ records_b,
                       const float *__restrict__ object_lut, const float *__restrict__ ground,
                       const int *__restrict__ vhor_arr, const float *__restrict__ inverse_height, float4 *dp_out,
                       unsigned long long *__restrict__ units_evaluated, const int *__restrict__ col_flags, KParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int kThreads = WARPS * 32;
  const unsigned full_mask = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gcol = blockIdx.x;  // frame * C + column
  const int H = p.rows, C = p.realcols;
  constexpr int Hp = HP;  // == p.rec_stride
  const int f = gcol / C;
  const int vhor = vhor_arr[f];
  const float inf = inf_f();
  const PruneLayout L(H, WARPS);
  const int nt = (H + kChunk - 1) / kChunk;

  uint32_t *stage_w = reinterpret_cast<uint32_t *>(smem_raw + L.off_stage) + (size_t)warp * 2 * kSlotWords;
  uint64_t *bars_w = reinterpret_cast<uint64_t *>(smem_raw + L.off_bars) + warp * 2;
  float *ihs = reinterpret_cast<float *>(smem_raw + L.off_ih);
  int *tile_next = reinterpret_cast<int *>(smem_raw + L.off_misc);
  float *norm_g_min_s = reinterpret_cast<float *>(smem_raw + L.off_misc + 4);

  DpConsts c;
  c.pw = p.prior_weight; c.dw = p.disparity_weight; c.sw = p.segmentation_weight; c.iw = p.instance_weight;
  c.dm1f = (float)(p.max_dis - 1);
  c.lut_stride4 = (unsigned)p.lut_stride * 4u;
  c.epsilon = p.epsilon;
  const uint32_t *recb = records_b + (size_t)gcol * Hp * kRecBWords;
  const unsigned long long lut_addr = lut_column_address((unsigned long long)object_lut, (size_t)gcol, p.lut_cols,
                                                         (size_t)p.max_dis * p.lut_stride * 4);
  c.lut_hi = (unsigned)(lut_addr >> 32);
  const unsigned lutb = (unsigned)lut_addr - 0x4B000000u * c.lut_stride4;
  float4 *out = dp_out + (size_t)gcol * H;

  // ---- one-time setup ----
  if (tid == 0) {
    uint64_t *bars_all = reinterpret_cast<uint64_t *>(smem_raw + L.off_bars);
    for (int i = 0; i < 2 * WARPS; i++) mbar_init(&bars_all[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    *tile_next = nt;
  }
  for (int i = tid; i <= H; i += kThreads) ihs[i] = __ldg(inverse_height + i);
  if (warp == 0) {
    // smallest normalization_ground over the rows that HAVE a ground cost (v < vhor; at/above the horizon ground_lut
    // is +inf, :437-446, while normalization_ground itself runs to -inf there: log of a vanishing range,
    // Stixels.cu:86, 812-814): per-row ground cost >= min(puniform, it) + ... (:217-234)
    const float *norm_g = ground + (size_t)f * 3 * H + H;
    float m = inf;
    for (int v = lane; v < min(H, vhor); v += 32) m = fminf(m, __ldg(norm_g + v));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) m = fminf(m, __shfl_xor_sync(full_mask, m, d));
    if (lane == 0) *norm_g_min_s = m;
  }
  __syncthreads();
  // smallest possible per-row data cost of the three models (StixelsKernels.cu:201-234, Stixels.cu:842-854):
  // the squared term is >= 0, fmin / fadd are monotone
  const float lb_g = fminf(p.pnexists_given_ground_log,
                           fadd(fminf(p.puniform, *norm_g_min_s), p.nopnexists_given_ground_log));
  const float lb_s = fminf(p.pnexists_given_sky_log,
                           fadd(fminf(p.puniform_sky, p.normalization_sky), p.nopnexists_given_sky_log));
  const float lb_o = p.obj_cost_min;
  // largest magnitude of a per-row data cost of each model: what the rounding of their float prefix sums scales with
  const float cmax_g = fmaxf(fabsf(p.pnexists_given_ground_log),
                             fmaxf(fabsf(fadd(p.puniform, p.nopnexists_given_ground_log)), fabsf(lb_g)));
  const float cmax_s = fmaxf(fabsf(p.pnexists_given_sky_log),
                             fmaxf(fabsf(fadd(p.puniform_sky, p.nopnexists_given_sky_log)), fabsf(lb_s)));
  const float cmax_o = p.obj_cost_absmax;
  // the bounds assume non-negative weights (NaN fails the test too) and non-negative class values without int32
  // wrap-around (col_flags, column_tables_kernel): otherwise every chunk is evaluated
  const bool prune_ok = ISX_UNARY_PRUNE && c.sw >= 0.0f && c.dw >= 0.0f && c.pw >= 0.0f && c.iw >= 0.0f &&
                        p.prune_unary != 0 && col_flags[gcol] == 0;

  unsigned ph0 = 0, ph1 = 0;  // phase parity of this warp's two buffers
  auto stage = [&](int ch, int b) {
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive_expect_tx(&bars_w[b], kSlotBytes);
      bulk_g2s(stage_w + (size_t)b * kSlotWords, recb + (size_t)ch * kSlotWords, kSlotBytes, &bars_w[b]);
    }
  };
  auto wait = [&](int b) {
    if (b) { mbar_wait(&bars_w[1], ph1); ph1 ^= 1u; }
    else { mbar_wait(&bars_w[0], ph0); ph0 ^= 1u; }
  };
  unsigned long long my_units = 0;

  while (true) {
    int t = 0;
    if (lane == 0) t = atomicSub(tile_next, 1) - 1;
    t = __shfl_sync(full_mask, t, 0);
    if (t < 0) break;
    const int vT = t * kChunk + lane;
    const bool row_ok = vT < H;
    const int vTc = row_ok ? vT : H - 1;
    stage(t, 0);

    uint32_t A[kRecWords];
    load_a_side(A, recb, vTc + 1);
    const unsigned ca = lutb + 4u * (unsigned)vTc;
    // ---- what the bounds of this tile are made of ----
    const int vTmaxc = min(t * kChunk + kChunk - 1, H - 1);
    float sq = 0.0f;
    if (lane == 0) {
      sq = fadd(fadd(f_(rec_word(recb, vTmaxc + 1, kRecMx2Hi)), f_(rec_word(recb, vTmaxc + 1, kRecMx2Lo))),
                fadd(f_(rec_word(recb, vTmaxc + 1, kRecMy2Hi)), f_(rec_word(recb, vTmaxc + 1, kRecMy2Lo))));
    }
    sq = __shfl_sync(full_mask, sq, 0);
    const float ic_lb = -fmul(fmul(sq, c.iw), 1.9073486328125e-06f);  // 2^-19: > 5 roundings + MUFU.RCP, relative
    const float nmaxf = (float)(vTmaxc + 1);
    const float dneg_o = fmul(c.dw, fmul(nmaxf, fminf(lb_o, 0.0f)));
    const float dneg_gs = fmul(c.dw, fmul(nmaxf, fminf(vTc < vhor ? lb_g : lb_s, 0.0f)));
    // slack of the data terms (prune_bound above): dw * data_err<HP>() * rows * largest per-row cost
    const float dslack_o = fmul(c.dw, fmul(fmul(nmaxf, cmax_o), data_err<HP>()));
    const float dslack_gs = fmul(c.dw, fmul(fmul(nmaxf, vTc < vhor ? cmax_g : cmax_s), data_err<HP>()));

    Best carried{inf, inf, 0, 0};
    int buf = 0;
    wait(0);
    for (int j = t;; j--) {
      if (j > 0) stage(j - 1, buf ^ 1);  // needed for the bound below, and for the next unit if the walk goes on
      const uint32_t *bchunk = stage_w + (size_t)buf * kSlotWords;
      const int vb0 = j * kChunk;
      const int nsteps = min(kChunk, H - vb0);
      const int kg = max(0, min(nsteps, vhor + 1 - vb0));  // steps with vB <= vhor are on the ground side
      const unsigned cb0 = lutb + 4u * (unsigned)(vb0 - 1);
      const int n0 = vTc + 1 - vb0;
      Best local{inf, inf, 0, 0};
      int k0 = 0;
      if (j == 0) {
        // first segment, vB = 0 (:481-594)
        const CellBase b = cell_base<true, 1, HAS_INVALID>(A, bchunk, ca, lutb, (float)n0, c);
        RowInfo q{};
        float cost_gs, cost_o;
        cell_finish<false, true, 1>(b, ihs[n0], q, 0.0f, 0.0f, c, cost_gs, cost_o);
        if (cost_gs < local.gs) { local.gs = cost_gs; local.vb_gs = 0; }
        if (cost_o < local.o) { local.o = cost_o; local.vb_o = 0; }
        k0 = 1;
      }
      if (j == t) {
        dp_steps<false, 1, true, HAS_INVALID>(A, bchunk, cb0, ca, ihs, nullptr, vb0, k0, max(k0, kg), n0, lane, c,
                                              local);
        dp_steps<false, 0, true, HAS_INVALID>(A, bchunk, cb0, ca, ihs, nullptr, vb0, max(k0, kg), nsteps, n0, lane, c,
                                              local);
      } else {
        if (t * kChunk >= vhor)
          dp_steps<false, 3, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, nullptr, vb0, k0, max(k0, kg), n0, lane, c,
                                                 local);
        else
          dp_steps<false, 1, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, nullptr, vb0, k0, max(k0, kg), n0, lane, c,
                                                 local);
        dp_steps<false, 0, false, HAS_INVALID>(A, bchunk, cb0, ca, ihs, nullptr, vb0, max(k0, kg), nsteps, n0, lane, c,
                                               local);
      }
      // this chunk lies below the ones seen so far: it wins ties
      if (local.gs <= carried.gs) { carried.gs = local.gs; carried.vb_gs = local.vb_gs; }
      if (local.o <= carried.o) { carried.o = local.o; carried.vb_o = local.vb_o; }
      my_units++;
      __syncwarp();
      if (j == 0) break;
      // ---- can a segment that starts in chunk j-1 or below still win a row of this tile? ----
      wait(buf ^ 1);
      bool stop = false;
      if (prune_ok) {
        // Row vT against the LAST row of chunk j-1 (all of them are full chunks): the class sums of the shortest
        // segment that is still to come; every other one contains it, and the sums only grow (non-negative terms).
        const int vbm = (j - 1) * kChunk + kChunk - 1;
        const uint32_t *blast = stage_w + (size_t)(buf ^ 1) * kSlotWords + (kChunk - 1) * kRecBWords;
        uint32_t Bl[20];
        {
          const uint4 *b4 = reinterpret_cast<const uint4 *>(blast);
#pragma unroll
          for (int k = 0; k < 5; k++) {
            const uint4 q4 = b4[k];
            Bl[4 * k] = q4.x; Bl[4 * k + 1] = q4.y; Bl[4 * k + 2] = q4.z; Bl[4 * k + 3] = q4.w;
          }
        }
        int l_ni = (int)(A[2] - Bl[2]);
#pragma unroll
        for (int k = 3; k < 10; k++) l_ni = min(l_ni, (int)(A[k] - Bl[k]));
        int l_in = (int)(A[11] - Bl[11]);
#pragma unroll
        for (int k = 12; k < 19; k++) l_in = min(l_in, (int)(A[k] - Bl[k]));
        const int l_g = min((int)(A[0] - Bl[0]), (int)(A[1] - Bl[1]));
        const int l_s = (int)(A[kSkyClass] - Bl[kSkyClass]);
        // object slot: seg_o >= min(0 + S_ni, ic + S_in), prior >= 0
        const float seg_o_lb = fminf((float)l_ni, fadd(ic_lb, (float)l_in));
        const float lbo = prune_bound(ffma(seg_o_lb, c.sw, dneg_o), dneg_o, 0.0f, dslack_o);
        // ground / sky slot of this lane's row; sky cells need vB > vhor, ground rows always have candidates
        const bool gs_possible = vTc < vhor || vbm > vhor;
        const float seg_gs_lb = (float)(vTc < vhor ? l_g : l_s);
        const float lbgs = prune_bound(ffma(seg_gs_lb, c.sw, dneg_gs), dneg_gs, 0.0f, dslack_gs);
        const bool lane_done = !row_ok || (lbo > carried.o && (!gs_possible || lbgs > carried.gs));
        stop = __all_sync(full_mask, lane_done);
      }
      if (stop) break;
      buf ^= 1;
    }
    if (row_ok) store_best(out + vT, carried);
    __syncwarp();
  }
  if (lane == 0 && my_units) atomicAdd(units_evaluated, my_units);
}


// ---------------------------------------------------------------------------
// Pairwise mode, tile-major with exact pruning.
//
// The pairwise cost of a cell is  dw*data + pw*min_k(C[vB-1][k] + pw*trans_k) + sw*seg : the best total cost of the
// rows below plus what the segment itself costs.  A segment that runs across a region of another class pays for
// every row of it, so most far cells cannot win -- but proving it needs the row's near candidates first, and the
// chunk-major schedule of dp_kernel evaluates the far chunks first.  Here a column is processed TILE by tile behind
// the diagonal chain:
//   for tile t:  (1) the units (t, j), j = t-1 ... 0, interleaved over the warps of the CTA, each unit only if a
//                    lower bound of its cells does not already exceed the minima carried so far in some row;
//                (2) the diagonal unit (t, t) -- the wavefront -- by warp 0, which finalises the rows of the tile,
//                    writes their transition records Q[vB] for all later tiles and the smallest priors of the chunk.
// Bound of unit (t, j) for row vT (the slots separately) -- per class, because the cost of a cell is a minimum over
// classes of terms that SEPARATE into a part of the top row and a part of the bottom row:
//     cost_o(vB, vT) >= min_c [ sw * (w_c * dO + dP_c) ] + kmin_o(vB) + dw * data_lb       (dX = X(vT+1) - X(vB))
//                     = min_c [ F_c(vT+1) + (kmin_o(vB) - F_c(vB)) ] + ...,   F_c(v) = sw * (w_c * O(v) + P_c(v)),
//   with P_c the class prefix, O the squared-offset prefix (w_c = iw for the non-instance classes; the instance
//   classes carry the variance term instead, >= -2^-19 * iw * sum(means^2)), kmin_o(vB) the smallest object prior any
//   cell of row vB can get.  So the diagonal of chunk j leaves M_c[j] = min over its rows of (kmin_o(vB) - F_c(vB)),
//   16 numbers, and a later tile tests  min_c (F_c(vT+1) + M_c[j])  against its carried minima.  The ground / sky
//   slot is even exact: its prior k_gs(vB) and its data term (a prefix difference) separate too, classes {road,
//   sidewalk} or {sky}.
// r1 bounded the class sums by those of the SHORTEST segment into the chunk and the prior by the chunk's smallest:
// loose by a whole chunk of accumulated cost (hundreds of units), while the candidates of a column lie more than 5
// units apart (measured: with an exact bound 0.8 off-diagonal units per tile are needed, the old bound let 5.5
// through).  The envelopes are floats of magnitude up to 1e6; the slack 2^-21 * (|F| + |M|) covers their <= 6
// roundings (relative 2^-24 each) with a factor 2, the data terms keep prune_bound()'s slack.  Minima are merged
// lexicographically by (cost, vB): the reference's "lowest vB wins ties" whatever the order of evaluation.
// ---------------------------------------------------------------------------
#ifndef ISX_WALK_CTAS
#define ISX_WALK_CTAS 4
#endif
#ifndef ISX_WALK_WARPS_PER_SM
#define ISX_WALK_WARPS_PER_SM 16   // one-warp CTAs per SM the register budget of the walk kernel aims at (128 registers)
#endif
#ifndef ISX_PAIRWISE_WALK_DEFAULT
#define ISX_PAIRWISE_WALK_DEFAULT 1
#endif

// envelope words per chunk: 0..7 classes 2..9 | 8..15 classes 11..18 | 16, 17 road, sidewalk (ground slot) |
// 18 sky (sky slot) | 19 largest finite |entry| (scale of the slack)
constexpr int kMWords = 20;
constexpr float kEnvErr = 4.76837158203125e-07f;   // 2^-21

struct WalkLayout {
  int nt;
  size_t off_stage, off_bars, off_q, off_sst, off_odr, off_merge, off_mtab, off_seed, off_qnext, total;
  __host__ __device__ WalkLayout(int H, int D, int warps) {
    nt = (H + kChunk - 1) / kChunk;
    size_t o = 0;
    off_stage = o; o += (size_t)warps * kSlotBytes;
    off_bars = o; o += (size_t)warps * 8;
    o = (o + 15) & ~(size_t)15;
    off_q = o; o += (size_t)warps * kChunk * kDynWords * 4;
    off_sst = o; o += (size_t)kSstWords * 4;
    off_odr = o; o += (size_t)((D + 3) & ~3) * 4;
    off_merge = o; o += (size_t)warps * 32 * 16;
    off_mtab = o; o += (size_t)nt * kMWords * 4;  // per chunk: the class envelopes M_c[j] (see the kernel's header)
    o = (o + 15) & ~(size_t)15;
    off_seed = o; o += (size_t)warps * (kRecBWords + kDynWords + 4) * 4 + 16;  // one B row + one Q row per warp | seeds
    off_qnext = o; o += (size_t)kDynWords * 4;
    total = (o + 15) & ~(size_t)15;
  }
};

// (cost, vB) lexicographic: the lowest vB among equal costs, NaN never wins
__device__ __forceinline__ void merge_best(Best &c, const Best &l) {
  if (l.gs < c.gs || (l.gs == c.gs && l.vb_gs < c.vb_gs)) { c.gs = l.gs; c.vb_gs = l.vb_gs; }
  if (l.o < c.o || (l.o == c.o && l.vb_o < c.vb_o)) { c.o = l.o; c.vb_o = l.vb_o; }
}

// smallest prior any object cell of row vB can get (object_priors picks one of these), times pw like the cell
__device__ __forceinline__ float object_prior_floor(const RowInfo &q, bool ground_side, float pw) {
  float m = fminf(q.p2_hi, fminf(q.p2_lo, q.p2_mid));
  m = fminf(m, fminf(q.a1, q.a2));
  if (ground_side) m = fminf(m, q.a3);
  return fmul(m, pw);
}

template <bool HAS_INVALID, int WARPS, int HP>
__global__ void __launch_bounds__(WARPS * 32, WARPS == 1 ? ISX_WALK_WARPS_PER_SM : WARPS == kDpWarps ? ISX_WALK_CTAS : 2)
dp_pairwise_walk_kernel(const uint32_t *__restrict__ records_b,
                        const float *__restrict__ object_lut, const float *__restrict__ stat,
                        const float *__restrict__ ground, float *__restrict__ pm_out, float *__restrict__ qrows,
                        const int *__restrict__ vhor_arr, const float *__restrict__ object_disparity_range,
                        float4 *dp_out, unsigned long long *__restrict__ units_evaluated,
                        const int *__restrict__ col_flags, KParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int kThreads = WARPS * 32;
  const unsigned full_mask = 0xffffffffu;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gcol = blockIdx.x;
  const int H = p.rows, C = p.realcols;
  constexpr int Hp = HP;  // == p.rec_stride
  const int f = gcol / C;
  const int vhor = vhor_arr[f];
  const float inf = inf_f();
  const WalkLayout L(H, p.max_dis, WARPS);
  const int nt = L.nt;

  uint32_t *stage_w = reinterpret_cast<uint32_t *>(smem_raw + L.off_stage) + (size_t)warp * kSlotWords;
  uint64_t *bar_w = reinterpret_cast<uint64_t *>(smem_raw + L.off_bars) + warp;
  float *q_w = reinterpret_cast<float *>(smem_raw + L.off_q) + (size_t)warp * kChunk * kDynWords;
  float *sst = reinterpret_cast<float *>(smem_raw + L.off_sst);
  float *odr = reinterpret_cast<float *>(smem_raw + L.off_odr);
  float4 *merge = reinterpret_cast<float4 *>(smem_raw + L.off_merge);
  float *mtab = reinterpret_cast<float *>(smem_raw + L.off_mtab);
  int *seeds = reinterpret_cast<int *>(smem_raw + L.off_seed);                      // [2] argmin vB of the row below the tile
  uint32_t *seed_row = reinterpret_cast<uint32_t *>(smem_raw + L.off_seed + 16) + warp * (kRecBWords + kDynWords + 4);
  float *seed_q = reinterpret_cast<float *>(seed_row + kRecBWords);
  float *qnext = reinterpret_cast<float *>(smem_raw + L.off_qnext);

  DpConsts c;
  c.pw = p.prior_weight; c.dw = p.disparity_weight; c.sw = p.segmentation_weight; c.iw = p.instance_weight;
  c.dm1f = (float)(p.max_dis - 1);
  c.lut_stride4 = (unsigned)p.lut_stride * 4u;
  c.epsilon = p.epsilon;
  const uint32_t *recb = records_b + (size_t)gcol * Hp * kRecBWords;
  const unsigned long long lut_addr = lut_column_address((unsigned long long)object_lut, (size_t)gcol, p.lut_cols,
                                                         (size_t)p.max_dis * p.lut_stride * 4);
  c.lut_hi = (unsigned)(lut_addr >> 32);
  const unsigned lutb = (unsigned)lut_addr - 0x4B000000u * c.lut_stride4;
  const float *S = stat + (size_t)f * H * kStatWords;
  float *pm_col = pm_out + (size_t)gcol * H;
  float *qg = qrows + (size_t)gcol * Hp * kDynWords;  // Q[vB] of every row of this column
  float4 *out = dp_out + (size_t)gcol * H;

  if (tid == 0) {
    uint64_t *bars_all = reinterpret_cast<uint64_t *>(smem_raw + L.off_bars);
    for (int i = 0; i < WARPS; i++) mbar_init(&bars_all[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < p.max_dis; i += kThreads) odr[i] = __ldg(object_disparity_range + i);
  float norm_g_min = inf;
  {
    const float *norm_g = ground + (size_t)f * 3 * H + H;   // rows below the horizon only (see dp_unary_pruned_kernel)
    for (int v = lane; v < min(H, vhor); v += 32) norm_g_min = fminf(norm_g_min, __ldg(norm_g + v));
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) norm_g_min = fminf(norm_g_min, __shfl_xor_sync(full_mask, norm_g_min, d));
  }
  __syncthreads();
  const float lb_g = fminf(p.pnexists_given_ground_log, fadd(fminf(p.puniform, norm_g_min), p.nopnexists_given_ground_log));
  const float lb_s = fminf(p.pnexists_given_sky_log,
                           fadd(fminf(p.puniform_sky, p.normalization_sky), p.nopnexists_given_sky_log));
  const float lb_o = p.obj_cost_min;
  const float cmax_g = fmaxf(fabsf(p.pnexists_given_ground_log),
                             fmaxf(fabsf(fadd(p.puniform, p.nopnexists_given_ground_log)), fabsf(lb_g)));
  const float cmax_s = fmaxf(fabsf(p.pnexists_given_sky_log),
                             fmaxf(fabsf(fadd(p.puniform_sky, p.nopnexists_given_sky_log)), fabsf(lb_s)));
  const float cmax_o = p.obj_cost_absmax;
  const bool prune_ok = c.sw >= 0.0f && c.dw >= 0.0f && c.pw >= 0.0f && c.iw >= 0.0f && p.prune_pairwise != 0 &&
                        col_flags[gcol] == 0;
  // first-segment priors (:189-199)
  const float first_k_gs = fmul(ffma(1.0f, kLn2, p.rows_log), c.pw);

  unsigned ph = 0;  // phase parity of this warp's buffer
  auto stage = [&](int ch) {
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_arrive_expect_tx(bar_w, kSlotBytes);
      bulk_g2s(stage_w, recb + (size_t)ch * kSlotWords, kSlotBytes, bar_w);
    }
  };
  auto wait = [&]() { mbar_wait(bar_w, ph); ph ^= 1u; };
  unsigned long long my_units = 0;

  for (int t = 0; t < nt; t++) {
    const int vT = t * kChunk + lane;
    const bool row_ok = vT < H;
    const int vTc = row_ok ? vT : H - 1;
    uint32_t A[kRecWords];
    load_a_side(A, recb, vTc + 1);
    const unsigned ca = lutb + 4u * (unsigned)vTc;
    // bound ingredients of this tile (see dp_unary_pruned_kernel)
    const int vTmaxc = min(t * kChunk + kChunk - 1, H - 1);
    float sq = 0.0f;
    if (lane == 0) {
      sq = fadd(fadd(f_(rec_word(recb, vTmaxc + 1, kRecMx2Hi)), f_(rec_word(recb, vTmaxc + 1, kRecMx2Lo))),
                fadd(f_(rec_word(recb, vTmaxc + 1, kRecMy2Hi)), f_(rec_word(recb, vTmaxc + 1, kRecMy2Lo))));
    }
    sq = __shfl_sync(full_mask, sq, 0);
    const float ic_lb = -fmul(fmul(sq, c.iw), 1.9073486328125e-06f);
    const float nmaxf = (float)(vTmaxc + 1);
    const float dneg_o = fmul(c.dw, fmul(nmaxf, fminf(lb_o, 0.0f)));
    const float dneg_gs = fmul(c.dw, fmul(nmaxf, fminf(vTc < vhor ? lb_g : lb_s, 0.0f)));
    const float dslack_o = fmul(c.dw, fmul(fmul(nmaxf, cmax_o), data_err<HP>()));
    const float dslack_gs = fmul(c.dw, fmul(fmul(nmaxf, vTc < vhor ? cmax_g : cmax_s), data_err<HP>()));
    const float nicA = fmul((float)(int)A[kRecOff], c.iw);   // iw * O(vT + 1)
    (void)dneg_gs;

    // ================= (1) the chunks below the diagonal, nearest first, interleaved over the warps =================
    Best carried{inf, inf, 0, 0};
    // Seeds: the row just below the tile is final, and the best segments of the tile's rows mostly start where ITS best
    // segments start (the same region goes on).  Those two cells (one step each) give the carried minima a value to
    // prune against before any unit is walked -- otherwise the nearest chunk is always evaluated.  They are cells of
    // the column like any other, so the result does not depend on them.
    if (prune_ok && t > 0) {
      const int s0 = seeds[0], s1 = seeds[1];
#pragma unroll 1
      for (int si = 0; si < 2; si++) {
        const int vB = si == 0 ? s0 : s1;
        if ((si == 1 && s1 == s0) || vB < 0 || vB >= t * kChunk) continue;   // only candidates below the tile's own chunk
        Best local{inf, inf, 0, 0};
        __syncwarp();
        seed_row[lane] = __ldg(recb + (size_t)vB * kRecBWords + lane);
        if (lane < kDynWords) seed_q[lane] = __ldcg(qg + (size_t)vB * kDynWords + lane);
        __syncwarp();
        const float nf = (float)(vTc + 1 - vB);
        if (vB == 0) {
          // first segment, vB = 0 (:481-594)
          const CellBase b = cell_base<true, 1, HAS_INVALID>(A, seed_row, ca, lutb, nf, c);
          RowInfo q{};
          const float first_k_o = fmul(fadd(fadd((vT <= vhor) ? kLn2 : 0.0f, p.rows_log), p.max_dis_log), c.pw);
          float cost_gs, cost_o;
          cell_finish<true, true, 1>(b, 0.0f, q, first_k_gs, first_k_o, c, cost_gs, cost_o);
          if (cost_gs < local.gs) { local.gs = cost_gs; local.vb_gs = 0; }
          if (cost_o < local.o) { local.o = cost_o; local.vb_o = 0; }
        } else {
          const unsigned cbs = lutb + 4u * (unsigned)(vB - 1);
          if (vB > vhor)
            dp_step<true, 0, false, HAS_INVALID, 0>(A, seed_row, ca, cbs, nullptr, nullptr, 0, seed_q, vB, 0, lane, nf, c, local);
          else if (t * kChunk >= vhor)
            dp_step<true, 3, false, HAS_INVALID, 0>(A, seed_row, ca, cbs, nullptr, nullptr, 0, seed_q, vB, 0, lane, nf, c, local);
          else
            dp_step<true, 1, false, HAS_INVALID, 0>(A, seed_row, ca, cbs, nullptr, nullptr, 0, seed_q, vB, 0, lane, nf, c, local);
        }
        merge_best(carried, local);
      }
    }
    for (int j = t - 1 - warp; j >= 0; j -= WARPS) {
      const int vb0 = j * kChunk;
      bool skip = false;
      if (prune_ok) {
        const float4 *M4 = reinterpret_cast<const float4 *>(mtab + j * kMWords);
        float M[kMWords];
#pragma unroll
        for (int k = 0; k < kMWords / 4; k++) {
          const float4 m4 = M4[k];
          M[4 * k] = m4.x; M[4 * k + 1] = m4.y; M[4 * k + 2] = m4.z; M[4 * k + 3] = m4.w;
        }
        // object slot: min over the classes of F_c(vT + 1) + M_c[j]
        float lbo = inf, fmax_o = 0.0f;
#pragma unroll
        for (int k = 2; k < 10; k++) {
          const float F = fmul(c.sw, fadd(nicA, (float)(int)A[k]));
          fmax_o = fmaxf(fmax_o, F);
          lbo = fminf(lbo, fadd(F, M[k - 2]));
        }
#pragma unroll
        for (int k = 11; k < 19; k++) {
          const float F = fmul(c.sw, fadd(ic_lb, (float)(int)A[k]));
          fmax_o = fmaxf(fmax_o, F);
          lbo = fminf(lbo, fadd(F, M[8 + k - 11]));
        }
        if (lbo < inf) lbo = prune_bound(fadd(lbo, dneg_o), dneg_o, 0.0f, ffma(fadd(fmax_o, M[19]), kEnvErr, dslack_o));
        // ground / sky slot of this lane's row
        float lbgs = inf, fmax_gs = 0.0f;
        if (vTc < vhor) {
#pragma unroll
          for (int k = 0; k < 2; k++) {
            const float F = ffma(c.dw, f_(A[kRecGround]), fmul(c.sw, fadd(nicA, (float)(int)A[k])));
            fmax_gs = fmaxf(fmax_gs, fabsf(F));
            lbgs = fminf(lbgs, fadd(F, M[16 + k]));
          }
        } else {
          const float F = ffma(c.dw, f_(A[kRecSky]), fmul(c.sw, fadd(nicA, (float)(int)A[kSkyClass])));
          fmax_gs = fabsf(F);
          lbgs = fadd(F, M[18]);
        }
        if (lbgs < inf) lbgs = prune_bound(lbgs, 0.0f, 0.0f, ffma(fadd(fmax_gs, M[19]), kEnvErr, dslack_gs));
        const bool lane_done = !row_ok || ((lbo > carried.o || lbo == inf) && (lbgs > carried.gs || lbgs == inf));
        skip = __all_sync(full_mask, lane_done);
      }
      if (skip) continue;
      __syncwarp();
      stage(j);
      // Q[vB] of the chunk: global -> this warp's shared copy (row k by lane k)
      {
        const float4 *src = reinterpret_cast<const float4 *>(qg + (size_t)(vb0 + lane) * kDynWords);
        float4 *dst = reinterpret_cast<float4 *>(q_w + lane * kDynWords);
        const float4 x0 = __ldcg(src), x1 = __ldcg(src + 1), x2 = __ldcg(src + 2);
        dst[0] = x0; dst[1] = x1; dst[2] = x2;
      }
      __syncwarp();
      wait();
      const uint32_t *bchunk = stage_w;
      const int nsteps = kChunk;
      const int kg = max(0, min(nsteps, vhor + 1 - vb0));
      const unsigned cb0 = lutb + 4u * (unsigned)(vb0 - 1);
      const int n0 = vTc + 1 - vb0;
      Best local{inf, inf, 0, 0};
      int k0 = 0;
      if (j == 0) {
        // first segment, vB = 0 (:481-594)
        const CellBase b = cell_base<true, 1, HAS_INVALID>(A, bchunk, ca, lutb, (float)n0, c);
        RowInfo q{};
        const float first_k_o = fmul(fadd(fadd((vT <= vhor) ? kLn2 : 0.0f, p.rows_log), p.max_dis_log), c.pw);
        float cost_gs, cost_o;
        cell_finish<true, true, 1>(b, 0.0f, q, first_k_gs, first_k_o, c, cost_gs, cost_o);
        if (cost_gs < local.gs) { local.gs = cost_gs; local.vb_gs = 0; }
        if (cost_o < local.o) { local.o = cost_o; local.vb_o = 0; }
        k0 = 1;
      }
      if (t * kChunk >= vhor)
        dp_steps<true, 3, false, HAS_INVALID>(A, bchunk, cb0, ca, nullptr, q_w, vb0, k0, max(k0, kg), n0, lane, c, local);
      else
        dp_steps<true, 1, false, HAS_INVALID>(A, bchunk, cb0, ca, nullptr, q_w, vb0, k0, max(k0, kg), n0, lane, c, local);
      dp_steps<true, 0, false, HAS_INVALID>(A, bchunk, cb0, ca, nullptr, q_w, vb0, max(k0, kg), nsteps, n0, lane, c, local);
      merge_best(carried, local);
      my_units++;
    }
    // ---- the warps' minima -> warp 0 ----
    merge[warp * 32 + lane] = make_float4(carried.gs, carried.o, __int_as_float(carried.vb_gs), __int_as_float(carried.vb_o));
    __syncthreads();

    // ================= (2) the diagonal unit: the wavefront =================
    if (warp == 0) {
      Best best = carried;
#pragma unroll
      for (int w = 1; w < WARPS; w++) {
        const float4 m4 = merge[w * 32 + lane];
        merge_best(best, Best{m4.x, m4.y, __float_as_int(m4.z), __float_as_int(m4.w)});
      }
      const int j = t, vb0 = t * kChunk;
      const int nsteps = min(kChunk, H - vb0);
      const int kg = max(0, min(nsteps, vhor + 1 - vb0));
      stage(j);
      for (int i = lane; i < (kChunk + 1) * kStatWords; i += 32)
        sst[i] = (vb0 + i / kStatWords) < H ? __ldg(S + (size_t)vb0 * kStatWords + i) : 0.0f;
      __syncwarp();
      wait();
      const uint32_t *bchunk = stage_w;
      float *qs_slot = q_w;  // Q[vb0 .. vb0+31] as they become known
      // prefix values at the start row of the best object segment so far (previous_mean needs them)
      float lo_d = f_(rec_word(recb, best.vb_o, kRecDisp));
      float lo_v = f_(rec_word(recb, best.vb_o, kRecValid));
      if (j > 0) {
        if (lane < kDynWords) qs_slot[lane] = qnext[lane];
        __syncwarp();
      }
      auto finish_row = [&](int vB, int src_lane, float hi_d, float hi_v) {
        const float c_gs = __shfl_sync(full_mask, best.gs, src_lane), c_o = __shfl_sync(full_mask, best.o, src_lane);
        const int o_vb = __shfl_sync(full_mask, best.vb_o, src_lane);
        const float l_d = __shfl_sync(full_mask, lo_d, src_lane), l_v = __shfl_sync(full_mask, lo_v, src_lane);
        const bool ground_side = vB - 1 < vhor;
        const float pm = segment_mean(hi_d, l_d, hi_v, l_v, vB - o_vb, HAS_INVALID);
        RowPriors rp;
        return make_row_info(sst + (vB - vb0) * kStatWords, ground_side, ground_side ? c_gs : inf, c_o,
                             ground_side ? inf : c_gs, pm, odr, p, &rp);
      };
      auto base_of = [&](int k) {
        const int vB = vb0 + k;
        return cell_base<false, 2, HAS_INVALID>(A, bchunk + k * kRecBWords, ca, lutb + 4u * (unsigned)(vB - 1),
                                                (float)max(vTc + 1 - vB, 1), c, k < kg);
      };
      CellBase b_cur = (j == 0) ? cell_base<true, 1, HAS_INVALID>(A, bchunk, ca, lutb, (float)(vTc + 1), c)
                                : base_of(0);
      for (int k = 0; k < nsteps; k++) {
        const int vB = vb0 + k;
        const float ps_d = f_(bchunk[k * kRecBWords + kRecDisp]), ps_v = f_(bchunk[k * kRecBWords + kRecValid]);
        CellBase b_next = b_cur;
        if (k + 1 < nsteps) b_next = base_of(k + 1);
        RowInfo q{};
        if (k > 0) {
          q = finish_row(vB, k - 1, ps_d, ps_v);
          if (lane == 0) {
            store_row_info(qs_slot + k * kDynWords, q);
            pm_col[vB] = q.pm;
          }
        } else if (vB > 0) {
          q = load_row_info(qs_slot);
        }
        float cost_gs, cost_o;
        if (vB == 0) {
          const float first_k_o = fmul(fadd(fadd((vT <= vhor) ? kLn2 : 0.0f, p.rows_log), p.max_dis_log), c.pw);
          cell_finish<true, true, 1>(b_cur, 0.0f, q, first_k_gs, first_k_o, c, cost_gs, cost_o);
        } else {
          cell_finish<true, false, 2>(b_cur, 0.0f, q, 0.0f, 0.0f, c, cost_gs, cost_o, k < kg);
        }
        const bool live = row_ok && lane >= k;
        if (live && cost_gs < best.gs) { best.gs = cost_gs; best.vb_gs = vB; }
        if (live && cost_o < best.o) { best.o = cost_o; best.vb_o = vB; lo_d = ps_d; lo_v = ps_v; }
        b_cur = b_next;
      }
      // Q[vb0 + 32] for the next diagonal (row vb0 + 31 is final now)
      if (vb0 + kChunk < H) {
        const int vB = vb0 + kChunk;
        const RowInfo q = finish_row(vB, 31, f_(rec_word(recb, vB, kRecDisp)),
                                     f_(rec_word(recb, vB, kRecValid)));
        if (lane == 0) {
          store_row_info(qnext, q);
          pm_col[vB] = q.pm;
        }
      }
      if (row_ok) store_best(out + vT, best);
      {
        // the seeds of the next tile: where the best segments of the tile's last row start
        const int last = nsteps - 1;
        const int so = __shfl_sync(full_mask, best.vb_o, last), sg = __shfl_sync(full_mask, best.vb_gs, last);
        const float cg = __shfl_sync(full_mask, best.gs, last);
        if (lane == 0) {
          seeds[0] = so;
          seeds[1] = cg < inf ? sg : -1;
        }
      }
      __syncwarp();
      // publish Q of the chunk for the later tiles: shared copy -> global (row k by lane k), and its smallest priors
      {
        const float4 *srcq = reinterpret_cast<const float4 *>(qs_slot + lane * kDynWords);
        float4 *dstq = reinterpret_cast<float4 *>(qg + (size_t)(vb0 + lane) * kDynWords);
        if (lane < nsteps) { __stcg(dstq, srcq[0]); __stcg(dstq + 1, srcq[1]); __stcg(dstq + 2, srcq[2]); }
      }
      // ---- the class envelopes M_c[t] of this chunk for the bounds of the later tiles (header): lane = row vB ----
      {
        const int vBl = vb0 + lane;
        const bool in_rows = lane < nsteps;
        float kmin_o = inf, kgs = inf;
        bool ground_side = true;
        if (in_rows) {
          if (vBl == 0) {
            // the first-segment priors (:189-199), the smaller of the two object variants
            kmin_o = fmul(fadd(fadd(0.0f, p.rows_log), p.max_dis_log), c.pw);
            kgs = first_k_gs;
          } else {
            const RowInfo ql = load_row_info(qs_slot + lane * kDynWords);
            ground_side = vBl - 1 < vhor;
            kmin_o = object_prior_floor(ql, ground_side, c.pw);
            kgs = ql.gs_k;
          }
        }
        // the record of this lane's row of the staged chunk (per-lane rows: bank conflicts, once per tile)
        const uint4 *b4 = reinterpret_cast<const uint4 *>(bchunk + lane * kRecBWords);
        uint32_t Bw[20];
#pragma unroll
        for (int k = 0; k < 5; k++) {
          const uint4 q4 = b4[k];
          Bw[4 * k] = q4.x; Bw[4 * k + 1] = q4.y; Bw[4 * k + 2] = q4.z; Bw[4 * k + 3] = q4.w;
        }
        const uint4 gsw = b4[7];   // words 28 .. 31: ground and sky prefix
        const float nicB = fmul((float)(int)Bw[kRecOff], c.iw);
        float mabs = 0.0f;
        auto publish = [&](int slot, float m) {
          if (!in_rows) m = inf;
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) m = fminf(m, __shfl_xor_sync(full_mask, m, d));
          if (m < inf) mabs = fmaxf(mabs, fabsf(m));
          if (lane == 0) mtab[t * kMWords + slot] = m;
        };
#pragma unroll
        for (int k = 2; k < 10; k++) publish(k - 2, fsub(kmin_o, fmul(c.sw, fadd(nicB, (float)(int)Bw[k]))));
#pragma unroll
        for (int k = 11; k < 19; k++) publish(8 + k - 11, fsub(kmin_o, fmul(c.sw, (float)(int)Bw[k])));
        // ground slot candidates come from rows at/below the horizon, sky slot candidates from rows above it
        const float fg0 = ffma(c.dw, f_(gsw.x), fmul(c.sw, fadd(nicB, (float)(int)Bw[0])));
        const float fg1 = ffma(c.dw, f_(gsw.x), fmul(c.sw, fadd(nicB, (float)(int)Bw[1])));
        const float fs = ffma(c.dw, f_(gsw.y), fmul(c.sw, fadd(nicB, (float)(int)Bw[kSkyClass])));
        publish(16, ground_side ? fsub(kgs, fg0) : inf);
        publish(17, ground_side ? fsub(kgs, fg1) : inf);
        publish(18, ground_side ? inf : fsub(kgs, fs));
        if (lane == 0) mtab[t * kMWords + 19] = mabs;
      }
      my_units++;
    }
    __syncthreads();
  }
  if (lane == 0 && my_units) atomicAdd(units_evaluated, my_units);
}

}  // namespace

size_t dp_smem_bytes(const KParams &p, bool pairwise) {
  return DpLayout(p.rows, p.max_dis, pairwise).total;
}

template <bool PAIRWISE, bool HAS_INVALID, int WARPS, int HP>
static void launch_dp_warps(const KParams &p, const BatchBuffers &b, int ncolumns, size_t smem, cudaStream_t s) {
  static SmemOptIn optin;
  opt_in_smem(dp_kernel<PAIRWISE, HAS_INVALID, WARPS, HP>, optin);
  dp_kernel<PAIRWISE, HAS_INVALID, WARPS, HP><<<ncolumns, WARPS * 32, smem, s>>>(
      b.records_b, b.object_lut, b.stat, b.pm, b.vhor, b.object_disparity_range, b.inverse_height, b.dp, p);
}

template <bool PAIRWISE, bool HAS_INVALID, int HP>
static void launch_dp_variant(const KParams &p, const BatchBuffers &b, int ncolumns, size_t smem, cudaStream_t s) {
  const int sms = device_sm_count();
  bool latency = ncolumns < 2 * sms;
  if (const char *e = std::getenv("ISX_DP_WARPS")) {  // tests pin the variant
    if (std::atoi(e) == kDpWarps) latency = false;
    if (std::atoi(e) == kDpWarpsLatency) latency = true;
  }
  if (latency) launch_dp_warps<PAIRWISE, HAS_INVALID, kDpWarpsLatency, HP>(p, b, ncolumns, smem, s);
  else launch_dp_warps<PAIRWISE, HAS_INVALID, kDpWarps, HP>(p, b, ncolumns, smem, s);
}

template <bool HAS_INVALID, int WARPS, int HP>
static void launch_unary_pruned_warps(const KParams &p, const BatchBuffers &b, int ncolumns, cudaStream_t s) {
  const size_t smem = PruneLayout(p.rows, WARPS).total;
  static SmemOptIn optin;
  opt_in_smem(dp_unary_pruned_kernel<HAS_INVALID, WARPS, HP>, optin);
  dp_unary_pruned_kernel<HAS_INVALID, WARPS, HP><<<ncolumns, WARPS * 32, smem, s>>>(
      b.records_b, b.object_lut, b.ground, b.vhor, b.inverse_height, b.dp, b.dp_units, b.col_flags, p);
}

template <bool HAS_INVALID, int HP>
static void launch_unary_pruned(const KParams &p, const BatchBuffers &b, int ncolumns, cudaStream_t s) {
  const int sms = device_sm_count();
  bool latency = ncolumns < 2 * sms;
  if (const char *e = std::getenv("ISX_DP_WARPS")) {  // tests pin the variant
    if (std::atoi(e) == kDpWarps) latency = false;
    if (std::atoi(e) == kDpWarpsLatency) latency = true;
  }
  if (latency) launch_unary_pruned_warps<HAS_INVALID, kDpWarpsLatency, HP>(p, b, ncolumns, s);
  else launch_unary_pruned_warps<HAS_INVALID, kDpWarps, HP>(p, b, ncolumns, s);
}

template <bool HAS_INVALID, int WARPS, int HP>
static void launch_pairwise_walk_warps(const KParams &p, const BatchBuffers &b, int ncolumns, cudaStream_t s) {
  const size_t smem = WalkLayout(p.rows, p.max_dis, WARPS).total;
  static SmemOptIn optin;
  opt_in_smem(dp_pairwise_walk_kernel<HAS_INVALID, WARPS, HP>, optin);
  dp_pairwise_walk_kernel<HAS_INVALID, WARPS, HP><<<ncolumns, WARPS * 32, smem, s>>>(
      b.records_b, b.object_lut, b.stat, b.ground, b.pm, b.qrows, b.vhor, b.object_disparity_range, b.dp,
      b.dp_units, b.col_flags, p);
}

template <bool HAS_INVALID, int HP>
static void launch_pairwise_walk(const KParams &p, const BatchBuffers &b, int ncolumns, cudaStream_t s) {
  const int sms = device_sm_count();
  bool latency = ncolumns < 2 * sms;
  if (const char *e = std::getenv("ISX_DP_WARPS")) {
    if (std::atoi(e) == kDpWarps) latency = false;
    if (std::atoi(e) == kDpWarpsLatency) latency = true;
  }
  // throughput: ONE warp per column (16 columns per SM, no barrier between the tiles of a column, the warp's
  // carried minima see every chunk it evaluated); ISX_WALK_WARPS=4 keeps the 4-warp CTA per column for A/B runs
  int tw = 1;
  if (const char *e = std::getenv("ISX_WALK_WARPS")) tw = std::atoi(e);
  if (latency) launch_pairwise_walk_warps<HAS_INVALID, kDpWarpsLatency, HP>(p, b, ncolumns, s);
  else if (tw == kDpWarps) launch_pairwise_walk_warps<HAS_INVALID, kDpWarps, HP>(p, b, ncolumns, s);
  else launch_pairwise_walk_warps<HAS_INVALID, 1, HP>(p, b, ncolumns, s);
}

// Which pairwise kernel runs: the tile-major walk (ISX_PAIRWISE_WALK=1) or the chunk-major exhaustive one.
bool pairwise_walk_enabled() {
  const char *e = std::getenv("ISX_PAIRWISE_WALK");
  return e ? std::atoi(e) != 0 : (ISX_PAIRWISE_WALK_DEFAULT != 0);
}

// The tile-major walk runs one warp per column: it needs a launch that fills the 16 warp slots of every SM (ten
// 1024 x 2048 frames at width 8); smaller launches keep the chunk-major kernel, whose 4 or 8 warps per column are
// what a few hundred columns need.  ISX_DP_WARPS / ISX_WALK_WARPS (tests) force the walk's variants.
bool pairwise_walk_used(int ncolumns, bool have_qrows) {
  const int sm_count = device_sm_count();
  const bool forced = std::getenv("ISX_DP_WARPS") != nullptr || std::getenv("ISX_WALK_WARPS") != nullptr;
  return pairwise_walk_enabled() && have_qrows && (ncolumns >= 16 * sm_count || forced);
}

// HP: the record stride (kRecStride, or kRecStrideTall for frames of more than kShortRows rows)
template <int HP>
static void launch_dp_rows(const KParams &p, const BatchBuffers &b, int nframes, bool pairwise, cudaStream_t s) {
  const int ncolumns = nframes * p.realcols;
  const size_t smem = dp_smem_bytes(p, pairwise);
  const bool has_invalid = p.invalid_disparity >= 0.0f;  // ComputeMean's two modes (StixelsKernels.cu:47-60)
  // ISX_UNARY_EXHAUSTIVE=1: the unary DP without the walk from the diagonal (every unit of every tile)
  const char *ex = std::getenv("ISX_UNARY_EXHAUSTIVE");
  const bool exhaustive = ex && std::atoi(ex) != 0;
  if (pairwise && pairwise_walk_used(ncolumns, b.qrows != nullptr)) {
    if (has_invalid) launch_pairwise_walk<true, HP>(p, b, ncolumns, s);
    else launch_pairwise_walk<false, HP>(p, b, ncolumns, s);
  } else if (pairwise) {
    if (has_invalid) launch_dp_variant<true, true, HP>(p, b, ncolumns, smem, s);
    else launch_dp_variant<true, false, HP>(p, b, ncolumns, smem, s);
  } else if (!exhaustive) {
    if (has_invalid) launch_unary_pruned<true, HP>(p, b, ncolumns, s);
    else launch_unary_pruned<false, HP>(p, b, ncolumns, s);
  } else {
    if (has_invalid) launch_dp_variant<false, true, HP>(p, b, ncolumns, smem, s);
    else launch_dp_variant<false, false, HP>(p, b, ncolumns, smem, s);
  }
  g_launch_count++;
}

void launch_dp(const KParams &p, const BatchBuffers &b, int nframes, bool pairwise, cudaStream_t s) {
  if (p.rec_stride == kRecStrideTall) launch_dp_rows<kRecStrideTall>(p, b, nframes, pairwise, s);
  else launch_dp_rows<kRecStride>(p, b, nframes, pairwise, s);
}

}  // namespace isx
