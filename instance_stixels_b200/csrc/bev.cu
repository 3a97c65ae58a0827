// Bird's-eye-view grid of a computed batch (isx_bev_grid_device): free, occupied and unknown cells on the ground
// plane, each occupied cell linked to its nearest OBJECT stixel.  The definition is in include/instance_stixels_b200.h;
// Stixels::GetBevGrid (Stixels.hpp) states it on the host, and this file computes the same bytes.
//
//   export_column_scan_kernel (export.cu) : frame-local index of the first stixel of every column
//   memset 0xFF                           : every cell starts as the empty 64-bit key
//   bev_occupancy_kernel                  : one warp per (frame, column), one lane per stixel; an OBJECT stixel
//                                           takes the 64-bit atomicMin of (order key of z) << 32 | i over its cells
//   bev_finalize_kernel                   : one thread per cell decodes the key, or runs the free test with a binary
//                                           search of the column's stixels (as rasterize_kernel does), and rewrites
//                                           the 8 bytes as {stixel, state}
// The library builds with -ftz=true; the new arithmetic below is spelled in PTX without .ftz, so subnormals are kept
// as the host keeps them.  The corners come from stixel_vertices, the code of the export's vertices.
#include "kernels.h"
#include "vertices.cuh"

namespace isx {
namespace {

constexpr int kBevThreads = 256;
constexpr int kBevWarps = kBevThreads / 32;
constexpr unsigned long long kEmptyCell = ~0ull;   // above the key of every non-NaN z

// IEEE binary32 operations and comparisons, rounded to nearest, subnormals kept whatever -ftz says.
__device__ __forceinline__ float add_keep(float a, float b) {
  float r;
  asm("add.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float sub_keep(float a, float b) {
  float r;
  asm("sub.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float mul_keep(float a, float b) {
  float r;
  asm("mul.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float div_keep(float a, float b) {
  float r;
  asm("div.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ bool ge_keep(float a, float b) {
  unsigned r;
  asm("{ .reg .pred p; setp.ge.f32 p, %1, %2; selp.u32 %0, 1, 0, p; }" : "=r"(r) : "f"(a), "f"(b));
  return r != 0;
}
__device__ __forceinline__ bool gt_keep(float a, float b) {
  unsigned r;
  asm("{ .reg .pred p; setp.gt.f32 p, %1, %2; selp.u32 %0, 1, 0, p; }" : "=r"(r) : "f"(a), "f"(b));
  return r != 0;
}
__device__ __forceinline__ bool lt_keep(float a, float b) {
  unsigned r;
  asm("{ .reg .pred p; setp.lt.f32 p, %1, %2; selp.u32 %0, 1, 0, p; }" : "=r"(r) : "f"(a), "f"(b));
  return r != 0;
}

// (order key of z) << 32 | i: unsigned comparison of the keys is the order of z (-0.0 taken as +0.0), then of i.
__device__ __forceinline__ unsigned long long occupant_key(float z, int i) {
  unsigned b = __float_as_uint(z);
  if ((b << 1) == 0) b = 0;
  b ^= (b >> 31) ? 0xffffffffu : 0x80000000u;
  return (unsigned long long)b << 32 | (unsigned)i;
}

__global__ void __launch_bounds__(kBevThreads)
bev_occupancy_kernel(BevArgs a, int nframes) {
  const int C = a.realcols, lane = threadIdx.x & 31;
  const int w = blockIdx.x * kBevWarps + (threadIdx.x >> 5);
  if (w >= nframes * C) return;
  const int f = w / C, col = w - f * C;
  const int n = a.n_sections[w], base = a.col_local[w];
  const isx_section *src = a.sections + (size_t)w * kMaxSections;
  const isx_bev_params &p = a.p;
  unsigned long long *cells = reinterpret_cast<unsigned long long *>(a.cells) + (size_t)f * p.nz * p.nx;
  const float fnx = (float)p.nx, fnz = (float)p.nz;
  for (int j = lane; j < n; j += 32) {
    const isx_section s = src[j];
    if (s.type != OBJECT) continue;
    float v[12];
    stixel_vertices(s, col, a, 0.0f, 0, v);   // OBJECT stixels: no road enters
    const float z = v[2];
    const float rz = div_keep(sub_keep(z, p.z_min), p.cell);
    if (!(ge_keep(rz, 0.0f) && lt_keep(rz, fnz))) continue;   // NaN fails both
    const float l = div_keep(sub_keep(v[0], p.x_min), p.cell), r = div_keep(sub_keep(v[3], p.x_min), p.cell);
    if (!(ge_keep(r, 0.0f) && lt_keep(l, fnx))) continue;
    const int ix0 = lt_keep(l, 0.0f) ? 0 : (int)l, ix1 = ge_keep(r, fnx) ? p.nx - 1 : (int)r;
    const unsigned long long key = occupant_key(z, base + j);
    unsigned long long *row = cells + (size_t)(int)rz * p.nx;
    for (int ix = ix0; ix <= ix1; ix++) atomicMin(row + ix, key);
  }
}

// Whether the ground is seen at the centre of cell (iz, ix) of frame f (the free test of the definition).
__device__ __forceinline__ bool ground_visible(const BevArgs &a, int f, int iz, int ix, float alpha, int vhor) {
  const isx_bev_params &p = a.p;
  const float xc = add_keep(p.x_min, mul_keep(add_keep((float)ix, 0.5f), p.cell));
  const float zc = add_keep(p.z_min, mul_keep(add_keep((float)iz, 0.5f), p.cell));
  if (!gt_keep(zc, 0.0f)) return false;
  const float u = add_keep(a.camera_center_x, mul_keep(a.focal, div_keep(xc, zc)));
  if (!(ge_keep(u, 0.0f) && lt_keep(u, (float)(a.realcols * a.column_step)))) return false;
  const int c = (int)u / a.column_step;
  const float t = div_keep(a.bf, mul_keep(alpha, zc));
  const float vf = sub_keep((float)vhor, t);
  if (!(gt_keep(t, 0.0f) && ge_keep(vf, 0.0f) && lt_keep(vf, (float)a.rows))) return false;
  const int v = (int)vf;
  const size_t fc = (size_t)f * a.realcols + c;
  const int n = a.n_sections[fc];
  if (n < 1) return false;
  const isx_section *col = a.sections + fc * kMaxSections;
  int lo = 0, hi = n - 1;   // vB decreases with the index: smallest index with vB <= v
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (col[mid].vB <= v) hi = mid; else lo = mid + 1;
  }
  const isx_section s = col[lo];
  return s.vB <= v && v <= s.vT && s.type == GROUND;
}

__global__ void __launch_bounds__(kBevThreads)
bev_finalize_kernel(BevArgs a, ExportFrames fr, int f0) {
  const int f = f0 + blockIdx.y, nx = a.p.nx, per = a.p.nz * nx;
  const int k = blockIdx.x * kBevThreads + threadIdx.x;
  if (k >= per) return;
  unsigned long long *cell = reinterpret_cast<unsigned long long *>(a.cells) + (size_t)f * per + k;
  const unsigned long long key = *cell;
  int stixel = -1, state = ISX_BEV_UNKNOWN;
  if (key != kEmptyCell) {
    stixel = (int)(unsigned)key;
    state = ISX_BEV_OCCUPIED;
  } else {
    const float alpha = a.roads ? a.roads[f].alpha_ground : fr.alpha_ground[blockIdx.y];
    const int vhor = a.roads ? a.rows - a.roads[f].vhor - 1 : fr.vhor[blockIdx.y];   // flipped (Stixels.cu:377)
    if (ground_visible(a, f, k / nx, k - (k / nx) * nx, alpha, vhor)) state = ISX_BEV_FREE;
  }
  *reinterpret_cast<int2 *>(cell) = make_int2(stixel, state);
}

}  // namespace

void launch_bev_grid(const BevArgs &a, int nframes, const float *alpha_ground, const int *vhor, cudaStream_t s) {
  launch_export_column_scan(a.n_sections, a.realcols, a.col_local, a.frame_totals, nframes, s);
  const size_t per = (size_t)a.p.nz * a.p.nx;
  cudaMemsetAsync(a.cells, 0xff, sizeof(isx_bev_cell) * per * nframes, s);
  const int warps = nframes * a.realcols;
  bev_occupancy_kernel<<<(warps + kBevWarps - 1) / kBevWarps, kBevThreads, 0, s>>>(a, nframes);
  g_launch_count++;
  // the road scalars travel as kernel parameters, kExportFramesPerLaunch frames per launch, as in the export
  for (int f0 = 0; f0 < nframes; f0 += kExportFramesPerLaunch) {
    const int gn = nframes - f0 < kExportFramesPerLaunch ? nframes - f0 : kExportFramesPerLaunch;
    ExportFrames fr;
    for (int i = 0; i < gn; i++) {
      fr.alpha_ground[i] = a.roads ? 0.0f : alpha_ground[f0 + i];
      fr.vhor[i] = a.roads ? 0 : vhor[f0 + i];
    }
    bev_finalize_kernel<<<dim3((unsigned)((per + kBevThreads - 1) / kBevThreads), gn), kBevThreads, 0, s>>>(a, fr, f0);
    g_launch_count++;
  }
}

}  // namespace isx
