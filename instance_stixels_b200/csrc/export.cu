// Stixels of a computed batch -> caller device buffers (isx_export_batch_device), for consumers on the GPU.
// The layout is CSR over the frames and columns of the batch: the used Sections of frame f lie at
// [frame_offsets[f], frame_offsets[f+1]), column 0 first, each column top to bottom (the order of
// isx_wait_batch_packed and of Stixels::Get3DVertices); column c of frame f starts at column_offsets[f*C + c].
// Per stixel there is an instance label (the map GetInstanceStixels returns, -2 for stixels outside it) and the
// four corner points Get3DVertices computes (Stixels.hpp, Stixels.cu:683-742).
// Unlike pack_results_kernel, which places frames with atomicAdd, every position follows from the scans: the bytes
// are the same from run to run.
#include "kernels.h"

namespace isx {
namespace {

constexpr int kExportThreads = 256;
constexpr int kExportWarps = kExportThreads / 32;
constexpr int kFrameScanThreads = 1024;

// One CTA per frame: the exclusive prefix of the stixel counts over the columns (the scan of pack_results_kernel)
// into col_local[f*C + c], relative to the frame; the frame's total into frame_offsets[f + 1].
__global__ void __launch_bounds__(kExportThreads)
export_column_scan_kernel(const int *__restrict__ n_sections, int C, int *__restrict__ col_local,
                          int *__restrict__ frame_offsets) {
  __shared__ int warp_tot[kExportWarps];
  __shared__ int s_running;
  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int *ns = n_sections + (size_t)f * C;
  if (tid == 0) s_running = 0;
  __syncthreads();
  for (int base = 0; base < C; base += kExportThreads) {
    const int col = base + tid;
    const int n = col < C ? ns[col] : 0;
    int incl = n;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = s_running;
    for (int w = 0; w < warp; w++) before += warp_tot[w];
    if (col < C) col_local[(size_t)f * C + col] = before + incl - n;
    __syncthreads();
    if (tid == 0) {
      int t = s_running;
      for (int w = 0; w < kExportWarps; w++) t += warp_tot[w];
      s_running = t;
    }
    __syncthreads();
  }
  if (tid == 0) frame_offsets[f + 1] = s_running;
}

// One CTA: the frame totals in frame_offsets[1..n] -> their inclusive prefix (frame_offsets[0] = 0), in place.
__global__ void __launch_bounds__(kFrameScanThreads)
export_frame_scan_kernel(int *__restrict__ frame_offsets, int *__restrict__ column_offsets, int n, int C) {
  __shared__ int warp_tot[kFrameScanThreads / 32];
  __shared__ int s_running;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_running = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kFrameScanThreads) {
    const int f = base + tid;
    int incl = f < n ? frame_offsets[f + 1] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = s_running;
    for (int w = 0; w < warp; w++) before += warp_tot[w];
    if (f < n) frame_offsets[f + 1] = before + incl;
    __syncthreads();
    if (tid == 0) {
      int t = s_running;
      for (int w = 0; w < kFrameScanThreads / 32; w++) t += warp_tot[w];
      s_running = t;
    }
    __syncthreads();
  }
  if (tid == 0) {
    frame_offsets[0] = 0;
    if (column_offsets) column_offsets[(size_t)n * C] = s_running;
  }
}

// Stixels::Get3DVertices for one Section, in the header's operation order (xl = i * step, xr = xl + step,
// yt = rows - vT - 1, yb = rows - vB; z = bf / disparity for objects, bf / (alpha_ground * (vhor - v)) for ground,
// 0 for sky; then per corner -z / f * (c - x), -z / f * (c - y), z), with every operation rounded on its own.
__device__ __forceinline__ void stixel_vertices(const isx_section &s, int col, const ExportArgs &a, float alpha,
                                                int vhor, float *v) {
  const float xl = (float)(col * a.column_step), xr = __fadd_rn(xl, (float)a.column_step);
  const float yt = (float)(a.rows - s.vT - 1), yb = (float)(a.rows - s.vB);
  float zt = 0.0f, zb = 0.0f;
  if (s.type == OBJECT) {
    zt = zb = __fdiv_rn(a.bf, s.disparity);
  } else if (s.type == GROUND) {
    zt = __fdiv_rn(a.bf, __fmul_rn(alpha, (float)(vhor - s.vT)));
    zb = __fdiv_rn(a.bf, __fmul_rn(alpha, (float)(vhor - s.vB)));
  }
  const float cx[4] = {xl, xr, xr, xl}, cy[4] = {yt, yt, yb, yb}, cz[4] = {zt, zt, zb, zb};
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const float q = __fdiv_rn(-cz[k], a.focal);
    v[3 * k + 0] = __fmul_rn(q, __fsub_rn(a.camera_center_x, cx[k]));
    v[3 * k + 1] = __fmul_rn(q, __fsub_rn(a.camera_center_y, cy[k]));
    v[3 * k + 2] = cz[k];
  }
}

// One CTA per frame, one warp per column.  Column offsets and the error word are always written; Sections, labels
// and vertices only if the whole frame fits `capacity`.  Labels start at -2 and the frame's instance records
// (column, index, label, class) overwrite theirs after the CTA barrier.
__global__ void __launch_bounds__(kExportThreads)
export_stixels_kernel(ExportArgs a, ExportFrames fr, int f0) {
  __shared__ float s_vert[kExportWarps][32 * 12];
  const int f = f0 + blockIdx.x, C = a.realcols;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const isx_device_results &o = a.out;
  const int *ns = a.n_sections + (size_t)f * C;
  const int *loc = a.col_local + (size_t)f * C;
  const int base = o.frame_offsets[f];
  const bool fits = o.frame_offsets[f + 1] <= o.capacity;
  if (o.column_offsets)
    for (int col = tid; col < C; col += kExportThreads) o.column_offsets[(size_t)f * C + col] = base + loc[col];
  if (tid == 0 && o.frame_errors) o.frame_errors[f] = a.frames[f].error;
  if (!fits) return;
  const float alpha = a.roads ? a.roads[f].alpha_ground : fr.alpha_ground[blockIdx.x];
  const int vhor = a.roads ? a.rows - a.roads[f].vhor - 1 : fr.vhor[blockIdx.x];   // flipped (Stixels.cu:377)
  for (int col = warp; col < C; col += kExportWarps) {
    const int n = ns[col], dst0 = base + loc[col];
    const isx_section *src = a.sections + ((size_t)f * C + col) * kMaxSections;
    if (o.sections) {
      const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
      uint4 *d4 = reinterpret_cast<uint4 *>(o.sections + dst0);
      for (int j = lane; j < 2 * n; j += 32) d4[j] = s4[j];
    }
    if (o.labels)
      for (int j = lane; j < n; j += 32) o.labels[dst0 + j] = -2;
    if (o.vertices) {
      // 32 stixels per pass: each lane computes its 12 floats into shared memory, the warp stores the 1.5 KB back
      // to back
      float *sv = s_vert[warp];
      for (int j0 = 0; j0 < n; j0 += 32) {
        const int j = j0 + lane, cnt = min(32, n - j0);
        if (j < n) stixel_vertices(src[j], col, a, alpha, vhor, sv + 12 * lane);
        __syncwarp();
        float *dv = o.vertices + (size_t)(dst0 + j0) * 12;
        for (int k = lane; k < 12 * cnt; k += 32) dv[k] = sv[k];
        __syncwarp();
      }
    }
  }
  if (!o.labels) return;
  __syncthreads();
  const int ni = min(a.inst_count[f], a.inst_cap);
  const isx_instance *rec = a.inst + (size_t)f * a.inst_cap;
  for (int i = tid; i < ni; i += kExportThreads) {
    const isx_instance r = rec[i];
    o.labels[base + loc[r.column] + r.index] = r.label;
  }
}

}  // namespace

void launch_export_results(const ExportArgs &a, int nframes, const float *alpha_ground, const int *vhor,
                           cudaStream_t s) {
  export_column_scan_kernel<<<nframes, kExportThreads, 0, s>>>(a.n_sections, a.realcols, a.col_local,
                                                               a.out.frame_offsets);
  export_frame_scan_kernel<<<1, kFrameScanThreads, 0, s>>>(a.out.frame_offsets, a.out.column_offsets, nframes,
                                                           a.realcols);
  g_launch_count += 2;
  // the road scalars of the frames travel as kernel parameters, kExportFramesPerLaunch frames per launch (unless they
  // are in device memory, a.roads)
  for (int f0 = 0; f0 < nframes; f0 += kExportFramesPerLaunch) {
    const int gn = nframes - f0 < kExportFramesPerLaunch ? nframes - f0 : kExportFramesPerLaunch;
    ExportFrames fr;
    for (int i = 0; i < gn; i++) {
      fr.alpha_ground[i] = a.roads ? 0.0f : alpha_ground[f0 + i];
      fr.vhor[i] = a.roads ? 0 : vhor[f0 + i];
    }
    export_stixels_kernel<<<gn, kExportThreads, 0, s>>>(a, fr, f0);
    g_launch_count++;
  }
}

}  // namespace isx
