// Stixels of a computed batch -> caller device buffers (isx_export_batch_device), for consumers on the GPU.
// The layout is CSR over the frames and columns of the batch: the used Sections of frame f lie at
// [frame_offsets[f], frame_offsets[f+1]), column 0 first, each column top to bottom (the order of
// isx_wait_batch_packed and of Stixels::Get3DVertices); column c of frame f starts at column_offsets[f*C + c].
// Per stixel there is an instance label (the map GetInstanceStixels returns, -2 for stixels outside it) and the
// four corner points Get3DVertices computes (Stixels.hpp, Stixels.cu:683-742, vertices.cuh).
// Unlike pack_results_kernel, which places frames with atomicAdd, every position follows from the scans: the bytes
// are the same from run to run.
#include "kernels.h"
#include "vertices.cuh"

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

// ---- device objects (isx_export_objects_device): one record per (frame, class, label) of the instance records ----
constexpr int kObjectThreads = 256;
constexpr int kClasses = ISX_INSTANCE_CLASSES;
constexpr int kKeyEmpty = 0x7fffffff;   // "no value" of a minimum: the key of no float but a NaN
constexpr int kKeyEmptyMax = -kKeyEmpty - 1;

// Order-preserving int key of a non-NaN float: signed comparison of the keys is the float order, with -0.0 below
// +0.0.  The map is its own inverse.
__device__ __forceinline__ int float_key(float x) {
  const int b = __float_as_int(x);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
// key -> float bits; the empty key -> 0x7FC00000 (every member NaN)
__device__ __forceinline__ int key_bits(int k, int empty) {
  return k == empty ? 0x7fc00000 : (k >= 0 ? k : k ^ 0x7fffffff);
}

// One CTA per frame: objects of instance class 11+k = 1 + the largest label of the frame's records of that class, into
// class_start[8f + k + 1].  The frame scan then makes class_start the exclusive prefix over (frame, class).
__global__ void __launch_bounds__(kObjectThreads)
object_count_kernel(const isx_instance *__restrict__ inst, const int *__restrict__ inst_count, int inst_cap,
                    int *__restrict__ class_start) {
  __shared__ int s_max[kClasses];
  const int f = blockIdx.x, tid = threadIdx.x;
  if (tid < kClasses) s_max[tid] = -1;
  __syncthreads();
  const int ni = min(inst_count[f], inst_cap);
  const isx_instance *rec = inst + (size_t)f * inst_cap;
  for (int i = tid; i < ni; i += kObjectThreads) {
    const isx_instance r = rec[i];
    const int k = r.semantic_class - ISX_FIRST_INSTANCE_CLASS;
    if (r.label >= 0 && k >= 0 && k < kClasses) atomicMax(&s_max[k], r.label);
  }
  __syncthreads();
  if (tid < kClasses) class_start[(size_t)f * kClasses + tid + 1] = s_max[tid] + 1;
}

// One CTA per frame.  Offsets are always written; the frame's objects and extents only if they all fit `capacity`.
// Three passes over global memory, separated by CTA barriers: initialise the frame's records (minima at the empty key,
// maxima at its negation), let every instance record fold its Section into its object with integer atomics (floats as
// order-preserving keys, NaN skipped), then turn the keys back into floats and the column range into the image box.
// Every update is a sum, a minimum or a maximum of integers, so the result does not depend on their order.
__global__ void __launch_bounds__(kObjectThreads)
export_objects_kernel(ObjectArgs a) {
  __shared__ int s_start[kClasses + 1];
  const int f = blockIdx.x, tid = threadIdx.x, last = gridDim.x - 1;
  const isx_device_objects &o = a.out;
  if (tid <= kClasses) {
    const int v = a.class_start[(size_t)f * kClasses + tid];
    s_start[tid] = v;
    if (o.class_offsets && (tid < kClasses || f == last)) o.class_offsets[(size_t)f * kClasses + tid] = v;
    if (tid == 0 || (tid == kClasses && f == last)) o.frame_offsets[f + tid / kClasses] = v;
  }
  __syncthreads();
  const int lo = s_start[0], hi = s_start[kClasses];
  int *obj = reinterpret_cast<int *>(o.objects);   // 12 words per object
  int *ext = reinterpret_cast<int *>(o.extents);   // 6 words per object
  if (hi > o.capacity || (!obj && !ext)) return;
  for (int j = lo + tid; j < hi; j += kObjectThreads) {
    int k = 0;
    while (j >= s_start[k + 1]) k++;
    if (obj) {
      int4 *w = reinterpret_cast<int4 *>(obj + (size_t)j * 12);
      w[0] = make_int4(ISX_FIRST_INSTANCE_CLASS + k, j - s_start[k], 0, 0);    // class, label, stixels, pixels
      w[1] = make_int4(kKeyEmpty, kKeyEmptyMax, 0, kKeyEmpty);                 // col_min, col_max, x0, y0
      w[2] = make_int4(0, kKeyEmptyMax, kKeyEmpty, kKeyEmptyMax);              // x1, y1, disparity_min, _max
    }
    if (ext)
      for (int q = 0; q < 3; q++) {
        ext[(size_t)j * 6 + q] = kKeyEmpty;
        ext[(size_t)j * 6 + 3 + q] = kKeyEmptyMax;
      }
  }
  __syncthreads();
  const int ni = min(a.inst_count[f], a.inst_cap);
  const isx_instance *rec = a.inst + (size_t)f * a.inst_cap;
  for (int i = tid; i < ni; i += kObjectThreads) {
    const isx_instance r = rec[i];
    const int k = r.semantic_class - ISX_FIRST_INSTANCE_CLASS;
    if (r.label < 0 || k < 0 || k >= kClasses) continue;
    const size_t j = (size_t)(s_start[k] + r.label);
    const isx_section s = a.sections[((size_t)f * a.realcols + r.column) * kMaxSections + r.index];
    if (obj) {
      int *w = obj + j * 12;
      atomicAdd(w + 2, 1);
      atomicAdd(w + 3, a.column_step * (s.vT - s.vB + 1));
      atomicMin(w + 4, r.column);
      atomicMax(w + 5, r.column);
      atomicMin(w + 7, a.rows - 1 - s.vT);
      atomicMax(w + 9, a.rows - 1 - s.vB);
      if (!isnan(s.disparity)) {
        const int key = float_key(s.disparity);
        atomicMin(w + 10, key);
        atomicMax(w + 11, key);
      }
    }
    if (ext) {
      float v[12];
      stixel_vertices(s, r.column, a, 0.0f, 0, v);   // members are OBJECT stixels: no road enters
      int mn[3] = {kKeyEmpty, kKeyEmpty, kKeyEmpty}, mx[3] = {kKeyEmptyMax, kKeyEmptyMax, kKeyEmptyMax};
#pragma unroll
      for (int c = 0; c < 12; c++) {
        if (isnan(v[c])) continue;
        const int key = float_key(v[c]);
        mn[c % 3] = min(mn[c % 3], key);
        mx[c % 3] = max(mx[c % 3], key);
      }
      int *e = ext + j * 6;
#pragma unroll
      for (int q = 0; q < 3; q++)
        if (mn[q] != kKeyEmpty) {
          atomicMin(e + q, mn[q]);
          atomicMax(e + 3 + q, mx[q]);
        }
    }
  }
  __syncthreads();
  // the atomics ran in L2: read their results past L1
  for (int j = lo + tid; j < hi; j += kObjectThreads) {
    if (obj) {
      int *w = obj + (size_t)j * 12;
      w[6] = __ldcg(w + 4) * a.column_step;
      w[8] = __ldcg(w + 5) * a.column_step + a.column_step - 1;
      w[10] = key_bits(__ldcg(w + 10), kKeyEmpty);
      w[11] = key_bits(__ldcg(w + 11), kKeyEmptyMax);
    }
    if (ext)
      for (int q = 0; q < 6; q++) {
        int *e = ext + (size_t)j * 6 + q;
        *e = key_bits(__ldcg(e), q < 3 ? kKeyEmpty : kKeyEmptyMax);
      }
  }
}

}  // namespace

void launch_export_objects(const ObjectArgs &a, int nframes, cudaStream_t s) {
  object_count_kernel<<<nframes, kObjectThreads, 0, s>>>(a.inst, a.inst_count, a.inst_cap, a.class_start);
  // the frame scan over the n*8 counts in class_start[1..n*8]: class_start[i] = objects before (frame, class) i
  export_frame_scan_kernel<<<1, kFrameScanThreads, 0, s>>>(a.class_start, nullptr, nframes * kClasses, 0);
  export_objects_kernel<<<nframes, kObjectThreads, 0, s>>>(a);
  g_launch_count += 3;
}

void launch_export_column_scan(const int *n_sections, int realcols, int *col_local, int *frame_totals, int nframes,
                               cudaStream_t s) {
  export_column_scan_kernel<<<nframes, kExportThreads, 0, s>>>(n_sections, realcols, col_local, frame_totals);
  g_launch_count++;
}

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
