// Launchers of the sm_100a kernels (one translation unit per stage).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <string>

#include "../../include/instance_stixels_b200.h"
#include "common.cuh"

namespace isx {

// Device buffers of one batch (B frames).  Layouts are documented in DESIGN.md.
struct BatchBuffers {
  // inputs
  const float *disparity = nullptr;    // [B][H][W]
  const int32_t *segmentation = nullptr;  // [B][C][21][Hs2]
  // per-frame road tables
  float *ground = nullptr;             // [B][3][H]: ground_function | normalization | inv_sigma2
  int *vhor = nullptr;                 // [B] flipped horizon row
  float *stat = nullptr;               // [B][H][kStatWords] static transition records (pairwise)
  // intermediates
  float *joined = nullptr;             // [B][C][H]
  uint32_t *records_b = nullptr;       // [B][C][rec_stride][kRecBWords]: one 128-byte record per row (common.cuh)
  float *object_lut = nullptr;         // [B][C][D][lut_stride]
  float *pm = nullptr;                 // [B][C][H] previous_mean of row vB-1 (pairwise; backtracking re-derives priors)
  float *qrows = nullptr;              // [B][C][rec_stride][kDynWords] transition records Q[vB] (pairwise tile-major walk)
  float4 *dp = nullptr;                // [B][C][H]: {cost_gs, cost_obj, as_float(vB_gs), as_float(vB_obj)}
  // model tables (device copies of HostModel vectors)
  const float *obj_cost_lut = nullptr;       // [D][D]
  const float *obj_cost_lut_t = nullptr;     // [D][D rounded up to 32], transposed: [dis][fn]
  const float *object_disparity_range = nullptr;  // [D]
  const float *inverse_height = nullptr;     // [H+1]
  // outputs
  isx_section *sections = nullptr;     // [B][C][200]
  int *n_sections = nullptr;           // [B][C] stixels per column
  // instance candidates, per frame and instance class, column-major stable order
  int *cand_count = nullptr;           // [B][8]
  int *cand_offset = nullptr;          // [B][C+1][8] exclusive prefix over columns (per class)
  float2 *cand_xy = nullptr;           // [B][8][C*200]
  int2 *cand_idx = nullptr;            // [B][8][C*200] (column, index)
  uint8_t *cand_core = nullptr;        // [B][8][C*200] size filter
  int *cand_label = nullptr;           // [B][8][C*200]
  int *cand_scratch = nullptr;         // [B][8][C*200] component representatives
  int *error_flag = nullptr;           // [B] per frame: kErr* bits (column overflowed 200 stixels, offsets out of range)
  int *pack_offset = nullptr;          // [B][C+1] exclusive prefix of the stixel counts over columns (result packing)
  int *col_flags = nullptr;            // [B][C] 1: the column has negative class values -> no pruning in the DP
  unsigned long long *dp_units = nullptr;  // [1] 32 x 32-cell units the unary DP evaluated (it prunes the rest)
};

void launch_join_columns(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s);
void launch_frame_tables(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s);
void launch_column_tables(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s);
void launch_dp(const KParams &p, const BatchBuffers &b, int nframes, bool pairwise, cudaStream_t s);
bool pairwise_walk_enabled();
// whether launch_dp takes the tile-major walk for a pairwise launch of `ncolumns` columns
bool pairwise_walk_used(int ncolumns, bool have_qrows);
void launch_emit(const KParams &p, const BatchBuffers &b, int nframes, bool pairwise, cudaStream_t s);
// segmentation ingest (FlipAndPad, ingest.cu): cnn float [n][channels][hs][ws] -> seg int32 [n][C][channels][hs2]
void launch_flip_and_pad(const KParams &p, const float *cnn, int32_t *seg, int nframes, int hs, int ws,
                         cudaStream_t s);
// stixels -> label / instance / disparity images (raster.cu)
void launch_rasterize(const KParams &p, const isx_section *sections, const int *n_sections, const isx_instance *inst,
                      const int *inst_count, int inst_cap, int *table, int nframes, uint8_t *label_img,
                      int32_t *instance_img, float *disparity_img, cudaStream_t s);
void launch_grouping(const KParams &p, const BatchBuffers &b, int nframes, cudaStream_t s);
// Result packing (emit.cu): everything pack_results_kernel reads and writes for the frames of one chunk.
struct PackArgs {
  const isx_section *sections;   // [n][C][200] padded device results of the chunk
  const int *n_sections;         // [n][C]
  const int *cand_count;         // [n][8]
  const int2 *cand_idx;          // [n][8][C*200]
  const int *cand_label;         // [n][8][C*200]
  const int *err;                // [n] kErr* bits per frame
  int *col_offset;               // [n][C+1] scratch
  isx_instance *inst_out;        // [n][inst_cap] device copy of the records
  int *inst_count_out;           // [n]
  int inst_cap;
  int *cursors;                  // [2] device: next free packed section / instance record of the result set
  // pinned host memory, mapped (device-visible addresses)
  isx_section *h_sections;       // packed sections of the whole batch
  int h_sections_cap;
  isx_instance *h_inst;          // packed instance records of the whole batch
  int h_inst_cap;
  isx_section *h_padded;         // the caller's own [n][C][200] array when it is pinned and mapped (else null): the
                                 // used Sections and the terminator of every column are written straight into it
                                 // and the packed copy is skipped
  int *h_counts;                 // [n][C] stixels per column
  isx_packed_frame *h_frames;    // [n]
};
void launch_pack(const KParams &p, const PackArgs &a, int nframes, cudaStream_t s);
// Device export of a computed batch (export.cu): frames [0, n) of the arrays below, into the caller's buffers.
struct ExportArgs {
  const isx_section *sections;   // [n][C][200] padded device results
  const int *n_sections;         // [n][C]
  const isx_instance *inst;      // [n][inst_cap]
  const int *inst_count;         // [n]
  int inst_cap;
  const isx_packed_frame *frames;  // [n] descriptors the packing wrote (mapped host memory): the error words
  int *col_local;                // [n][C] scratch: column offsets relative to the frame
  int realcols, rows, column_step;
  float focal, bf, camera_center_x, camera_center_y;   // bf = baseline * focal
  // [n] roads of the frames in device memory (batches whose roads were estimated on the device), or null: the road
  // scalars then travel as kernel parameters (ExportFrames)
  const isx_road *roads;
  isx_device_results out;
};
constexpr int kExportFramesPerLaunch = 128;
struct ExportFrames {              // per-frame road scalars of one launch: alpha_ground and the flipped horizon row
  float alpha_ground[kExportFramesPerLaunch];
  int vhor[kExportFramesPerLaunch];
};
void launch_export_results(const ExportArgs &a, int nframes, const float *alpha_ground, const int *vhor,
                           cudaStream_t s);
// Road estimation in front of a device batch (road.cu, isx_compute_batch_device_road): the checks (nothing enqueued),
// then the Hough kernels, the device line selection and the keep-last rule on the road handle's stream, ordered after
// and before `caller`.  d_roads [n]: the road every frame is computed with.  0 or an isx_status, text in `msg`.
int road_check_batch(isx_road_handle road, int device, int rows, int cols, int max_dis, int n, bool has_fallback,
                     std::string &msg);
int road_enqueue_batch(isx_road_handle road, cudaStream_t caller, int n, const float *d_disparity,
                       const isx_road *fallback, isx_road_estimate *d_estimates, isx_road *d_roads_out,
                       isx_road *d_roads, std::string &msg);
// u16 disparity / i16 segmentation staging -> the float / int32 layouts of the path (ingest.cu)
void launch_widen_inputs(const KParams &p, const uint16_t *disp16, float scale, const int16_t *seg16, float *disp,
                         int32_t *seg, int nframes, cudaStream_t s);
// one point set through the grouping kernel, host buffers; 0 or a cudaError_t
int dbscan_fit_host(const float *xy, int n, float eps, int min_pts, const uint8_t *core_candidates, int *labels,
                    int threads);
// reference-format views for the parity tests
void launch_export_tables(const KParams &p, const BatchBuffers &b, int frame, bool pairwise, float *cost_table,
                          int *index_table, cudaStream_t s);

extern std::atomic<unsigned long long> g_launch_count;

// ---- per-device launch state ----
// cudaFuncSetAttribute applies to the CURRENT device only and the SM count is a property of the device, so neither
// may be cached process-wide: one process can hold contexts on several GPUs (isx_create(&h, device), isx_pool_*),
// each driven by its own host thread.
constexpr int kMaxDevices = 64;
inline int current_device() {
  int d = 0;
  cudaGetDevice(&d);
  return (d < 0 || d >= kMaxDevices) ? 0 : d;
}
// SM count of the current device.
inline int device_sm_count() {
  static std::atomic<int> sms[kMaxDevices];
  const int d = current_device();
  int n = sms[d].load(std::memory_order_relaxed);
  if (n == 0) {
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, d);
    sms[d].store(n, std::memory_order_relaxed);
  }
  return n;
}
// Opt-in to more than 48 KB of dynamic shared memory for `kernel` on the current device: once per (kernel, device),
// always to the device's maximum, so that concurrent callers can only ever write the same value.
struct SmemOptIn {
  std::atomic<int> done[kMaxDevices];
};
template <class Kernel>
inline cudaError_t opt_in_smem(Kernel kernel, SmemOptIn &state) {
  const int d = current_device();
  if (state.done[d].load(std::memory_order_acquire)) return cudaSuccess;
  int max_optin = 0;
  cudaError_t e = cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, d);
  if (e != cudaSuccess) return e;
  cudaFuncAttributes fa;
  e = cudaFuncGetAttributes(&fa, kernel);   // the limit covers static + dynamic shared memory together
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - (int)fa.sharedSizeBytes);
  if (e == cudaSuccess) state.done[d].store(1, std::memory_order_release);
  return e;
}

}  // namespace isx
