// Road estimation on the device (SURVEY.md 8f rank 1).
// Replaces RoadEstimation (InstanceStixels/src/RoadEstimation.cu:24-193, RoadEstimationKernels.cu:25-60)
// and the cv::HoughLines call inside it (RoadEstimation.cu:152; OpenCV's standard Hough transform:
// createTrigTable / accumulate / findLocalMaximums / sort by votes).
//
//   vdisp_kernel      : CTA per image row; the row's histogram of (int)d lives in shared memory (the
//                       reference does one global atomicAdd per pixel), one coalesced store per row and
//                       one atomicMax per row for the maximum.
//   binarize_kernel   : (float)p > max * threshold -> 255/0, and the set pixels are compacted into a
//                       point list (the Hough accumulation is order-independent integer counting).
//   hough_kernel      : CTA per angle; its accumulator row (2 (W + H) + 3 ints) lives in shared memory,
//                       r = cvRound(j * tabCos[n] + i * tabSin[n]) with the same float products/sum.
//   maxima_kernel     : OpenCV's local-maximum test, candidates compacted as (index, votes).
// The candidates go to the host, which orders them like OpenCV (votes descending, index ascending) and
// applies RoadEstimation::ComputeHough / ComputeCameraProperties with glibc's sinf/cosf/atanf.
//
// isx_compute_batch_device_road selects on the device instead, with nothing on the host in between:
//   select_kernel     : per frame, the argmax of (votes, -index) over the cells that pass the local-maximum test, the
//                       vote threshold and the pitch range -- the first line the host's ordered walk accepts.  Whether
//                       a cell's pitch is in range, and its camera properties, depend on the cell alone: a table
//                       built once per handle on the host with the very code of the host walk (cell_estimate).
//   resolve_kernel    : cells -> estimates, and the reference's keep-last rule across the frames of the batch (or, for
//                       the frame pool, every frame on its own: its estimate or the seed).
//   pull_tables_kernel: host batches with estimated roads -- the staged ground tables of a chunk from mapped pinned
//                       memory into the road ring, read by the SMs, so that no copy queues on the copy engine.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>

#include "cuda_resources.h"
#include "kernels.h"

namespace isx {
namespace {

constexpr int kHoughThreshold = 25;  // m_HoughAccumThr, RoadEstimation.cu:45
constexpr int kMaxCandidates = 1 << 16;

__global__ void __launch_bounds__(256)
vdisp_kernel(const float *__restrict__ disparity, int *__restrict__ vdisp, int *__restrict__ maximum, int rows,
             int cols, int max_dis) {
  extern __shared__ int hist[];
  const int row = blockIdx.x, f = blockIdx.y;
  for (int i = threadIdx.x; i < max_dis; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const float *src = disparity + ((size_t)f * rows + row) * cols;
  const int lane = threadIdx.x & 31;
  auto vote = [&](float d) {
    // RoadEstimationKernels.cu:32-36: d != 0 -> bin (int)d.  The reference writes out of bounds for
    // d < 0 or d >= max_dis; those pixels are ignored here.  Neighbouring pixels of a row mostly fall
    // into the same bin (the road surface), so the votes of a warp are merged before the atomic.
    int c = (d != 0.0f) ? (int)d : -1;
    if (c >= max_dis) c = -1;
    const unsigned peers = __match_any_sync(__activemask(), c);
    if (c >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hist[c], __popc(peers));
  };
  if ((cols & 3) == 0 && ((size_t)src & 15) == 0) {
    const float4 *s4 = reinterpret_cast<const float4 *>(src);
    for (int i = threadIdx.x; i < cols / 4; i += blockDim.x) {
      const float4 v = __ldg(s4 + i);
      vote(v.x); vote(v.y); vote(v.z); vote(v.w);
    }
  } else {
    for (int i = threadIdx.x; i < cols; i += blockDim.x) vote(__ldg(src + i));
  }
  __syncthreads();
  int m = 0;
  int *dst = vdisp + ((size_t)f * rows + row) * max_dis;
  for (int i = threadIdx.x; i < max_dis; i += blockDim.x) {
    const int v = hist[i];
    dst[i] = v;
    m = max(m, v);
  }
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0 && m > 0) atomicMax(maximum + f, m);
}

__global__ void __launch_bounds__(256)
binarize_kernel(const int *__restrict__ vdisp, const int *__restrict__ maximum, uint8_t *__restrict__ binary,
                int2 *__restrict__ points, int *__restrict__ n_points, float threshold, int rows, int max_dis) {
  const int f = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int total = rows * max_dis;
  bool set = false;
  if (idx < total) {
    // RoadEstimationKernels.cu:56-58: (float)p > (*maximum) * threshold
    const float p = (float)vdisp[(size_t)f * total + idx];
    set = p > __fmul_rn((float)maximum[f], threshold);
    binary[(size_t)f * total + idx] = set ? 255 : 0;
  }
  const unsigned ballot = __ballot_sync(0xffffffffu, set);
  if (ballot) {
    int base = 0;
    const int lane = threadIdx.x & 31;
    if (lane == 0) base = atomicAdd(n_points + f, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (set) points[(size_t)f * total + base + __popc(ballot & ((1u << lane) - 1))] = make_int2(idx / max_dis, idx % max_dis);
  }
}

__global__ void __launch_bounds__(256)
hough_kernel(const int2 *__restrict__ points, const int *__restrict__ n_points, const float *__restrict__ tab_sin,
             const float *__restrict__ tab_cos, int *__restrict__ accum, int numangle, int numrho, int total) {
  extern __shared__ int row_acc[];  // [numrho + 2]
  const int n = blockIdx.x, f = blockIdx.y;
  for (int i = threadIdx.x; i < numrho + 2; i += blockDim.x) row_acc[i] = 0;
  __syncthreads();
  const float s = tab_sin[n], c = tab_cos[n];
  const int np = n_points[f];
  const int2 *pts = points + (size_t)f * total;
  const int half = (numrho - 1) / 2;
  for (int k = threadIdx.x; k < np; k += blockDim.x) {
    const int2 pt = pts[k];  // (i = row, j = column)
    // cvRound(j * tabCos[n] + i * tabSin[n]): two float products, one float sum, round half to even
    const float v = __fadd_rn(__fmul_rn((float)pt.y, c), __fmul_rn((float)pt.x, s));
    const int r = __float2int_rn(v) + half;
    atomicAdd(&row_acc[r + 1], 1);
  }
  __syncthreads();
  int *dst = accum + ((size_t)f * (numangle + 2) + (n + 1)) * (numrho + 2);
  for (int i = threadIdx.x; i < numrho + 2; i += blockDim.x) dst[i] = row_acc[i];
}

__global__ void __launch_bounds__(256)
maxima_kernel(const int *__restrict__ accum, int2 *__restrict__ cand, int *__restrict__ n_cand, int numangle,
              int numrho, int threshold, int cap) {
  const int f = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= numangle * numrho) return;
  const int n = idx / numrho, r = idx - n * numrho;
  const int W = numrho + 2;
  const int *a = accum + (size_t)f * (numangle + 2) * W;
  const int base = (n + 1) * W + r + 1;
  const int v = a[base];
  // findLocalMaximums: > threshold, > left, >= right, > previous angle, >= next angle
  if (v > threshold && v > a[base - 1] && v >= a[base + 1] && v > a[base - W] && v >= a[base + W]) {
    const int k = atomicAdd(n_cand + f, 1);
    if (k < cap) cand[(size_t)f * cap + k] = make_int2(base, v);
  }
}

// The cell the host walk of road_run accepts, as a 64-bit key (votes << 32 | ~cell): the walk goes through the local
// maxima above the threshold by votes descending, then accumulator index ascending (the index grows with the cell),
// and stops at the first in-range pitch -- the largest key among the cells that pass all three tests.  Integer
// maxima do not depend on the order of the atomics: the same key on every run.  sel[f] == 0: no line.
__global__ void __launch_bounds__(256)
select_kernel(const int *__restrict__ accum, const isx_road_estimate *__restrict__ cells,
              unsigned long long *__restrict__ sel, int numangle, int numrho, int threshold) {
  const int f = blockIdx.y;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long key = 0;
  if (idx < numangle * numrho) {
    const int n = idx / numrho, r = idx - n * numrho;
    const int W = numrho + 2;
    const int *a = accum + (size_t)f * (numangle + 2) * W;
    const int base = (n + 1) * W + r + 1;
    const int v = a[base];
    if (v > threshold && v > a[base - 1] && v >= a[base + 1] && v > a[base - W] && v >= a[base + W] && cells[idx].ok)
      key = ((unsigned long long)(unsigned)v << 32) | (unsigned)~(unsigned)idx;
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
    key = other > key ? other : key;
  }
  if ((threadIdx.x & 31) == 0 && key) atomicMax(sel + f, key);
}

// One thread walks the frames in order: the estimate of every frame (zeros when no line was accepted, like road_run)
// and the road it is computed with -- its own estimate, else the last accepted one (RoadEstimation.cu:123-133 only
// overwrites the getters on success), else the seed.  *state = the cell behind the last accepted estimate, -1 = seed.
// carry == 0: no frame inherits from another (the frame pool's per-frame rule): its own estimate, else the seed.
__global__ void resolve_kernel(const unsigned long long *__restrict__ sel, const isx_road_estimate *__restrict__ cells,
                               int *__restrict__ state, int reset, int carry, isx_road seed, int n,
                               isx_road_estimate *__restrict__ estimates, isx_road *__restrict__ roads_out,
                               isx_road *__restrict__ roads) {
  if (threadIdx.x != 0) return;
  int cur = reset ? -1 : *state;
  for (int f = 0; f < n; f++) {
    if (!carry) cur = -1;
    const unsigned long long key = sel[f];
    isx_road_estimate e = {0, 0, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (key) {
      cur = (int)~(unsigned)(key & 0xffffffffu);
      e = cells[cur];
    }
    isx_road r = seed;
    if (cur >= 0) {
      const isx_road_estimate &k = cells[cur];
      r = isx_road{k.horizon_point, k.pitch, k.camera_height, k.slope};   // apps/run_cityscapes.cu:396-407
    }
    if (estimates) estimates[f] = e;
    if (roads_out) roads_out[f] = r;
    roads[f] = r;
  }
  *state = cur;
}

// [n][3][H] ground tables + [n] horizon rows: mapped pinned staging -> a slot of the road ring (under a MB per 64-frame
// chunk of 1024 rows).  The loads cross the host link as reads of the SMs, beside whatever the copy engine is doing.
__global__ void __launch_bounds__(256)
pull_tables_kernel(const float *__restrict__ src_ground, float *__restrict__ dst_ground, size_t n_ground,
                   const int *__restrict__ src_vhor, int *__restrict__ dst_vhor, int n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_ground; i += stride) dst_ground[i] = src_ground[i];
  if (blockIdx.x == 0)
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst_vhor[i] = src_vhor[i];
}

}  // namespace

// Everything one isx_road_initialize acquires, and the state of the device selection since then.
struct InitializedRoad {
  explicit InitializedRoad(int device) : res(device) {}
  cudaStream_t stream = nullptr;
  float *d_disparity = nullptr;  // staging for host images
  int *d_vdisp = nullptr, *d_counters = nullptr;  // counters: [3][max_batch] maximum | n_points | n_cand
  uint8_t *d_binary = nullptr;
  int2 *d_points = nullptr, *d_cand = nullptr;
  int *d_accum = nullptr;
  float *d_tab = nullptr;  // sin | cos
  int *h_counters = nullptr;
  int2 *h_cand = nullptr;
  // device selection (isx_compute_batch_device_road): the estimate of every Hough cell [numangle][numrho], uploaded on
  // first use; the selected key per frame; the keep-last state (cell of the last accepted estimate, -1 = seed)
  isx_road_estimate *d_cells = nullptr;
  bool cells_ready = false;
  unsigned long long *d_sel = nullptr;   // [max_batch]
  int *d_state = nullptr;
  bool has_seed = false;
  isx_road seed{0, 0.f, 0.f, 0.f};
  cudaEvent_t ev_in = nullptr, ev_done = nullptr;   // hand-off from / back to the stixel handle's stream
  CudaResources res;   // owns every stream, event and allocation above
};

}  // namespace isx

struct isx_road_estimator {
  int device = 0;
  float cy = 0, baseline = 0, focal = 0, threshold = 0.2f;
  int rows = 0, cols = 0, max_dis = 0, max_batch = 1;
  int numangle = 0, numrho = 0;
  float theta_step = 0;
  float min_pitch = 0, max_pitch = 0;
  int last_n = 0;
  std::unique_ptr<isx::InitializedRoad> init;   // null: not initialised
  std::string last_error;
};

namespace {
std::string g_road_error;
int road_fail(isx_road_estimator *h, int code, const std::string &msg) {
  g_road_error = msg;
  if (h) h->last_error = msg;
  return code;
}
#define ROAD_TRY(h, expr)                                                                        \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return road_fail(h, ISX_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));    \
  } while (0)

// RoadEstimation::ComputeCameraProperties (RoadEstimation.cu:172-193), same float expressions and libm calls.
void camera_properties(const isx_road_estimator *h, float rho, float theta, float &horizon, float &pitch,
                       float &camera_height, float &slope) {
  horizon = rho / sinf(theta);
  pitch = -atanf((h->cy - horizon) / (h->focal));
  const float last_row = (float)(h->rows - 1);
  const float vdisp_down = (rho - last_row * sinf(theta)) / cosf(theta);
  slope = (0 - vdisp_down) / (horizon - last_row);
  camera_height = h->baseline * cosf(pitch) / slope;
}

// RoadEstimation::ComputeHough for the Hough cell (angle nidx, rho bin r): the line cv::HoughLines reports for it
// (RoadEstimation.cu:155-157), its camera properties, and whether the pitch lies inside +-50 degrees (:163).
void cell_estimate(const isx_road_estimator *h, int nidx, int r, isx_road_estimate &e) {
  const float line_rho = (r - (h->numrho - 1) * 0.5f) * 1.0f;
  const float theta = 0.0f + nidx * h->theta_step;
  const float rho = std::fabs(line_rho);  // RoadEstimation.cu:157
  float horizon, pitch, height, slope;
  camera_properties(h, rho, theta, horizon, pitch, height, slope);
  e = isx_road_estimate{0, 0, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (pitch >= h->min_pitch && pitch <= h->max_pitch) {  // :163
    e.ok = 1;
    e.horizon_point = (int)ceil(horizon);  // :127
    e.pitch = pitch; e.camera_height = height; e.slope = slope; e.rho = rho; e.theta = theta;
  }
}

int road_run(isx_road_estimator *h, int n, const float *d_disparity, isx_road_estimate *out) {
  using namespace isx;
  isx::InitializedRoad &I = *h->init;
  const int rows = h->rows, cols = h->cols, D = h->max_dis, total = rows * D;
  const int B = h->max_batch;
  cudaStream_t s = I.stream;
  ROAD_TRY(h, cudaMemsetAsync(I.d_counters, 0, sizeof(int) * 3 * B, s));
  vdisp_kernel<<<dim3(rows, n), 256, D * sizeof(int), s>>>(d_disparity, I.d_vdisp, I.d_counters, rows, cols, D);
  binarize_kernel<<<dim3((total + 255) / 256, n), 256, 0, s>>>(I.d_vdisp, I.d_counters, I.d_binary, I.d_points,
                                                               I.d_counters + B, h->threshold, rows, D);
  hough_kernel<<<dim3(h->numangle, n), 256, (h->numrho + 2) * sizeof(int), s>>>(
      I.d_points, I.d_counters + B, I.d_tab, I.d_tab + h->numangle, I.d_accum, h->numangle, h->numrho, total);
  maxima_kernel<<<dim3((h->numangle * h->numrho + 255) / 256, n), 256, 0, s>>>(
      I.d_accum, I.d_cand, I.d_counters + 2 * B, h->numangle, h->numrho, kHoughThreshold, kMaxCandidates);
  g_launch_count += 4;
  ROAD_TRY(h, cudaGetLastError());
  ROAD_TRY(h, cudaMemcpyAsync(I.h_counters, I.d_counters, sizeof(int) * 3 * B, cudaMemcpyDeviceToHost, s));
  ROAD_TRY(h, cudaStreamSynchronize(s));
  // only the used part of every frame's candidate array travels
  int most = 0;
  for (int f = 0; f < n; f++) most = std::max(most, std::min(I.h_counters[2 * B + f], kMaxCandidates));
  if (most > 0) {
    ROAD_TRY(h, cudaMemcpy2DAsync(I.h_cand, sizeof(int2) * kMaxCandidates, I.d_cand, sizeof(int2) * kMaxCandidates,
                                  sizeof(int2) * most, n, cudaMemcpyDeviceToHost, s));
    ROAD_TRY(h, cudaStreamSynchronize(s));
  }
  h->last_n = n;
  const int W = h->numrho + 2;
  for (int f = 0; f < n; f++) {
    isx_road_estimate &e = out[f];
    e = isx_road_estimate{0, 0, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int nc = I.h_counters[2 * B + f];
    if (nc > kMaxCandidates) return road_fail(h, ISX_ERR_CAPACITY, "more Hough line candidates than the buffer holds");
    int2 *c = I.h_cand + (size_t)f * kMaxCandidates;
    // hough_cmp_gt: votes descending, accumulator index ascending
    std::sort(c, c + nc, [](const int2 &a, const int2 &b) { return a.y > b.y || (a.y == b.y && a.x < b.x); });
    for (int k = 0; k < nc; k++) {
      const int nidx = c[k].x / W - 1;
      const int r = c[k].x - (nidx + 1) * W - 1;
      cell_estimate(h, nidx, r, e);
      if (e.ok) break;
    }
  }
  return ISX_OK;
}
}  // namespace

extern "C" {

int isx_road_create(isx_road_handle *out, int device) {
  if (!out) return road_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null out pointer");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return road_fail(nullptr, ISX_ERR_CUDA, std::string("no CUDA device: road estimation has no CPU fallback (") +
                                                cudaGetErrorString(e) + ")");
  if (device < 0 || device >= count) return road_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "no such device");
  *out = new isx_road_estimator();
  (*out)->device = device;
  return ISX_OK;
}

void isx_road_destroy(isx_road_handle h) { delete h; }

const char *isx_road_last_error(isx_road_handle h) { return h ? h->last_error.c_str() : g_road_error.c_str(); }
int isx_road_is_initialized(isx_road_handle h) { return h && h->init; }

int isx_road_initialize(isx_road_handle h, float camera_center_y, float baseline, float focal, int rows, int cols,
                        int max_dis, float road_vdisparity_threshold, int max_batch) {
  if (!h) return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  if (rows < 1 || cols < 1 || max_dis < 1 || max_batch < 1)
    return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "rows, cols, max_dis and max_batch must be positive");
  h->init.reset();
  ROAD_TRY(h, cudaSetDevice(h->device));
  h->cy = camera_center_y; h->baseline = baseline; h->focal = focal; h->threshold = road_vdisparity_threshold;
  h->rows = rows; h->cols = cols; h->max_dis = max_dis; h->max_batch = max_batch;
  // RoadEstimation.cu:47-58
  h->max_pitch = 50 * (float)M_PI / 180.0f;
  h->min_pitch = -50 * (float)M_PI / 180.0f;
  // cv::HoughLines(img, lines, rho = 1.0, theta = CV_PI/180, ...): the image is [rows][max_dis]
  const double theta_d = M_PI / 180;
  h->theta_step = (float)theta_d;
  int numangle = (int)std::floor((M_PI - 0.0) / (double)h->theta_step) + 1;  // computeNumangle
  if (numangle > 1 && std::fabs(M_PI - (numangle - 1) * (double)h->theta_step) < (double)h->theta_step / 2) --numangle;
  h->numangle = numangle;
  const int max_rho = max_dis + rows;
  h->numrho = (int)std::lrint(((2 * max_rho) + 1) / 1.0);
  std::vector<float> tab(2 * numangle);
  {
    // createTrigTable: float angle accumulation, double sin/cos, irho = 1
    float ang = 0.0f;
    const float irho = 1.0f;
    for (int n = 0; n < numangle; ang += h->theta_step, n++) {
      tab[n] = (float)(sin((double)ang) * irho);
      tab[numangle + n] = (float)(cos((double)ang) * irho);
    }
  }
  const size_t B = max_batch, total = (size_t)rows * max_dis;
  // built here and kept only on success: an early return releases what was acquired
  auto init = std::make_unique<isx::InitializedRoad>(h->device);
  isx::InitializedRoad &I = *init;
  ROAD_TRY(h, I.res.stream(&I.stream));
  ROAD_TRY(h, I.res.device(&I.d_disparity, sizeof(float) * rows * cols));
  ROAD_TRY(h, I.res.device(&I.d_vdisp, sizeof(int) * B * total));
  ROAD_TRY(h, I.res.device(&I.d_counters, sizeof(int) * 3 * B));
  ROAD_TRY(h, I.res.device(&I.d_binary, B * total));
  ROAD_TRY(h, I.res.device(&I.d_points, sizeof(int2) * B * total));
  ROAD_TRY(h, I.res.device(&I.d_cand, sizeof(int2) * B * isx::kMaxCandidates));
  const size_t acc = (size_t)(numangle + 2) * (h->numrho + 2);
  ROAD_TRY(h, I.res.device(&I.d_accum, sizeof(int) * B * acc));
  ROAD_TRY(h, cudaMemset(I.d_accum, 0, sizeof(int) * B * acc));  // border rows n = 0 and numangle + 1 stay zero
  ROAD_TRY(h, I.res.device(&I.d_tab, sizeof(float) * 2 * numangle));
  ROAD_TRY(h, cudaMemcpy(I.d_tab, tab.data(), sizeof(float) * 2 * numangle, cudaMemcpyHostToDevice));
  ROAD_TRY(h, I.res.host(&I.h_counters, sizeof(int) * 3 * B));
  ROAD_TRY(h, I.res.host(&I.h_cand, sizeof(int2) * B * isx::kMaxCandidates));
  ROAD_TRY(h, I.res.device(&I.d_cells, sizeof(isx_road_estimate) * numangle * h->numrho));
  ROAD_TRY(h, I.res.device(&I.d_sel, sizeof(unsigned long long) * B));
  ROAD_TRY(h, I.res.device(&I.d_state, sizeof(int)));
  ROAD_TRY(h, I.res.event(&I.ev_in));
  ROAD_TRY(h, I.res.event(&I.ev_done));
  if ((h->numrho + 2) * sizeof(int) > 48 * 1024)
    ROAD_TRY(h, cudaFuncSetAttribute(isx::hough_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)((h->numrho + 2) * sizeof(int))));
  h->init = std::move(init);
  return ISX_OK;
}

int isx_road_finish(isx_road_handle h) {
  if (!h) return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  h->init.reset();
  return ISX_OK;
}

static int road_ready(isx_road_handle h) {
  if (!h) return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  if (!h->init) return road_fail(h, ISX_ERR_NOT_INITIALIZED, "Initialize() has not been called");
  cudaError_t e = cudaSetDevice(h->device);
  if (e != cudaSuccess) return road_fail(h, ISX_ERR_CUDA, cudaGetErrorString(e));
  return ISX_OK;
}

int isx_road_compute_host(isx_road_handle h, const float *disparity, size_t n_pixels, isx_road_estimate *out) {
  if (int rc = road_ready(h)) return rc;
  if (!disparity || !out || n_pixels != (size_t)h->rows * h->cols)
    return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "disparity image must hold rows * cols pixels");
  ROAD_TRY(h, cudaMemcpyAsync(h->init->d_disparity, disparity, sizeof(float) * n_pixels, cudaMemcpyHostToDevice,
                              h->init->stream));
  return road_run(h, 1, h->init->d_disparity, out);
}

int isx_road_compute_device(isx_road_handle h, const float *d_disparity, isx_road_estimate *out) {
  if (int rc = road_ready(h)) return rc;
  if (!d_disparity || !out) return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  return road_run(h, 1, d_disparity, out);
}

int isx_road_compute_batch_device(isx_road_handle h, int n, const float *d_disparity, isx_road_estimate *out) {
  if (int rc = road_ready(h)) return rc;
  if (!d_disparity || !out) return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  if (n < 1 || n > h->max_batch) return road_fail(h, ISX_ERR_CAPACITY, "batch size exceeds isx_road_initialize(max_batch)");
  return road_run(h, n, d_disparity, out);
}

size_t isx_road_tensor_bytes(isx_road_handle h, int tensor) {
  if (!h || !h->init) return 0;
  const size_t total = (size_t)h->rows * h->max_dis;
  switch (tensor) {
    case 0: return total * sizeof(int);
    case 1: return total;
    case 2: return (size_t)(h->numangle + 2) * (h->numrho + 2) * sizeof(int);
    default: return 0;
  }
}

int isx_road_read_tensor(isx_road_handle h, int tensor, int frame, void *host, size_t bytes) {
  if (int rc = road_ready(h)) return rc;
  const size_t need = isx_road_tensor_bytes(h, tensor);
  if (need == 0 || !host || bytes < need || frame < 0 || frame >= h->last_n)
    return road_fail(h, ISX_ERR_INVALID_ARGUMENT, "bad tensor id, frame or buffer");
  const char *src = tensor == 0 ? (const char *)h->init->d_vdisp
                    : tensor == 1 ? (const char *)h->init->d_binary : (const char *)h->init->d_accum;
  // isx_compute_batch_device_road leaves its work queued on the road stream, which does not synchronise with the
  // legacy stream of cudaMemcpy
  ROAD_TRY(h, cudaStreamSynchronize(h->init->stream));
  ROAD_TRY(h, cudaMemcpy(host, src + need * frame, need, cudaMemcpyDeviceToHost));
  return ISX_OK;
}

}  // extern "C"

namespace isx {

int road_check_batch(isx_road_handle h, int device, int rows, int cols, int max_dis, int n, bool has_fallback,
                     std::string &msg) {
  if (!h || !h->init) return msg = "the road handle is not initialised", ISX_ERR_INVALID_ARGUMENT;
  if (h->device != device) return msg = "the road handle computes on another device", ISX_ERR_INVALID_ARGUMENT;
  if (h->rows != rows || h->cols != cols || h->max_dis != max_dis)
    return msg = "the road handle was initialised for other rows, cols or max_dis", ISX_ERR_INVALID_ARGUMENT;
  if (n > h->max_batch) return msg = "batch size exceeds isx_road_initialize(max_batch)", ISX_ERR_CAPACITY;
  if (!has_fallback && !h->init->has_seed)
    return msg = "no fallback road: the road handle has no state to continue from", ISX_ERR_INVALID_ARGUMENT;
  return ISX_OK;
}

// The road step of isx_compute_batch_device_road, in stream order: the road stream waits for `caller`, runs the
// Hough kernels and the device selection of n frames, and `caller` waits for it.  d_roads [n] receives the road each
// frame is computed with.  Checked by road_check_batch before.
int road_enqueue_batch(isx_road_handle h, cudaStream_t caller, int n, const float *d_disparity,
                       const isx_road *fallback, isx_road_estimate *d_estimates, isx_road *d_roads_out,
                       isx_road *d_roads, std::string &msg, bool carry) {
  auto cuda = [&](cudaError_t e, const char *what) -> int {
    if (e == cudaSuccess) return ISX_OK;
    msg = std::string(what) + ": " + cudaGetErrorString(e);
    return road_fail(h, ISX_ERR_CUDA, msg);
  };
#define ROAD_ENQ(expr) \
  if (int _rc = cuda((expr), #expr)) return _rc
  isx::InitializedRoad &I = *h->init;
  if (!I.cells_ready) {
    // once per handle: the estimate of every Hough cell, by the code of the host walk (road_run)
    std::vector<isx_road_estimate> cells((size_t)h->numangle * h->numrho);
    for (int a = 0; a < h->numangle; a++)
      for (int r = 0; r < h->numrho; r++) cell_estimate(h, a, r, cells[(size_t)a * h->numrho + r]);
    // pageable source: returns once the driver has staged it, without waiting for other streams
    ROAD_ENQ(cudaMemcpyAsync(I.d_cells, cells.data(), sizeof(isx_road_estimate) * cells.size(),
                             cudaMemcpyHostToDevice, I.stream));
    I.cells_ready = true;
  }
  if (fallback) {
    I.seed = *fallback;
    I.has_seed = true;
  }
  const int rows = h->rows, cols = h->cols, D = h->max_dis, total = rows * D;
  const int B = h->max_batch;
  cudaStream_t s = I.stream;
  ROAD_ENQ(cudaEventRecord(I.ev_in, caller));
  ROAD_ENQ(cudaStreamWaitEvent(s, I.ev_in, 0));
  ROAD_ENQ(cudaMemsetAsync(I.d_counters, 0, sizeof(int) * 3 * B, s));
  ROAD_ENQ(cudaMemsetAsync(I.d_sel, 0, sizeof(unsigned long long) * n, s));
  vdisp_kernel<<<dim3(rows, n), 256, D * sizeof(int), s>>>(d_disparity, I.d_vdisp, I.d_counters, rows, cols, D);
  binarize_kernel<<<dim3((total + 255) / 256, n), 256, 0, s>>>(I.d_vdisp, I.d_counters, I.d_binary, I.d_points,
                                                               I.d_counters + B, h->threshold, rows, D);
  hough_kernel<<<dim3(h->numangle, n), 256, (h->numrho + 2) * sizeof(int), s>>>(
      I.d_points, I.d_counters + B, I.d_tab, I.d_tab + h->numangle, I.d_accum, h->numangle, h->numrho, total);
  select_kernel<<<dim3((h->numangle * h->numrho + 255) / 256, n), 256, 0, s>>>(I.d_accum, I.d_cells, I.d_sel,
                                                                               h->numangle, h->numrho, kHoughThreshold);
  resolve_kernel<<<1, 32, 0, s>>>(I.d_sel, I.d_cells, I.d_state, fallback ? 1 : 0, carry ? 1 : 0, I.seed, n,
                                  d_estimates, d_roads_out, d_roads);
  g_launch_count += 5;
  ROAD_ENQ(cudaGetLastError());
  ROAD_ENQ(cudaEventRecord(I.ev_done, s));
  ROAD_ENQ(cudaStreamWaitEvent(caller, I.ev_done, 0));
#undef ROAD_ENQ
  h->last_n = n;
  return ISX_OK;
}

void launch_pull_road_tables(const float *src_ground, float *dst_ground, size_t ground_floats, const int *src_vhor,
                             int *dst_vhor, int n, cudaStream_t s) {
  const int blocks = (int)std::min<size_t>((ground_floats + 255) / 256, 512);
  pull_tables_kernel<<<blocks < 1 ? 1 : blocks, 256, 0, s>>>(src_ground, dst_ground, ground_floats, src_vhor, dst_vhor,
                                                            n);
  g_launch_count++;
}

}  // namespace isx
