// Object tracking on the device (isx_tracker_*): persistent ids for the objects isx_export_objects_device writes.
// The definition is in include/instance_stixels_b200.h; include/InstanceStixels/ObjectTracker.hpp states it on the
// host (HostObjectTracker), and this file computes the same bytes.
//
//   track_classes_kernel : one CTA per instance class walks the frames of the call in order.  The class's track table
//                          lives in shared memory.  The greedy association runs as rounds of locally dominant pairs: every
//                          free track picks its best free candidate object, every object picked that way picks its
//                          best free candidate track, and mutual picks are accepted.  Under a strict total order a pair
//                          that comes first among all pairs of its track and of its object belongs to the greedy
//                          matching, so the rounds give exactly the sequential walk.  Tracks born in the call get
//                          provisional ids (kProvisional | frame | class | rank), whose order within a class is the
//                          order of the global ids.
//   track_ids_kernel     : one CTA scans the births over (frame, class), replaces the provisional ids of the outputs and
//                          of the tables by global ids, advances the id counter and writes the frame flags.
#include <algorithm>
#include <cmath>
#include <memory>
#include <string>
#include <vector>

#include "cuda_resources.h"
#include "kernels.h"

namespace isx {
namespace {

constexpr int kTrackThreads = 512;
constexpr int kClassCount = ISX_INSTANCE_CLASSES;
constexpr long long kProvisional = 1LL << 62;   // above every global id; | frame << 32 | class << 28 | rank
constexpr long long kFree = -2, kPicked = -3;   // object states during the association (in d_track_ids)
static_assert(ISX_TRACK_MAX_TRACKS <= 2 * kTrackThreads, "the table compaction handles two tracks per thread");
static_assert(ISX_TRACK_MAX_FRAMES <= (1 << 30), "frame index of the provisional ids");

// Device state of a tracker: per class a table of max_tracks tracks (structure of arrays), the live counts and the
// id counter.
struct TrackState {
  long long *id;    // [8][T]
  int4 *box;        // [8][T] x0, y0, x1, y1
  float2 *disp;     // [8][T] disparity min, max
  int2 *hm;         // [8][T] hits, misses
  int *count;       // [8]
  long long *next_id;
};

struct TrackArgs {
  const isx_object *objects;
  const int *frame_offsets, *class_offsets;
  int capacity, n;
  long long *ids;           // [capacity]
  int *hits;                // [capacity] or null
  int *flags;               // [n] or null
  int *births, *left;       // [n][8] scratch: new tracks / objects left over per (frame, class)
  TrackState st;
  int T;                    // max_tracks
  int iou_min_permille, max_age;
  float margin;
};

// IEEE add and compare with subnormals kept, whatever -ftz says: the host computes the gate that way.
__device__ __forceinline__ float add_keep_subnormals(float a, float b) {
  float r;
  asm("add.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ bool greater_keep_subnormals(float a, float b) {
  unsigned r;
  asm("{ .reg .pred p; setp.gt.f32 p, %1, %2; selp.u32 %0, 1, 0, p; }" : "=r"(r) : "f"(a), "f"(b));
  return r != 0;
}

__device__ __forceinline__ long long box_area(int4 b) { return ((long long)b.z - b.x + 1) * ((long long)b.w - b.y + 1); }

// Whether (track box a, disparity da) and (object box b, disparity db) are a candidate pair; I and U of the boxes.
__device__ __forceinline__ bool candidate(int4 a, float2 da, int4 b, float2 db, const TrackArgs &p, long long &I,
                                          long long &U) {
  const long long w = (long long)min(a.z, b.z) - max(a.x, b.x) + 1;
  const long long h = (long long)min(a.w, b.w) - max(a.y, b.y) + 1;
  if (w <= 0 || h <= 0) return false;
  I = w * h;
  U = box_area(a) + box_area(b) - I;
  if (1000 * I < (long long)p.iou_min_permille * U) return false;
  if (isnan(da.x) || isnan(da.y) || isnan(db.x) || isnan(db.y)) return true;
  return !greater_keep_subnormals(db.x, add_keep_subnormals(da.y, p.margin)) &&
         !greater_keep_subnormals(da.x, add_keep_subnormals(db.y, p.margin));
}

__device__ __forceinline__ int4 object_box(const isx_object &o) { return make_int4(o.x0, o.y0, o.x1, o.y1); }

// Exclusive prefix of `flag` over the threads of the CTA and the CTA total.  Every thread must call it.
__device__ __forceinline__ int block_scan(int flag, int *s_warp, int &total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned b = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_warp[warp] = __popc(b);
  __syncthreads();
  int before = 0;
  total = 0;
  for (int w = 0; w < kTrackThreads / 32; w++) {
    const int c = s_warp[w];
    before += w < warp ? c : 0;
    total += c;
  }
  __syncthreads();
  return before + __popc(b & ((1u << lane) - 1));
}

__global__ void __launch_bounds__(kTrackThreads)
track_classes_kernel(TrackArgs p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int T = p.T;
  int4 *s_box = reinterpret_cast<int4 *>(smem);
  long long *s_id = reinterpret_cast<long long *>(s_box + T);
  float2 *s_disp = reinterpret_cast<float2 *>(s_id + T);
  int2 *s_hm = reinterpret_cast<int2 *>(s_disp + T);
  int *s_best = reinterpret_cast<int *>(s_hm + T);     // best free object of a free track in this round, -1: none
  int *s_match = s_best + T;                           // matched object of a track, -1: none
  __shared__ int s_warp[kTrackThreads / 32];
  __shared__ int s_any;
  const int k = blockIdx.x, tid = threadIdx.x;
  const size_t tab = (size_t)k * T;
  int live = p.st.count[k];
  for (int t = tid; t < live; t += kTrackThreads) {
    s_id[t] = p.st.id[tab + t];
    s_box[t] = p.st.box[tab + t];
    s_disp[t] = p.st.disp[tab + t];
    s_hm[t] = p.st.hm[tab + t];
  }
  __syncthreads();
  for (int f = 0; f < p.n; f++) {
    const bool written = p.frame_offsets[f + 1] <= p.capacity;
    const int lo = written ? p.class_offsets[f * kClassCount + k] : 0;
    const int m = written ? p.class_offsets[f * kClassCount + k + 1] - lo : 0;
    const isx_object *obj = p.objects + lo;
    long long *ids = p.ids + lo;
    for (int o = tid; o < m; o += kTrackThreads) ids[o] = kFree;
    for (int t = tid; t < live; t += kTrackThreads) s_match[t] = -1;
    __syncthreads();
    // ---- greedy association in rounds of locally dominant pairs ----
    while (m > 0 && live > 0) {
      if (tid == 0) s_any = 0;
      __syncthreads();
      for (int t = tid; t < live; t += kTrackThreads) {
        int best = -1;
        if (s_match[t] < 0) {
          const int4 tb = s_box[t];
          const float2 td = s_disp[t];
          long long bI = 0, bU = 1;
          for (int o = 0; o < m; o++) {
            if (ids[o] >= 0) continue;   // taken
            long long I, U;
            const isx_object &ob = obj[o];
            if (!candidate(tb, td, object_box(ob), make_float2(ob.disparity_min, ob.disparity_max), p, I, U)) continue;
            if (best < 0 || I * bU > bI * U) best = o, bI = I, bU = U;   // ties: the lower label stays
          }
          if (best >= 0) {
            ids[best] = kPicked;
            s_any = 1;
          }
        }
        s_best[t] = best;
      }
      __syncthreads();
      if (!s_any) break;
      for (int o = tid; o < m; o += kTrackThreads) {
        if (ids[o] != kPicked) continue;
        const isx_object &ob = obj[o];
        const int4 obx = object_box(ob);
        const float2 od = make_float2(ob.disparity_min, ob.disparity_max);
        int best = -1;
        long long bI = 0, bU = 1;
        for (int t = 0; t < live; t++) {
          if (s_match[t] >= 0) continue;
          long long I, U;
          if (!candidate(s_box[t], s_disp[t], obx, od, p, I, U)) continue;
          const long long l = I * bU, r = bI * U;
          if (best < 0 || l > r || (l == r && s_id[t] < s_id[best])) best = t, bI = I, bU = U;
        }
        ids[o] = (best >= 0 && s_best[best] == o) ? best : kFree;
      }
      __syncthreads();
      for (int t = tid; t < live; t += kTrackThreads)
        if (s_match[t] < 0 && s_best[t] >= 0 && ids[s_best[t]] == t) s_match[t] = s_best[t];
      __syncthreads();
    }
    // ---- matched tracks take their object, the others age; removal keeps the order (ids ascending) ----
    long long e_id[2];
    int4 e_box[2];
    float2 e_disp[2];
    int2 e_hm[2];
    int keep[2], pos[2], kept[2];
#pragma unroll
    for (int i = 0; i < 2; i++) {
      const int t = tid + i * kTrackThreads;
      keep[i] = 0;
      if (t < live) {
        e_id[i] = s_id[t];
        e_box[i] = s_box[t];
        e_disp[i] = s_disp[t];
        e_hm[i] = s_hm[t];
        const int o = s_match[t];
        if (o >= 0) {
          const isx_object &ob = obj[o];
          e_box[i] = object_box(ob);
          e_disp[i] = make_float2(ob.disparity_min, ob.disparity_max);
          e_hm[i] = make_int2(e_hm[i].x + 1, 0);
          ids[o] = e_id[i];
          if (p.hits) p.hits[lo + o] = e_hm[i].x;
        } else {
          e_hm[i].y += 1;
        }
        keep[i] = e_hm[i].y <= p.max_age;
      }
    }
    pos[0] = block_scan(keep[0], s_warp, kept[0]);
    pos[1] = kept[0] + block_scan(keep[1], s_warp, kept[1]);
#pragma unroll
    for (int i = 0; i < 2; i++)
      if (keep[i]) {
        s_id[pos[i]] = e_id[i];
        s_box[pos[i]] = e_box[i];
        s_disp[pos[i]] = e_disp[i];
        s_hm[pos[i]] = e_hm[i];
      }
    live = kept[0] + kept[1];
    __syncthreads();
    // ---- unmatched objects become tracks in label order while the class has room ----
    int born = 0, unmatched = 0;
    for (int o0 = 0; o0 < m; o0 += kTrackThreads) {
      const int o = o0 + tid;
      const int u = o < m && ids[o] == kFree;
      int chunk;
      const int rank = unmatched + block_scan(u, s_warp, chunk);
      if (u) {
        const int slot = live + rank;
        if (slot < T) {
          const long long id = kProvisional | ((long long)f << 32) | ((long long)k << 28) | rank;
          const isx_object &ob = obj[o];
          s_id[slot] = id;
          s_box[slot] = object_box(ob);
          s_disp[slot] = make_float2(ob.disparity_min, ob.disparity_max);
          s_hm[slot] = make_int2(1, 0);
          ids[o] = id;
          if (p.hits) p.hits[lo + o] = 1;
        } else {
          ids[o] = -1;
          if (p.hits) p.hits[lo + o] = 0;
        }
      }
      unmatched += chunk;
    }
    born = min(unmatched, T - live);
    if (tid == 0) {
      p.births[f * kClassCount + k] = born;
      p.left[f * kClassCount + k] = unmatched > born;
    }
    live += born;
    __syncthreads();
  }
  for (int t = tid; t < live; t += kTrackThreads) {
    p.st.id[tab + t] = s_id[t];
    p.st.box[tab + t] = s_box[t];
    p.st.disp[tab + t] = s_disp[t];
    p.st.hm[tab + t] = s_hm[t];
  }
  if (tid == 0) p.st.count[k] = live;
}

constexpr int kIdThreads = 1024;

__device__ __forceinline__ long long global_id(long long v, long long next0, const int *base) {
  if (v < kProvisional) return v;
  const long long r = v - kProvisional;
  const int f = (int)(r >> 32), k = (int)((r >> 28) & 15), rank = (int)(r & ((1 << 28) - 1));
  return next0 + base[f * kClassCount + k] + rank;
}

// births [n][8] -> their exclusive prefix (in place), then the global ids.  One CTA.
__global__ void __launch_bounds__(kIdThreads)
track_ids_kernel(TrackArgs p) {
  __shared__ int s_warp[kIdThreads / 32];
  __shared__ int s_end;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long next0 = *p.st.next_id;
  const int cells = p.n * kClassCount;
  if (tid == 0) s_end = 0;
  int carry = 0;
  for (int c0 = 0; c0 < cells; c0 += kIdThreads) {
    const int c = c0 + tid;
    const int v = c < cells ? p.births[c] : 0;
    int x = v;   // inclusive warp scan
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int before = 0, total = 0;
    for (int w = 0; w < kIdThreads / 32; w++) {
      before += w < warp ? s_warp[w] : 0;
      total += s_warp[w];
    }
    __syncthreads();
    if (c < cells) p.births[c] = carry + before + x - v;
    carry += total;
  }
  for (int f = tid; f < p.n; f += kIdThreads) {
    const int end = p.frame_offsets[f + 1];
    const bool written = end <= p.capacity;
    if (written) atomicMax(&s_end, end);
    if (p.flags) {
      int fl = written ? 0 : ISX_TRACK_NOT_WRITTEN;
      for (int k = 0; k < kClassCount; k++) fl |= p.left[f * kClassCount + k] ? ISX_TRACK_UNMATCHED : 0;
      p.flags[f] = fl;
    }
  }
  __syncthreads();   // births hold their prefix; s_end = objects of the written frames
  for (int j = tid; j < s_end; j += kIdThreads) p.ids[j] = global_id(p.ids[j], next0, p.births);
  for (int k = 0; k < kClassCount; k++)
    for (int t = tid; t < p.st.count[k]; t += kIdThreads) {
      long long *id = p.st.id + (size_t)k * p.T + t;
      *id = global_id(*id, next0, p.births);
    }
  if (tid == 0) *p.st.next_id = next0 + carry;
}

size_t track_smem_bytes(int T) { return (size_t)T * (sizeof(int4) + sizeof(long long) + sizeof(float2) + sizeof(int2) + 2 * sizeof(int)); }

}  // namespace

struct TrackerState {
  explicit TrackerState(int device) : res(device) {}
  cudaStream_t stream = nullptr;   // reset and read_state
  cudaEvent_t ev_last = nullptr;   // recorded after every update and reset
  bool recorded = false;
  TrackState st{};
  int *d_births = nullptr, *d_left = nullptr;
  CudaResources res;
};

}  // namespace isx

struct isx_tracker {
  int device = 0;
  isx_track_params params{};
  std::unique_ptr<isx::TrackerState> s;
  std::string last_error;
};

namespace {
std::string g_track_error;
int track_fail(isx_tracker *t, int code, const std::string &msg) {
  g_track_error = msg;
  if (t) t->last_error = msg;
  return code;
}
#define TRACK_TRY(t, expr)                                                                       \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return track_fail(t, ISX_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));   \
  } while (0)

// Whether `p` is device memory of `device` (or managed memory).
bool on_device(const void *p, int device) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == device;
}

// The next update (or reset, read) on `s` waits for the previous update of the tracker.
int after_previous(isx_tracker *t, cudaStream_t s) {
  if (t->s->recorded) TRACK_TRY(t, cudaStreamWaitEvent(s, t->s->ev_last, 0));
  return ISX_OK;
}
int record(isx_tracker *t, cudaStream_t s) {
  TRACK_TRY(t, cudaEventRecord(t->s->ev_last, s));
  t->s->recorded = true;
  return ISX_OK;
}
}  // namespace

extern "C" {

void isx_track_params_init(isx_track_params *p) {
  if (p) *p = isx_track_params{300, 2, 2.0f, 1024};
}

const char *isx_tracker_last_error(isx_tracker_handle t) { return t ? t->last_error.c_str() : g_track_error.c_str(); }

int isx_tracker_create(isx_tracker_handle *out, int device, const isx_track_params *params) {
  if (!out) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null out pointer");
  isx_track_params p;
  isx_track_params_init(&p);
  if (params) p = *params;
  if (p.iou_min_permille < 1 || p.iou_min_permille > 1000)
    return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "iou_min_permille must be in 1..1000");
  if (p.max_age < 0) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "max_age must be >= 0");
  if (std::isnan(p.disparity_margin) || p.disparity_margin < 0)
    return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "disparity_margin must be >= 0 and not NaN");
  if (p.max_tracks < 1) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "max_tracks must be >= 1");
  if (p.max_tracks > ISX_TRACK_MAX_TRACKS)
    return track_fail(nullptr, ISX_ERR_UNSUPPORTED, "max_tracks above ISX_TRACK_MAX_TRACKS (1024)");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return track_fail(nullptr, ISX_ERR_CUDA, std::string("no CUDA device: the tracker has no CPU fallback (") +
                                                 cudaGetErrorString(e) + ")");
  if (device < 0 || device >= count) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "no such device");
  TRACK_TRY(nullptr, cudaSetDevice(device));
  auto s = std::make_unique<isx::TrackerState>(device);
  const size_t T = (size_t)p.max_tracks, C = isx::kClassCount;
  isx::TrackState &st = s->st;
  TRACK_TRY(nullptr, s->res.stream(&s->stream));
  TRACK_TRY(nullptr, s->res.event(&s->ev_last));
  TRACK_TRY(nullptr, s->res.device(&st.id, sizeof(long long) * C * T));
  TRACK_TRY(nullptr, s->res.device(&st.box, sizeof(int4) * C * T));
  TRACK_TRY(nullptr, s->res.device(&st.disp, sizeof(float2) * C * T));
  TRACK_TRY(nullptr, s->res.device(&st.hm, sizeof(int2) * C * T));
  TRACK_TRY(nullptr, s->res.device(&st.count, sizeof(int) * C));
  TRACK_TRY(nullptr, s->res.device(&st.next_id, sizeof(long long)));
  TRACK_TRY(nullptr, s->res.device(&s->d_births, sizeof(int) * C * ISX_TRACK_MAX_FRAMES));
  TRACK_TRY(nullptr, s->res.device(&s->d_left, sizeof(int) * C * ISX_TRACK_MAX_FRAMES));
  TRACK_TRY(nullptr, cudaMemsetAsync(st.count, 0, sizeof(int) * C, s->stream));
  TRACK_TRY(nullptr, cudaMemsetAsync(st.next_id, 0, sizeof(long long), s->stream));
  TRACK_TRY(nullptr, cudaStreamSynchronize(s->stream));
  TRACK_TRY(nullptr, cudaFuncSetAttribute(isx::track_classes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)isx::track_smem_bytes(ISX_TRACK_MAX_TRACKS)));
  isx_tracker *t = new isx_tracker();
  t->device = device;
  t->params = p;
  t->s = std::move(s);
  *out = t;
  return ISX_OK;
}

int isx_tracker_destroy(isx_tracker_handle t) {
  if (!t) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null tracker");
  cudaSetDevice(t->device);
  if (t->s->recorded) cudaEventSynchronize(t->s->ev_last);
  delete t;   // CudaResources synchronises the device and releases the state
  return ISX_OK;
}

int isx_tracker_reset(isx_tracker_handle t) {
  if (!t) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null tracker");
  TRACK_TRY(t, cudaSetDevice(t->device));
  isx::TrackerState &S = *t->s;
  if (int rc = after_previous(t, S.stream)) return rc;
  TRACK_TRY(t, cudaMemsetAsync(S.st.count, 0, sizeof(int) * isx::kClassCount, S.stream));
  TRACK_TRY(t, cudaMemsetAsync(S.st.next_id, 0, sizeof(long long), S.stream));
  return record(t, S.stream);
}

int isx_tracker_update_device(isx_tracker_handle t, uint64_t stream, int n, const isx_device_objects *in,
                              int64_t *d_track_ids, int32_t *d_hits, int32_t *d_frame_flags) {
  if (!t) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null tracker");
  if (n < 1 || n > ISX_TRACK_MAX_FRAMES)
    return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "n must be in 1..ISX_TRACK_MAX_FRAMES (4096)");
  if (!in || !in->objects || !in->frame_offsets || !in->class_offsets || !d_track_ids)
    return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "objects, frame_offsets, class_offsets and track_ids are required");
  if ((uintptr_t)in->objects % 16 || (uintptr_t)in->frame_offsets % 4 || (uintptr_t)in->class_offsets % 4 ||
      (uintptr_t)d_track_ids % 8 || (uintptr_t)d_hits % 4 || (uintptr_t)d_frame_flags % 4)
    return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "misaligned pointer");
  if (in->capacity < 0) return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "capacity must be >= 0");
  TRACK_TRY(t, cudaSetDevice(t->device));
  const void *ptrs[] = {in->objects, in->frame_offsets, in->class_offsets, d_track_ids, d_hits, d_frame_flags};
  for (const void *q : ptrs)
    if (q && !on_device(q, t->device))
      return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "a pointer is not device memory of the tracker's device");
  isx::TrackerState &S = *t->s;
  cudaStream_t s = (cudaStream_t)(uintptr_t)stream;
  if (int rc = after_previous(t, s)) return rc;
  isx::TrackArgs a;
  a.objects = in->objects;
  a.frame_offsets = in->frame_offsets;
  a.class_offsets = in->class_offsets;
  a.capacity = in->capacity;
  a.n = n;
  a.ids = reinterpret_cast<long long *>(d_track_ids);
  a.hits = d_hits;
  a.flags = d_frame_flags;
  a.births = S.d_births;
  a.left = S.d_left;
  a.st = S.st;
  a.T = t->params.max_tracks;
  a.iou_min_permille = t->params.iou_min_permille;
  a.max_age = t->params.max_age;
  a.margin = t->params.disparity_margin;
  isx::track_classes_kernel<<<isx::kClassCount, isx::kTrackThreads, isx::track_smem_bytes(a.T), s>>>(a);
  isx::track_ids_kernel<<<1, isx::kIdThreads, 0, s>>>(a);
  isx::g_launch_count += 2;
  TRACK_TRY(t, cudaGetLastError());
  return record(t, s);
}

int isx_tracker_read_state(isx_tracker_handle t, isx_track *host, int capacity, int *n, int64_t *next_id) {
  if (!t) return track_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null tracker");
  if (capacity < 0 || (capacity > 0 && !host)) return track_fail(t, ISX_ERR_INVALID_ARGUMENT, "bad host buffer");
  TRACK_TRY(t, cudaSetDevice(t->device));
  isx::TrackerState &S = *t->s;
  const size_t C = isx::kClassCount, T = (size_t)t->params.max_tracks;
  std::vector<long long> id(C * T);
  std::vector<int4> box(C * T);
  std::vector<float2> disp(C * T);
  std::vector<int2> hm(C * T);
  int count[isx::kClassCount];
  long long next = 0;
  if (int rc = after_previous(t, S.stream)) return rc;
  TRACK_TRY(t, cudaMemcpyAsync(id.data(), S.st.id, sizeof(long long) * C * T, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaMemcpyAsync(box.data(), S.st.box, sizeof(int4) * C * T, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaMemcpyAsync(disp.data(), S.st.disp, sizeof(float2) * C * T, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaMemcpyAsync(hm.data(), S.st.hm, sizeof(int2) * C * T, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaMemcpyAsync(count, S.st.count, sizeof count, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaMemcpyAsync(&next, S.st.next_id, sizeof next, cudaMemcpyDeviceToHost, S.stream));
  TRACK_TRY(t, cudaStreamSynchronize(S.stream));
  std::vector<isx_track> live;
  for (size_t k = 0; k < C; k++)
    for (int i = 0; i < count[k]; i++) {
      const size_t j = k * T + i;
      live.push_back(isx_track{id[j], (int32_t)(ISX_FIRST_INSTANCE_CLASS + k), hm[j].x, hm[j].y, box[j].x, box[j].y,
                               box[j].z, box[j].w, disp[j].x, disp[j].y, 0});
    }
  std::sort(live.begin(), live.end(), [](const isx_track &a, const isx_track &b) { return a.id < b.id; });
  for (int i = 0; i < capacity && i < (int)live.size(); i++) host[i] = live[(size_t)i];
  if (n) *n = (int)live.size();
  if (next_id) *next_id = next;
  return ISX_OK;
}

}  // extern "C"
