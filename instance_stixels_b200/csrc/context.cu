// C ABI of the library (include/instance_stixels_b200.h): object lifetime,
// configuration, device memory, streams and the per-batch kernel sequence.
// Host orchestration of the reference: Stixels::Initialize / Compute /
// ClusterInstances / GetInstanceStixels (InstanceStixels/src/Stixels.cu:43-283,
// 449-681, 744-776).
//
// Differences in mechanism (not in results): batches of independent frames go
// through every kernel in one launch; frames are processed in chunks so that a
// chunk's H2D copy, the previous chunk's kernels and the one before's D2H copy
// overlap on three streams; there is no per-frame cudaMalloc, handle
// construction or device-wide synchronisation.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "host_model.h"
#include "kernels.h"

namespace isx {

static thread_local std::string g_last_error;
constexpr int kStageSlots = 8;    // pinned staging buffers of the road tables (see isx_context::h_ground)
constexpr int kRoadSlots = 4;     // device copies of a chunk's road tables (isx_context::roads)
constexpr int kResultSets = 4;    // result sets: up to kResultSets - 1 submitted batches in flight + the one waited last
constexpr int kProfEvents = 9;    // profiling events per enqueued chunk (enqueue_chunk)
constexpr int kTraceStamps = 11;  // time stamps per chunk of isx_get_chunk_trace

static int fail(isx_context *ctx, int code, const std::string &msg);

struct RoadKey {
  int vhor;
  float tilt, height, alpha;
  bool operator<(const RoadKey &o) const {
    if (vhor != o.vhor) return vhor < o.vhor;
    if (tilt != o.tilt) return tilt < o.tilt;
    if (height != o.height) return height < o.height;
    return alpha < o.alpha;
  }
};

}  // namespace isx

struct isx_context {
  int device = 0;
  bool configured_parts[8] = {false, false, false, false, false, false, false, false};
  bool initialized = false;
  isx::HostModel model;
  isx::KParams kp{};
  int max_batch = 0, chunk = 0;   // chunk: frames the intermediates hold = frames per pairwise launch
  int chunk_unary = 0;            // frames per unary launch
  int last_launch_frames = 0;     // of the last enqueued batch (isx_chunk_frames)
  std::string last_error;

  // s_tables: join + table build (HBM-bound), s_compute: the DP (issue-bound), s_emit: backtracking, grouping, packing
  // (short, latency-bound).  The tables of chunk k+1 are built WHILE the DP of chunk k runs: their CTAs take the
  // places DP CTAs vacate (12 K registers against 16 K), so the memory-bound and the issue-bound kernel share the SMs.
  cudaStream_t s_tables = nullptr, s_compute = nullptr, s_emit = nullptr, s_h2d = nullptr, s_d2h = nullptr;
  cudaEvent_t ev_dp_done[2] = {nullptr, nullptr}, ev_emit_done[2] = {nullptr, nullptr};
  cudaEvent_t ev_tab_done[2] = {nullptr, nullptr};   // tables of the chunk in this set are complete
  cudaEvent_t ev_user = nullptr;                     // the caller's work on isx_stream() before a device batch
  cudaEvent_t ev_in_ready[2] = {nullptr, nullptr}, ev_in_free[2] = {nullptr, nullptr};
  cudaEvent_t ev_chunk_done = nullptr;
  // narrow host inputs (isx_*_u16): staging for the raw uint16 / int16 data, allocated on first use
  uint16_t *d_in_disp16[2] = {nullptr, nullptr};  // [chunk][H][W]
  int16_t *d_in_seg16[2] = {nullptr, nullptr};    // [chunk][C][21][ceil(H/8)]

  // device memory
  std::vector<void *> allocations;
  float *d_in_disp[2] = {nullptr, nullptr};       // staging for host batches: [chunk][H][W]
  int32_t *d_in_seg[2] = {nullptr, nullptr};      // [chunk][seg_elems]
  float *d_single_disp = nullptr;                 // SetDisparityImage target (d_disparity_big)
  int32_t *d_single_seg = nullptr;                // SetSegmentation target
  isx::BatchBuffers buf;                          // intermediates sized `chunk`, results sized `max_batch`
  // Buffers the emission stream still reads while the compute stream works on the next chunk exist
  // twice; chunk k uses set k & 1.
  struct ChunkSet {
    float *stat = nullptr;
    uint32_t *records_b = nullptr;
    float4 *dp = nullptr;
    float *pm = nullptr;
    int *err = nullptr;   // [chunk] kErr* bits per frame, zeroed when the chunk is enqueued
    float *joined = nullptr;      // [chunk][C][H]
    float *object_lut = nullptr;  // [chunk][C][D][lut_stride]
    int *col_flags = nullptr;     // [chunk][C]
  } sets[2];
  int last_set = 0;
  // The road tables of a chunk ([chunk][3][H] + [chunk] horizon rows) arrive on the copy stream in front of the chunk's
  // images.  They have their own ring: as members of the chunk set their copy had to wait for the emission two chunks
  // back, and with it every image copy queued behind -- the input copies of a pipelined host batch then started a
  // whole DP late.  `ev_free` = the emission of the chunk that last read the slot.
  struct RoadSlot {
    float *ground = nullptr;
    int *vhor = nullptr;
    cudaEvent_t ev_free = nullptr;
  } roads[isx::kRoadSlots];
  unsigned long long road_next = 0;
  int last_road_slot = 0;
  bool overlap_tables = true;      // table build of chunk k+1 beside the DP of chunk k (ISX_OVERLAP_TABLES)
  bool emit_join_pending = false;  // results of the last device batch are not yet ordered on isx_stream()
  // Results of one batch.  The padded device arrays feed the rasteriser and the fallback copy; what a host caller
  // gets is packed by pack_results_kernel (emit.cu) straight into pinned host memory that is mapped into the
  // device address space (h_* = host address, m_* = the device's address of the same memory).
  struct ResultSet {
    bool allocated = false;
    isx_section *d_sections = nullptr;            // [max_batch][C][200]
    int *d_nsections = nullptr;                   // [max_batch][C]
    isx_instance *d_inst = nullptr;               // [max_batch][inst_cap]
    int *d_inst_count = nullptr;                  // [max_batch]
    int *d_cursors = nullptr;                     // [2] next free packed section / instance record
    isx_section *h_sections = nullptr, *m_sections = nullptr;   // packed Sections of the batch
    isx_instance *h_inst = nullptr, *m_inst = nullptr;          // packed instance records of the batch
    int *h_counts = nullptr, *m_counts = nullptr;               // [max_batch][C] stixels per column
    isx_packed_frame *h_frames = nullptr, *m_frames = nullptr;  // [max_batch]
    int sections_cap = 0, inst_cap = 0;           // entries of the packed arrays
  } rs[isx::kResultSets];
  int cur = 0;                                    // result set of the batch being enqueued / of the last batch
  int *d_raster_table = nullptr;                  // [max_batch][C][200] instance id per stixel (rasteriser)
  int *d_export_col = nullptr;                    // [max_batch][C] frame-relative column offsets (device export)
  int inst_cap = 0;                               // instance records per frame of the device arrays: C * 200
  float *d_export_cost = nullptr;
  int *d_export_index = nullptr;

  // pinned host staging
  // road tables on their way to the device: a ring of kStageSlots pinned buffers, each with the event of the copy
  // that last read it, so that the enqueueing host thread may run several chunks ahead of the device
  float *h_ground = nullptr;                      // [kStageSlots][chunk][3][H]
  int *h_vhor = nullptr;                          // [kStageSlots][chunk]
  cudaEvent_t ev_stage_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  unsigned long long stage_next = 0;
  // isx_submit_batch_host keeps up to kResultSets - 1 batches in flight: rs[cur] belongs to the batch submitted last;
  // a new batch takes the lowest set that is neither in flight nor the one handed out by the last wait (allocated on
  // first use: a caller with two batches in flight only ever touches three).  Indexed by ticket % kResultSets:
  cudaEvent_t ev_batch_done[isx::kResultSets] = {};       // behind the packing of the batch's last chunk
  int batch_n[isx::kResultSets] = {};                     // frames of the batch in flight with that ticket, 0 = none
  int batch_set[isx::kResultSets] = {};                   // its result set
  isx_section *batch_sections[isx::kResultSets] = {};     // the caller's padded array the wait expands into
  bool batch_direct[isx::kResultSets] = {};               // ... or that the device has already filled (mapped memory)
  isx_section *direct_sections = nullptr;               // device address of the caller's array for the batch being enqueued
  bool results_stay_on_device = false;                  // set while a device batch is enqueued
  int last_waited_set = -1;                           // result set of the batch waited for last (isx_wait_batch_packed)
  unsigned long long submitted = 0, waited = 0;       // tickets: batches [waited, submitted) are in flight
  unsigned long long dp_units_pairwise = 0;           // ... of which in pairwise mode (never pruned)
  unsigned long long dp_units_total = 0;              // 32 x 32-cell units of all DP launches so far
  int host_slot = 0;                                  // input slot / chunk set of the next host chunk (alternates across batches)

  std::map<isx::RoadKey, std::vector<float>> road_cache;
  isx_road single_road{0, 0.f, 0.f, 0.f};
  bool single_has_road = false;
  int last_batch = 0;          // frames of the last batch (results valid for these)
  int last_chunk_first = 0;    // first frame whose intermediates are still in `buf`
  int last_chunk_n = 0;
  bool last_pairwise = false;
  std::vector<isx_road> last_roads;

  // optional per-stage CUDA-event timing (isx_set_profiling)
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;   // kStages+1 events per enqueued chunk
  size_t prof_used = 0;
  std::vector<cudaEvent_t> prof_h2d;      // host batches: begin / end of every chunk's input copies (copy stream)
  size_t prof_h2d_used = 0;
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long stage_launches[8] = {0, 0, 0, 0, 0, 0, 0, 0};
};

namespace isx {

static int fail(isx_context *ctx, int code, const std::string &msg) {
  g_last_error = msg;
  if (ctx) ctx->last_error = msg;
  return code;
}

int fail_cuda(cudaError_t e, const char *expr, const char *file, int line) {
  char buf[512];
  std::snprintf(buf, sizeof buf, "%s returned %s(%d) at %s:%d", expr, cudaGetErrorString(e), (int)e, file, line);
  g_last_error = buf;
  return ISX_ERR_CUDA;
}

#define ISX_TRY(ctx, expr)                                            \
  do {                                                                \
    cudaError_t _e = (expr);                                          \
    if (_e != cudaSuccess) {                                          \
      int _c = ::isx::fail_cuda(_e, #expr, __FILE__, __LINE__);       \
      (ctx)->last_error = ::isx::g_last_error;                        \
      return _c;                                                      \
    }                                                                 \
  } while (0)

template <typename T>
static cudaError_t dev_alloc(isx_context *c, T **p, size_t count) {
  void *q = nullptr;
  cudaError_t e = cudaMalloc(&q, count * sizeof(T) + 256);
  if (e == cudaSuccess) {
    c->allocations.push_back(q);
    *p = static_cast<T *>(q);
  }
  return e;
}

// Device bytes per frame of a chunk: both chunk sets, both input staging slots and the transition records of the
// pairwise walk (the allocations of isx_initialize that scale with the chunk).
static size_t chunk_frame_bytes(int rows, int cols, int rec_stride, int realcols, int max_dis) {
  const size_t H = rows, C = realcols, D = max_dis, lut_stride = (H + 31) & ~(size_t)31;
  const size_t hs2 = H > (size_t)kShortRows ? 256 : 128;   // rows_power2_segmentation, an upper bound below 1025 rows
  const size_t set = H * kStatWords * 4 + C * rec_stride * kRecBWords * 4 + C * H * (4 + 16 + 4) + C * D * lut_stride * 4;
  const size_t inputs = H * (size_t)cols * 4 + hs2 * C * 21 * 4;
  return 2 * (set + inputs) + C * rec_stride * kDynWords * 4;
}

static size_t seg_elems(const isx_context *c) {
  return (size_t)c->model.rows_power2_seg * c->model.realcols * c->model.n_channels;
}

static void fill_kparams(isx_context *c) {
  const HostModel &m = c->model;
  KParams &k = c->kp;
  k.rows = m.rows;
  k.cols = m.cols;
  k.realcols = m.realcols;
  k.column_step = m.column_step;
  k.width_margin = m.width_margin;
  k.max_dis = m.max_dis;
  k.hs2 = m.rows_power2_seg;
  k.n_classes = m.n_classes;
  k.n_channels = m.n_channels;
  k.median_join = m.median_join ? 1 : 0;
  k.size_filter = m.size_filter;
  k.min_pts = m.min_pts;
  k.eps_cluster = m.eps;
  k.invalid_disparity = m.invalid_disparity;
  k.max_disf = m.max_disf;
  k.rows_log = m.rows_log;
  k.max_dis_log = m.max_dis_log;
  k.pnexists_given_sky_log = m.pnexists_given_sky_log;
  k.normalization_sky = m.normalization_sky;
  k.inv_sigma2_sky = m.inv_sigma2_sky;
  k.puniform_sky = m.puniform_sky;
  k.nopnexists_given_sky_log = m.nopnexists_given_sky_log;
  k.pnexists_given_ground_log = m.pnexists_given_ground_log;
  k.puniform = m.puniform;
  k.nopnexists_given_ground_log = m.nopnexists_given_ground_log;
  k.pord = m.pord;
  k.epsilon = m.epsilon;
  k.pgrav = m.pgrav;
  k.pblg = m.pblg;
  k.prior_weight = m.prior_weight;
  k.disparity_weight = m.disparity_weight;
  k.segmentation_weight = m.segmentation_weight;
  k.instance_weight = m.instance_weight;
  k.rec_stride = rec_stride_for_rows(m.rows);
  k.lut_stride = (m.rows + 31) & ~31;
  float mn = m.obj_cost_lut.empty() ? 0.0f : m.obj_cost_lut[0];
  float amax = 0.0f;
  for (float v : m.obj_cost_lut) {
    mn = v < mn ? v : mn;
    const float a = v < 0.0f ? -v : v;
    amax = a > amax ? a : amax;   // NaN entries are skipped; an infinite one makes the slack infinite: no pruning
  }
  k.obj_cost_min = mn;
  k.obj_cost_absmax = amax;
  const char *e = std::getenv("ISX_UNARY_PRUNE");
  k.prune_unary = (e && std::atoi(e) == 0) ? 0 : 1;
  const char *e2 = std::getenv("ISX_PAIRWISE_PRUNE");
  k.prune_pairwise = (e2 && std::atoi(e2) == 0) ? 0 : 1;
}

static const float *road_tables(isx_context *c, const isx_road &r) {
  RoadKey key{r.vhor, r.camera_tilt, r.camera_height, r.alpha_ground};
  auto it = c->road_cache.find(key);
  if (it == c->road_cache.end()) {
    if (c->road_cache.size() > 64) c->road_cache.clear();
    std::vector<float> t((size_t)3 * c->model.rows);
    c->model.ground_tables(r, t.data());
    it = c->road_cache.emplace(key, std::move(t)).first;
  }
  return it->second.data();
}

// Enqueue the kernel sequence for `n` frames whose inputs are at d_disp/d_seg.
// `slot` selects the pinned ground-table staging half and the ChunkSet; results
// land at frame offset `first` of the per-batch result arrays.
//
// Three streams: join -> tables -> LUT on s_tables, the DP on s_compute; backtracking, candidate
// collection, grouping and packing (short, latency-bound launches) on s_emit, so
// that they overlap the next chunk's DP.
// The per-frame road tables of a chunk (Stixels.cu:463-493: three blocking copies per frame in the reference) go
// through a pinned staging buffer to the next slot of the road ring on stream `st`, behind the emission that last read
// that slot (kRoadSlots chunks ago).  Returns the slot (>= 0) or an error (< 0).
static int stage_road_tables(isx_context *c, const isx_road *roads, int n, cudaStream_t st) {
  const int H = c->kp.rows;
  const int stage = (int)(c->stage_next++ % kStageSlots);
  // the copy that read this staging buffer kStageSlots chunks ago must be done (a never-recorded event is complete)
  ISX_TRY(c, cudaEventSynchronize(c->ev_stage_done[stage]));
  float *hg = c->h_ground + (size_t)stage * c->chunk * 3 * H;
  int *hv = c->h_vhor + (size_t)stage * c->chunk;
  for (int i = 0; i < n; i++) {
    std::memcpy(hg + (size_t)i * 3 * H, road_tables(c, roads[i]), sizeof(float) * 3 * H);
    hv[i] = H - roads[i].vhor - 1;  // Stixels.cu:377
  }
  const int rslot = (int)(c->road_next++ % kRoadSlots);
  const isx_context::RoadSlot &rd = c->roads[rslot];
  ISX_TRY(c, cudaStreamWaitEvent(st, rd.ev_free, 0));
  ISX_TRY(c, cudaMemcpyAsync(rd.ground, hg, sizeof(float) * 3 * H * n, cudaMemcpyHostToDevice, st));
  ISX_TRY(c, cudaMemcpyAsync(rd.vhor, hv, sizeof(int) * n, cudaMemcpyHostToDevice, st));
  ISX_TRY(c, cudaEventRecord(c->ev_stage_done[stage], st));
  return rslot;
}

// `road_slot` >= 0: the caller has already copied the road tables of the chunk into that slot of the ring (host
// batches send them on the copy stream IN FRONT of the chunk's images: as a copy on the compute stream they would
// queue on the copy engine behind the next chunk's images -- several milliseconds of an idle GPU per chunk, measured
// with isx_get_chunk_trace).
static int enqueue_chunk(isx_context *c, bool pairwise, int first, int n, const float *d_disp,
                         const int32_t *d_seg, const isx_road *roads, int slot, int road_slot = -1) {
  const KParams &kp = c->kp;
  const int H = kp.rows, C = kp.realcols;
  const isx_context::ChunkSet &cs = c->sets[slot];
  cudaStream_t st = c->s_tables, s = c->s_compute, se = c->s_emit;
  // the emission of the chunk that used this set two chunks ago must be done with it (it follows that chunk's DP)
  ISX_TRY(c, cudaStreamWaitEvent(st, c->ev_emit_done[slot], 0));
  // ISX_OVERLAP_TABLES=0: the table build waits for the DP of the chunk before it (one kernel at a time on the SMs)
  if (!c->overlap_tables) ISX_TRY(c, cudaStreamWaitEvent(st, c->ev_dp_done[slot ^ 1], 0));
  if (road_slot < 0) {
    road_slot = stage_road_tables(c, roads, n, st);
    if (road_slot < 0) return road_slot;
  }
  const isx_context::RoadSlot &rd = c->roads[road_slot];
  ISX_TRY(c, cudaMemsetAsync(cs.err, 0, sizeof(int) * n, st));  // the error words of THIS chunk's frames
  isx_context::ResultSet &R = c->rs[c->cur];
  BatchBuffers b = c->buf;
  b.ground = rd.ground; b.vhor = rd.vhor; b.stat = cs.stat;
  b.records_b = cs.records_b; b.dp = cs.dp; b.pm = cs.pm;
  b.joined = cs.joined; b.object_lut = cs.object_lut; b.col_flags = cs.col_flags;
  b.error_flag = cs.err;
  b.disparity = d_disp;
  b.segmentation = d_seg;
  b.sections = R.d_sections + (size_t)first * C * kMaxSections;
  b.n_sections = R.d_nsections + (size_t)first * C;
  // profiling events per chunk: 0 join | 1 frame tables | 2 column tables + LUT | 3 end (s_tables); 4 dp | 5 dp end
  //                             (s_compute); 6 backtrack + collect | 7 grouping + pack | 8 end (s_emit)
  auto mark = [&](cudaStream_t st) {
    if (!c->profiling) return;
    if (c->prof_used >= c->prof_events.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      c->prof_events.push_back(e);
    }
    cudaEventRecord(c->prof_events[c->prof_used++], st);
  };
  mark(st);
  launch_join_columns(kp, b, n, st);
  mark(st);
  if (pairwise) launch_frame_tables(kp, b, n, st);
  mark(st);
  launch_column_tables(kp, b, n, st);
  mark(st);
  ISX_TRY(c, cudaEventRecord(c->ev_tab_done[slot], st));
  ISX_TRY(c, cudaStreamWaitEvent(s, c->ev_tab_done[slot], 0));
  mark(s);
  launch_dp(kp, b, n, pairwise, s);
  {
    const unsigned long long nt = (unsigned long long)(H + 31) / 32;
    c->dp_units_total += (unsigned long long)n * C * (nt * (nt + 1) / 2);
    const char *ex = std::getenv("ISX_UNARY_EXHAUSTIVE");
    // the pruning kernels count on the device
    const bool walks_all = (pairwise && !pairwise_walk_used(n * C, b.qrows != nullptr)) || (!pairwise && ex && std::atoi(ex) != 0);
    c->dp_units_pairwise += walks_all ? (unsigned long long)n * C * (nt * (nt + 1) / 2) : 0;
  }
  mark(s);
  ISX_TRY(c, cudaEventRecord(c->ev_dp_done[slot], s));
  ISX_TRY(c, cudaStreamWaitEvent(se, c->ev_dp_done[slot], 0));
  mark(se);
  launch_emit(kp, b, n, pairwise, se);
  mark(se);
  launch_grouping(kp, b, n, se);
  {
    PackArgs a;
    a.sections = b.sections; a.n_sections = b.n_sections;
    a.cand_count = b.cand_count; a.cand_idx = b.cand_idx; a.cand_label = b.cand_label;
    a.err = cs.err; a.col_offset = b.pack_offset;
    a.inst_out = R.d_inst + (size_t)first * c->inst_cap; a.inst_count_out = R.d_inst_count + first;
    a.inst_cap = c->inst_cap; a.cursors = R.d_cursors;
    a.h_padded = c->direct_sections ? c->direct_sections + (size_t)first * C * kMaxSections : nullptr;
    // a device batch leaves its results on the device (isx_compute_batch_device): only the counts and descriptors
    // cross the host link, a later fetch reads the padded device arrays (the frames are flagged like overflows)
    a.h_sections = R.m_sections; a.h_sections_cap = c->results_stay_on_device ? 0 : R.sections_cap;
    a.h_inst = R.m_inst; a.h_inst_cap = c->results_stay_on_device ? 0 : R.inst_cap;
    a.h_counts = R.m_counts + (size_t)first * C; a.h_frames = R.m_frames + first;
    launch_pack(kp, a, n, se);
  }
  mark(se);
  ISX_TRY(c, cudaEventRecord(c->ev_emit_done[slot], se));
  ISX_TRY(c, cudaEventRecord(rd.ev_free, se));
  ISX_TRY(c, cudaGetLastError());
  c->last_chunk_first = first;
  c->last_chunk_n = n;
  c->last_pairwise = pairwise;
  c->last_set = slot;
  c->last_road_slot = road_slot;
  return ISX_OK;
}

// If the caller's Section array is pinned and mapped (cudaHostAlloc / cudaHostRegister / torch pin_memory), the
// device writes the padded layout straight into it: returns the device address of `sections`, or null for
// pageable memory (then the packed arrays are expanded on the host).  ISX_NO_DIRECT=1 forces the packed path.
static isx_section *device_view_of(isx_section *sections) {
  if (!sections) return nullptr;
  if (const char *e = std::getenv("ISX_NO_DIRECT"))
    if (std::atoi(e) != 0) return nullptr;
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, sections) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (attr.type != cudaMemoryTypeHost || !attr.devicePointer) return nullptr;
  return static_cast<isx_section *>(attr.devicePointer);
}

// Every batch starts its packed result arrays from the front (ordered on the emission stream behind the packing of
// whatever batch used this result set before).
static int begin_batch(isx_context *c) {
  ISX_TRY(c, cudaMemsetAsync(c->rs[c->cur].d_cursors, 0, 2 * sizeof(int), c->s_emit));
  return ISX_OK;
}

// The result arrays of one batch: padded device arrays + packed arrays in mapped pinned host memory.
static int alloc_result_set(isx_context *c, int i) {
  isx_context::ResultSet &R = c->rs[i];
  if (R.allocated) return ISX_OK;
  const size_t C = c->kp.realcols, MB = c->max_batch;
  ISX_TRY(c, dev_alloc(c, &R.d_sections, MB * C * kMaxSections));
  // entries after a column's terminator are never written: start them from zero
  ISX_TRY(c, cudaMemset(R.d_sections, 0, MB * C * kMaxSections * sizeof(isx_section)));
  ISX_TRY(c, dev_alloc(c, &R.d_nsections, MB * C));
  ISX_TRY(c, dev_alloc(c, &R.d_inst, MB * (size_t)c->inst_cap));
  ISX_TRY(c, dev_alloc(c, &R.d_inst_count, MB));
  ISX_TRY(c, dev_alloc(c, &R.d_cursors, 2));
  ISX_TRY(c, cudaMemset(R.d_cursors, 0, 2 * sizeof(int)));
  // Packed arrays: sized for `budget` stixels per column on average over a batch (the pairwise model yields about
  // ten per column on street scenes, the unary model with its 1/n prior sixty to seventy; the capacity of the
  // reference's array is 200).  A batch that needs more falls back to the padded arrays frame by frame.
  // Frames taller than 1024 rows have proportionally more stixels per column (synthetic unary frames: 80 at 1280
  // rows, 129 at 2047): the budget grows with the rows there, up to the capacity of 200.
  size_t budget = 100;
  if (c->kp.rows > kShortRows) budget = ((size_t)c->kp.rows * 100 + kShortRows - 1) / kShortRows;
  if (const char *e = std::getenv("ISX_PACK_BUDGET")) budget = std::atoi(e) > 0 ? (size_t)std::atoi(e) : budget;
  budget = budget < (size_t)kMaxSections ? budget : (size_t)kMaxSections;
  R.sections_cap = R.inst_cap = (int)(MB * C * budget);
  const unsigned flags = cudaHostAllocMapped | cudaHostAllocPortable;
  ISX_TRY(c, cudaHostAlloc(&R.h_sections, sizeof(isx_section) * (size_t)R.sections_cap, flags));
  ISX_TRY(c, cudaHostAlloc(&R.h_inst, sizeof(isx_instance) * (size_t)R.inst_cap, flags));
  ISX_TRY(c, cudaHostAlloc(&R.h_counts, sizeof(int) * MB * C, flags));
  ISX_TRY(c, cudaHostAlloc(&R.h_frames, sizeof(isx_packed_frame) * MB, flags));
  ISX_TRY(c, cudaHostGetDevicePointer(&R.m_sections, R.h_sections, 0));
  ISX_TRY(c, cudaHostGetDevicePointer(&R.m_inst, R.h_inst, 0));
  ISX_TRY(c, cudaHostGetDevicePointer(&R.m_counts, R.h_counts, 0));
  ISX_TRY(c, cudaHostGetDevicePointer(&R.m_frames, R.h_frames, 0));
  std::memset(R.h_frames, 0, sizeof(isx_packed_frame) * MB);
  R.allocated = true;
  return ISX_OK;
}

// Results of every enqueued chunk become visible to work ordered after this on isx_stream() (the table stream: the
// first stream of the pipeline, where a caller's producers of device inputs and consumers of results run).
static int join_emit_stream(isx_context *c) {
  ISX_TRY(c, cudaStreamWaitEvent(c->s_tables, c->ev_emit_done[c->last_set], 0));
  c->emit_join_pending = false;
  return ISX_OK;
}
// isx_compute_batch_device leaves the join to whoever touches the results next (or to isx_flush), so that the
// first kernels of a following batch do not wait for the emission tail of this one.
static int ensure_joined(isx_context *c) { return c->emit_join_pending ? join_emit_stream(c) : ISX_OK; }

static int check_ready(isx_context *c) {
  if (!c) return fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null handle");
  if (!c->initialized) return fail(c, ISX_ERR_NOT_INITIALIZED, "Initialize() has not been called");
  cudaError_t e = cudaSetDevice(c->device);
  if (e != cudaSuccess) return fail(c, ISX_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  return ISX_OK;
}

}  // namespace isx

using namespace isx;

extern "C" {

int isx_abi_version(void) { return ISX_ABI_VERSION; }
uint64_t isx_kernel_launch_count(void) { return g_launch_count; }
const char *isx_last_error(isx_handle h) { return h ? h->last_error.c_str() : g_last_error.c_str(); }

void isx_config_init(isx_config *c) {
  // default member initialisers of StixelConfig (types.h:30-141)
  c->rows = -1; c->cols = -1; c->max_dis = -1; c->invalid_disparity = -1.0f;
  c->eps = -1; c->min_pts = -1; c->size_filter = -1;
  c->n_semantic_classes = -1; c->n_offset_channels = -1;
  c->prior_weight = -1; c->segmentation_weight = -1; c->instance_weight = -1; c->disparity_weight = -1;
  c->pairwise = 0; c->column_step = -1;
  c->focal = -1; c->baseline = -1; c->camera_center_x = -1; c->camera_center_y = -1;
  c->sigma_disparity_object = 1.0f; c->sigma_disparity_ground = 2.0f; c->sigma_sky = 0.1f;
  c->pout = 0.15f; c->pout_sky = 0.4f; c->pord = 0.2f; c->pgrav = 0.1f; c->pblg = 0.04f;
  c->pground_given_nexist = 0.28; c->pobject_given_nexist = 0.44; c->psky_given_nexist = 0.28;
  c->pnexist_dis = 0.25f;
  c->pground = 1.0f / 3.0f; c->pobject = 1.0f / 3.0f; c->psky = 1.0f / 3.0f;
  c->width_margin = 0;
  c->sigma_camera_tilt = 0.05f; c->sigma_camera_height = 0.05f;
  c->median_join = 0; c->epsilon = 3.0f; c->range_objects_z = 10.20f;
  c->road_vdisparity_threshold = 0.2f;
}

int isx_create(isx_handle *out, int device) {
  if (!out) return fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null out pointer");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(nullptr, ISX_ERR_CUDA,
                std::string("no CUDA device: the stixel path has no CPU fallback (") + cudaGetErrorString(e) + ")");
  if (device < 0 || device >= count) return fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "device ordinal out of range");
  isx_context *c = new isx_context();
  c->device = device;
  *out = c;
  return ISX_OK;
}

int isx_destroy(isx_handle h) {
  if (!h) return ISX_OK;
  if (h->initialized) isx_finish(h);
  delete h;
  return ISX_OK;
}

int isx_set_config(isx_handle h, const isx_config *cfg) {
  if (!h || !cfg) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  const std::string err = validate_config(*cfg);
  if (!err.empty()) return fail(h, ISX_ERR_INVALID_ARGUMENT, err);
  h->model.apply(*cfg);
  return ISX_OK;
}

int isx_set_disparity_parameters(isx_handle h, int rows, int cols, int max_dis, float invalid_disparity,
                                 float sigma_disparity_object, float sigma_disparity_ground, float sigma_sky) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  HostModel &m = h->model;
  m.rows = rows; m.cols = cols; m.max_dis = max_dis; m.invalid_disparity = invalid_disparity;
  m.sigma_disparity_object = sigma_disparity_object; m.sigma_disparity_ground = sigma_disparity_ground;
  m.sigma_sky = sigma_sky;
  return ISX_OK;
}
int isx_set_segmentation_parameters(isx_handle h, int classes, int instance_channels) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  h->model.n_classes = classes;
  h->model.n_channels = classes + instance_channels;
  return ISX_OK;
}
int isx_set_clustering_parameters(isx_handle h, float eps, int min_pts, int size_filter) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  h->model.eps = eps; h->model.min_pts = min_pts; h->model.size_filter = size_filter;
  if (h->initialized) {  // the reference writes these straight into m_params (Stixels.cu:395-400)
    h->kp.eps_cluster = eps; h->kp.min_pts = min_pts; h->kp.size_filter = size_filter;
  }
  return ISX_OK;
}
int isx_set_weight_parameters(isx_handle h, float prior_weight, float disparity_weight, float segmentation_weight,
                              float instance_weight) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  HostModel &m = h->model;
  m.prior_weight = prior_weight; m.disparity_weight = disparity_weight; m.segmentation_weight = segmentation_weight;
  m.instance_weight = 0.0;
  if (segmentation_weight > 1e-5) {
    m.instance_weight = instance_weight / segmentation_weight;
    if (instance_weight < 1e-8) m.instance_weight = 0.0;
  }
  return ISX_OK;
}
int isx_set_probabilities(isx_handle h, float pout, float pout_sky, float pground_given_nexist,
                          float pobject_given_nexist, float psky_given_nexist, float pnexist_dis, float pground,
                          float pobject, float psky, float pord, float pgrav, float pblg) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  HostModel &m = h->model;
  m.pout = pout; m.pout_sky = pout_sky;
  m.pnexists_given_ground = (pground_given_nexist * pnexist_dis) / pground;
  m.pnexists_given_object = (pobject_given_nexist * pnexist_dis) / pobject;
  m.pnexists_given_sky = (psky_given_nexist * pnexist_dis) / psky;
  m.pord = pord; m.pgrav = pgrav; m.pblg = pblg;
  return ISX_OK;
}
int isx_set_camera_parameters(isx_handle h, float focal, float baseline, float sigma_camera_tilt,
                              float sigma_camera_height, float camera_center_x, float camera_center_y) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  HostModel &m = h->model;
  m.focal = focal; m.baseline = baseline;
  m.sigma_camera_tilt = sigma_camera_tilt * (3.1416f) / 180.0f;
  m.sigma_camera_height = sigma_camera_height;
  m.camera_center_x = camera_center_x; m.camera_center_y = camera_center_y;
  return ISX_OK;
}
int isx_set_model_parameters(isx_handle h, int column_step, int median_join, float epsilon, float range_objects_z,
                             int width_margin) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  HostModel &m = h->model;
  m.column_step = column_step; m.median_join = median_join != 0; m.epsilon = epsilon;
  m.range_objects_z = range_objects_z; m.width_margin = width_margin;
  return ISX_OK;
}

int isx_initialize(isx_handle h, int max_batch) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  if (h->initialized) return fail(h, ISX_ERR_INVALID_ARGUMENT, "already initialized: call Finish() first");
  if (max_batch < 1) return fail(h, ISX_ERR_INVALID_ARGUMENT, "max_batch must be >= 1");
  HostModel &m = h->model;
  if (m.rows <= 0 || m.cols <= 0 || m.max_dis <= 0 || m.column_step <= 0)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "configuration is not set");
  // The reference stops at 1024 rows (its one-thread-per-row block, apps/run_cityscapes.cu:129-134); up to
  // ISX_MAX_ROWS its padded sizes, and so the segmentation layout and the scan orders, stay defined (DESIGN.md 1, 2).
  if (m.rows > ISX_MAX_ROWS) return fail(h, ISX_ERR_UNSUPPORTED, "rows > ISX_MAX_ROWS (2047) is not supported");
  if (m.max_dis > 256) return fail(h, ISX_ERR_UNSUPPORTED, "max_dis > 256 is not supported");
  if (m.n_classes != 19 || m.n_channels != 21)
    return fail(h, ISX_ERR_UNSUPPORTED, "the Cityscapes layout (19 classes + 2 offsets) is hard-wired like Cityscapes.h");
  if (m.column_step > 16) return fail(h, ISX_ERR_UNSUPPORTED, "column_step > 16 is not supported");
  ISX_TRY(h, cudaSetDevice(h->device));
  m.derive();
  fill_kparams(h);
  const KParams &kp = h->kp;
  const size_t H = kp.rows, W = kp.cols, C = kp.realcols, D = kp.max_dis;
  if (C == 0) return fail(h, ISX_ERR_INVALID_ARGUMENT, "no stixel columns");
  h->max_batch = max_batch;
  // Frames per launch.  Every DP launch ends with a partly filled wave, so few large launches beat many small
  // ones; but the copies of a host batch only overlap kernels of OTHER chunks.  Measured (B200, 64-frame batches,
  // frames/s resident | end to end): unary 16 / 32 / 64 frames per launch = 7095 | 4614, 7999 | 4628, 8083 | 4525;
  // pairwise 2691 | 2473, 2940 | 2817, 3041 | 2855 -- the pairwise walk kernel runs ONE warp per column, 2368 at a
  // time: 32 frames are 3.46 waves of them, 64 frames 6.9.  So the buffers hold 64 frames (two sets, about 23 GB at
  // width 8) and unary launches take 32 of them.
  int chunk = 64, chunk_unary = 32;
  if (m.rows > kShortRows) {
    // Frames taller than 1024 rows: as many frames per chunk as keep the two chunk sets within the footprint of two
    // 64-frame sets of 1024 x 2048 frames at width 4 and the same max_dis (the largest before tall frames existed).
    const size_t budget = 64 * chunk_frame_bytes(kShortRows, 2048, kRecStride, 2048 / 4, m.max_dis);
    const size_t per_frame = chunk_frame_bytes(m.rows, m.cols, rec_stride_for_rows(m.rows), m.realcols, m.max_dis);
    const size_t fit = budget / per_frame;
    chunk = fit < 1 ? 1 : fit < 64 ? (int)fit : 64;
    chunk_unary = chunk < 32 ? chunk : 32;
  }
  if (const char *e = std::getenv("ISX_CHUNK")) chunk = chunk_unary = std::atoi(e) > 0 ? std::atoi(e) : chunk;
  h->chunk = chunk < max_batch ? chunk : max_batch;
  h->chunk_unary = chunk_unary < h->chunk ? chunk_unary : h->chunk;
  h->last_launch_frames = h->chunk_unary;
  h->kp.lut_cols = h->chunk * (int)C;
  const size_t ch = h->chunk, MB = max_batch;
  const size_t cap = C * kMaxSections;
  h->inst_cap = (int)cap;  // every stixel of a frame can be an instance stixel (the reference sizes 8 x this)

  {
    // The emission stream's short kernels should not queue behind the DP's thousands of CTAs: highest priority.
    // The table build runs at the DP's own (lowest) priority: its CTAs then fill the SMs as the DP of the chunk
    // before drains (B200, 64-frame batches: unary 7581 -> 7995 frames/s, pairwise 2761 -> 2942 against one kernel
    // at a time); ABOVE the DP they push its CTAs out as they retire and both kernels lose (7581 / 2566).
    int prio_lo = 0, prio_hi = 0;
    ISX_TRY(h, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    int prio_mid = prio_lo;
    if (const char *e = std::getenv("ISX_TABLES_PRIO"))   // A/B runs: 1 = between the DP and the emission kernels
      prio_mid = (std::atoi(e) != 0 && prio_hi < prio_lo - 1) ? prio_hi + 1 : prio_lo;
    ISX_TRY(h, cudaStreamCreateWithPriority(&h->s_compute, cudaStreamNonBlocking, prio_lo));
    ISX_TRY(h, cudaStreamCreateWithPriority(&h->s_tables, cudaStreamNonBlocking, prio_mid));
    ISX_TRY(h, cudaStreamCreateWithPriority(&h->s_emit, cudaStreamNonBlocking, prio_hi));
  }
  ISX_TRY(h, cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
  ISX_TRY(h, cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_in_ready[i], cudaEventDisableTiming));
    ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_in_free[i], cudaEventDisableTiming));
    ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_dp_done[i], cudaEventDisableTiming));
    ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_emit_done[i], cudaEventDisableTiming));
    ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_tab_done[i], cudaEventDisableTiming));
  }
  ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_chunk_done, cudaEventDisableTiming));
  ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_user, cudaEventDisableTiming));

  BatchBuffers &b = h->buf;
  for (int i = 0; i < kRoadSlots; i++) {
    ISX_TRY(h, dev_alloc(h, &h->roads[i].ground, ch * 3 * H));
    ISX_TRY(h, dev_alloc(h, &h->roads[i].vhor, ch));
    ISX_TRY(h, cudaEventCreateWithFlags(&h->roads[i].ev_free, cudaEventDisableTiming));
  }
  h->road_next = 0;
  for (int i = 0; i < 2; i++) {
    ISX_TRY(h, dev_alloc(h, &h->d_in_disp[i], ch * H * W));
    ISX_TRY(h, dev_alloc(h, &h->d_in_seg[i], ch * seg_elems(h)));
    ISX_TRY(h, cudaMemset(h->d_in_seg[i], 0, ch * seg_elems(h) * sizeof(int32_t)));
  }
  ISX_TRY(h, dev_alloc(h, &h->d_single_disp, H * W));
  ISX_TRY(h, dev_alloc(h, &h->d_single_seg, seg_elems(h)));
  for (int i = 0; i < 2; i++) {
    isx_context::ChunkSet &cs = h->sets[i];
    ISX_TRY(h, dev_alloc(h, &cs.stat, ch * H * kStatWords));
    ISX_TRY(h, dev_alloc(h, &cs.records_b, ch * C * kRecBWords * (size_t)kp.rec_stride));
    ISX_TRY(h, cudaMemset(cs.records_b, 0, ch * C * kRecBWords * (size_t)kp.rec_stride * sizeof(uint32_t)));
    ISX_TRY(h, dev_alloc(h, &cs.pm, ch * C * H));
    ISX_TRY(h, cudaMemset(cs.pm, 0, ch * C * H * sizeof(float)));
    ISX_TRY(h, dev_alloc(h, &cs.dp, ch * C * H));
    ISX_TRY(h, dev_alloc(h, &cs.err, ch));
    ISX_TRY(h, dev_alloc(h, &cs.joined, ch * C * H));
    ISX_TRY(h, dev_alloc(h, &cs.object_lut, lut_buffer_bytes(ch * C, D * (size_t)kp.lut_stride * 4) / 4));
    ISX_TRY(h, dev_alloc(h, &cs.col_flags, ch * C));
    ISX_TRY(h, cudaMemset(cs.col_flags, 0, ch * C * sizeof(int)));
  }
  ISX_TRY(h, dev_alloc(h, &b.cand_count, ch * kInstanceClasses));
  ISX_TRY(h, dev_alloc(h, &b.cand_offset, ch * (C + 1) * kInstanceClasses));
  ISX_TRY(h, dev_alloc(h, &b.cand_xy, ch * kInstanceClasses * cap));
  ISX_TRY(h, dev_alloc(h, &b.cand_idx, ch * kInstanceClasses * cap));
  ISX_TRY(h, dev_alloc(h, &b.cand_core, ch * kInstanceClasses * cap));
  ISX_TRY(h, dev_alloc(h, &b.cand_label, ch * kInstanceClasses * cap));
  ISX_TRY(h, dev_alloc(h, &b.cand_scratch, ch * kInstanceClasses * cap));
  ISX_TRY(h, dev_alloc(h, &b.pack_offset, ch * (C + 1)));
  ISX_TRY(h, dev_alloc(h, &b.dp_units, 1));
  if (pairwise_walk_enabled()) {
    ISX_TRY(h, dev_alloc(h, &b.qrows, ch * C * (size_t)kp.rec_stride * kDynWords));
    ISX_TRY(h, cudaMemset(b.qrows, 0, ch * C * (size_t)kp.rec_stride * kDynWords * sizeof(float)));
  }
  ISX_TRY(h, cudaMemset(b.dp_units, 0, sizeof(unsigned long long)));
  h->cur = 0;
  if (int rc = alloc_result_set(h, 0)) return rc;
  ISX_TRY(h, dev_alloc(h, &h->d_raster_table, MB * C * kMaxSections));
  ISX_TRY(h, dev_alloc(h, &h->d_export_col, MB * C));
  ISX_TRY(h, dev_alloc(h, &h->d_export_cost, C * H * 3));
  ISX_TRY(h, dev_alloc(h, &h->d_export_index, C * H * 3));

  float *d_tmp = nullptr;
  ISX_TRY(h, dev_alloc(h, &d_tmp, D * D));
  ISX_TRY(h, cudaMemcpy(d_tmp, m.obj_cost_lut.data(), sizeof(float) * D * D, cudaMemcpyHostToDevice));
  b.obj_cost_lut = d_tmp;
  {
    // transposed copy [dis][fn], fn padded to 32: the LUT kernel reads one 128-byte line per (row, 32 fn)
    const size_t Dp = (D + 31) & ~(size_t)31;
    std::vector<float> t(D * Dp, 0.0f);
    for (size_t fn = 0; fn < D; fn++)
      for (size_t dis = 0; dis < D; dis++) t[dis * Dp + fn] = m.obj_cost_lut[fn * D + dis];
    // object_lut_kernel addresses the table with 32-bit arithmetic on one upper address word: keep it inside one
    // 4 GB window (room for two copies; the second cannot straddle if the first does)
    ISX_TRY(h, dev_alloc(h, &d_tmp, 2 * D * Dp));
    const unsigned long long a0 = (unsigned long long)d_tmp, bytes = sizeof(float) * D * Dp;
    if (((a0 ^ (a0 + bytes - 1)) >> 32) != 0) d_tmp += D * Dp;
    ISX_TRY(h, cudaMemcpy(d_tmp, t.data(), bytes, cudaMemcpyHostToDevice));
    b.obj_cost_lut_t = d_tmp;
  }
  ISX_TRY(h, dev_alloc(h, &d_tmp, D));
  ISX_TRY(h, cudaMemcpy(d_tmp, m.object_disparity_range.data(), sizeof(float) * D, cudaMemcpyHostToDevice));
  b.object_disparity_range = d_tmp;
  ISX_TRY(h, dev_alloc(h, &d_tmp, H + 1));
  ISX_TRY(h, cudaMemcpy(d_tmp, m.inverse_height.data(), sizeof(float) * (H + 1), cudaMemcpyHostToDevice));
  b.inverse_height = d_tmp;

  ISX_TRY(h, cudaMallocHost(&h->h_ground, sizeof(float) * kStageSlots * ch * 3 * H));
  ISX_TRY(h, cudaMallocHost(&h->h_vhor, sizeof(int) * kStageSlots * ch));
  for (int i = 0; i < kStageSlots; i++) ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_stage_done[i], cudaEventDisableTiming));
  h->stage_next = 0;
  h->road_cache.clear();
  h->overlap_tables = true;
  if (const char *e = std::getenv("ISX_OVERLAP_TABLES")) h->overlap_tables = std::atoi(e) != 0;
  h->initialized = true;
  h->last_batch = 0;
  return ISX_OK;
}

int isx_finish(isx_handle h) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  if (!h->initialized) return ISX_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (void *p : h->allocations) cudaFree(p);
  h->allocations.clear();
  cudaFreeHost(h->h_ground);
  cudaFreeHost(h->h_vhor);
  for (int i = 0; i < kStageSlots; i++) {
    if (h->ev_stage_done[i]) cudaEventDestroy(h->ev_stage_done[i]);
    h->ev_stage_done[i] = nullptr;
  }
  for (int i = 0; i < kRoadSlots; i++) {
    if (h->roads[i].ev_free) cudaEventDestroy(h->roads[i].ev_free);
    h->roads[i] = isx_context::RoadSlot();
  }
  for (int i = 0; i < kResultSets; i++) {
    isx_context::ResultSet &R = h->rs[i];
    if (R.allocated) {
      cudaFreeHost(R.h_sections);
      cudaFreeHost(R.h_inst);
      cudaFreeHost(R.h_counts);
      cudaFreeHost(R.h_frames);
    }
    R = isx_context::ResultSet();
    if (h->ev_batch_done[i]) cudaEventDestroy(h->ev_batch_done[i]);
    h->ev_batch_done[i] = nullptr;
    h->batch_sections[i] = nullptr;
    h->batch_n[i] = 0;
  }
  for (int i = 0; i < 2; i++) {
    h->d_in_disp16[i] = nullptr;
    h->d_in_seg16[i] = nullptr;
  }
  h->cur = 0;
  h->submitted = h->waited = 0;
  h->last_waited_set = -1;
  h->host_slot = 0;
  h->dp_units_total = h->dp_units_pairwise = 0;
  h->emit_join_pending = false;
  for (int i = 0; i < 2; i++) {
    cudaEventDestroy(h->ev_in_ready[i]);
    cudaEventDestroy(h->ev_in_free[i]);
    cudaEventDestroy(h->ev_dp_done[i]);
    cudaEventDestroy(h->ev_emit_done[i]);
    cudaEventDestroy(h->ev_tab_done[i]);
  }
  cudaEventDestroy(h->ev_chunk_done);
  cudaEventDestroy(h->ev_user);
  cudaStreamDestroy(h->s_tables);
  cudaStreamDestroy(h->s_compute);
  cudaStreamDestroy(h->s_emit);
  cudaStreamDestroy(h->s_h2d);
  cudaStreamDestroy(h->s_d2h);
  h->buf = BatchBuffers();
  h->initialized = false;
  return ISX_OK;
}

int isx_is_initialized(isx_handle h) { return h && h->initialized; }
int isx_real_cols(isx_handle h) { return h ? (h->initialized ? h->kp.realcols : 0) : 0; }
int isx_max_sections(isx_handle h) { (void)h; return kMaxSections; }
size_t isx_segmentation_elems(isx_handle h) { return (h && h->initialized) ? seg_elems(h) : 0; }

int isx_set_disparity_image(isx_handle h, const float *host, size_t n) {
  if (int rc = check_ready(h)) return rc;
  if (!host || n != (size_t)h->kp.rows * h->kp.cols)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "disparity image must hold rows*cols floats");
  ISX_TRY(h, cudaMemcpyAsync(h->d_single_disp, host, n * sizeof(float), cudaMemcpyHostToDevice, h->s_tables));
  return ISX_OK;
}

float *isx_input_disparity_device(isx_handle h) {
  if (!h || !h->initialized) return nullptr;
  // the caller hands the pointer to its own kernels (RoadEstimation::Compute(pixel_t *d_im), RoadEstimation.cu:107):
  // the image SetDisparityImage is still copying must have arrived
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->s_tables);
  return h->d_single_disp;
}

int isx_set_segmentation(isx_handle h, const int32_t *host, size_t n) {
  if (int rc = check_ready(h)) return rc;
  if (!host || n != seg_elems(h))
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "segmentation must hold realcols*channels*rows_power2_segmentation ints");
  ISX_TRY(h, cudaMemcpyAsync(h->d_single_seg, host, n * sizeof(int32_t), cudaMemcpyHostToDevice, h->s_tables));
  return ISX_OK;
}

// FlipAndPad on the device (ingest.cu).  The CNN grid is [channels][rows/8][cols/8]; width_margin must be 0 and
// column_step must divide 8, as in every configuration the reference ships.
static int check_cnn_grid(isx_handle h, int cnn_rows, int cnn_cols) {
  const KParams &kp = h->kp;
  if (kp.width_margin != 0 || kp.column_step < 1 || kDownsample % kp.column_step != 0)
    return fail(h, ISX_ERR_UNSUPPORTED, "segmentation ingest needs width_margin == 0 and column_step dividing 8");
  if (cnn_rows != kp.rows / kDownsample || cnn_cols * (kDownsample / kp.column_step) != kp.realcols)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "CNN output must be [channels][rows/8][cols/8]");
  return ISX_OK;
}

int isx_set_segmentation_from_cnn_device(isx_handle h, const float *d_cnn, int cnn_rows, int cnn_cols) {
  if (int rc = check_ready(h)) return rc;
  if (!d_cnn) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  if (int rc = check_cnn_grid(h, cnn_rows, cnn_cols)) return rc;
  launch_flip_and_pad(h->kp, d_cnn, h->d_single_seg, 1, cnn_rows, cnn_cols, h->s_tables);
  ISX_TRY(h, cudaGetLastError());
  return ISX_OK;
}

int isx_flip_and_pad_batch_device(isx_handle h, int n, const float *d_cnn, int cnn_rows, int cnn_cols,
                                  int32_t *d_segmentation) {
  if (int rc = check_ready(h)) return rc;
  if (!d_cnn || !d_segmentation || n < 1) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument or empty batch");
  if (int rc = check_cnn_grid(h, cnn_rows, cnn_cols)) return rc;
  launch_flip_and_pad(h->kp, d_cnn, d_segmentation, n, cnn_rows, cnn_cols, h->s_tables);
  ISX_TRY(h, cudaGetLastError());
  return ISX_OK;
}

int isx_set_road_parameters(isx_handle h, int vhor, float camera_tilt, float camera_height, float alpha_ground) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  h->single_road = isx_road{vhor, camera_tilt, camera_height, alpha_ground};
  h->single_has_road = true;
  return ISX_OK;
}

static int no_batches_in_flight(isx_handle h);

// Hands the results of n frames of result set R to the caller: the packed Sections are expanded into the caller's
// padded [n][C][200] array (used entries + the type == -1 terminator of every column; entries behind a terminator
// are not touched, like the reference's d_stixels, StixelsKernels.cu:951-955), the instance records are copied
// frame after frame.  Everything comes from pinned host memory the device has already written (the caller has
// waited for the emission stream); only a frame that did not fit the packed arrays costs a device -> host copy.
// Returns the first per-frame error AFTER delivering what there is.
static int deliver(isx_handle h, isx_context::ResultSet &R, int n, isx_section *sections, isx_instance *instances,
                   int instances_capacity, int32_t *instance_offsets, bool direct = false) {
  if (direct) sections = nullptr;   // the device has written the caller's array itself
  const size_t C = h->kp.realcols;
  int rc = ISX_OK;
  int total = 0;
  for (int f = 0; f < n; f++) {
    const isx_packed_frame &d = R.h_frames[f];
    if (d.error && rc == ISX_OK) {
      char msg[160];
      if (d.error & kErrOffsetRange) {
        std::snprintf(msg, sizeof msg, "frame %d: instance offsets out of range: |sum of instance means| of a column "
                      "must stay below 2^24", f);
        rc = fail(h, ISX_ERR_UNSUPPORTED, msg);
      } else {
        std::snprintf(msg, sizeof msg, "frame %d: a column produced >= 200 stixels (MAX_STIXELS_PER_COLUMN)", f);
        rc = fail(h, ISX_ERR_CAPACITY, msg);
      }
    }
    if (sections) {
      isx_section *dst = sections + (size_t)f * C * kMaxSections;
      if (d.overflow & 1) {
        ISX_TRY(h, cudaMemcpy(dst, R.d_sections + (size_t)f * C * kMaxSections, sizeof(isx_section) * C * kMaxSections,
                              cudaMemcpyDeviceToHost));
      } else {
        const isx_section *src = R.h_sections + d.section_offset;
        const int *cnt = R.h_counts + (size_t)f * C;
        isx_section term;
        term.type = -1;
        term.vB = term.vT = 0;
        term.disparity = term.cost = term.instance_meanx = term.instance_meany = 0.0f;
        term.semantic_class = 0;
        for (size_t c = 0; c < C; c++) {
          const int k = cnt[c];
          std::memcpy(dst + c * kMaxSections, src, sizeof(isx_section) * (size_t)k);
          dst[c * kMaxSections + k] = term;
          src += k;
        }
      }
    }
    if (instance_offsets) instance_offsets[f] = total;
    if (instances) {
      const int room = instances_capacity - total;
      const int take = d.instance_count < room ? d.instance_count : (room > 0 ? room : 0);
      if (take > 0) {
        if (d.overflow & 2)
          ISX_TRY(h, cudaMemcpy(instances + total, R.d_inst + (size_t)f * h->inst_cap, sizeof(isx_instance) * take,
                                cudaMemcpyDeviceToHost));
        else
          std::memcpy(instances + total, R.h_inst + d.instance_offset, sizeof(isx_instance) * (size_t)take);
      }
    }
    total += d.instance_count;
  }
  if (instance_offsets) instance_offsets[n] = total;
  return rc;
}

// Waits until the results of the last enqueued batch are in host memory.
static int wait_last_emission(isx_handle h) {
  ISX_TRY(h, cudaEventSynchronize(h->ev_emit_done[h->last_set]));
  return ISX_OK;
}

int isx_compute(isx_handle h, int pairwise, isx_section *sections, isx_frame_meta *meta,
                const int32_t *d_segmentation_local) {
  if (int rc = check_ready(h)) return rc;
  if (!h->single_has_road) return fail(h, ISX_ERR_INVALID_ARGUMENT, "SetRoadParameters has not been called");
  if (int rc = no_batches_in_flight(h)) return rc;
  const int32_t *seg = d_segmentation_local ? d_segmentation_local : h->d_single_seg;
  if (int rc = begin_batch(h)) return rc;
  h->direct_sections = device_view_of(sections);
  const bool direct = h->direct_sections != nullptr;
  const int erc = enqueue_chunk(h, pairwise != 0, 0, 1, h->d_single_disp, seg, &h->single_road, 0);
  h->direct_sections = nullptr;
  if (erc) return erc;
  ISX_TRY(h, cudaEventRecord(h->ev_in_free[0], h->s_tables));
  if (int rc = join_emit_stream(h)) return rc;
  h->last_batch = 1;
  h->last_roads.assign(1, h->single_road);
  if (int rc = wait_last_emission(h)) return rc;
  if (int rc = deliver(h, h->rs[h->cur], 1, sections, nullptr, 0, nullptr, direct)) return rc;
  if (meta) {
    meta->rows = h->kp.rows; meta->cols = h->kp.cols; meta->realcols = h->kp.realcols;
    meta->max_sections = kMaxSections; meta->max_dis = h->kp.max_dis; meta->column_step = h->kp.column_step;
    meta->semantic_classes = h->kp.n_classes; meta->alpha_ground = h->single_road.alpha_ground;
    meta->vhor = h->kp.rows - h->single_road.vhor - 1;
  }
  return ISX_OK;
}

int isx_cluster_instances(isx_handle h) { return check_ready(h); }

int isx_dbscan_fit_host(int device, const float *xy, int n, float eps, int min_pts,
                        const unsigned char *core_candidates, int *labels) {
  if (n < 0 || (n > 0 && (!xy || !core_candidates || !labels)))
    return fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "isx_dbscan_fit_host: null argument");
  if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, ISX_ERR_CUDA, "isx_dbscan_fit_host: no such CUDA device");
  // both launch shapes of the kernel (ISX_GROUP_THREADS=256: the batch shape; default: the single-frame shape)
  const char *e = std::getenv("ISX_GROUP_THREADS");
  if (isx::dbscan_fit_host(xy, n, eps, min_pts, core_candidates, labels, e ? std::atoi(e) : 1024) != 0)
    return fail(nullptr, ISX_ERR_CUDA, "isx_dbscan_fit_host: CUDA error");
  return ISX_OK;
}

int isx_get_instance_stixels(isx_handle h, isx_instance *out, int capacity, int *n) {
  if (int rc = check_ready(h)) return rc;
  if (h->last_batch < 1) return fail(h, ISX_ERR_INVALID_ARGUMENT, "Compute has not been called");
  if (int rc = no_batches_in_flight(h)) return rc;
  if (int rc = wait_last_emission(h)) return rc;
  int32_t offs[2] = {0, 0};
  if (int rc = deliver(h, h->rs[h->cur], 1, nullptr, out, out ? capacity : 0, offs)) return rc;
  if (n) *n = offs[1];
  return ISX_OK;
}

int isx_compute_batch_device(isx_handle h, int pairwise, int n, const float *d_disparity,
                             const int32_t *d_segmentation, const isx_road *roads) {
  if (int rc = check_ready(h)) return rc;
  if (int rc = no_batches_in_flight(h)) return rc;
  if (n < 1 || n > h->max_batch) return fail(h, ISX_ERR_CAPACITY, "batch size exceeds isx_initialize(max_batch)");
  if (!d_disparity || !d_segmentation || !roads) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  const size_t hw = (size_t)h->kp.rows * h->kp.cols, se = seg_elems(h);
  int slot = h->host_slot;  // keeps alternating across batches (see enqueue_host_batch)
  if (int rc = begin_batch(h)) return rc;
  const int chunk = pairwise ? h->chunk : h->chunk_unary;
  h->last_launch_frames = chunk;
  for (int first = 0; first < n; first += chunk) {
    const int cn = (n - first) < chunk ? (n - first) : chunk;
    h->results_stay_on_device = true;
    const int erc = enqueue_chunk(h, pairwise != 0, first, cn, d_disparity + first * hw, d_segmentation + first * se,
                                  roads + first, slot);
    h->results_stay_on_device = false;
    if (erc) return erc;
    ISX_TRY(h, cudaEventRecord(h->ev_in_free[slot], h->s_tables));
    slot ^= 1;
  }
  h->host_slot = slot;
  h->emit_join_pending = true;  // joined lazily: isx_flush / isx_synchronize / any result access
  h->last_batch = n;
  h->last_roads.assign(roads, roads + n);
  return ISX_OK;
}

int isx_flush(isx_handle h) {
  if (int rc = check_ready(h)) return rc;
  return ensure_joined(h);
}

int isx_synchronize(isx_handle h) {
  if (int rc = check_ready(h)) return rc;
  if (int rc = ensure_joined(h)) return rc;
  ISX_TRY(h, cudaStreamSynchronize(h->s_tables));
  return ISX_OK;
}

int isx_fetch_batch_results(isx_handle h, int n, isx_section *sections, isx_instance *instances,
                            int instances_capacity, int32_t *instance_offsets) {
  if (int rc = check_ready(h)) return rc;
  if (n < 1 || n > h->last_batch) return fail(h, ISX_ERR_INVALID_ARGUMENT, "no results for that many frames");
  if (int rc = no_batches_in_flight(h)) return rc;
  if (int rc = ensure_joined(h)) return rc;
  if (int rc = wait_last_emission(h)) return rc;
  return deliver(h, h->rs[h->cur], n, sections, instances, instances_capacity, instance_offsets);
}

// Host inputs of one batch: the reference's types (float disparity, int32 segmentation with its padding), or the
// narrow forms of the isx_*_u16 entry points.
struct HostInputs {
  const float *disparity = nullptr;
  const int32_t *segmentation = nullptr;
  const uint16_t *disparity16 = nullptr;
  float scale = 0.0f;
  const int16_t *segmentation16 = nullptr;
  bool narrow() const { return disparity16 != nullptr; }
};

static size_t narrow_seg_elems(const isx_context *c) {
  const size_t used = (size_t)(c->kp.rows + kDownsample - 1) / kDownsample;
  return (size_t)c->kp.realcols * c->kp.n_channels * (used < (size_t)c->kp.hs2 ? used : (size_t)c->kp.hs2);
}

static int ensure_narrow_staging(isx_handle h) {
  if (h->d_in_disp16[0]) return ISX_OK;
  const size_t hw = (size_t)h->kp.rows * h->kp.cols, ch = h->chunk;
  for (int i = 0; i < 2; i++) {
    ISX_TRY(h, dev_alloc(h, &h->d_in_disp16[i], ch * hw));
    ISX_TRY(h, dev_alloc(h, &h->d_in_seg16[i], ch * narrow_seg_elems(h)));
  }
  return ISX_OK;
}

// The copy/kernel pipeline of one host batch: H2D on s_h2d, kernels on s_compute / s_emit; the results reach host
// memory through pack_results_kernel (no D2H copies).  Blocks the caller only for the reuse of an input slot (two
// chunks behind).
// `caller_waits`: a synchronous call -- the kernels of the last chunk run with nothing beside them while the caller
// waits, so the tail goes in quarter pieces like the head.
static int enqueue_host_batch(isx_handle h, int pairwise, int n, const HostInputs &in, const isx_road *roads,
                              bool caller_waits) {
  const size_t hw = (size_t)h->kp.rows * h->kp.cols, se = seg_elems(h), se16 = narrow_seg_elems(h);
  if (in.narrow()) {
    if (hw % 8 != 0) return fail(h, ISX_ERR_UNSUPPORTED, "the uint16 disparity path needs rows*cols to be a multiple of 8");
    if (int rc = ensure_narrow_staging(h)) return rc;
  }
  if (int rc = begin_batch(h)) return rc;
  // The slots keep alternating across batches, so that the first copy of a pipelined batch only waits for the
  // second-to-last chunk of the batch before it.
  int slot = h->host_slot;
  int cn = 0;
  const int chunk = pairwise ? h->chunk : h->chunk_unary;
  h->last_launch_frames = chunk;
  const bool pipeline_idle = h->submitted == h->waited;
  for (int first = 0; first < n; first += cn) {
    cn = (n - first) < chunk ? (n - first) : chunk;
    // Nothing is running: no kernel hides the input copies, so the first `chunk` frames go in quarter pieces and the
    // kernels of a piece run under the copy of the next (a synchronous 64-frame pairwise call: copy 13 ms + tables and
    // DP of the last piece instead of copy + tables and DP of all 64 frames); likewise the last `chunk` frames of a
    // call whose caller waits.  The shorter launches cost the DP a few per cent -- in between, and once the pipeline
    // of a streaming caller is filled, launches are whole chunks.
    const bool head = pipeline_idle && first < chunk, tail = caller_waits && n - first <= chunk;
    if ((head || tail) && chunk >= 32) cn = cn < chunk / 4 ? cn : chunk / 4;
    // H2D of this chunk on the copy stream, once the table build that last read this input slot is done (a
    // device-side wait: the host thread runs ahead)
    ISX_TRY(h, cudaStreamWaitEvent(h->s_h2d, h->ev_in_free[slot], 0));
    auto mark_h2d = [&]() {
      if (!h->profiling) return;
      if (h->prof_h2d_used >= h->prof_h2d.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->prof_h2d.push_back(e);
      }
      cudaEventRecord(h->prof_h2d[h->prof_h2d_used++], h->s_h2d);
    };
    mark_h2d();
    const int road_slot = stage_road_tables(h, roads + first, cn, h->s_h2d);
    if (road_slot < 0) return road_slot;
    if (in.narrow()) {
      ISX_TRY(h, cudaMemcpyAsync(h->d_in_disp16[slot], in.disparity16 + first * hw, sizeof(uint16_t) * hw * cn,
                                 cudaMemcpyHostToDevice, h->s_h2d));
      ISX_TRY(h, cudaMemcpyAsync(h->d_in_seg16[slot], in.segmentation16 + first * se16, sizeof(int16_t) * se16 * cn,
                                 cudaMemcpyHostToDevice, h->s_h2d));
    } else {
      ISX_TRY(h, cudaMemcpyAsync(h->d_in_disp[slot], in.disparity + first * hw, sizeof(float) * hw * cn,
                                 cudaMemcpyHostToDevice, h->s_h2d));
      // Only the first rows/8 entries of every [rows_power2_segmentation] channel row are ever read
      // (StixelsKernels.cu:393-405, 462-468 index v/8 with v < rows); the zero padding of FlipAndPad does not
      // travel: a 2-D copy of the used part, the rest of the staging buffer stays zero from isx_initialize.
      const size_t hs2 = (size_t)h->kp.hs2;
      size_t used = (size_t)(h->kp.rows + kDownsample - 1) / kDownsample;
      used = used < hs2 ? used : hs2;
      ISX_TRY(h, cudaMemcpy2DAsync(h->d_in_seg[slot], hs2 * sizeof(int32_t), in.segmentation + first * se,
                                   hs2 * sizeof(int32_t), used * sizeof(int32_t), (se / hs2) * cn,
                                   cudaMemcpyHostToDevice, h->s_h2d));
    }
    mark_h2d();
    ISX_TRY(h, cudaEventRecord(h->ev_in_ready[slot], h->s_h2d));
    ISX_TRY(h, cudaStreamWaitEvent(h->s_tables, h->ev_in_ready[slot], 0));
    if (in.narrow())
      launch_widen_inputs(h->kp, h->d_in_disp16[slot], in.scale, h->d_in_seg16[slot], h->d_in_disp[slot],
                          h->d_in_seg[slot], cn, h->s_tables);
    if (int rc = enqueue_chunk(h, pairwise != 0, first, cn, h->d_in_disp[slot], h->d_in_seg[slot], roads + first,
                               slot, road_slot))
      return rc;
    ISX_TRY(h, cudaEventRecord(h->ev_in_free[slot], h->s_tables));   // the inputs are read by the table build only
    slot ^= 1;
  }
  h->host_slot = slot;
  h->last_batch = n;
  h->last_roads.assign(roads, roads + n);
  return ISX_OK;
}

static int no_batches_in_flight(isx_handle h) {
  if (h->submitted != h->waited)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "submitted batches are in flight: call isx_wait_batch_host first");
  return ISX_OK;
}

static int compute_batch_host(isx_handle h, int pairwise, int n, const HostInputs &in, const isx_road *roads,
                              isx_section *sections, isx_instance *instances, int instances_capacity,
                              int32_t *instance_offsets) {
  if (int rc = check_ready(h)) return rc;
  if (int rc = no_batches_in_flight(h)) return rc;
  if (n < 1 || n > h->max_batch) return fail(h, ISX_ERR_CAPACITY, "batch size exceeds isx_initialize(max_batch)");
  if (!roads) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  h->direct_sections = device_view_of(sections);
  const bool direct = h->direct_sections != nullptr;
  const int erc = enqueue_host_batch(h, pairwise, n, in, roads, /*caller_waits=*/true);
  h->direct_sections = nullptr;
  if (erc) return erc;
  if (int rc = join_emit_stream(h)) return rc;
  if (int rc = wait_last_emission(h)) return rc;
  return deliver(h, h->rs[h->cur], n, sections, instances, instances_capacity, instance_offsets, direct);
}

int isx_compute_batch_host(isx_handle h, int pairwise, int n, const float *disparity, const int32_t *segmentation,
                           const isx_road *roads, isx_section *sections, isx_instance *instances,
                           int instances_capacity, int32_t *instance_offsets) {
  if (!disparity || !segmentation) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  HostInputs in;
  in.disparity = disparity;
  in.segmentation = segmentation;
  return compute_batch_host(h, pairwise, n, in, roads, sections, instances, instances_capacity, instance_offsets);
}

int isx_compute_batch_host_u16(isx_handle h, int pairwise, int n, const uint16_t *disparity, float disparity_scale,
                               const int16_t *segmentation, const isx_road *roads, isx_section *sections,
                               isx_instance *instances, int instances_capacity, int32_t *instance_offsets) {
  if (!disparity || !segmentation) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  HostInputs in;
  in.disparity16 = disparity;
  in.scale = disparity_scale;
  in.segmentation16 = segmentation;
  return compute_batch_host(h, pairwise, n, in, roads, sections, instances, instances_capacity, instance_offsets);
}

size_t isx_narrow_segmentation_elems(isx_handle h) { return (h && h->initialized) ? narrow_seg_elems(h) : 0; }

static int submit_batch_host(isx_handle h, int pairwise, int n, const HostInputs &in, const isx_road *roads,
                             isx_section *sections) {
  if (int rc = check_ready(h)) return rc;
  if (n < 1 || n > h->max_batch) return fail(h, ISX_ERR_CAPACITY, "batch size exceeds isx_initialize(max_batch)");
  if (!roads) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  if (h->submitted - h->waited >= (unsigned long long)(kResultSets - 1))
    return fail(h, ISX_ERR_CAPACITY, "three batches are already in flight: call isx_wait_batch_host first");
  int next = 0;
  {
    bool busy[kResultSets] = {};
    for (unsigned long long t = h->waited; t < h->submitted; t++) busy[h->batch_set[t % kResultSets]] = true;
    if (h->last_waited_set >= 0) busy[h->last_waited_set] = true;  // its packed arrays may still be read
    while (busy[next]) next++;
  }
  if (int rc = alloc_result_set(h, next)) return rc;
  for (int i = 0; i < kResultSets; i++)
    if (!h->ev_batch_done[i]) ISX_TRY(h, cudaEventCreateWithFlags(&h->ev_batch_done[i], cudaEventDisableTiming));
  h->cur = next;
  h->direct_sections = device_view_of(sections);
  const bool direct = h->direct_sections != nullptr;
  const int erc = enqueue_host_batch(h, pairwise, n, in, roads, /*caller_waits=*/false);
  h->direct_sections = nullptr;
  if (erc) return erc;
  const int par = (int)(h->submitted % kResultSets);
  h->batch_direct[par] = direct;
  ISX_TRY(h, cudaEventRecord(h->ev_batch_done[par], h->s_emit));  // behind the packing of the last chunk
  h->batch_n[par] = n;
  h->batch_set[par] = h->cur;
  h->batch_sections[par] = sections;
  h->submitted++;
  h->emit_join_pending = true;  // isx_stream() itself has not been ordered behind the emission stream
  return ISX_OK;
}

int isx_submit_batch_host(isx_handle h, int pairwise, int n, const float *disparity, const int32_t *segmentation,
                          const isx_road *roads, isx_section *sections) {
  if (!disparity || !segmentation) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  HostInputs in;
  in.disparity = disparity;
  in.segmentation = segmentation;
  return submit_batch_host(h, pairwise, n, in, roads, sections);
}

int isx_submit_batch_host_u16(isx_handle h, int pairwise, int n, const uint16_t *disparity, float disparity_scale,
                              const int16_t *segmentation, const isx_road *roads, isx_section *sections) {
  if (!disparity || !segmentation) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null argument");
  HostInputs in;
  in.disparity16 = disparity;
  in.scale = disparity_scale;
  in.segmentation16 = segmentation;
  return submit_batch_host(h, pairwise, n, in, roads, sections);
}

int isx_reserve_in_flight(isx_handle h, int batches) {
  if (int rc = check_ready(h)) return rc;
  if (batches < 1 || batches > kResultSets - 1)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "isx_reserve_in_flight: between one and three batches");
  cudaSetDevice(h->device);
  for (int i = 0; i <= batches && i < kResultSets; i++)
    if (int rc = alloc_result_set(h, i)) return rc;
  return ISX_OK;
}

// Waits for the oldest batch in flight; returns its ticket slot (>= 0) or an error (< 0).
static int wait_oldest(isx_handle h) {
  if (int rc = check_ready(h)) return rc;
  if (h->submitted == h->waited) return fail(h, ISX_ERR_INVALID_ARGUMENT, "no submitted batch is in flight");
  const int par = (int)(h->waited % kResultSets);
  ISX_TRY(h, cudaEventSynchronize(h->ev_batch_done[par]));
  h->last_waited_set = h->batch_set[par];
  h->waited++;
  return par;
}

int isx_wait_batch_host(isx_handle h, isx_instance *instances, int instances_capacity, int32_t *instance_offsets) {
  const int par = wait_oldest(h);
  if (par < 0) return par;
  const int n = h->batch_n[par];
  h->batch_n[par] = 0;
  return deliver(h, h->rs[h->batch_set[par]], n, h->batch_sections[par], instances, instances_capacity,
                 instance_offsets, h->batch_direct[par]);
}

int isx_wait_batch_packed(isx_handle h, const isx_section **sections, const int32_t **counts,
                          const isx_instance **instances, const isx_packed_frame **frames, int *n) {
  const int par = wait_oldest(h);
  if (par < 0) return par;
  const isx_context::ResultSet &R = h->rs[h->batch_set[par]];
  if (sections) *sections = R.h_sections;
  if (counts) *counts = R.h_counts;
  if (instances) *instances = R.h_inst;
  if (frames) *frames = R.h_frames;
  if (n) *n = h->batch_n[par];
  int rc = ISX_OK;
  for (int f = 0; f < h->batch_n[par] && rc == ISX_OK; f++) {
    if (R.h_frames[f].error & kErrOffsetRange) rc = fail(h, ISX_ERR_UNSUPPORTED, "instance offsets out of range in a frame of the batch");
    else if (R.h_frames[f].error) rc = fail(h, ISX_ERR_CAPACITY, "a column produced >= 200 stixels (MAX_STIXELS_PER_COLUMN)");
  }
  h->batch_n[par] = 0;
  return rc;
}

int isx_rasterize_batch_device(isx_handle h, int first, int n, uint8_t *d_label_ids, int32_t *d_instance_ids,
                               float *d_disparity) {
  if (int rc = check_ready(h)) return rc;
  if (first < 0 || n < 1 || first + n > h->last_batch)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "frames outside the last computed batch");
  if (!d_label_ids && !d_instance_ids && !d_disparity) return fail(h, ISX_ERR_INVALID_ARGUMENT, "no output image");
  if (int rc = ensure_joined(h)) return rc;
  const size_t C = h->kp.realcols;
  const isx_context::ResultSet &R = h->rs[h->cur];
  launch_rasterize(h->kp, R.d_sections + (size_t)first * C * kMaxSections, R.d_nsections + (size_t)first * C,
                   R.d_inst + (size_t)first * h->inst_cap, R.d_inst_count + first, h->inst_cap,
                   h->d_raster_table, n, d_label_ids, d_instance_ids, d_disparity, h->s_tables);
  ISX_TRY(h, cudaGetLastError());
  return ISX_OK;
}

// Reads result set rs[cur] on s_tables.  A later batch cannot overwrite it underneath: every kernel of a batch queues
// behind the table build of its first chunk on s_tables (the DP waits for ev_tab_done, the emission for ev_dp_done),
// so it starts after whatever was enqueued here.
int isx_export_batch_device(isx_handle h, int first, int n, const isx_device_results *out) {
  if (int rc = check_ready(h)) return rc;
  if (first < 0 || n < 1 || first + n > h->last_batch)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "frames outside the last computed batch");
  if (!out || !out->frame_offsets) return fail(h, ISX_ERR_INVALID_ARGUMENT, "frame_offsets is required");
  if ((uintptr_t)out->sections % 16 != 0)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "sections must be 16-byte aligned");
  if (out->capacity < 0) return fail(h, ISX_ERR_INVALID_ARGUMENT, "capacity must be >= 0");
  const HostModel &m = h->model;
  if (out->vertices && (m.camera_center_x == -1 || m.camera_center_y == -1))
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "Camera parameters are not set.");  // Get3DVertices (Stixels.cu:685-687)
  if (int rc = no_batches_in_flight(h)) return rc;
  if (int rc = ensure_joined(h)) return rc;
  const size_t C = h->kp.realcols;
  const isx_context::ResultSet &R = h->rs[h->cur];
  ExportArgs a;
  a.sections = R.d_sections + (size_t)first * C * kMaxSections;
  a.n_sections = R.d_nsections + (size_t)first * C;
  a.inst = R.d_inst + (size_t)first * h->inst_cap;
  a.inst_count = R.d_inst_count + first;
  a.inst_cap = h->inst_cap;
  a.frames = R.m_frames + first;
  a.col_local = h->d_export_col;
  a.realcols = h->kp.realcols;
  a.rows = h->kp.rows;
  a.column_step = h->kp.column_step;
  a.focal = m.focal;
  a.bf = m.baseline * m.focal;
  a.camera_center_x = m.camera_center_x;
  a.camera_center_y = m.camera_center_y;
  a.out = *out;
  std::vector<float> alpha((size_t)n);
  std::vector<int> vhor((size_t)n);
  for (int f = 0; f < n; f++) {
    alpha[f] = h->last_roads[first + f].alpha_ground;
    vhor[f] = h->kp.rows - h->last_roads[first + f].vhor - 1;   // isx_frame_meta.vhor (Stixels.cu:377)
  }
  launch_export_results(a, n, alpha.data(), vhor.data(), h->s_tables);
  ISX_TRY(h, cudaGetLastError());
  return ISX_OK;
}

uint64_t isx_stream(isx_handle h) { return (h && h->initialized) ? (uint64_t)(uintptr_t)h->s_tables : 0; }

size_t isx_tensor_elems(isx_handle h, int tensor) {
  if (!h || !h->initialized) return 0;
  const size_t H = h->kp.rows, C = h->kp.realcols, D = h->kp.max_dis;
  switch (tensor) {
    case ISX_T_JOINED_DISPARITY: return C * H;
    case ISX_T_OBJECT_LUT: return C * D * (H + 1);
    case ISX_T_DISPARITY_PS:
    case ISX_T_VALID_PS:
    case ISX_T_GROUND_PS:
    case ISX_T_SKY_PS: return C * (H + 1);
    case ISX_T_COST_TABLE:
    case ISX_T_INDEX_TABLE: return C * H * 3;
    case ISX_T_GROUND_TABLES: return 3 * H;
    case ISX_T_OBJ_COST_LUT: return D * D;
    case ISX_T_OBJECT_DISPARITY_RANGE: return D;
    default: return 0;
  }
}

int isx_read_tensor(isx_handle h, int tensor, int frame, void *host, size_t bytes) {
  if (int rc = check_ready(h)) return rc;
  const size_t need = isx_tensor_elems(h, tensor) * 4;
  if (need == 0 || !host || bytes < need) return fail(h, ISX_ERR_INVALID_ARGUMENT, "bad tensor id or buffer too small");
  const int local = frame - h->last_chunk_first;
  if (local < 0 || local >= h->last_chunk_n)
    return fail(h, ISX_ERR_INVALID_ARGUMENT, "intermediates are only kept for the last chunk of the last batch");
  if (int rc = ensure_joined(h)) return rc;
  ISX_TRY(h, cudaStreamSynchronize(h->s_tables));
  ISX_TRY(h, cudaStreamSynchronize(h->s_compute));
  const KParams &kp = h->kp;
  const size_t H = kp.rows, C = kp.realcols, D = kp.max_dis;
  BatchBuffers b = h->buf;
  {
    const isx_context::ChunkSet &cs = h->sets[h->last_set];
    b.ground = h->roads[h->last_road_slot].ground; b.vhor = h->roads[h->last_road_slot].vhor; b.stat = cs.stat;
    b.records_b = cs.records_b; b.dp = cs.dp; b.pm = cs.pm;
    b.joined = cs.joined; b.object_lut = cs.object_lut; b.col_flags = cs.col_flags;
  }
  if (tensor == ISX_T_GROUND_TABLES) {
    ISX_TRY(h, cudaMemcpy(host, b.ground + (size_t)local * 3 * H, need, cudaMemcpyDeviceToHost));
  } else if (tensor == ISX_T_OBJ_COST_LUT) {
    ISX_TRY(h, cudaMemcpy(host, b.obj_cost_lut, need, cudaMemcpyDeviceToHost));
  } else if (tensor == ISX_T_OBJECT_DISPARITY_RANGE) {
    ISX_TRY(h, cudaMemcpy(host, b.object_disparity_range, need, cudaMemcpyDeviceToHost));
  } else if (tensor == ISX_T_JOINED_DISPARITY) {
    ISX_TRY(h, cudaMemcpy(host, b.joined + (size_t)local * C * H, need, cudaMemcpyDeviceToHost));
  } else if (tensor == ISX_T_OBJECT_LUT) {
    // device rows hold LUT[fn][1..H]; the reference layout has a leading 0 (StixelsKernels.cu:283-285)
    float *dst = static_cast<float *>(host);
    for (size_t r = 0; r < C * D; r++) dst[r * (H + 1)] = 0.0f;
    for (size_t col = 0; col < C; col++) {
      const void *src = reinterpret_cast<const void *>(lut_column_address(
          (unsigned long long)b.object_lut, (size_t)local * C + col, kp.lut_cols, D * (size_t)kp.lut_stride * 4));
      ISX_TRY(h, cudaMemcpy2D(dst + 1 + col * D * (H + 1), (H + 1) * 4, src, (size_t)kp.lut_stride * 4, H * 4, D,
                              cudaMemcpyDeviceToHost));
    }
  } else if (tensor >= ISX_T_DISPARITY_PS && tensor <= ISX_T_SKY_PS) {
    const int word = tensor == ISX_T_DISPARITY_PS ? kRecDisp
                     : tensor == ISX_T_VALID_PS   ? kRecValid
                     : tensor == ISX_T_GROUND_PS  ? kRecGround
                                                  : kRecSky;
    // records [column][row][32 words] -> word `word` of rows 0 .. H of every column: [column][H+1]
    for (size_t col = 0; col < C; col++)
      ISX_TRY(h, cudaMemcpy2D(static_cast<float *>(host) + col * (H + 1), 4,
                              b.records_b + (((size_t)local * C + col) * kp.rec_stride) * kRecBWords + word,
                              (size_t)kRecBWords * 4, 4, H + 1, cudaMemcpyDeviceToHost));
  } else {
    launch_export_tables(kp, b, local, h->last_pairwise, h->d_export_cost, h->d_export_index, h->s_compute);
    ISX_TRY(h, cudaStreamSynchronize(h->s_compute));
    ISX_TRY(h, cudaMemcpy(host, tensor == ISX_T_COST_TABLE ? (void *)h->d_export_cost : (void *)h->d_export_index,
                          need, cudaMemcpyDeviceToHost));
  }
  return ISX_OK;
}

void *isx_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void isx_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

int isx_set_profiling(isx_handle h, int enable) {
  if (!h) return fail(h, ISX_ERR_INVALID_ARGUMENT, "null handle");
  h->profiling = enable != 0;
  return ISX_OK;
}

int isx_get_stage_times(isx_handle h, double *ms, long *chunks, int n_stages, int reset) {
  if (int rc = check_ready(h)) return rc;
  ISX_TRY(h, cudaStreamSynchronize(h->s_tables));
  ISX_TRY(h, cudaStreamSynchronize(h->s_compute));
  ISX_TRY(h, cudaStreamSynchronize(h->s_emit));
  // 9 events per chunk (enqueue_chunk): stages 0..2 = events i..i+1 on s_tables, stage 3 = events 4..5 on s_compute,
  // stages 4, 5 = events 6..8 on s_emit.  The table build of a chunk overlaps the DP of the chunk before it, so the
  // stage times of a stream of chunks add up to more than the wall time.
  const int per = kProfEvents;
  for (size_t base = 0; base + per <= h->prof_used; base += per) {
    for (int i = 0; i < 6; i++) {
      const int e0 = i < 3 ? i : i + 1;
      float t = 0.f;
      if (cudaEventElapsedTime(&t, h->prof_events[base + e0], h->prof_events[base + e0 + 1]) == cudaSuccess) {
        h->stage_ms[i] += t;
        h->stage_launches[i]++;
      }
    }
  }
  h->prof_used = 0;
  h->prof_h2d_used = 0;
  for (int i = 0; i < n_stages && i < 6; i++) {
    if (ms) ms[i] = h->stage_ms[i];
    if (chunks) chunks[i] = h->stage_launches[i];
  }
  if (reset)
    for (int i = 0; i < 8; i++) { h->stage_ms[i] = 0; h->stage_launches[i] = 0; }
  return ISX_OK;
}

// Developer trace of the host-batch pipeline (profiling enabled): per profiled chunk 11 time stamps in ms relative
// to the first one -- input copy begin | end (copy stream); join | frame tables | column tables | tables end (table
// stream); DP begin | DP end (compute stream); emission begin | grouping begin | emission end (emission stream).
// Returns the number of chunks written; call before isx_get_stage_times (which consumes the events).
int isx_get_chunk_trace(isx_handle h, double *ms, int max_chunks) {
  if (int rc = check_ready(h)) return rc;
  ISX_TRY(h, cudaStreamSynchronize(h->s_tables));
  ISX_TRY(h, cudaStreamSynchronize(h->s_compute));
  ISX_TRY(h, cudaStreamSynchronize(h->s_emit));
  ISX_TRY(h, cudaStreamSynchronize(h->s_h2d));
  const size_t chunks = std::min(h->prof_used / kProfEvents, h->prof_h2d_used / 2);
  int n = 0;
  if (chunks == 0) return 0;
  cudaEvent_t t0 = h->prof_h2d[0];
  for (size_t c = 0; c < chunks && n < max_chunks; c++, n++) {
    for (int i = 0; i < kTraceStamps; i++) {
      cudaEvent_t e = i < 2 ? h->prof_h2d[2 * c + i] : h->prof_events[kProfEvents * c + (i - 2)];
      float t = 0.f;
      cudaEventElapsedTime(&t, t0, e);
      ms[(size_t)n * kTraceStamps + i] = t;
    }
  }
  h->prof_h2d_used = 0;
  return n;
}

int isx_get_dp_units(isx_handle h, unsigned long long *evaluated, unsigned long long *total) {
  if (int rc = check_ready(h)) return rc;
  unsigned long long dev = 0;
  ISX_TRY(h, cudaStreamSynchronize(h->s_compute));
  ISX_TRY(h, cudaMemcpy(&dev, h->buf.dp_units, sizeof dev, cudaMemcpyDeviceToHost));
  if (evaluated) *evaluated = dev + h->dp_units_pairwise;
  if (total) *total = h->dp_units_total;
  return ISX_OK;
}
int isx_chunk_frames(isx_handle h) { return (h && h->initialized) ? h->last_launch_frames : 0; }
int isx_instance_capacity(isx_handle h) { return (h && h->initialized) ? h->inst_cap : 0; }

}  // extern "C"
