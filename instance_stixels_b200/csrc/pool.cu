// Frame pool: one context and one host worker thread per GPU inside one process (SURVEY.md 8e: "frame f -> GPU
// f*G/N, one host worker thread + >= 2 streams per GPU, pinned double-buffered staging").  Pure host code over the
// C ABI of context.cu -- the reference has no counterpart, its Compute() takes one frame on one GPU
// (InstanceStixels/src/Stixels.cu:449-637, frame loop apps/run_cityscapes.cu:249-449).
//
// A call shards its n frames into contiguous blocks, worker w OWNS frames [n*w/G, n*(w+1)/G) and streams them from the
// front through isx_submit_batch_host / isx_wait_batch_host in sub-batches of at most `max_batch` frames, three in
// flight.  A worker whose block is used up takes sub-batches from the BACK of the block with the most frames left: the
// GPUs of a box are not equally fast at this (measured on the 8-GPU VM of this pool: 20 GB/s of host-to-device copies
// for four of the GPUs, 35 GB/s for the others, and one GPU whose kernels run 8 % slower), and with fixed shards the
// call takes as long as the slowest of them.  Frames are independent, so there is no collective: every sub-batch
// writes its frames' Sections into the caller's array at their place; the instance records are concatenated in frame
// order when all workers are done.
//
// isx_pool_compute_host_road estimates the road of every frame on the device inside the same pipeline (the road step of
// isx_submit_batch_host_road): every worker owns a road handle on its GPU, created on the first such call.  A frame is
// computed with its OWN accepted estimate, else with the caller's fallback -- never with another frame's: which frames
// a worker sees, and in which order, depends on the schedule, so a keep-last rule would make the results depend on it.
#include <algorithm>
#include <condition_variable>
#include <deque>
#include <memory>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/instance_stixels_b200.h"

namespace isx {
// context.cu
int pool_submit_batch_host_road(isx_handle h, isx_road_handle road, int pairwise, int n, const float *disparity,
                                const int32_t *segmentation, const isx_road *fallback, isx_road_estimate *estimates,
                                isx_road *roads_out, isx_section *sections);
int largest_chunk(isx_handle h);
}  // namespace isx

namespace {

// One call's frames: per worker the part of its block nobody has taken yet.
struct Job {
  int pairwise = 0, n = 0;
  const float *disparity = nullptr;
  const int32_t *segmentation = nullptr;
  const isx_road *roads = nullptr;
  // road estimation on the device (isx_pool_compute_host_road): `roads` is null, these are set
  const isx_road *fallback = nullptr;
  isx_road_estimate *estimates = nullptr;
  isx_road *roads_out = nullptr;
  isx_section *sections = nullptr;
  bool want_instances = false;
  std::mutex m;
  std::vector<int> lo, hi;   // worker w's block: frames [lo[w], hi[w]) are still unclaimed
};

// What one sub-batch produced (kept per worker, merged in frame order at the end of the call).
struct Piece {
  int first = 0, count = 0;
  std::vector<isx_instance> inst;
  std::vector<int32_t> inst_count;   // per frame of the piece
};

struct Worker {
  isx_handle h = nullptr;
  isx_road_handle road = nullptr;    // created by the first isx_pool_compute_host_road
  int device = 0, index = 0;
  std::thread thread;
  std::mutex m;
  std::condition_variable cv;
  bool has_job = false, done = false, quit = false;
  Job *job = nullptr;
  int rc = ISX_OK;
  std::string error;
  std::vector<Piece> pieces;         // results of the last job
  int frames_done = 0;
  std::unique_ptr<isx_instance[]> tmp;
  size_t tmp_cap = 0;
};

}  // namespace

struct isx_pool {
  std::vector<Worker *> workers;
  isx_config cfg;                    // for the road handles of the workers
  int max_batch = 0;
  size_t hw = 0, seg_elems = 0, sec_per_frame = 0;
  int realcols = 0, inst_cap = 0;
  std::string last_error;
  std::vector<int> last_frames;      // frames every worker processed in the last call
};

namespace {

thread_local std::string g_pool_error;

int pool_fail(isx_pool *p, int code, const std::string &msg) {
  g_pool_error = msg;
  if (p) p->last_error = msg;
  return code;
}

// The next sub-batch of worker w: the front of its own block, else the back of the fullest other block.
bool claim(Job &j, int w, int max_batch, int *first, int *count) {
  std::lock_guard<std::mutex> lk(j.m);
  if (j.lo[(size_t)w] < j.hi[(size_t)w]) {
    const int take = std::min(max_batch, j.hi[(size_t)w] - j.lo[(size_t)w]);
    *first = j.lo[(size_t)w];
    *count = take;
    j.lo[(size_t)w] += take;
    return true;
  }
  int victim = -1, most = 0;
  for (int v = 0; v < (int)j.lo.size(); v++)
    if (j.hi[(size_t)v] - j.lo[(size_t)v] > most) {
      most = j.hi[(size_t)v] - j.lo[(size_t)v];
      victim = v;
    }
  if (victim < 0) return false;
  const int take = std::min(max_batch, most);
  j.hi[(size_t)victim] -= take;
  *first = j.hi[(size_t)victim];
  *count = take;
  return true;
}

// Sub-batches of <= max_batch frames through one context, three in flight, until no frames are left to claim.
void run_job(isx_pool *p, Worker *w) {
  Job &j = *w->job;
  w->rc = ISX_OK;
  w->error.clear();
  w->pieces.clear();
  w->frames_done = 0;
  const int mb = p->max_batch;
  // scratch for the records of one sub-batch: kept across calls, never zero-filled (52 MB at 64 frames)
  const size_t tmp_need = j.want_instances ? (size_t)mb * p->inst_cap : 0;
  if (tmp_need > w->tmp_cap) {
    w->tmp.reset(new isx_instance[tmp_need]);
    w->tmp_cap = tmp_need;
  }
  isx_instance *tmp = w->tmp.get();
  std::vector<int32_t> offs((size_t)mb + 1);
  std::deque<std::pair<int, int>> in_flight;   // (first frame, frames) in submission order
  bool more = true;
  while (true) {
    while (more && in_flight.size() < 3 && w->rc == ISX_OK) {
      int f0 = 0, cn = 0;
      more = claim(j, w->index, mb, &f0, &cn);
      if (!more) break;
      isx_section *sec = j.sections ? j.sections + (size_t)f0 * p->sec_per_frame : nullptr;
      const int rc = j.roads ? isx_submit_batch_host(w->h, j.pairwise, cn, j.disparity + (size_t)f0 * p->hw,
                                                     j.segmentation + (size_t)f0 * p->seg_elems, j.roads + f0, sec)
                             : isx::pool_submit_batch_host_road(
                                   w->h, w->road, j.pairwise, cn, j.disparity + (size_t)f0 * p->hw,
                                   j.segmentation + (size_t)f0 * p->seg_elems, j.fallback,
                                   j.estimates ? j.estimates + f0 : nullptr, j.roads_out ? j.roads_out + f0 : nullptr,
                                   sec);
      if (rc != ISX_OK) {
        w->rc = rc;
        w->error = isx_last_error(w->h);
        break;
      }
      in_flight.emplace_back(f0, cn);
    }
    if (in_flight.empty()) break;   // nothing left to claim (or a submit failed) and nothing in flight any more
    const std::pair<int, int> oldest = in_flight.front();
    in_flight.pop_front();
    const int rc = isx_wait_batch_host(w->h, j.want_instances ? tmp : nullptr, (int)tmp_need,
                                       j.want_instances ? offs.data() : nullptr);
    if (rc != ISX_OK && w->rc == ISX_OK) {
      w->rc = rc;
      w->error = isx_last_error(w->h);
    }
    if (rc == ISX_OK) {
      w->frames_done += oldest.second;
      if (j.want_instances) {
        Piece pc;
        pc.first = oldest.first;
        pc.count = oldest.second;
        pc.inst.assign(tmp, tmp + offs[(size_t)oldest.second]);
        pc.inst_count.resize((size_t)oldest.second);
        for (int f = 0; f < oldest.second; f++) pc.inst_count[(size_t)f] = offs[(size_t)f + 1] - offs[(size_t)f];
        w->pieces.push_back(std::move(pc));
      }
    }
  }
}

void worker_main(isx_pool *p, Worker *w) {
  std::unique_lock<std::mutex> lk(w->m);
  while (true) {
    w->cv.wait(lk, [&] { return w->has_job || w->quit; });
    if (w->quit) return;
    lk.unlock();
    run_job(p, w);
    lk.lock();
    w->has_job = false;
    w->done = true;
    w->cv.notify_all();
  }
}

}  // namespace

extern "C" {

int isx_pool_create(isx_pool_handle *out, const int *devices, int n_devices, const isx_config *cfg, int max_batch) {
  if (!out || !devices || n_devices < 1 || !cfg || max_batch < 1)
    return pool_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "isx_pool_create: bad argument");
  isx_pool *p = new isx_pool();
  p->max_batch = max_batch;
  p->cfg = *cfg;
  for (int i = 0; i < n_devices; i++) {
    Worker *w = new Worker();
    w->device = devices[i];
    w->index = i;
    int rc = isx_create(&w->h, devices[i]);
    if (rc == ISX_OK) rc = isx_set_config(w->h, cfg);
    if (rc == ISX_OK) rc = isx_initialize(w->h, max_batch);
    if (rc == ISX_OK) rc = isx_reserve_in_flight(w->h, 3);   // run_job keeps three sub-batches in flight
    if (rc != ISX_OK) {
      const std::string msg = std::string("isx_pool_create, device ") + std::to_string(devices[i]) + ": " +
                              isx_last_error(w->h ? w->h : nullptr);
      if (w->h) isx_destroy(w->h);
      delete w;
      for (Worker *v : p->workers) { isx_destroy(v->h); delete v; }
      delete p;
      return pool_fail(nullptr, rc, msg);
    }
    p->workers.push_back(w);
  }
  isx_handle h0 = p->workers[0]->h;
  p->realcols = isx_real_cols(h0);
  p->seg_elems = isx_segmentation_elems(h0);
  p->hw = (size_t)cfg->rows * (size_t)cfg->cols;
  p->sec_per_frame = (size_t)p->realcols * isx_max_sections(h0);
  p->inst_cap = isx_instance_capacity(h0);
  p->last_frames.assign(p->workers.size(), 0);
  for (Worker *w : p->workers) w->thread = std::thread(worker_main, p, w);
  *out = p;
  return ISX_OK;
}

int isx_pool_destroy(isx_pool_handle p) {
  if (!p) return ISX_OK;
  for (Worker *w : p->workers) {
    {
      std::lock_guard<std::mutex> lk(w->m);
      w->quit = true;
    }
    w->cv.notify_all();
    if (w->thread.joinable()) w->thread.join();
    isx_destroy(w->h);
    isx_road_destroy(w->road);
    delete w;
  }
  delete p;
  return ISX_OK;
}

int isx_pool_size(isx_pool_handle p) { return p ? (int)p->workers.size() : 0; }
int isx_pool_real_cols(isx_pool_handle p) { return p ? p->realcols : 0; }
size_t isx_pool_segmentation_elems(isx_pool_handle p) { return p ? p->seg_elems : 0; }
const char *isx_pool_last_error(isx_pool_handle p) { return p ? p->last_error.c_str() : g_pool_error.c_str(); }

int isx_pool_frames_by_worker(isx_pool_handle p, int *frames, int capacity) {
  if (!p || !frames) return 0;
  const int n = (int)p->last_frames.size() < capacity ? (int)p->last_frames.size() : capacity;
  for (int i = 0; i < n; i++) frames[i] = p->last_frames[(size_t)i];
  return n;
}

}  // extern "C"

namespace {

// One call: the frames of `job` (inputs and road arguments set) through all workers.
int pool_run(isx_pool *p, Job &job, int n, isx_section *sections, isx_instance *instances, int instances_capacity,
             int32_t *instance_offsets) {
  job.n = n;
  job.sections = sections;
  job.want_instances = instances != nullptr || instance_offsets != nullptr;
  const int G = (int)p->workers.size();
  job.lo.resize((size_t)G);
  job.hi.resize((size_t)G);
  // worker g owns frames [n * g / G, n * (g + 1) / G): contiguous blocks (SURVEY.md 8e)
  for (int g = 0; g < G; g++) {
    job.lo[(size_t)g] = (int)((long long)n * g / G);
    job.hi[(size_t)g] = (int)((long long)n * (g + 1) / G);
  }
  for (int g = 0; g < G; g++) {
    Worker *w = p->workers[(size_t)g];
    std::lock_guard<std::mutex> lk(w->m);
    w->job = &job;
    w->done = false;
    w->has_job = true;   // a worker with an empty block starts by taking from the others
    w->cv.notify_all();
  }
  int rc = ISX_OK;
  for (int g = 0; g < G; g++) {
    Worker *w = p->workers[(size_t)g];
    std::unique_lock<std::mutex> lk(w->m);
    w->cv.wait(lk, [&] { return w->done; });
    w->job = nullptr;
    p->last_frames[(size_t)g] = w->frames_done;
    if (w->rc != ISX_OK && rc == ISX_OK)
      rc = pool_fail(p, w->rc, "worker " + std::to_string(g) + " (device " + std::to_string(w->device) + "): " + w->error);
  }
  if (rc != ISX_OK) return rc;
  if (job.want_instances) {
    // the pieces of all workers in frame order
    std::vector<const Piece *> order;
    for (Worker *w : p->workers)
      for (const Piece &pc : w->pieces) order.push_back(&pc);
    std::sort(order.begin(), order.end(), [](const Piece *a, const Piece *b) { return a->first < b->first; });
    int total = 0, f = 0;
    for (const Piece *pc : order) {
      if (pc->first != f) return pool_fail(p, ISX_ERR_CUDA, "frame pool: the sub-batches do not tile the frames");
      if (instances) {
        const int room = instances_capacity - total;
        const int take = (int)pc->inst.size() < room ? (int)pc->inst.size() : (room > 0 ? room : 0);
        if (take > 0) std::memcpy(instances + total, pc->inst.data(), sizeof(isx_instance) * (size_t)take);
      }
      for (int32_t c : pc->inst_count) {
        if (instance_offsets) instance_offsets[f] = total;
        total += c;
        f++;
      }
    }
    if (f != n) return pool_fail(p, ISX_ERR_CUDA, "frame pool: the sub-batches do not cover the frames");
    if (instance_offsets) instance_offsets[n] = total;
  }
  return ISX_OK;
}

}  // namespace

extern "C" {

int isx_pool_compute_host(isx_pool_handle p, int pairwise, int n, const float *disparity,
                          const int32_t *segmentation, const isx_road *roads, isx_section *sections,
                          isx_instance *instances, int instances_capacity, int32_t *instance_offsets) {
  if (!p) return pool_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null pool");
  if (n < 1 || !disparity || !segmentation || !roads) return pool_fail(p, ISX_ERR_INVALID_ARGUMENT, "bad argument");
  Job job;
  job.pairwise = pairwise;
  job.disparity = disparity;
  job.segmentation = segmentation;
  job.roads = roads;
  return pool_run(p, job, n, sections, instances, instances_capacity, instance_offsets);
}

int isx_pool_compute_host_road(isx_pool_handle p, int pairwise, int n, const float *disparity,
                               const int32_t *segmentation, const isx_road *fallback, isx_road_estimate *estimates,
                               isx_road *roads_out, isx_section *sections, isx_instance *instances,
                               int instances_capacity, int32_t *instance_offsets) {
  if (!p) return pool_fail(nullptr, ISX_ERR_INVALID_ARGUMENT, "null pool");
  if (n < 1 || !disparity || !segmentation || !fallback)
    return pool_fail(p, ISX_ERR_INVALID_ARGUMENT, "bad argument (the fallback road is required)");
  for (Worker *w : p->workers) {
    if (w->road) continue;
    // one road handle per worker, on its GPU, for the largest chunk its context cuts a sub-batch into
    const isx_config &c = p->cfg;
    int rc = isx_road_create(&w->road, w->device);
    if (rc == ISX_OK)
      rc = isx_road_initialize(w->road, c.camera_center_y, c.baseline, c.focal, (int)c.rows, (int)c.cols, c.max_dis,
                               c.road_vdisparity_threshold, isx::largest_chunk(w->h));
    if (rc != ISX_OK) {
      const std::string msg = std::string("isx_pool_compute_host_road, device ") + std::to_string(w->device) + ": " +
                              isx_road_last_error(w->road);
      isx_road_destroy(w->road);
      w->road = nullptr;
      return pool_fail(p, rc, msg);
    }
  }
  Job job;
  job.pairwise = pairwise;
  job.disparity = disparity;
  job.segmentation = segmentation;
  job.fallback = fallback;
  job.estimates = estimates;
  job.roads_out = roads_out;
  return pool_run(p, job, n, sections, instances, instances_capacity, instance_offsets);
}

}  // extern "C"
