// Drop-in replacement for InstanceStixels/include/InstanceStixels/Stixels.hpp:40-96.
//
// `class Stixels` with the reference's public method names and signatures,
// implemented header-only on top of the C ABI (include/instance_stixels_b200.h,
// libinstance_stixels_b200.so).  apps/run_cityscapes.cu and
// apps/stixels_wrapper.cu compile against it unchanged: same include name,
// same call sequence, same exceptions (std::invalid_argument from SetConfig /
// Get3DVertices), CUDA failures print and exit(1) like CUDA_CHECK_RETURN.
// Host-only code: no CUDA headers are needed to include it.
#ifndef ISX_DROPIN_STIXELS_HPP_
#define ISX_DROPIN_STIXELS_HPP_

#include <stdint.h>

#include <cmath>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <memory>
#include <stdexcept>
#include <utility>
#include <vector>

#include "../instance_stixels_b200.h"
#include "RoadEstimation.h"
#include "configuration.h"
#include "types.h"
#include "util.h"

constexpr float PIFLOAT = 3.1416f;

class Stixels {
public:
    Stixels() {
        if (isx_create(&h_, device_from_env()) != ISX_OK) die();
    }
    ~Stixels() { isx_destroy(h_); }
    Stixels(const Stixels&) = delete;
    Stixels& operator=(const Stixels&) = delete;

    // Extension: frames per batched call (the reference is always 1).
    void Initialize(int max_batch) { check(isx_initialize(h_, max_batch)); }
    void Initialize() { Initialize(1); }
    void Finish() { check(isx_finish(h_)); }
    bool IsInitialized() { return isx_is_initialized(h_) != 0; }

    float Compute(bool pairwise, StixelsData& stixels, int32_t* d_segmentation_local = nullptr) {
        stixels.sections.resize((size_t)GetRealCols() * GetMaxSections());
        isx_frame_meta m;
        check(isx_compute(h_, pairwise ? 1 : 0, reinterpret_cast<isx_section*>(stixels.sections.data()), &m,
                          d_segmentation_local));
        stixels.rows = m.rows;
        stixels.cols = m.cols;
        stixels.realcols = m.realcols;
        stixels.max_sections = m.max_sections;
        stixels.max_dis = m.max_dis;
        stixels.column_step = m.column_step;
        stixels.semantic_classes = m.semantic_classes;
        stixels.alpha_ground = m.alpha_ground;
        stixels.vhor = m.vhor;
        meta_ = m;
        return -1;  // the reference's timing code is commented out and it returns -1 too
    }
    float ClusterInstances() {
        check(isx_cluster_instances(h_));
        return -1;
    }
    std::map<std::pair<int, int>, int> GetInstanceStixels() {
        int n = 0;
        check(isx_get_instance_stixels(h_, nullptr, 0, &n));
        std::vector<isx_instance> v((size_t)(n > 0 ? n : 1));
        check(isx_get_instance_stixels(h_, v.data(), n, &n));
        std::map<std::pair<int, int>, int> out;
        for (int i = 0; i < n; i++) out[std::make_pair(v[i].column, v[i].index)] = v[i].label;
        return out;
    }
    int GetRealCols() { return isx_real_cols(h_); }
    int GetMaxSections() { return isx_max_sections(h_); }

    static isx_config ToIsxConfig(const StixelConfig& c) {
        isx_config k;
        isx_config_init(&k);
        k.rows = c.rows; k.cols = c.cols; k.max_dis = c.max_dis; k.invalid_disparity = c.invalid_disparity;
        k.eps = c.eps; k.min_pts = c.min_pts; k.size_filter = c.size_filter;
        k.n_semantic_classes = c.n_semantic_classes; k.n_offset_channels = c.n_offset_channels;
        k.prior_weight = c.prior_weight; k.segmentation_weight = c.segmentation_weight;
        k.instance_weight = c.instance_weight; k.disparity_weight = c.disparity_weight;
        k.pairwise = c.pairwise; k.column_step = c.column_step;
        k.focal = c.focal; k.baseline = c.baseline;
        k.camera_center_x = c.camera_center_x; k.camera_center_y = c.camera_center_y;
        k.sigma_disparity_object = c.sigma_disparity_object; k.sigma_disparity_ground = c.sigma_disparity_ground;
        k.sigma_sky = c.sigma_sky;
        k.pout = c.pout; k.pout_sky = c.pout_sky; k.pord = c.pord; k.pgrav = c.pgrav; k.pblg = c.pblg;
        k.pground_given_nexist = c.pground_given_nexist; k.pobject_given_nexist = c.pobject_given_nexist;
        k.psky_given_nexist = c.psky_given_nexist; k.pnexist_dis = c.pnexist_dis;
        k.pground = c.pground; k.pobject = c.pobject; k.psky = c.psky;
        k.width_margin = c.width_margin;
        k.sigma_camera_tilt = c.sigma_camera_tilt; k.sigma_camera_height = c.sigma_camera_height;
        k.median_join = c.median_join; k.epsilon = c.epsilon; k.range_objects_z = c.range_objects_z;
        k.road_vdisparity_threshold = c.road_vdisparity_threshold;
        return k;
    }
    void SetConfig(const StixelConfig& c) {
        const isx_config k = ToIsxConfig(c);
        check(isx_set_config(h_, &k));
        cfg_ = c;
    }
    void SetSegmentation(const std::vector<int32_t>& segmentation) {
        check(isx_set_segmentation(h_, segmentation.data(), segmentation.size()));
    }
    void SetSegmentationParameters(const int classes, const int instance_channels) {
        check(isx_set_segmentation_parameters(h_, classes, instance_channels));
    }
    void SetClusteringParameters(const float eps, const int min_pts, const int size_filter) {
        check(isx_set_clustering_parameters(h_, eps, min_pts, size_filter));
    }
    void SetWeightParameters(const float prior_weight, const float disparity_weight,
                             const float segmentation_weight, const float instance_weight) {
        check(isx_set_weight_parameters(h_, prior_weight, disparity_weight, segmentation_weight, instance_weight));
    }
    void SetDisparityImage(const std::vector<pixel_t>& disp_im) {
        check(isx_set_disparity_image(h_, disp_im.data(), disp_im.size()));
    }
    pixel_t* GetInputDisparityImageOnDevice() { return isx_input_disparity_device(h_); }
    void SetProbabilities(float pout, float pout_sky, float pground_given_nexist, float pobject_given_nexist,
                          float psky_given_nexist, float pnexist_dis, float pground, float pobject, float psky,
                          float pord, float pgrav, float pblg) {
        check(isx_set_probabilities(h_, pout, pout_sky, pground_given_nexist, pobject_given_nexist,
                                    psky_given_nexist, pnexist_dis, pground, pobject, psky, pord, pgrav, pblg));
    }
    void SetRoadParameters(int vhor, float camera_tilt, float camera_height, float alpha_ground) {
        check(isx_set_road_parameters(h_, vhor, camera_tilt, camera_height, alpha_ground));
    }
    void SetCameraParameters(float focal, float baseline, float sigma_camera_tilt, float sigma_camera_height,
                             float camera_center_x = -1, float camera_center_y = -1) {
        check(isx_set_camera_parameters(h_, focal, baseline, sigma_camera_tilt, sigma_camera_height,
                                        camera_center_x, camera_center_y));
        cfg_.focal = focal; cfg_.baseline = baseline;
        cfg_.camera_center_x = camera_center_x; cfg_.camera_center_y = camera_center_y;
    }
    void SetDisparityParameters(const int rows, const int cols, const int max_dis, const float invalid_disparity,
                                const float sigma_disparity_object, const float sigma_disparity_ground,
                                float sigma_sky) {
        check(isx_set_disparity_parameters(h_, rows, cols, max_dis, invalid_disparity, sigma_disparity_object,
                                           sigma_disparity_ground, sigma_sky));
        cfg_.rows = rows;
    }
    void SetModelParameters(const int column_step, const bool median_join, float epsilon, float range_objects_z,
                            int width_margin) {
        check(isx_set_model_parameters(h_, column_step, median_join, epsilon, range_objects_z, width_margin));
        cfg_.column_step = column_step;
    }

    // Corner points of every stixel in camera coordinates, 4 x (x, y, z) per stixel, clockwise
    // from the top-left corner (Stixels.cu:683-742).  Pure function of the result.
    std::vector<float> Get3DVertices(const StixelsData& d) {
        if (cfg_.camera_center_x == -1 || cfg_.camera_center_y == -1)
            throw std::invalid_argument("Camera parameters are not set.");
        const float f = cfg_.focal, bf = cfg_.baseline * cfg_.focal;
        const float cx = cfg_.camera_center_x, cy = cfg_.camera_center_y;
        const int step = d.column_step;
        std::vector<float> v;
        for (size_t i = 0; i < (size_t)d.realcols; i++) {
            for (size_t j = 0; j < (size_t)d.max_sections; j++) {
                const Section& s = d.sections[i * d.max_sections + j];
                if (s.type == -1) break;
                const float xl = i * step, xr = xl + step;
                const float yt = d.rows - s.vT - 1, yb = d.rows - s.vB;
                float zt = 0.0, zb = 0.0;  // sky stays at depth 0
                if (s.type == OBJECT) {
                    zt = zb = bf / s.disparity;
                } else if (s.type == GROUND) {
                    zt = bf / (d.alpha_ground * (d.vhor - s.vT));
                    zb = bf / (d.alpha_ground * (d.vhor - s.vB));
                }
                const float corner[4][3] = {{xl, yt, zt}, {xr, yt, zt}, {xr, yb, zb}, {xl, yb, zb}};
                for (const auto& c : corner) {
                    v.push_back(-c[2] / f * (cx - c[0]));
                    v.push_back(-c[2] / f * (cy - c[1]));
                    v.push_back(c[2]);
                }
            }
        }
        return v;
    }

    // The `.stixels` text format read by tools/visualization (Stixels.cu:889-926): one line per
    // column, "type,vB,vT,disparity,class,cost,meanx,meany[,label];" per stixel, then the ground plane.
    static void SaveStixels(Section* stixels, std::map<std::pair<int, int>, int> instance_stixels,
                            const float alpha_ground, const int vhor, const int real_cols,
                            const int max_segments, const char* fname) {
        std::ofstream fp(fname, std::ofstream::out | std::ofstream::trunc);
        if (!fp.is_open()) {
            std::cerr << "Counldn't write file: " << fname << std::endl;
            return;
        }
        for (size_t i = 0; i < (size_t)real_cols; i++) {
            for (size_t j = 0; j < (size_t)max_segments; j++) {
                const Section& s = stixels[i * max_segments + j];
                if (s.type == -1) break;
                fp << s.type << "," << s.vB << "," << s.vT << "," << s.disparity << "," << s.semantic_class << ","
                   << s.cost << "," << s.instance_meanx << "," << s.instance_meany;
                const auto it = instance_stixels.find(std::make_pair((int)i, (int)j));
                if (it != instance_stixels.end()) fp << "," << it->second;
                fp << ";";
            }
            fp << std::endl;
        }
        fp << "groundplane" << alpha_ground << "," << vhor << "\n";
    }

    // ---- extensions: batches of independent frames (the reference takes one frame per Compute) ----
    // Road parameters of one frame of a batch (the arguments of SetRoadParameters).
    typedef isx_road Road;
    // Instance ids of one frame of a batch, the map GetInstanceStixels returns.
    typedef std::map<std::pair<int, int>, int> InstanceMap;

    // n frames, host buffers: disparity [n][rows][cols], segmentation [n][realcols][21][rows_power2_segmentation],
    // one Road per frame.  Fills `frames` (one StixelsData per frame) and, if given, `instances`.  Synchronous;
    // n <= Initialize(max_batch).
    void ComputeBatch(bool pairwise, int n, const pixel_t* disparity, const int32_t* segmentation, const Road* roads,
                      std::vector<StixelsData>& frames, std::vector<InstanceMap>* instances = nullptr) {
        sections_.resize((size_t)n * GetRealCols() * GetMaxSections());
        inst_.resize((size_t)n * (size_t)isx_instance_capacity(h_));
        offs_.resize((size_t)n + 1);
        check(isx_compute_batch_host(h_, pairwise ? 1 : 0, n, disparity, segmentation, roads,
                                     reinterpret_cast<isx_section*>(sections_.data()), inst_.data(), (int)inst_.size(),
                                     offs_.data()));
        unpack(n, roads, sections_.data(), frames, instances);
    }
    // Streaming form: SubmitBatch enqueues a batch and returns; WaitBatch delivers the OLDEST one.  At most three in
    // flight (submit, submit, submit, wait, submit, wait, ...); the input buffers must stay valid until their
    // WaitBatch.  ReserveInFlight allocates the result arrays of that many batches up front (otherwise the first
    // submits do).
    void ReserveInFlight(int batches) { check(isx_reserve_in_flight(h_, batches)); }
    void SubmitBatch(bool pairwise, int n, const pixel_t* disparity, const int32_t* segmentation, const Road* roads) {
        Pending& p = pending_[submitted_ % 3];
        p.n = n;
        p.roads.assign(roads, roads + n);
        p.sections.resize((size_t)n * GetRealCols() * GetMaxSections());
        check(isx_submit_batch_host(h_, pairwise ? 1 : 0, n, disparity, segmentation, roads,
                                    reinterpret_cast<isx_section*>(p.sections.data())));
        submitted_++;
    }
    void WaitBatch(std::vector<StixelsData>& frames, std::vector<InstanceMap>* instances = nullptr) {
        Pending& p = pending_[waited_ % 3];
        inst_.resize((size_t)p.n * (size_t)isx_instance_capacity(h_));
        offs_.resize((size_t)p.n + 1);
        check(isx_wait_batch_host(h_, inst_.data(), (int)inst_.size(), offs_.data()));
        waited_++;
        unpack(p.n, p.roads.data(), p.sections.data(), frames, instances);
    }

    // n frames resident on the device (isx_compute_batch_device): results stay there for ExportBatchDevice /
    // isx_fetch_batch_results; asynchronous on isx_stream().
    void ComputeBatchDevice(bool pairwise, int n, const pixel_t* d_disparity, const int32_t* d_segmentation,
                            const Road* roads) {
        check(isx_compute_batch_device(h_, pairwise ? 1 : 0, n, d_disparity, d_segmentation, roads));
    }
    // The same with the road of every frame estimated on the device by `road` from the frame's own disparity
    // (isx_compute_batch_device_road): a frame without an accepted line keeps the last accepted estimate, before the
    // first one `fallback` is used; fallback == nullptr continues from the previous call on `road`.  d_estimates /
    // d_roads: optional device arrays [n].  No host round trip between road estimation and stixels.
    void ComputeBatchDevice(bool pairwise, int n, const pixel_t* d_disparity, const int32_t* d_segmentation,
                            RoadEstimation& road, const Road* fallback, isx_road_estimate* d_estimates = nullptr,
                            Road* d_roads = nullptr) {
        check(isx_compute_batch_device_road(h_, road.handle(), pairwise ? 1 : 0, n, d_disparity, d_segmentation,
                                            fallback, d_estimates, d_roads));
    }

    // Frames [first, first + n) of the last batch into the caller's device buffers (isx_export_batch_device):
    // packed frame-ordered Sections, offsets, instance labels and Get3DVertices, asynchronous on isx_stream().
    void ExportBatchDevice(int first, int n, const isx_device_results& out) {
        check(isx_export_batch_device(h_, first, n, &out));
    }

    isx_handle handle() { return h_; }  // for the other C entry points

private:
    isx_handle h_ = nullptr;
    StixelConfig cfg_;
    isx_frame_meta meta_{};
    struct Pending {
        int n = 0;
        std::vector<Road> roads;
        std::vector<Section> sections;
    } pending_[3];
    unsigned long long submitted_ = 0, waited_ = 0;
    std::vector<Section> sections_;
    std::vector<isx_instance> inst_;
    std::vector<int32_t> offs_;

    void unpack(int n, const Road* roads, const Section* sections, std::vector<StixelsData>& frames,
                std::vector<InstanceMap>* instances) {
        const size_t per = (size_t)GetRealCols() * GetMaxSections();
        frames.resize((size_t)n);
        if (instances) instances->assign((size_t)n, InstanceMap());
        for (int f = 0; f < n; f++) {
            StixelsData& d = frames[(size_t)f];
            d.sections.assign(sections + (size_t)f * per, sections + (size_t)(f + 1) * per);
            d.rows = (int)cfg_.rows;
            d.cols = (int)cfg_.cols;
            d.realcols = GetRealCols();
            d.max_sections = GetMaxSections();
            d.max_dis = cfg_.max_dis;
            d.column_step = cfg_.column_step;
            d.semantic_classes = cfg_.n_semantic_classes;
            d.alpha_ground = roads[f].alpha_ground;
            d.vhor = (int)cfg_.rows - roads[f].vhor - 1;
            if (instances)
                for (int32_t i = offs_[(size_t)f]; i < offs_[(size_t)f + 1]; i++)
                    (*instances)[(size_t)f][std::make_pair(inst_[(size_t)i].column, inst_[(size_t)i].index)] = inst_[(size_t)i].label;
        }
    }

    static int device_from_env() {
        const char* e = std::getenv("ISX_DEVICE");
        return e ? std::atoi(e) : 0;
    }
    [[noreturn]] void die() {
        std::cerr << "instance_stixels_b200: " << isx_last_error(h_) << std::endl;
        std::exit(1);
    }
    void check(int rc) {
        if (rc == ISX_OK) return;
        if (rc == ISX_ERR_INVALID_ARGUMENT) throw std::invalid_argument(isx_last_error(h_));
        die();
    }
};

// Extension: one context and worker thread per GPU in this process (isx_pool_*, SURVEY.md 8e): a call shards its
// frames into contiguous blocks over the GPUs, frame f -> GPU f * G / n.
class StixelsPool {
public:
    typedef isx_road Road;
    typedef std::map<std::pair<int, int>, int> InstanceMap;

    StixelsPool(const StixelConfig& c, const std::vector<int>& devices, int max_batch) {
        cfg_ = c;
        const isx_config k = to_isx(c);
        if (isx_pool_create(&p_, devices.data(), (int)devices.size(), &k, max_batch) != ISX_OK) {
            std::cerr << "instance_stixels_b200: " << isx_pool_last_error(nullptr) << std::endl;
            std::exit(1);
        }
    }
    ~StixelsPool() { isx_pool_destroy(p_); }
    StixelsPool(const StixelsPool&) = delete;
    StixelsPool& operator=(const StixelsPool&) = delete;

    int Size() { return isx_pool_size(p_); }
    int GetRealCols() { return isx_pool_real_cols(p_); }
    int GetMaxSections() { return ISX_MAX_STIXELS_PER_COLUMN; }
    // Frames every worker processed in the last ComputeBatch: its contiguous block, less or plus the sub-batches a
    // worker that was done took over from the back of another block.
    std::vector<int> FramesByWorker() {
        std::vector<int> f((size_t)Size());
        f.resize((size_t)isx_pool_frames_by_worker(p_, f.data(), (int)f.size()));
        return f;
    }

    // Any n >= 1; layouts as Stixels::ComputeBatch.  `sections` receives [n][realcols][200].
    void ComputeBatch(bool pairwise, int n, const pixel_t* disparity, const int32_t* segmentation, const Road* roads,
                      std::vector<Section>& sections, std::vector<InstanceMap>* instances = nullptr) {
        sections.resize((size_t)n * (size_t)GetRealCols() * GetMaxSections());
        ComputeBatch(pairwise, n, disparity, segmentation, roads, sections.data(), instances);
    }
    // The same into a caller-owned array of n * realcols * 200 Sections; when it is pinned (isx_host_alloc,
    // cudaHostAlloc, cudaHostRegister) the device writes into it directly and nothing is expanded on the host.
    void ComputeBatch(bool pairwise, int n, const pixel_t* disparity, const int32_t* segmentation, const Road* roads,
                      Section* sections, std::vector<InstanceMap>* instances = nullptr) {
        std::vector<isx_instance> inst;
        std::vector<int32_t> offs;
        ComputeBatch(pairwise, n, disparity, segmentation, roads, sections, instances ? &inst : nullptr, &offs);
        if (instances) {
            instances->assign((size_t)n, InstanceMap());
            for (int f = 0; f < n; f++) (*instances)[(size_t)f] = MapOf(inst, offs, f);
        }
    }
    // ... with the instance ids as packed records (column, index, label, class), frame f = [offsets[f], offsets[f+1]):
    // what a throughput caller wants inside its timed region; MapOf builds the reference's std::map per frame later.
    void ComputeBatch(bool pairwise, int n, const pixel_t* disparity, const int32_t* segmentation, const Road* roads,
                      Section* sections, std::vector<isx_instance>* records, std::vector<int32_t>* offsets) {
        const size_t per = (size_t)GetRealCols() * GetMaxSections();
        // Worst-case capacity (every stixel an instance stixel) as UNINITIALISED scratch: pages that are never written
        // cost nothing, while value-initialising a vector of this size would take longer than the GPU work.
        if (records && scratch_cap_ < (size_t)n * per) {
            scratch_.reset(new isx_instance[(size_t)n * per]);
            scratch_cap_ = (size_t)n * per;
        }
        std::vector<int32_t> local_offsets;
        if (records && !offsets) offsets = &local_offsets;
        if (offsets) offsets->resize((size_t)n + 1);
        if (isx_pool_compute_host(p_, pairwise ? 1 : 0, n, disparity, segmentation, roads,
                                  reinterpret_cast<isx_section*>(sections), records ? scratch_.get() : nullptr,
                                  records ? (int)scratch_cap_ : 0, offsets ? offsets->data() : nullptr) != ISX_OK) {
            std::cerr << "instance_stixels_b200: " << isx_pool_last_error(p_) << std::endl;
            std::exit(1);
        }
        if (records) records->assign(scratch_.get(), scratch_.get() + (*offsets)[(size_t)n]);
    }
    static InstanceMap MapOf(const std::vector<isx_instance>& records, const std::vector<int32_t>& offsets, int frame) {
        InstanceMap m;
        for (int32_t i = offsets[(size_t)frame]; i < offsets[(size_t)frame + 1]; i++)
            m[std::make_pair(records[(size_t)i].column, records[(size_t)i].index)] = records[(size_t)i].label;
        return m;
    }

private:
    isx_pool_handle p_ = nullptr;
    StixelConfig cfg_;
    std::unique_ptr<isx_instance[]> scratch_;
    size_t scratch_cap_ = 0;
    static isx_config to_isx(const StixelConfig& c) { return Stixels::ToIsxConfig(c); }
};

#endif  // ISX_DROPIN_STIXELS_HPP_
