// Drop-in replacement for InstanceStixels/include/InstanceStixels/RoadEstimation.h:31-93.
//
// `class RoadEstimation` with the reference's public method names and signatures, header-only on
// top of the C ABI (include/instance_stixels_b200.h, isx_road_*).  Unlike the reference it needs no
// OpenCV: the Hough transform behind cv::HoughLines (RoadEstimation.cu:152) runs on the device.
// apps/run_cityscapes.cu:246, 332-343, 390-400 and apps/stixels_node.cu compile against it unchanged.
// CUDA failures print and exit(1) like CUDA_CHECK_RETURN (util.h:27-42).
#ifndef ISX_DROPIN_ROADESTIMATION_H_
#define ISX_DROPIN_ROADESTIMATION_H_

#include <cstdlib>
#include <iostream>
#include <vector>

#include "../instance_stixels_b200.h"
#include "configuration.h"
#include "util.h"

class RoadEstimation {
public:
    RoadEstimation() {
        const char* e = std::getenv("ISX_DEVICE");
        if (isx_road_create(&h_, e ? std::atoi(e) : 0) != ISX_OK) die();
    }
    ~RoadEstimation() { isx_road_destroy(h_); }
    RoadEstimation(const RoadEstimation&) = delete;
    RoadEstimation& operator=(const RoadEstimation&) = delete;

    // Extension: `max_batch` frames per batched call (Stixels::ComputeBatchDevice with road estimation).
    void Initialize(const float camera_center_y, const float baseline, const float focal, const int rows,
                    const int cols, const int max_dis, const float road_vdisparity_threshold = 0.2f,
                    int max_batch = 1) {
        check(isx_road_initialize(h_, camera_center_y, baseline, focal, rows, cols, max_dis,
                                  road_vdisparity_threshold, max_batch));
    }
    void Finish() { check(isx_road_finish(h_)); }

    bool Compute(const std::vector<pixel_t>& im) {
        isx_road_estimate e;
        check(isx_road_compute_host(h_, im.data(), im.size(), &e));
        return keep(e);
    }
    bool Compute(pixel_t* d_im) {
        isx_road_estimate e;
        check(isx_road_compute_device(h_, d_im, &e));
        return keep(e);
    }

    float GetCameraHeight() { return est_.camera_height; }
    float GetPitch() { return est_.pitch; }
    float GetSlope() { return est_.slope; }
    int GetHorizonPoint() { return est_.horizon_point; }
    bool IsInitialized() { return isx_road_is_initialized(h_) != 0; }

    isx_road_handle handle() { return h_; }  // for the other C entry points

private:
    // the reference only overwrites its members when a line was accepted (RoadEstimation.cu:123-133)
    bool keep(const isx_road_estimate& e) {
        if (e.ok) est_ = e;
        return e.ok != 0;
    }
    [[noreturn]] void die() {
        std::cerr << "instance_stixels_b200: " << isx_road_last_error(h_) << std::endl;
        std::exit(1);
    }
    void check(int rc) {
        if (rc != ISX_OK) die();
    }
    isx_road_handle h_ = nullptr;
    isx_road_estimate est_{0, 0, 0.f, 0.f, 0.f, 0.f, 0.f};
};

#endif  // ISX_DROPIN_ROADESTIMATION_H_
