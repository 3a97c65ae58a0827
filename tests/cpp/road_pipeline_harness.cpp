// The drop-in classes on the stream-ordered path: `Stixels::ComputeBatchDevice(..., RoadEstimation&, fallback, ...)`
// on n frames resident on the device, road estimation included, then the results of the batch through handle():
//   road_pipeline_harness <disparity.f32> <segmentation.i32> <n> <rows> <cols> <pairwise> <fallback_vhor>
//                         <fallback_alpha> <out prefix>
// Writes <prefix>.sections ([n][realcols][200] isx_section), <prefix>.instances (packed isx_instance records),
// <prefix>.offsets (int32 [n+1]), <prefix>.roads ([n] isx_road) and <prefix>.estimates ([n] isx_road_estimate).
// Exit code 0 on success.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "RoadEstimation.h"
#include "Stixels.hpp"
#include "configuration.h"

template <typename T>
static std::vector<T> read_all(const char* path, size_t n) {
    std::vector<T> v(n);
    std::ifstream f(path, std::ios::binary);
    f.read(reinterpret_cast<char*>(v.data()), n * sizeof(T));
    if (!f) { std::cerr << "short read: " << path << "\n"; std::exit(2); }
    return v;
}

template <typename T>
static void write_all(const std::string& path, const T* p, size_t n) {
    std::ofstream f(path, std::ios::binary);
    f.write(reinterpret_cast<const char*>(p), n * sizeof(T));
}

static void cuda_check(cudaError_t e) {
    if (e != cudaSuccess) { std::cerr << cudaGetErrorString(e) << "\n"; std::exit(4); }
}

int main(int argc, char* argv[]) {
    if (argc < 10) return 2;
    const int n = atoi(argv[3]), rows = atoi(argv[4]), cols = atoi(argv[5]);
    const bool pairwise = atoi(argv[6]);
    const Stixels::Road fallback{atoi(argv[7]), 0.0f, 1.18f, (float)atof(argv[8])};
    const std::string prefix = argv[9];

    StixelConfig cfg;
    cfg.rows = rows;
    cfg.cols = cols;
    cfg.column_step = 8;
    cfg.max_dis = 128;
    cfg.invalid_disparity = 0.0f;
    cfg.n_semantic_classes = 19;
    cfg.n_offset_channels = 2;
    cfg.prior_weight = pairwise ? 1 : 1e4;
    cfg.segmentation_weight = pairwise ? 4.709500548254913f : 11.241965032069425f;
    cfg.instance_weight = pairwise ? 0.0031312903639774976f : 0.0017313017435431333f;
    cfg.disparity_weight = pairwise ? 0.0001f : 0.0069935800364145494f;
    cfg.eps = pairwise ? 18.82232269133926f : 23.89408062110343f;
    cfg.min_pts = pairwise ? 3 : 4;
    cfg.size_filter = pairwise ? 25 : 42;
    cfg.baseline = 0.209313f;
    cfg.focal = 2262.52f;
    cfg.camera_center_x = 1024.0f;
    cfg.camera_center_y = 512.0f;
    cfg.pground = cfg.pobject = cfg.psky = 0.33f;

    Stixels stixels;
    stixels.SetConfig(cfg);
    stixels.Initialize(n);
    RoadEstimation road;
    road.Initialize(cfg.camera_center_y, cfg.baseline, cfg.focal, rows, cols, cfg.max_dis,
                    cfg.road_vdisparity_threshold, n);

    const size_t C = (size_t)stixels.GetRealCols(), seg_elems = isx_segmentation_elems(stixels.handle());
    const auto disparity = read_all<pixel_t>(argv[1], (size_t)n * rows * cols);
    const auto segmentation = read_all<int32_t>(argv[2], (size_t)n * seg_elems);
    pixel_t* d_disparity = nullptr;
    int32_t* d_segmentation = nullptr;
    isx_road_estimate* d_estimates = nullptr;
    Stixels::Road* d_roads = nullptr;
    cuda_check(cudaMalloc(&d_disparity, sizeof(pixel_t) * disparity.size()));
    cuda_check(cudaMalloc(&d_segmentation, sizeof(int32_t) * segmentation.size()));
    cuda_check(cudaMalloc(&d_estimates, sizeof(isx_road_estimate) * n));
    cuda_check(cudaMalloc(&d_roads, sizeof(Stixels::Road) * n));
    cuda_check(cudaMemcpy(d_disparity, disparity.data(), sizeof(pixel_t) * disparity.size(), cudaMemcpyHostToDevice));
    cuda_check(cudaMemcpy(d_segmentation, segmentation.data(), sizeof(int32_t) * segmentation.size(),
                          cudaMemcpyHostToDevice));

    stixels.ComputeBatchDevice(pairwise, n, d_disparity, d_segmentation, road, &fallback, d_estimates, d_roads);

    std::vector<isx_section> sections((size_t)n * C * 200);
    std::vector<isx_instance> instances((size_t)n * isx_instance_capacity(stixels.handle()));
    std::vector<int32_t> offsets((size_t)n + 1);
    if (isx_fetch_batch_results(stixels.handle(), n, sections.data(), instances.data(), (int)instances.size(),
                                offsets.data()) != ISX_OK) {
        std::cerr << isx_last_error(stixels.handle()) << "\n";
        return 3;
    }
    std::vector<Stixels::Road> roads((size_t)n);
    std::vector<isx_road_estimate> estimates((size_t)n);
    cuda_check(cudaMemcpy(roads.data(), d_roads, sizeof(Stixels::Road) * n, cudaMemcpyDeviceToHost));
    cuda_check(cudaMemcpy(estimates.data(), d_estimates, sizeof(isx_road_estimate) * n, cudaMemcpyDeviceToHost));
    write_all(prefix + ".sections", sections.data(), sections.size());
    write_all(prefix + ".instances", instances.data(), (size_t)offsets[n]);
    write_all(prefix + ".offsets", offsets.data(), offsets.size());
    write_all(prefix + ".roads", roads.data(), roads.size());
    write_all(prefix + ".estimates", estimates.data(), estimates.size());
    cudaFree(d_disparity);
    cudaFree(d_segmentation);
    cudaFree(d_estimates);
    cudaFree(d_roads);
    std::printf("frames %d instances %d\n", n, offsets[n]);
    return 0;
}
