// The drop-in classes on host batches with road estimation inside the pipeline:
//   * `Stixels::SubmitBatch(..., RoadEstimation&, fallback, estimates, roads_out)` + `WaitBatch` (keep-last rule),
//   * `StixelsPool::ComputeBatch(..., const Road& fallback, &estimates, ...)` on one GPU (per-frame rule).
//   host_road_harness <disparity.f32> <segmentation.i32> <n> <rows> <cols> <pairwise> <out prefix>
// Writes <prefix>.stixels.* and <prefix>.pool.*: sections ([n][realcols][200] isx_section), instances (packed
// isx_instance records), offsets (int32 [n+1]), roads ([n] isx_road), estimates ([n] isx_road_estimate); for
// SubmitBatch the instances are the per-frame maps WaitBatch fills, as int32 (column, index, label) in map order.
// The fallback road is vhor 100, tilt 0, height 1.18, alpha_ground 0.177384.  Exit code 0 on success.
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

int main(int argc, char* argv[]) {
    if (argc < 8) return 2;
    const int n = atoi(argv[3]), rows = atoi(argv[4]), cols = atoi(argv[5]);
    const bool pairwise = atoi(argv[6]);
    const Stixels::Road fallback{100, 0.0f, 1.18f, 0.177384f};
    const std::string prefix = argv[7];

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

    std::vector<pixel_t> disparity;
    std::vector<int32_t> segmentation;
    {
        Stixels stixels;
        stixels.SetConfig(cfg);
        stixels.Initialize(n);
        RoadEstimation road;
        road.Initialize(cfg.camera_center_y, cfg.baseline, cfg.focal, rows, cols, cfg.max_dis,
                        cfg.road_vdisparity_threshold, n);
        const size_t se = isx_segmentation_elems(stixels.handle());
        disparity = read_all<pixel_t>(argv[1], (size_t)n * rows * cols);
        segmentation = read_all<int32_t>(argv[2], (size_t)n * se);
        std::vector<isx_road_estimate> estimates((size_t)n);
        std::vector<Stixels::Road> roads((size_t)n);
        stixels.SubmitBatch(pairwise, n, disparity.data(), segmentation.data(), road, &fallback, estimates.data(),
                            roads.data());
        std::vector<StixelsData> frames;
        std::vector<Stixels::InstanceMap> maps;
        stixels.WaitBatch(frames, &maps);
        std::vector<Section> sections;
        std::vector<isx_instance> instances;
        std::vector<int32_t> offsets(1, 0);
        for (int f = 0; f < n; f++) {
            const StixelsData& d = frames[(size_t)f];
            sections.insert(sections.end(), d.sections.begin(), d.sections.end());
            if (d.alpha_ground != roads[(size_t)f].alpha_ground || d.vhor != rows - roads[(size_t)f].vhor - 1) {
                std::cerr << "frame " << f << ": StixelsData does not carry the road it was computed with\n";
                return 3;
            }
            offsets.push_back(offsets.back() + (int32_t)maps[(size_t)f].size());
        }
        write_all(prefix + ".stixels.sections", sections.data(), sections.size());
        write_all(prefix + ".stixels.roads", roads.data(), roads.size());
        write_all(prefix + ".stixels.estimates", estimates.data(), estimates.size());
        write_all(prefix + ".stixels.offsets", offsets.data(), offsets.size());
        std::vector<int32_t> flat;
        for (const auto& m : maps)
            for (const auto& kv : m) flat.insert(flat.end(), {kv.first.first, kv.first.second, kv.second});
        write_all(prefix + ".stixels.instances", flat.data(), flat.size());
        stixels.Finish();
    }
    {
        StixelsPool pool(cfg, std::vector<int>{0}, n);
        std::vector<Section> sections((size_t)n * pool.GetRealCols() * pool.GetMaxSections());
        std::vector<isx_road_estimate> estimates;
        std::vector<isx_instance> records;
        std::vector<int32_t> offsets;
        std::vector<Stixels::Road> roads;
        pool.ComputeBatch(pairwise, n, disparity.data(), segmentation.data(), fallback, &estimates, sections.data(),
                          &records, &offsets, &roads);
        write_all(prefix + ".pool.sections", sections.data(), sections.size());
        write_all(prefix + ".pool.instances", records.data(), records.size());
        write_all(prefix + ".pool.offsets", offsets.data(), offsets.size());
        write_all(prefix + ".pool.roads", roads.data(), roads.size());
        write_all(prefix + ".pool.estimates", estimates.data(), estimates.size());
        std::printf("frames %d instances %d\n", n, offsets[(size_t)n]);
    }
    return 0;
}
