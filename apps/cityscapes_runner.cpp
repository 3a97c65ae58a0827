// cityscapes_runner: the role of the reference's batch runner (apps/run_cityscapes.cu) on the drop-in classes.
//
//   cityscapes_runner <dir> <max_disparity> <segmentation_weight> <instance_weight> <disparity_weight> <pairwise>
//                     <stixel_width> <eps> <min_pts> <size_filter> [tensorrt]
//
// Contract kept from the reference so that tools/run_cityscapes.py can drive it unchanged:
//   * the ten positional arguments and their meaning (apps/run_cityscapes.cu:158-176; the Python side builds the
//     command line at tools/run_cityscapes.py:191-219); prior weight = 1 in pairwise mode, 1e4 otherwise;
//   * the directory layout: <dir>/disparities/<base>_disparity.png, <dir>/camera/<base>_camera.json,
//     <dir>/probs/<base>_probs.*, output <dir>/stixels/<base>.stixels (:199-268);
//   * per frame: disparity + segmentation in, road estimation, Compute, instance map, .stixels file out; the clock
//     runs from SetSegmentation to the end of Compute (:372-416) and the first frame is a warm-up (:420-426);
//   * the closing line "It took an average of X milliseconds, Y fps" (:453-459), which
//     tools/run_cityscapes.py:314-325 parses with a regular expression.
// Not kept: OpenCV, rapidjson and HDF5 (apps/loaders.h reads the PNG, the three camera numbers and an .npy copy of
// the "nlogprobs" dataset; tools/h5_to_npy.py converts), the TensorRT path (argument 11 is refused), readdir order
// (frames are processed in sorted order).  Rows >= 1024 are refused like the reference does (:129-134) unless
// ISX_ALLOW_1024=1: the library itself handles frames of up to ISX_MAX_ROWS (2047) rows.
#include <dirent.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <map>
#include <numeric>
#include <string>
#include <vector>

#include "RoadEstimation.h"  // RoadEstimation (drop-in)
#include "Stixels.hpp"       // Stixels (drop-in)
#include "configuration.h"   // pixel_t
#include "h5_reader.h"
#include "loaders.h"

namespace {

struct Options {
    std::string dataset;
    bool pairwise = false;
    StixelConfig config;  // everything that does not depend on the frame
    // extensions (not in the reference's CLI): --batch B frames per batched call, --gpus G GPUs of this box
    // and --road-on-device (below)
    int batch = 1, gpus = 1;
    int replicate = 1;   // --replicate K (measurement only): the timed call streams the loaded frames K times
    // --road-on-device (with --batch / --gpus): the road of every frame is estimated inside the timed pool call
    bool road_on_device = false;
};

bool parse_options(int argc, char** argv, Options* o) {
    // optional flags behind the reference's positional arguments
    std::vector<char*> pos;
    for (int i = 0; i < argc; i++) {
        const std::string a(argv[i]);
        if (a == "--road-on-device") {
            o->road_on_device = true;
            continue;
        }
        if ((a == "--batch" || a == "--gpus" || a == "--replicate") && i + 1 < argc) {
            (a == "--batch" ? o->batch : a == "--gpus" ? o->gpus : o->replicate) = std::max(1, std::atoi(argv[++i]));
            continue;
        }
        pos.push_back(argv[i]);
    }
    argc = (int)pos.size();
    argv = pos.data();
    if (argc < 11) {
        std::cerr << "Usage: stixels dir max_disparity segmentation_weight instance_weight disparity_weight "
                     "pairwise stixel_width eps min_pts size_filter\n";
        return false;
    }
    if (argc > 11 && std::atoi(argv[11]) == 1) {
        std::cerr << "The TensorRT path is not part of this build: provide <base>_probs.h5 (or .npy) files.\n";
        return false;
    }
    o->dataset = argv[1];
    o->pairwise = std::atoi(argv[6]) != 0;
    StixelConfig& c = o->config;
    c.max_dis = std::atoi(argv[2]);
    c.segmentation_weight = std::atof(argv[3]);
    c.instance_weight = std::atof(argv[4]);
    c.disparity_weight = std::atof(argv[5]);
    c.prior_weight = o->pairwise ? 1 : 1e4;
    c.column_step = std::atoi(argv[7]);
    c.eps = std::atof(argv[8]);
    c.min_pts = std::atoi(argv[9]);
    c.size_filter = std::atoi(argv[10]);
    c.invalid_disparity = 0.0f;  // holes of the Cityscapes disparity maps
    c.n_semantic_classes = 19;
    c.n_offset_channels = 2;
    return true;
}

bool exists(const std::string& path) {
    struct stat st;
    return stat(path.c_str(), &st) == 0;
}

// Frame base names (<base>_disparity.png), sorted.
std::vector<std::string> list_frames(const std::string& disparity_dir) {
    static const std::string suffix = "_disparity.png";
    std::vector<std::string> bases;
    DIR* d = opendir(disparity_dir.c_str());
    if (!d) {
        std::cerr << "Invalid directory: " << disparity_dir << std::endl;
        std::exit(EXIT_FAILURE);
    }
    while (const dirent* e = readdir(d)) {
        const std::string name(e->d_name);
        if (name.size() > suffix.size() && name.compare(name.size() - suffix.size(), suffix.size(), suffix) == 0)
            bases.push_back(name.substr(0, name.size() - suffix.size()));
    }
    closedir(d);
    std::sort(bases.begin(), bases.end());
    return bases;
}

// Cityscapes disparity PNG -> float disparities: 16-bit values are 1/256 px, 8-bit values whole pixels.
struct Disparity {
    int rows = 0, cols = 0;
    std::vector<pixel_t> values;
};

Disparity load_disparity(const std::string& path, int max_dis) {
    const isx_apps::GrayImage png = isx_apps::read_png_gray(path);
    if (png.rows < max_dis)
        throw std::invalid_argument("ERROR: Image height has to be equal or bigger than maximum disparity.");
    const char* allow = std::getenv("ISX_ALLOW_1024");
    const bool allow_1024 = allow && std::atoi(allow) != 0;
    if (png.rows >= 1024 && !allow_1024)
        throw std::invalid_argument("ERROR: Maximum image height has to be less than 1024.");
    if (png.rows > ISX_MAX_ROWS)
        throw std::invalid_argument("ERROR: Maximum image height is " + std::to_string(ISX_MAX_ROWS) + ".");
    Disparity d;
    d.rows = png.rows;
    d.cols = png.cols;
    d.values.resize(png.pixels.size());
    const float scale = png.bit_depth == 16 ? 1.0f / 256.0f : 1.0f;  // exact: a power of two
    std::transform(png.pixels.begin(), png.pixels.end(), d.values.begin(),
                   [scale](uint16_t v) { return (float)v * scale; });
    return d;
}

// The pipeline objects and what they are currently initialised for.
class Pipeline {
public:
    explicit Pipeline(const Options& o) : opt_(o), config_(o.config) {}

    // (Re)initialises when the image size or the camera changed, like the reference does per frame.
    void prepare(int rows, int cols, const isx_apps::Camera& cam) {
        const bool same = ready_ && config_.rows == rows && config_.cols == cols && config_.baseline == cam.baseline &&
                          config_.focal == cam.focal && config_.camera_center_y == cam.center_y;
        if (same) return;
        if (!ready_ || config_.baseline != cam.baseline || config_.focal != cam.focal ||
            config_.camera_center_y != cam.center_y)
            std::cout << "New camera parameters: baseline = " << cam.baseline << ", focal = " << cam.focal
                      << ", camera_center_y = " << cam.center_y << "\n";
        config_.rows = rows;
        config_.cols = cols;
        config_.baseline = cam.baseline;
        config_.focal = cam.focal;
        config_.camera_center_y = cam.center_y;
        shutdown();
        stixels_.SetConfig(config_);
        stixels_.Initialize();
        road_.Initialize(config_.camera_center_y, config_.baseline, config_.focal, rows, cols, config_.max_dis);
        ready_ = true;
    }

    // One frame; returns the milliseconds of the timed region or a negative value when the frame was skipped.
    double run(const Disparity& disparity, const isx_apps::NpyInt32& segmentation, const std::string& out_file) {
        stixels_.SetDisparityImage(disparity.values);
        const auto t0 = std::chrono::steady_clock::now();
        stixels_.SetSegmentation(segmentation.data);
        if (!road_.Compute(disparity.values)) {
            std::printf("Road estimation failed.\n");
            return -1.0;
        }
        const int horizon = road_.GetHorizonPoint();
        const float pitch = road_.GetPitch(), height = road_.GetCameraHeight(), slope = road_.GetSlope();
        if (pitch == 0 && height == 0 && horizon == 0 && slope == 0) {
            std::printf("Invalid road estimation.\n");
            return -1.0;
        }
        stixels_.SetRoadParameters(horizon, pitch, height, slope);
        stixels_.Compute(opt_.pairwise, data_);  // synchronous: the Sections are on the host when it returns
        const auto t1 = std::chrono::steady_clock::now();
        const double us = (double)std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
        std::cout << "Done. Time elapsed (s): " << us * 1e-6 << "\n";

        std::map<std::pair<int, int>, int> instances = stixels_.GetInstanceStixels();
        const int per_column = stixels_.GetMaxSections();
        for (const auto& kv : instances) {  // an instance id on a non-instance class would be a bug: say so
            const int cls = data_.sections[(size_t)kv.first.first * per_column + kv.first.second].semantic_class;
            if (cls < 11)
                std::cout << "(" << kv.first.first << "," << kv.first.second << "):" << kv.second << " and class id "
                          << cls << "\n";
        }
        Stixels::SaveStixels(data_.sections.data(), instances, slope, config_.rows - 1 - horizon,
                             stixels_.GetRealCols(), per_column, out_file.c_str());
        std::cout << "Finished.\n";
        return us * 1e-3;
    }

    void shutdown() {
        if (stixels_.IsInitialized()) stixels_.Finish();
        if (road_.IsInitialized()) road_.Finish();
        ready_ = false;
    }

    int rows() const { return (int)config_.rows; }
    int cols() const { return (int)config_.cols; }

private:
    const Options& opt_;
    StixelConfig config_;
    Stixels stixels_;
    RoadEstimation road_;
    StixelsData data_;
    bool ready_ = false;
};

// The segmentation tensor of a frame: the int32 dataset "nlogprobs" of <base>_probs.h5 like the reference
// (H5Segmentation.cpp:25-49, read without libhdf5 by apps/h5_reader.h), or the same array as <base>_probs.npy.
isx_apps::NpyInt32 load_segmentation(const std::string& probs) {
    if (exists(probs + ".h5")) {
        std::cout << "Opening file " << probs << ".h5\n";
        isx_apps::H5Int32 h = isx_apps::load_h5_int32(probs + ".h5", "nlogprobs");
        isx_apps::NpyInt32 out;
        out.shape = h.shape;
        out.data.swap(h.data);
        std::cout << "H5Segmentation shape = (" << (out.shape.empty() ? 0 : out.shape[0]);
        for (size_t i = 1; i < out.shape.size(); i++) std::cout << ", " << out.shape[i];
        std::cout << ")\n";
        return out;
    }
    return isx_apps::load_npy_int32(probs + ".npy");
}

// [cols / stixel_width][21][2^ceil(log2(rows / 8 + 1))]; the reference checks cols / 8 (:363), width 4 needs
// a tensor at cols / 4 columns (SURVEY 8c O3).
bool segmentation_fits(const isx_apps::NpyInt32& seg, int rows, int cols, int column_step) {
    const size_t padded_rows = (size_t)std::pow(2, std::ceil(std::log2(rows / 8 + 1)));
    if (seg.shape.size() != 3 || seg.shape[2] != padded_rows) {
        std::cout << "ERROR: Height of disparity (" << rows << ") and segmentation input ("
                  << (seg.shape.size() == 3 ? seg.shape[2] : 0) << ") do not match. Segmentation input should be "
                  << padded_rows << ".\n";
        return false;
    }
    if (seg.shape[0] != (size_t)(cols / column_step)) {
        std::cout << "ERROR: Width of disparity (" << cols << ") and segmentation input (" << seg.shape[0]
                  << ") do not match.\n";
        return false;
    }
    return true;
}

// ---- extension: --batch B / --gpus G ----
// The same dataset through the batched entry points: all frames are loaded, the road is estimated per frame, and
// runs of frames with one geometry go through a StixelsPool (one context + worker thread per GPU, sub-batches of B
// frames, three in flight) from pinned host buffers.  The .stixels files are the same bytes as the one-frame loop
// writes; the timed region is the pool call (host buffers in -> Sections and instance maps out), after one
// discarded warm-up call like the reference's first frame.
// --road-on-device: no road is estimated while loading.  The pool call estimates every frame's road on the device
// inside its pipeline (isx_pool_compute_host_road), so road estimation is inside the timed region as in the
// reference's loop.  Frames whose estimate failed or is all zeros are reported and skipped after the call, like the
// one-frame loop skips them; they were computed with the camera's nominal road, whose results are discarded.
struct LoadedFrame {
    std::string base;
    int rows = 0, cols = 0;
    isx_apps::Camera cam;
    Stixels::Road road{};
    size_t slot = 0;  // index inside its group's pinned buffers
};

template <typename T>
struct Pinned {
    T* p = nullptr;
    size_t n = 0;
    explicit Pinned(size_t count) : n(count) {
        p = static_cast<T*>(isx_host_alloc(count * sizeof(T)));
        if (!p) throw std::runtime_error("out of pinned host memory");
    }
    ~Pinned() { isx_host_free(p); }
    Pinned(const Pinned&) = delete;
    Pinned& operator=(const Pinned&) = delete;
};

// RoadEstimation's accepted estimate of all zeros, which the reference's loop refuses (apps/run_cityscapes.cu:401-405)
bool invalid_road(const Stixels::Road& r) {
    return r.camera_tilt == 0 && r.camera_height == 0 && r.vhor == 0 && r.alpha_ground == 0;
}

// The road a frame whose estimate fails is computed with under --road-on-device: horizon at the principal point, no
// pitch, a car's camera height.  Its results are discarded; it only has to be a plausible road.
Stixels::Road nominal_road(const isx_apps::Camera& cam) {
    const float height = 1.2f;
    return Stixels::Road{(int)cam.center_y, 0.0f, height, cam.baseline / height};
}

int run_batched(const Options& opt) {
    const std::vector<std::string> bases = list_frames(opt.dataset + "/disparities");
    double total_ms = 0;
    size_t total_frames = 0;
    size_t i = 0;
    RoadEstimation road;
    while (i < bases.size()) {
        // ---- one group: consecutive frames with the geometry of the first usable one ----
        std::vector<LoadedFrame> group;
        std::vector<std::vector<pixel_t>> disp;
        std::vector<std::vector<int32_t>> seg;
        for (; i < bases.size(); i++) {
            const std::string& base = bases[i];
            std::cout << base << "_disparity.png" << std::endl;
            const std::string camera_file = opt.dataset + "/camera/" + base + "_camera.json";
            try {
                Disparity d = load_disparity(opt.dataset + "/disparities/" + base + "_disparity.png", opt.config.max_dis);
                const isx_apps::Camera cam = isx_apps::load_camera(camera_file);
                if (!group.empty()) {
                    const LoadedFrame& g = group.front();
                    if (g.rows != d.rows || g.cols != d.cols || g.cam.baseline != cam.baseline || g.cam.focal != cam.focal ||
                        g.cam.center_y != cam.center_y)
                        break;  // next group starts here
                }
                isx_apps::NpyInt32 s = load_segmentation(opt.dataset + "/probs/" + base + "_probs");
                if (!segmentation_fits(s, d.rows, d.cols, opt.config.column_step)) continue;
                LoadedFrame f;
                f.base = base;
                f.rows = d.rows;
                f.cols = d.cols;
                f.cam = cam;
                if (!opt.road_on_device) {
                    if (group.empty()) {
                        if (road.IsInitialized()) road.Finish();
                        road.Initialize(cam.center_y, cam.baseline, cam.focal, d.rows, d.cols, opt.config.max_dis);
                    }
                    if (!road.Compute(d.values)) {
                        std::printf("Road estimation failed.\n");
                        continue;
                    }
                    f.road = Stixels::Road{road.GetHorizonPoint(), road.GetPitch(), road.GetCameraHeight(),
                                           road.GetSlope()};
                    if (invalid_road(f.road)) {
                        std::printf("Invalid road estimation.\n");
                        continue;
                    }
                }
                f.slot = group.size();
                group.push_back(f);
                disp.push_back(std::move(d.values));
                seg.push_back(std::move(s.data));
            } catch (const std::invalid_argument& err) {
                std::cerr << err.what() << "\n";
            }
        }
        if (group.empty()) continue;
        const int loaded = (int)group.size();
        const int n = loaded * opt.replicate;
        StixelConfig cfg = opt.config;
        cfg.rows = group[0].rows;
        cfg.cols = group[0].cols;
        cfg.baseline = group[0].cam.baseline;
        cfg.focal = group[0].cam.focal;
        cfg.camera_center_y = group[0].cam.center_y;
        std::vector<int> devices;
        for (int g = 0; g < opt.gpus; g++) devices.push_back(g);
        StixelsPool pool(cfg, devices, opt.batch);
        const size_t hw = disp[0].size(), se = seg[0].size();
        Pinned<pixel_t> h_disp((size_t)n * hw);
        Pinned<int32_t> h_seg((size_t)n * se);
        std::vector<Stixels::Road> roads;
        for (int f = 0; f < n; f++) {
            const size_t src = (size_t)(f % loaded);
            std::copy(disp[src].begin(), disp[src].end(), h_disp.p + (size_t)f * hw);
            std::copy(seg[src].begin(), seg[src].end(), h_seg.p + (size_t)f * se);
            roads.push_back(group[src].road);
        }
        const size_t per_frame = (size_t)pool.GetRealCols() * pool.GetMaxSections();
        Pinned<Section> sections((size_t)n * per_frame);   // pinned: the device writes the Sections into it itself
        std::vector<isx_instance> records;   // the reference builds its std::map after the timed region too (:430)
        std::vector<int32_t> offsets;
        const int warm = std::min(n, opt.batch * opt.gpus);
        const Stixels::Road fallback = nominal_road(group[0].cam);
        std::vector<isx_road_estimate> estimates;
        if (opt.road_on_device)   // warm-up
            pool.ComputeBatch(opt.pairwise, warm, h_disp.p, h_seg.p, fallback, &estimates, sections.p, &records, &offsets);
        else
            pool.ComputeBatch(opt.pairwise, warm, h_disp.p, h_seg.p, roads.data(), sections.p, &records, &offsets);
        const auto t0 = std::chrono::steady_clock::now();
        if (opt.road_on_device)
            pool.ComputeBatch(opt.pairwise, n, h_disp.p, h_seg.p, fallback, &estimates, sections.p, &records, &offsets,
                              &roads);
        else
            pool.ComputeBatch(opt.pairwise, n, h_disp.p, h_seg.p, roads.data(), sections.p, &records, &offsets);
        const auto t1 = std::chrono::steady_clock::now();
        const double ms = (double)std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count() * 1e-3;
        std::cout << "Done. Time elapsed (s): " << ms * 1e-3 << " for " << n << " frames on " << pool.Size()
                  << " GPU worker(s), sub-batches of " << opt.batch << "\n";
        {
            std::cerr << "frames by worker:";   // a worker that is done takes sub-batches over from the fullest block
            for (int fw : pool.FramesByWorker()) std::cerr << " " << fw;
            std::cerr << "\n";
        }
        total_ms += ms;
        total_frames += (size_t)n;
        const size_t per = per_frame;
        for (int f = 0; f < loaded; f++) {
            LoadedFrame& lf = group[(size_t)f];
            if (opt.road_on_device) {
                if (!estimates[(size_t)f].ok) {
                    std::cout << lf.base << ": ";
                    std::printf("Road estimation failed.\n");
                    continue;
                }
                lf.road = roads[(size_t)f];   // the frame's own estimate (the pool's per-frame rule)
                if (invalid_road(lf.road)) {
                    std::cout << lf.base << ": ";
                    std::printf("Invalid road estimation.\n");
                    continue;
                }
            }
            Stixels::SaveStixels(sections.p + (size_t)f * per, StixelsPool::MapOf(records, offsets, f), lf.road.alpha_ground,
                                 lf.rows - 1 - lf.road.vhor, pool.GetRealCols(), pool.GetMaxSections(),
                                 (opt.dataset + "/stixels/" + lf.base + ".stixels").c_str());
        }
        std::cout << "Finished.\n";
    }
    if (road.IsInitialized()) road.Finish();
    const float mean = (float)(total_ms / (double)total_frames);
    std::cout << "It took an average of " << mean << " milliseconds, " << 1000.0f / mean << " fps" << std::endl;
    return 0;
}

}  // namespace

int main(int argc, char* argv[]) {
    Options opt;
    if (!parse_options(argc, argv, &opt)) return -1;
    if (opt.road_on_device && opt.batch <= 1 && opt.gpus <= 1) {
        std::cerr << "--road-on-device applies to the batched mode: give --batch B (B > 1) or --gpus G (G > 1).\n";
        return -1;
    }
    if (opt.batch > 1 || opt.gpus > 1) return run_batched(opt);
    Pipeline pipeline(opt);
    std::vector<double> frame_ms;
    bool warm = false;
    for (const std::string& base : list_frames(opt.dataset + "/disparities")) {
        std::cout << base << "_disparity.png" << std::endl;
        const std::string camera_file = opt.dataset + "/camera/" + base + "_camera.json";
        const std::string probs = opt.dataset + "/probs/" + base + "_probs";
        try {
            const Disparity disparity = load_disparity(opt.dataset + "/disparities/" + base + "_disparity.png",
                                                       opt.config.max_dis);
            if (exists(camera_file)) std::cout << "File " << camera_file << " exists.\n";
            else std::cout << "Warning: Camera file " << camera_file
                           << " does not exist. Falling back to UEYE parameters!\n";
            pipeline.prepare(disparity.rows, disparity.cols, isx_apps::load_camera(camera_file));
            const isx_apps::NpyInt32 segmentation = load_segmentation(probs);
            if (!segmentation_fits(segmentation, disparity.rows, disparity.cols, opt.config.column_step)) continue;
            const double ms = pipeline.run(disparity, segmentation, opt.dataset + "/stixels/" + base + ".stixels");
            if (ms < 0) continue;
            if (warm) frame_ms.push_back(ms);  // the first frame is the warm-up
            warm = true;
        } catch (const std::invalid_argument& err) {
            std::cerr << err.what() << "\n";
        }
    }
    const float mean = (float)(std::accumulate(frame_ms.begin(), frame_ms.end(), 0.0) / frame_ms.size());
    std::cout << "It took an average of " << mean << " milliseconds, " << 1000.0f / mean << " fps" << std::endl;
    pipeline.shutdown();
    return 0;
}
