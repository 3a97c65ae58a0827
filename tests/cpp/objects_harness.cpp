// Stixels::GetInstanceObjects of the drop-in header over the frames of a batch, for comparison with the device objects:
//   objects_harness <sections.bin> <instances.bin> <offsets.bin> <n> <rows> <cols> <column_step> <focal> <baseline>
//                   <cx> <cy> <objects.out> <extents.out>
// sections.bin = [n][realcols][200] Sections; instances.bin = the packed isx_instance records of the frames, frame f
// at [offsets[f], offsets[f+1]); offsets.bin = n+1 int32.  Writes the objects of frame 0, 1, ... back to back (48
// bytes each) and their extents (6 floats each) and prints "objects <count>".  cx == -1: no camera centre; the
// extents are asked for once, the refusal is printed ("refused: <message>") and only the objects are written.
// Built with -ffp-contract=off, so every operation is rounded like the header says.  Needs no device.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <vector>

#include "Stixels.hpp"

template <typename T>
static std::vector<T> read_all(const char* path, size_t n) {
    std::vector<T> v(n);
    std::ifstream f(path, std::ios::binary);
    f.read(reinterpret_cast<char*>(v.data()), n * sizeof(T));
    if (!f) { std::cerr << "short read: " << path << "\n"; std::exit(2); }
    return v;
}

int main(int argc, char* argv[]) {
    if (argc < 14) return 2;
    const int n = atoi(argv[4]), rows = atoi(argv[5]), cols = atoi(argv[6]), step = atoi(argv[7]);
    StixelConfig camera;
    camera.focal = strtof(argv[8], nullptr);
    camera.baseline = strtof(argv[9], nullptr);
    camera.camera_center_x = strtof(argv[10], nullptr);
    camera.camera_center_y = strtof(argv[11], nullptr);
    const int realcols = cols / step, per = realcols * ISX_MAX_STIXELS_PER_COLUMN;
    const std::vector<Section> sections = read_all<Section>(argv[1], (size_t)n * per);
    const std::vector<int32_t> offsets = read_all<int32_t>(argv[3], (size_t)n + 1);
    const std::vector<isx_instance> inst = read_all<isx_instance>(argv[2], (size_t)offsets[(size_t)n]);
    const bool with_extents = camera.camera_center_x != -1;

    std::ofstream out_objects(argv[12], std::ios::binary), out_extents(argv[13], std::ios::binary);
    size_t total = 0;
    for (int f = 0; f < n; f++) {
        StixelsData d;
        d.sections.assign(sections.begin() + (size_t)f * per, sections.begin() + (size_t)(f + 1) * per);
        d.rows = rows;
        d.cols = cols;
        d.realcols = realcols;
        d.max_sections = ISX_MAX_STIXELS_PER_COLUMN;
        d.max_dis = 128;
        d.column_step = step;
        d.semantic_classes = 19;
        d.alpha_ground = 0.0f;
        d.vhor = 0;
        Stixels::InstanceMap map;
        for (int32_t i = offsets[(size_t)f]; i < offsets[(size_t)f + 1]; i++)
            map[std::make_pair(inst[(size_t)i].column, inst[(size_t)i].index)] = inst[(size_t)i].label;
        std::vector<float> extents;
        if (!with_extents && f == 0) {
            try {
                Stixels::GetInstanceObjects(camera, d, map, &extents);
                std::cerr << "extents without a camera centre were not refused\n";
                return 1;
            } catch (const std::invalid_argument& e) {
                std::cout << "refused: " << e.what() << std::endl;
            }
        }
        const std::vector<isx_object> objects =
            Stixels::GetInstanceObjects(camera, d, map, with_extents ? &extents : nullptr);
        out_objects.write(reinterpret_cast<const char*>(objects.data()),
                          (std::streamsize)(objects.size() * sizeof(isx_object)));
        out_extents.write(reinterpret_cast<const char*>(extents.data()),
                          (std::streamsize)(extents.size() * sizeof(float)));
        total += objects.size();
    }
    std::cout << "objects " << total << std::endl;
    return out_objects && out_extents ? 0 : 1;
}
