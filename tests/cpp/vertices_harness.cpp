// Stixels::Get3DVertices of the drop-in header over the frames of a batch, for comparison with the device export:
//   vertices_harness <sections.bin> <roads.bin> <n> <rows> <cols> <column_step> <focal> <baseline> <cx> <cy> <out.f32>
// sections.bin = [n][realcols][200] Sections as ComputeBatch returns them; roads.bin = n x {float alpha_ground,
// int32 vhor} with vhor flipped like StixelsData::vhor.  Writes the vertices of frame 0, 1, ... back to back and
// prints "vertices <floats>".  Built with -ffp-contract=off, so every operation is rounded like the header says.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
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
    if (argc < 12) return 2;
    const int n = atoi(argv[3]), rows = atoi(argv[4]), cols = atoi(argv[5]), step = atoi(argv[6]);
    const float focal = strtof(argv[7], nullptr), baseline = strtof(argv[8], nullptr);
    const float cx = strtof(argv[9], nullptr), cy = strtof(argv[10], nullptr);
    const int realcols = cols / step, per = realcols * ISX_MAX_STIXELS_PER_COLUMN;
    const std::vector<Section> sections = read_all<Section>(argv[1], (size_t)n * per);
    const std::vector<int32_t> roads = read_all<int32_t>(argv[2], (size_t)n * 2);

    Stixels stixels;
    stixels.SetCameraParameters(focal, baseline, 0.05f, 0.05f, cx, cy);
    std::ofstream out(argv[11], std::ios::binary);
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
        std::memcpy(&d.alpha_ground, &roads[(size_t)f * 2], sizeof(float));
        d.vhor = roads[(size_t)f * 2 + 1];
        const std::vector<float> v = stixels.Get3DVertices(d);
        out.write(reinterpret_cast<const char*>(v.data()), (std::streamsize)(v.size() * sizeof(float)));
        total += v.size();
    }
    std::cout << "vertices " << total << std::endl;
    return out ? 0 : 1;
}
