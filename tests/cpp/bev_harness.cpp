// Stixels::GetBevGrid of the drop-in header over the frames of a batch, for comparison with the device grid:
//   bev_harness <sections.bin> <roads.bin> <n> <rows> <realcols> <column_step> <focal> <baseline> <cx> <cy>
//               <x_min> <z_min> <cell> <nx> <nz> <cells.out>
// sections.bin = [n][realcols][200] Sections; roads.bin = n records {float alpha_ground; int32 vhor} with vhor the
// flipped horizon of StixelsData.  Writes the [nz][nx] cells of frame 0, 1, ... back to back (8 bytes each) and prints
// "cells <count>".  A refused call (no camera centre, parameters out of range) prints "refused: <message>" and writes
// nothing.  Built with -ffp-contract=off, so every operation is rounded like the header says.  Needs no device.
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

struct FrameRoad {
    float alpha_ground;
    int32_t vhor;
};

int main(int argc, char* argv[]) {
    if (argc < 17) return 2;
    const int n = atoi(argv[3]), rows = atoi(argv[4]), realcols = atoi(argv[5]), step = atoi(argv[6]);
    StixelConfig camera;
    camera.focal = strtof(argv[7], nullptr);
    camera.baseline = strtof(argv[8], nullptr);
    camera.camera_center_x = strtof(argv[9], nullptr);
    camera.camera_center_y = strtof(argv[10], nullptr);
    isx_bev_params p{strtof(argv[11], nullptr), strtof(argv[12], nullptr), strtof(argv[13], nullptr),
                     atoi(argv[14]), atoi(argv[15]), 0};
    const int per = realcols * ISX_MAX_STIXELS_PER_COLUMN;
    const std::vector<Section> sections = read_all<Section>(argv[1], (size_t)n * per);
    const std::vector<FrameRoad> roads = read_all<FrameRoad>(argv[2], (size_t)n);

    std::ofstream out(argv[16], std::ios::binary);
    size_t total = 0;
    for (int f = 0; f < n; f++) {
        StixelsData d;
        d.sections.assign(sections.begin() + (size_t)f * per, sections.begin() + (size_t)(f + 1) * per);
        d.rows = rows;
        d.cols = realcols * step;
        d.realcols = realcols;
        d.max_sections = ISX_MAX_STIXELS_PER_COLUMN;
        d.max_dis = 128;
        d.column_step = step;
        d.semantic_classes = 19;
        d.alpha_ground = roads[(size_t)f].alpha_ground;
        d.vhor = roads[(size_t)f].vhor;
        std::vector<isx_bev_cell> cells;
        try {
            cells = Stixels::GetBevGrid(camera, d, p);
        } catch (const std::invalid_argument& e) {
            std::cout << "refused: " << e.what() << std::endl;
            return 0;
        }
        out.write(reinterpret_cast<const char*>(cells.data()), (std::streamsize)(cells.size() * sizeof(isx_bev_cell)));
        total += cells.size();
    }
    std::cout << "cells " << total << std::endl;
    return out ? 0 : 1;
}
