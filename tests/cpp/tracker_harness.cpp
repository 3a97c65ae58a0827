// HostObjectTracker of the drop-in header over a record stream, for the tracking tests:
//   tracker_harness <iou_min_permille> <max_age> <margin_bits> <max_tracks> <objects.bin> <offsets.bin> <calls.txt>
//                   <ids.out> <hits.out> <flags.out> <state.out>
// objects.bin = isx_object records, offsets.bin = int32 frame offsets of the whole stream (frames back to back);
// calls.txt = one "n capacity reset" line per call: the call's n frames have the offsets of the stream rebased to the
// call's first object, `capacity` counts objects from there, reset != 0 resets the tracker before the call.
// margin_bits = the float's bit pattern.  Writes, per call, the outputs of isx_tracker_update_device aligned with the
// stream's objects (an object of an unwritten frame keeps the 0x5A fill), the flags of every frame, the live tracks
// after the last call (isx_track records ordered by id) and prints "next_id <id>".  Needs no device.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <vector>

#include "ObjectTracker.hpp"

template <typename T>
static std::vector<T> read_file(const char* path) {
    std::ifstream f(path, std::ios::binary);
    std::vector<char> bytes((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
    std::vector<T> v(bytes.size() / sizeof(T));
    if (!v.empty()) std::memcpy(v.data(), bytes.data(), v.size() * sizeof(T));
    return v;
}

template <typename T>
static void write_file(const char* path, const std::vector<T>& v) {
    std::ofstream f(path, std::ios::binary);
    f.write(reinterpret_cast<const char*>(v.data()), (std::streamsize)(v.size() * sizeof(T)));
}

int main(int argc, char* argv[]) {
    if (argc < 12) return 2;
    isx_track_params p;
    p.iou_min_permille = std::atoi(argv[1]);
    p.max_age = std::atoi(argv[2]);
    const uint32_t bits = (uint32_t)std::strtoul(argv[3], nullptr, 0);
    std::memcpy(&p.disparity_margin, &bits, sizeof bits);
    p.max_tracks = std::atoi(argv[4]);
    const std::vector<isx_object> objects = read_file<isx_object>(argv[5]);
    const std::vector<int32_t> offsets = read_file<int32_t>(argv[6]);
    const int frames = (int)offsets.size() - 1;
    std::vector<int64_t> ids(objects.size());
    std::vector<int32_t> hits(objects.size()), flags((size_t)frames);
    std::memset(ids.data(), 0x5A, ids.size() * sizeof(int64_t));
    std::memset(hits.data(), 0x5A, hits.size() * sizeof(int32_t));
    try {
        HostObjectTracker tracker(p);
        std::ifstream calls(argv[7]);
        int n = 0, capacity = 0, reset = 0, f0 = 0;
        while (calls >> n >> capacity >> reset) {
            if (reset) tracker.Reset();
            const int base = offsets[(size_t)f0];
            std::vector<int32_t> rel((size_t)n + 1);
            for (int f = 0; f <= n; f++) rel[(size_t)f] = offsets[(size_t)(f0 + f)] - base;
            tracker.UpdateBatch(n, objects.data() + base, rel.data(), capacity, ids.data() + base, hits.data() + base,
                                flags.data() + f0);
            f0 += n;
        }
        if (f0 != frames) {
            std::cerr << "calls cover " << f0 << " of " << frames << " frames\n";
            return 2;
        }
        write_file(argv[8], ids);
        write_file(argv[9], hits);
        write_file(argv[10], flags);
        write_file(argv[11], tracker.Tracks());
        std::cout << "next_id " << tracker.NextId() << std::endl;
    } catch (const std::invalid_argument& e) {
        std::cout << "refused: " << e.what() << std::endl;
        return 3;
    }
    return 0;
}
