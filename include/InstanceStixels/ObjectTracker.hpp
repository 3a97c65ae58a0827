// Persistent ids for the objects of a frame stream (no reference counterpart).
//
// The DBSCAN labels of a frame's objects (Stixels::GetInstanceObjects, isx_export_objects_device) are numbered in
// column order, per frame and per class: "car 0" of one frame and "car 0" of the next are unrelated.  A tracker links
// the objects of consecutive frames by their image boxes and disparity ranges and gives every chain one int64 id.
//
// HostObjectTracker is the statement of the definition, on the host; isx_tracker_update_device computes the same bytes
// on the device (the definition is also summarised in include/instance_stixels_b200.h).  It consumes the isx_object
// records of one frame per call, in export order (by class, then label).  Its state is a set of live tracks, each with
// an id, a class, the box and disparity range of its last matched object, `hits` (frames in which it was matched, its
// birth included) and `misses` (consecutive frames without a match).  For each frame, each class c in 11..18 on its own:
//   1. Candidates: every (live track t of class c, object o of class c) with
//      - overlapping inclusive boxes: I = intersection area > 0, U = area(t) + area(o) - I;
//      - 1000 * I >= iou_min_permille * U, in int64;
//      - the disparity gate !(o.min > t.max + margin) && !(t.min > o.max + margin), each sum one round-to-nearest float
//        add, subnormals kept.  The gate passes when any of the four bounds is NaN (an object whose members all have
//        NaN disparity holds 0x7FC00000), and a NaN sum passes its comparison, so margin = +inf turns the gate off.
//   2. Greedy association: candidates ordered by IoU descending (I1 * U2 against I2 * U1 in int64, no float), then
//      track id ascending, then object label ascending; walking that list, a pair is accepted when neither its track
//      nor its object is taken yet.  The order is strict, so the matching is unique.
//   3. A matched track takes the object's box and disparity range, hits += 1, misses = 0; the object gets the track's
//      id and its new hits.
//   4. An unmatched track gets misses += 1 and is removed when misses > max_age.  Its id is never used again.
//   5. Unmatched objects become new tracks with hits = 1, in label order, while the class holds fewer than max_tracks
//      live tracks.  An object left over gets id -1 and hits 0 and sets ISX_TRACK_UNMATCHED in the frame's flags.
// Ids come from one tracker-wide counter starting at 0, handed out in record order within a frame (class, then label);
// an object without a track uses up no id.  A frame whose records were not written (the export's capacity rule,
// frame_offsets[f+1] > capacity) sets ISX_TRACK_NOT_WRITTEN and counts as a frame without objects: every track ages.
// IoU products are exact while every box side stays below 2^15 pixels.  Compile without -ffast-math: the gate relies
// on IEEE float adds and comparisons.
//
// Out of scope: motion models (a track's box is that of its last object), optimal (Hungarian) assignment, 3D
// association and re-identification of removed tracks.
//
// ObjectTracker is the RAII handle over the device tracker (isx_tracker_*).  Like the other drop-in classes it throws
// std::invalid_argument for refused arguments and prints and exits on CUDA failures.
#ifndef ISX_DROPIN_OBJECTTRACKER_HPP_
#define ISX_DROPIN_OBJECTTRACKER_HPP_

#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <vector>

#include "../instance_stixels_b200.h"

class HostObjectTracker {
public:
    explicit HostObjectTracker(const isx_track_params& p) : p_(p) {
        if (p.iou_min_permille < 1 || p.iou_min_permille > 1000)
            throw std::invalid_argument("iou_min_permille must be in 1..1000");
        if (p.max_age < 0) throw std::invalid_argument("max_age must be >= 0");
        if (std::isnan(p.disparity_margin) || p.disparity_margin < 0)
            throw std::invalid_argument("disparity_margin must be >= 0 and not NaN");
        if (p.max_tracks < 1) throw std::invalid_argument("max_tracks must be >= 1");
    }

    // One frame: its `count` records in export order.  track_ids / hits [count] receive the id and hits of every
    // object (either may be null).  Returns the frame's flags.
    int Update(const isx_object* objects, int count, int64_t* track_ids, int32_t* hits) {
        int flags = 0;
        for (int k = 0; k < ISX_INSTANCE_CLASSES; k++) {
            std::vector<int> objs;
            for (int j = 0; j < count; j++)
                if (objects[j].semantic_class == ISX_FIRST_INSTANCE_CLASS + k) objs.push_back(j);
            flags |= UpdateClass(k, objects, objs, track_ids, hits);
        }
        return flags;
    }
    // A frame whose records were not written: every track ages.
    int UpdateNotWritten() {
        for (int k = 0; k < ISX_INSTANCE_CLASSES; k++) UpdateClass(k, nullptr, std::vector<int>(), nullptr, nullptr);
        return ISX_TRACK_NOT_WRITTEN;
    }
    // n frames laid out like isx_device_objects (host memory): what isx_tracker_update_device computes.  Outputs are
    // aligned with `objects`; only the objects of written frames are written.  frame_flags [n] may be null.
    void UpdateBatch(int n, const isx_object* objects, const int32_t* frame_offsets, int capacity, int64_t* track_ids,
                     int32_t* hits, int32_t* frame_flags) {
        for (int f = 0; f < n; f++) {
            const int lo = frame_offsets[f], hi = frame_offsets[f + 1];
            const int flags = hi <= capacity
                                  ? Update(objects + lo, hi - lo, track_ids ? track_ids + lo : nullptr,
                                           hits ? hits + lo : nullptr)
                                  : UpdateNotWritten();
            if (frame_flags) frame_flags[f] = flags;
        }
    }
    void Reset() {
        for (auto& v : tracks_) v.clear();
        next_id_ = 0;
    }
    // The live tracks, ordered by id.
    std::vector<isx_track> Tracks() const {
        std::vector<isx_track> out;
        for (const auto& v : tracks_) out.insert(out.end(), v.begin(), v.end());
        std::sort(out.begin(), out.end(), [](const isx_track& a, const isx_track& b) { return a.id < b.id; });
        return out;
    }
    int64_t NextId() const { return next_id_; }

    // The candidate test of step 1 for track t and object o: false, or true with the intersection and union areas.
    static bool Candidate(const isx_track_params& p, const isx_track& t, const isx_object& o, int64_t& I,
                          int64_t& U) {
        const int64_t w = (int64_t)std::min(t.x1, o.x1) - std::max(t.x0, o.x0) + 1;
        const int64_t h = (int64_t)std::min(t.y1, o.y1) - std::max(t.y0, o.y0) + 1;
        if (w <= 0 || h <= 0) return false;
        I = w * h;
        U = Area(t.x0, t.y0, t.x1, t.y1) + Area(o.x0, o.y0, o.x1, o.y1) - I;
        if (1000 * I < (int64_t)p.iou_min_permille * U) return false;
        if (std::isnan(t.disparity_min) || std::isnan(t.disparity_max) || std::isnan(o.disparity_min) ||
            std::isnan(o.disparity_max))
            return true;
        const float t_reach = t.disparity_max + p.disparity_margin, o_reach = o.disparity_max + p.disparity_margin;
        return !(o.disparity_min > t_reach) && !(t.disparity_min > o_reach);
    }

private:
    struct Pair {
        int64_t I, U;
        int t, o;   // index into the class's tracks, index into `objs`
    };

    static int64_t Area(int32_t x0, int32_t y0, int32_t x1, int32_t y1) {
        return ((int64_t)x1 - x0 + 1) * ((int64_t)y1 - y0 + 1);
    }

    // Steps 1-5 for class 11 + k; objs = indices of the class's objects in label order.  Returns the flags it sets.
    int UpdateClass(int k, const isx_object* objects, const std::vector<int>& objs, int64_t* track_ids,
                    int32_t* hits) {
        std::vector<isx_track>& tr = tracks_[k];
        std::vector<Pair> pairs;
        for (int t = 0; t < (int)tr.size(); t++)
            for (int o = 0; o < (int)objs.size(); o++) {
                Pair c{0, 0, t, o};
                if (Candidate(p_, tr[(size_t)t], objects[objs[(size_t)o]], c.I, c.U)) pairs.push_back(c);
            }
        std::sort(pairs.begin(), pairs.end(), [&](const Pair& a, const Pair& b) {
            const int64_t l = a.I * b.U, r = b.I * a.U;
            if (l != r) return l > r;
            if (tr[(size_t)a.t].id != tr[(size_t)b.t].id) return tr[(size_t)a.t].id < tr[(size_t)b.t].id;
            return objects[objs[(size_t)a.o]].label < objects[objs[(size_t)b.o]].label;
        });
        std::vector<int> track_of(objs.size(), -1), object_of(tr.size(), -1);
        for (const Pair& c : pairs)
            if (object_of[(size_t)c.t] < 0 && track_of[(size_t)c.o] < 0) {
                object_of[(size_t)c.t] = c.o;
                track_of[(size_t)c.o] = c.t;
            }
        std::vector<isx_track> kept;
        for (size_t t = 0; t < tr.size(); t++) {
            isx_track x = tr[t];
            if (object_of[t] >= 0) {
                const int j = objs[(size_t)object_of[t]];
                Take(x, objects[j]);
                x.hits += 1;
                x.misses = 0;
                if (track_ids) track_ids[j] = x.id;
                if (hits) hits[j] = x.hits;
            } else {
                x.misses += 1;
            }
            if (x.misses <= p_.max_age) kept.push_back(x);
        }
        tr.swap(kept);
        int flags = 0;
        for (size_t o = 0; o < objs.size(); o++) {
            if (track_of[o] >= 0) continue;
            const int j = objs[o];
            if ((int)tr.size() < p_.max_tracks) {
                isx_track x{next_id_++, ISX_FIRST_INSTANCE_CLASS + k, 1, 0, 0, 0, 0, 0, 0.0f, 0.0f, 0};
                Take(x, objects[j]);
                tr.push_back(x);
                if (track_ids) track_ids[j] = x.id;
                if (hits) hits[j] = 1;
            } else {
                if (track_ids) track_ids[j] = -1;
                if (hits) hits[j] = 0;
                flags |= ISX_TRACK_UNMATCHED;
            }
        }
        return flags;
    }
    static void Take(isx_track& t, const isx_object& o) {
        t.x0 = o.x0; t.y0 = o.y0; t.x1 = o.x1; t.y1 = o.y1;
        t.disparity_min = o.disparity_min;
        t.disparity_max = o.disparity_max;
    }

    isx_track_params p_;
    std::vector<isx_track> tracks_[ISX_INSTANCE_CLASSES];   // per class, ids ascending
    int64_t next_id_ = 0;
};

// RAII handle over the device tracker (isx_tracker_*).  params == nullptr: isx_track_params_init's defaults.
class ObjectTracker {
public:
    explicit ObjectTracker(int device = 0, const isx_track_params* params = nullptr) {
        check(isx_tracker_create(&t_, device, params));
    }
    ~ObjectTracker() { isx_tracker_destroy(t_); }
    ObjectTracker(const ObjectTracker&) = delete;
    ObjectTracker& operator=(const ObjectTracker&) = delete;

    // The n frames of `in` (isx_export_objects_device's output) as the next frames of the sequence; asynchronous on
    // `stream` (a cudaStream_t as an integer, e.g. isx_stream()).  Outputs as for isx_tracker_update_device.
    void UpdateDevice(uint64_t stream, int n, const isx_device_objects& in, int64_t* d_track_ids,
                      int32_t* d_hits = nullptr, int32_t* d_frame_flags = nullptr) {
        check(isx_tracker_update_device(t_, stream, n, &in, d_track_ids, d_hits, d_frame_flags));
    }
    void Reset() { check(isx_tracker_reset(t_)); }
    // Waits for the updates in flight; the live tracks ordered by id.
    std::vector<isx_track> State(int64_t* next_id = nullptr) {
        int n = 0;
        check(isx_tracker_read_state(t_, nullptr, 0, &n, nullptr));
        std::vector<isx_track> out((size_t)n);
        check(isx_tracker_read_state(t_, out.data(), n, &n, next_id));
        return out;
    }
    isx_tracker_handle handle() { return t_; }

private:
    void check(int rc) {
        if (rc == ISX_OK) return;
        if (rc == ISX_ERR_INVALID_ARGUMENT || rc == ISX_ERR_UNSUPPORTED)
            throw std::invalid_argument(isx_tracker_last_error(t_));
        std::cerr << "instance_stixels_b200: " << isx_tracker_last_error(t_) << std::endl;
        std::exit(1);
    }
    isx_tracker_handle t_ = nullptr;
};

#endif  // ISX_DROPIN_OBJECTTRACKER_HPP_
