"""The tracking definition (HostObjectTracker in include/InstanceStixels/ObjectTracker.hpp) on hand-built record
sequences with literal ids and hits, through tests/cpp/tracker_harness.cpp.  No device."""
import ctypes as C
import os
import re
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

from instance_stixels_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAN = float("nan")
DEFAULTS = dict(iou_min_permille=300, max_age=2, disparity_margin=2.0, max_tracks=1024)


def build_harness(tmp_path):
    exe = str(tmp_path / "tracker_harness")
    cmd = ["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include", "InstanceStixels"),
           os.path.join(ROOT, "tests", "cpp", "tracker_harness.cpp"), "-o", exe]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


class Bits(int):
    """A float32 disparity given by its bit pattern.  Subnormals written this way survive in a process that flushes
    them (a library loaded earlier may have set FTZ / DAZ, and a float conversion would then give 0)."""


def frame(*objs):
    """isx_object records of one frame in export order from (class, (x0, y0, x1, y1)[, dmin, dmax]) tuples: sorted by
    class (stable), labels numbered within each class.  Disparities are floats or Bits."""
    objs = sorted(objs, key=lambda o: o[0])
    out, bits, seen = [], [], {}
    for o in objs:
        cls, (x0, y0, x1, y1) = o[0], o[1]
        d = (o[2], o[3]) if len(o) > 2 else (5.0, 5.0)
        label = seen.get(cls, 0)
        seen[cls] = label + 1
        out.append((cls, label, 1, (x1 - x0 + 1) * (y1 - y0 + 1), 0, 0, x0, y0, x1, y1) +
                   tuple(0.0 if isinstance(v, Bits) else v for v in d))
        bits.append(d)
    arr = np.array(out, dtype=L.OBJECT_DTYPE)
    for i, d in enumerate(bits):
        for name, v in zip(("disparity_min", "disparity_max"), d):
            if isinstance(v, Bits):
                arr[name].view(np.uint32)[i] = int(v)
    return arr


def stream(frames):
    """(objects, frame offsets, class offsets) of frames back to back, as isx_export_objects_device lays them out."""
    objects = np.concatenate([np.asarray(f, dtype=L.OBJECT_DTYPE) for f in frames]) if frames else \
        np.zeros(0, L.OBJECT_DTYPE)
    counts = np.zeros((len(frames), 8), np.int64)
    for i, f in enumerate(frames):
        for c in np.asarray(f, dtype=L.OBJECT_DTYPE)["semantic_class"]:
            counts[i, int(c) - 11] += 1
    co = np.concatenate([[0], np.cumsum(counts.reshape(-1))]).astype(np.int32)
    return objects, co[::8].copy(), co


def margin_bits(m):
    return struct.unpack("<I", struct.pack("<f", m))[0]


def run_host(exe, tmp_path, objects, frame_offsets, calls, **params):
    """The harness over a stream.  calls = [(n, capacity, reset)], the frames of each call back to back.  Returns
    ids, hits (aligned with the objects, 0x5A where not written), flags, state and next_id."""
    p = dict(DEFAULTS, **params)
    objects.tofile(tmp_path / "objects.bin")
    np.asarray(frame_offsets, np.int32).tofile(tmp_path / "offsets.bin")
    (tmp_path / "calls.txt").write_text("".join(f"{n} {cap} {int(r)}\n" for n, cap, r in calls))
    out = [str(tmp_path / x) for x in ("ids.bin", "hits.bin", "flags.bin", "state.bin")]
    r = subprocess.run([exe, str(p["iou_min_permille"]), str(p["max_age"]), hex(margin_bits(p["disparity_margin"])),
                        str(p["max_tracks"]), str(tmp_path / "objects.bin"), str(tmp_path / "offsets.bin"),
                        str(tmp_path / "calls.txt")] + out, capture_output=True, text=True)
    if r.returncode == 3:
        return dict(refused=r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
    return dict(ids=np.fromfile(out[0], np.int64), hits=np.fromfile(out[1], np.int32),
                flags=np.fromfile(out[2], np.int32), state=np.fromfile(out[3], L.TRACK_DTYPE),
                next_id=int(re.search(r"next_id (-?\d+)", r.stdout).group(1)))


def track(exe, tmp_path, frames, **params):
    """One call over all frames; ids and hits per frame as lists."""
    objects, fo, _ = stream(frames)
    r = run_host(exe, tmp_path, objects, fo, [(len(frames), len(objects), 0)], **params)
    r["frame_ids"] = [r["ids"][fo[f]:fo[f + 1]].tolist() for f in range(len(frames))]
    r["frame_hits"] = [r["hits"][fo[f]:fo[f + 1]].tolist() for f in range(len(frames))]
    return r


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_harness(tmp_path_factory.mktemp("tracker"))


BOX = (100, 200, 139, 259)


def test_track_structs_are_16_and_48_bytes():
    assert C.sizeof(L.TrackParams) == 16 and L.TRACK_DTYPE.itemsize == 48


def test_static_object_keeps_id_0_while_hits_count(exe, tmp_path):
    r = track(exe, tmp_path, [frame((11, BOX))] * 10)
    assert r["frame_ids"] == [[0]] * 10
    assert r["frame_hits"] == [[h] for h in range(1, 11)]
    assert r["flags"].tolist() == [0] * 10 and r["next_id"] == 1
    assert r["state"][["id", "semantic_class", "hits", "misses", "x0", "y0", "x1", "y1"]].tolist() == \
        [(0, 11, 10, 0) + BOX]


def test_object_absent_for_max_age_frames_keeps_its_id(exe, tmp_path):
    r = track(exe, tmp_path, [frame((11, BOX)), frame(), frame(), frame((11, BOX))])
    assert r["frame_ids"] == [[0], [], [], [0]] and r["frame_hits"][3] == [2]
    assert r["next_id"] == 1


def test_object_absent_for_one_frame_more_gets_a_new_id_and_the_old_one_never_returns(exe, tmp_path):
    frames = [frame((11, BOX)), frame(), frame(), frame(), frame((11, BOX))] + [frame((11, BOX), (12, BOX))] * 3
    r = track(exe, tmp_path, frames)
    assert r["frame_ids"] == [[0], [], [], [], [1], [1, 2], [1, 2], [1, 2]]
    assert r["frame_hits"][4:] == [[1], [2, 1], [3, 2], [4, 3]]
    assert r["state"]["id"].tolist() == [1, 2] and r["next_id"] == 3
    # the same with max_age 3: the object is found again
    r = track(exe, tmp_path, frames[:5], max_age=3)
    assert r["frame_ids"][4] == [0]


def test_on_iou_ties_the_lower_track_id_wins(exe, tmp_path):
    left, right, middle = (0, 0, 9, 9), (10, 0, 19, 9), (5, 0, 14, 9)   # the middle box has IoU 1/3 with both
    # the right box is seen first, so its track has the lower id and the higher label in frame 1
    r = track(exe, tmp_path, [frame((11, right)), frame((11, left), (11, right)), frame((11, middle))])
    assert r["frame_ids"] == [[0], [1, 0], [0]]


def test_on_iou_ties_the_lower_label_wins(exe, tmp_path):
    r = track(exe, tmp_path, [frame((11, (5, 0, 14, 9))), frame((11, (0, 0, 9, 9)), (11, (10, 0, 19, 9)))])
    assert r["frame_ids"] == [[0], [0, 1]] and r["frame_hits"][1] == [2, 1]


def test_the_same_box_in_two_classes_makes_two_tracks(exe, tmp_path):
    r = track(exe, tmp_path, [frame((13, BOX), (11, BOX))] * 2)
    assert r["frame_ids"] == [[0, 1], [0, 1]]   # records by class: 11 first
    assert r["state"]["semantic_class"].tolist() == [11, 13]


def test_the_disparity_gate_blocks_a_pair_and_a_nan_bound_lets_it_pass(exe, tmp_path):
    frames = [frame((11, BOX, 10.0, 10.0)), frame((11, BOX, 20.0, 20.0)), frame((11, BOX, NAN, NAN))]
    r = track(exe, tmp_path, frames)
    # 20 > 10 + 2: blocked, a new track; the NaN object ties both tracks and takes the lower id
    assert r["frame_ids"] == [[0], [1], [0]]
    r = track(exe, tmp_path, frames[:2] + [frame((11, BOX, 20.0, 20.0))])
    assert r["frame_ids"][2] == [1]
    r = track(exe, tmp_path, frames[:2], disparity_margin=float("inf"))
    assert r["frame_ids"] == [[0], [0]]
    r = track(exe, tmp_path, [frame((11, BOX, 30.0, float("-inf"))), frame((11, BOX, float("inf"), 0.0))],
              disparity_margin=float("inf"))
    assert r["frame_ids"] == [[0], [0]]   # -inf + inf is NaN: a +inf margin passes every pair
    r = track(exe, tmp_path, frames[:2], disparity_margin=10.0)
    assert r["frame_ids"] == [[0], [0]]


def test_the_disparity_gate_keeps_subnormals(exe, tmp_path):
    tiny, two = Bits(1), Bits(2)   # the smallest subnormal and twice it
    r = track(exe, tmp_path, [frame((11, BOX, 0.0, tiny)), frame((11, BOX, two, two))], disparity_margin=0.0)
    assert r["frame_ids"] == [[0], [1]]    # 2 * tiny > tiny + 0; flushed to zero both would pass
    assert r["state"]["disparity_max"].view(np.uint32).tolist() == [1, 2]


def test_a_full_class_gives_id_minus_1_and_flag_bit_1(exe, tmp_path):
    boxes = [(0, 0, 9, 9), (20, 0, 29, 9), (40, 0, 49, 9)]
    r = track(exe, tmp_path, [frame(*[(11, b) for b in boxes]), frame(*[(11, b) for b in boxes] + [(12, BOX)])],
              max_tracks=2)
    assert r["frame_ids"] == [[0, 1, -1], [0, 1, -1, 2]]
    assert r["frame_hits"] == [[1, 1, 0], [2, 2, 0, 1]]
    assert r["flags"].tolist() == [1, 1] and r["next_id"] == 3


def test_greedy_not_the_maximum_sum_assignment(exe, tmp_path):
    # tracks A = [0, 9] (id 0), B = [6, 15] (id 1); objects X = [2, 11], Y = [-4, 5] (rows 0..0).
    # IoU: A-X 8/12, B-X 6/14, A-Y 6/16, B-Y none.  Greedy takes A-X; the maximum sum would be A-Y + B-X.
    row = lambda a, b: (a, 0, b, 0)
    r = track(exe, tmp_path, [frame((11, row(0, 9)), (11, row(6, 15))), frame((11, row(2, 11)), (11, row(-4, 5)))])
    assert r["frame_ids"] == [[0, 1], [0, 2]]
    assert r["state"][["id", "misses"]].tolist() == [(0, 0), (1, 1), (2, 0)]


def test_unwritten_frames_age_every_track_and_are_not_written(exe, tmp_path):
    frames = [frame((11, BOX), (12, BOX))] * 4
    objects, fo, _ = stream(frames)
    # capacity 3 ends inside frame 1: frames 1..3 are not written, the tracks age through them and die at max_age 2
    r = run_host(exe, tmp_path, objects, fo, [(4, 3, 0)])
    assert r["ids"][:2].tolist() == [0, 1] and r["flags"].tolist() == [0, 2, 2, 2]
    assert (r["ids"][2:].view(np.uint8) == 0x5A).all() and (r["hits"][2:].view(np.uint8) == 0x5A).all()
    assert len(r["state"]) == 0 and r["next_id"] == 2
    # one frame fewer: the tracks survive with 2 misses
    r = run_host(exe, tmp_path, objects[:6], fo[:4], [(3, 3, 0)])
    assert r["state"][["id", "hits", "misses"]].tolist() == [(0, 1, 2), (1, 1, 2)]


def test_calls_split_and_reset(exe, tmp_path):
    frames = [frame((11, BOX))] * 6
    objects, fo, _ = stream(frames)
    one = run_host(exe, tmp_path, objects, fo, [(6, 6, 0)])
    split = run_host(exe, tmp_path, objects, fo, [(1, 1, 0), (2, 2, 0), (3, 3, 0)])
    for k in ("ids", "hits", "flags"):
        assert np.array_equal(one[k], split[k]), k
    again = run_host(exe, tmp_path, objects, fo, [(3, 3, 0), (3, 3, 1)])
    assert again["ids"].tolist() == [0] * 6 and again["hits"].tolist() == [1, 2, 3, 1, 2, 3]


def test_parameters_outside_their_ranges_are_refused(exe, tmp_path):
    objects, fo, _ = stream([frame((11, BOX))])
    for bad in (dict(iou_min_permille=0), dict(iou_min_permille=1001), dict(max_age=-1),
                dict(disparity_margin=-1.0), dict(disparity_margin=NAN), dict(max_tracks=0)):
        assert "refused" in run_host(exe, tmp_path, objects, fo, [(1, 1, 0)], **bad), bad


def test_track_kernels_build_without_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(ROOT, "instance_stixels_b200", "csrc", "track.cu")
    r = subprocess.run([nvcc, "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-ftz=true",
                        "-fmad=false", "-Xptxas", "-v", "-c", src, "-o", str(tmp_path / "track.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert len(spills) == 2 and all(s == ("0", "0") for s in spills), r.stderr


def test_track_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "track_bench.py"), "--help"],
                       capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout
