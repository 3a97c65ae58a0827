"""Device objects (isx_export_objects_device, Stixels.ComputeBatchTensors(objects=True)): the instances of a batch as
one record per (class, label), equal byte for byte to Stixels::GetInstanceObjects of the drop-in header run on the
host results of the same frames, and consistent with the stixel export and the rasteriser."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from instance_stixels_b200 import _lib as L
from instance_stixels_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILL = 0x5A
NAN_BITS = 0x7FC00000
CAM = synth.CAMERA
FALLBACK = dict(vhor=100, camera_tilt=0.0, camera_height=1.18, alpha_ground=0.177384)


def _stixels(mode, rows, cols, w, max_batch, **over):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(over)
    return api.make_stixels(pre, max_batch=max_batch)


def _build_harness(tmp_path):
    exe = str(tmp_path / "objects_harness")
    libdir = os.path.join(ROOT, "instance_stixels_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include", "InstanceStixels"),
           os.path.join(ROOT, "tests", "cpp", "objects_harness.cpp"), "-L" + libdir, "-linstance_stixels_b200",
           "-Wl,-rpath," + libdir, "-o", exe]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


def _class_offsets(inst, offs, n):
    """[n*8+1] exclusive prefix of the objects per (frame, class): 1 + the largest label of the class in the frame."""
    counts = np.zeros((n, 8), np.int64)
    for f in range(n):
        for r in inst[offs[f]:offs[f + 1]]:
            k = int(r["semantic_class"]) - 11
            if r["label"] >= 0 and 0 <= k < 8:
                counts[f, k] = max(counts[f, k], int(r["label"]) + 1)
    return np.concatenate([[0], np.cumsum(counts.reshape(-1))]).astype(np.int32)


def _host(exe, tmp_path, sections, inst, offs, rows, cols, w, focal=CAM["focal"], baseline=CAM["baseline"],
          cx=CAM["camera_center_x"], cy=CAM["camera_center_y"]):
    """GetInstanceObjects of the header over the frames: objects, extents [m][6], class offsets, frame offsets."""
    n = sections.shape[0]
    np.ascontiguousarray(sections).tofile(tmp_path / "s.bin")
    np.ascontiguousarray(inst, dtype=L.INSTANCE_DTYPE).tofile(tmp_path / "i.bin")
    np.ascontiguousarray(offs, dtype=np.int32).tofile(tmp_path / "o.bin")
    p = subprocess.run([exe, str(tmp_path / "s.bin"), str(tmp_path / "i.bin"), str(tmp_path / "o.bin"), str(n),
                        str(rows), str(cols), str(w), repr(focal), repr(baseline), repr(cx), repr(cy),
                        str(tmp_path / "obj.bin"), str(tmp_path / "ext.bin")], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    objects = np.fromfile(tmp_path / "obj.bin", dtype=L.OBJECT_DTYPE)
    extents = np.fromfile(tmp_path / "ext.bin", dtype=np.float32).reshape(-1, 6)
    co = _class_offsets(inst, offs, n)
    return dict(objects=objects, extents=extents, class_offsets=co, frame_offsets=co[::8].copy(), stdout=p.stdout)


def _buffers(n, cap):
    import torch
    u8 = lambda nbytes: torch.full((nbytes,), FILL, dtype=torch.uint8, device="cuda")
    return dict(objects=u8(cap * 48), frame_offsets=u8((n + 1) * 4), class_offsets=u8((n * 8 + 1) * 4),
                extents=u8(cap * 24))


def _objects(st, first, n, capacity=None, extents=True):
    """ExportObjectsDevice into buffers pre-filled with 0x5A; returns their bytes as numpy arrays."""
    import torch
    cap = n * st.GetRealCols() * 200 if capacity is None else capacity
    b = _buffers(n, cap)
    torch.cuda.synchronize()
    st.ExportObjectsDevice(first, n, b["frame_offsets"].data_ptr(), objects=b["objects"].data_ptr(),
                           class_offsets=b["class_offsets"].data_ptr(),
                           extents=b["extents"].data_ptr() if extents else 0, capacity=cap)
    st.Synchronize()
    return {k: v.cpu().numpy() for k, v in b.items()}


def _check_equal(got, want, n, extents=True):
    fo = got["frame_offsets"].view(np.int32)
    assert np.array_equal(fo, want["frame_offsets"])
    assert np.array_equal(got["class_offsets"].view(np.int32), want["class_offsets"])
    total = int(fo[n])
    assert total == len(want["objects"]) > 0
    assert np.array_equal(got["objects"][:total * 48], want["objects"].view(np.uint8))
    assert (got["objects"][total * 48:] == FILL).all()
    if extents:
        assert np.array_equal(got["extents"][:total * 24], want["extents"].reshape(-1).view(np.uint8))
        assert (got["extents"][total * 24:] == FILL).all()
    else:
        assert (got["extents"] == FILL).all()


def _export(st, n):
    import torch
    C_ = st.GetRealCols()
    cap = n * C_ * 200
    b = dict(sections=torch.empty((cap, 8), dtype=torch.int32, device="cuda"),
             frame_offsets=torch.empty(n + 1, dtype=torch.int32, device="cuda"),
             column_offsets=torch.empty(n * C_ + 1, dtype=torch.int32, device="cuda"),
             labels=torch.empty(cap, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    st.ExportBatchDevice(0, n, b["frame_offsets"].data_ptr(), sections=b["sections"].data_ptr(),
                         column_offsets=b["column_offsets"].data_ptr(), labels=b["labels"].data_ptr(), capacity=cap)
    st.Synchronize()
    return {k: v.cpu().numpy() for k, v in b.items()}


def _check_consistency(st, got, n, rows, cols, w):
    """The objects against the stixel export (labels, rectangles) and the rasteriser's instance image (pixels)."""
    import torch
    C_ = st.GetRealCols()
    fo, co = got["frame_offsets"].view(np.int32), got["class_offsets"].view(np.int32)
    obj = got["objects"][:int(fo[n]) * 48].view(L.OBJECT_DTYPE)
    assert (obj["stixels"] >= 1).all()
    ex = _export(st, n)
    efo, eco = ex["frame_offsets"], ex["column_offsets"]
    sec = ex["sections"][:efo[n]].reshape(-1).view(L.SECTION_DTYPE)
    lab = ex["labels"][:efo[n]]
    for f in range(n):
        assert obj["stixels"][fo[f]:fo[f + 1]].sum() == (lab[efo[f]:efo[f + 1]] >= 0).sum()
    i = np.nonzero(lab >= 0)[0]
    assert len(i) > 0
    frame = np.searchsorted(efo, i, side="right") - 1
    col = np.searchsorted(eco, i, side="right") - 1 - frame * C_
    cls, s = sec["semantic_class"][i], sec[i]
    j = co[frame * 8 + cls - 11] + lab[i]
    assert (j < fo[frame + 1]).all()
    o = obj[j]
    assert np.array_equal(o["semantic_class"], cls) and np.array_equal(o["label"], lab[i])
    assert (o["x0"] <= col * w).all() and (col * w + w - 1 <= o["x1"]).all()
    assert (o["y0"] <= rows - 1 - s["vT"]).all() and (rows - 1 - s["vB"] <= o["y1"]).all()
    img = torch.zeros(n * rows * cols, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    st.RasterizeBatchDevice(0, n, d_instance_ids=img.data_ptr())
    st.Synchronize()
    img = img.cpu().numpy().reshape(n, rows * cols)
    for f in range(n):
        count = np.bincount(img[f], minlength=19000)
        fr = obj[fo[f]:fo[f + 1]]
        small = fr["label"] < 1000
        assert np.array_equal(fr["pixels"][small], count[fr["semantic_class"][small] * 1000 + fr["label"][small]])


# ---- CPU: the header function against a numpy statement of the definition ----

def test_objects_harness_compiles(tmp_path):
    assert os.path.exists(_build_harness(tmp_path))


def test_object_structs_are_48_and_40_bytes():
    assert C.sizeof(L.Object) == 48 and L.OBJECT_DTYPE.itemsize == 48
    assert C.sizeof(L.DeviceObjects) == 40


def test_objects_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "objects_bench.py"), "--help"],
                       capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout


def _f32_min(v, largest=False):
    """Minimum (maximum) of float32 values that skips NaN and orders -0.0 below +0.0; all NaN -> 0x7FC00000."""
    v = np.asarray(v, np.float32)
    v = v[~np.isnan(v)]
    if v.size == 0:
        return np.array([NAN_BITS], np.uint32).view(np.float32)[0]
    m = v.max() if largest else v.min()
    if m == 0:
        zeros = np.signbit(v[v == 0])
        negative = zeros.all() if largest else zeros.any()
        return np.float32(-0.0) if negative else np.float32(0.0)
    return m


def _corners(col, s, rows, w, focal, baseline, cx, cy):
    """Get3DVertices of one OBJECT stixel in float32, one rounding per operation."""
    f32 = np.float32
    f, bf = f32(focal), f32(baseline) * f32(focal)
    xl = f32(col * w)
    xr = xl + f32(w)
    yt, yb = f32(rows - s["vT"] - 1), f32(rows - s["vB"])
    z = bf / f32(s["disparity"])
    return [((-z / f) * (f32(cx) - x), (-z / f) * (f32(cy) - y), z) for x, y in ((xl, yt), (xr, yt), (xr, yb), (xl, yb))]


def _restate(sections, inst, offs, rows, w, focal, baseline, cx, cy):
    objects, extents = [], []
    for f in range(sections.shape[0]):
        members = {}
        for r in inst[offs[f]:offs[f + 1]]:
            s = sections[f, r["column"], r["index"]]
            c = int(s["semantic_class"])
            if r["label"] >= 0 and 11 <= c <= 18:
                members.setdefault((c, int(r["label"])), []).append((int(r["column"]), s))
        for c in range(11, 19):
            for label in range(1 + max([lb for cc, lb in members if cc == c], default=-1)):
                m = members[(c, label)]
                cols = [col for col, _ in m]
                vB, vT = [int(s["vB"]) for _, s in m], [int(s["vT"]) for _, s in m]
                dis = [s["disparity"] for _, s in m]
                objects.append((c, label, len(m), sum(w * (t - b + 1) for b, t in zip(vB, vT)), min(cols), max(cols),
                                min(cols) * w, rows - 1 - max(vT), max(cols) * w + w - 1, rows - 1 - min(vB),
                                _f32_min(dis), _f32_min(dis, largest=True)))
                pts = np.array([p for col, s in m for p in _corners(col, s, rows, w, focal, baseline, cx, cy)],
                               np.float32)
                extents.append([_f32_min(pts[:, q]) for q in range(3)] +
                               [_f32_min(pts[:, q], largest=True) for q in range(3)])
    return np.array(objects, dtype=L.OBJECT_DTYPE), np.array(extents, np.float32).reshape(-1, 6)


def _hand_made_frames():
    """Three 64 x 64 frames, width 8: frame 0 with several classes, noise, a NaN member, an all-NaN object,
    single-stixel objects and members at infinite / zero depth (-0.0 and +0.0 extents); frame 1 without instances;
    frame 2 with one object spanning columns 1..6."""
    rows, w, C_ = 64, 8, 8
    sec = np.zeros((3, C_, 200), dtype=L.SECTION_DTYPE)
    sec["type"] = -1
    inst = [[], [], []]

    def put(f, col, stixels):
        for j, (t, vB, vT, dis, cls, label) in enumerate(stixels):
            sec[f, col, j] = (t, vB, vT, dis, cls, 0.0, 0.0, 0.0)
            if label is not None:
                inst[f].append((col, j, label, cls))

    nan, inf = float("nan"), float("inf")
    put(0, 0, [(1, 40, 63, 5.0, 11, 0), (0, 0, 39, 1.0, 0, None)])
    put(0, 1, [(1, 40, 63, 5.5, 11, 0), (1, 20, 39, nan, 11, 0), (0, 0, 19, 1.0, 0, None)])
    put(0, 2, [(1, 30, 63, inf, 13, 0), (0, 0, 29, 1.0, 0, None)])
    put(0, 3, [(2, 50, 63, 0.0, 10, None), (1, 24, 49, -inf, 13, 1), (0, 0, 23, 1.0, 0, None)])
    put(0, 4, [(1, 44, 63, inf, 18, 0), (1, 20, 43, -inf, 18, 0), (0, 0, 19, 1.0, 0, None)])
    put(0, 5, [(1, 10, 63, nan, 11, 1), (0, 0, 9, 1.0, 0, None)])
    put(0, 6, [(1, 50, 63, 7.0, 11, -1), (1, 30, 49, 0.0, 11, 2), (1, 0, 29, 3.25, 12, 0)])
    put(0, 7, [(1, 32, 63, 9.5, 18, 1), (0, 0, 31, 1.0, 0, None)])
    for col in range(C_):
        put(1, col, [(2, 40, 63, 0.0, 10, None), (1, 20, 39, 4.0, 13, None), (0, 0, 19, 1.0, 0, None)])
    for col in range(C_):
        label = 0 if col in (1, 6) else (-1 if col == 3 else None)
        put(2, col, [(1, 16 + col, 63, 2.0 + col, 15, label), (0, 0, 15 + col, 1.0, 0, None)])
    recs = np.array([r for f in range(3) for r in sorted(inst[f], key=lambda r: (r[3], r[0], r[1]))],
                    dtype=L.INSTANCE_DTYPE)
    offs = np.concatenate([[0], np.cumsum([len(x) for x in inst])]).astype(np.int32)
    return sec, recs, offs, rows, C_ * w, w


def test_header_objects_equal_a_numpy_statement(tmp_path):
    exe = _build_harness(tmp_path)
    sec, recs, offs, rows, cols, w = _hand_made_frames()
    cam = dict(focal=1000.0, baseline=0.25, cx=16.0, cy=40.0)
    got = _host(exe, tmp_path, sec, recs, offs, rows, cols, w, **cam)
    with np.errstate(all="ignore"):     # divisions by +-0 and +-inf disparities are part of the cases
        objects, extents = _restate(sec, recs, offs, rows, w, cam["focal"], cam["baseline"], cam["cx"], cam["cy"])
    assert np.array_equal(got["objects"].view(np.uint8), objects.view(np.uint8))
    assert np.array_equal(got["extents"].view(np.uint32), extents.view(np.uint32))
    assert got["frame_offsets"].tolist() == [0, 8, 8, 9]
    # the cases the frames are meant to cover
    assert (got["objects"]["disparity_min"].view(np.uint32) == NAN_BITS).sum() == 1        # the all-NaN object
    assert (extents.view(np.uint32) == NAN_BITS).all(axis=1).sum() == 1
    bits = extents.view(np.uint32)
    assert (bits == 0x80000000).any() and (bits == 0).any()                                 # -0.0 and +0.0
    assert (got["objects"]["stixels"] == 1).sum() >= 4 and len(set(got["objects"]["semantic_class"])) == 5
    # without the camera centre the extents are refused like Get3DVertices; the objects stay the same
    nocam = _host(exe, tmp_path, sec, recs, offs, rows, cols, w, focal=1000.0, baseline=0.25, cx=-1.0, cy=-1.0)
    assert "refused: Camera parameters are not set." in nocam["stdout"]
    assert np.array_equal(nocam["objects"].view(np.uint8), objects.view(np.uint8)) and nocam["extents"].size == 0


# ---- GPU: the device objects against the header on the host results of the same frames ----

# The unary preset's size filter (42 stixels) leaves these small synthetic frames without clusters: a smaller one
# gives them objects.
DENSE = {"size_filter": 2, "min_pts": 2}
CASES = {
    "unary_w8_chunks": ("unary", 256, 512, 8, 6, DENSE, "4"),
    "pairwise_w8_chunks": ("pairwise", 256, 512, 8, 6, {}, "4"),
    "pairwise_w4": ("pairwise", 256, 512, 4, 3, {}, None),
    "median_join": ("pairwise", 256, 512, 8, 3, {"median_join": 1}, None),
    "tall_1208": ("pairwise", 1208, 512, 8, 1, {}, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_device_objects_equal_the_header(case, tmp_path, monkeypatch):
    import torch
    exe = _build_harness(tmp_path)
    mode, rows, cols, w, n, over, chunk = CASES[case]
    if chunk:
        monkeypatch.setenv("ISX_CHUNK", chunk)
    st = _stixels(mode, rows, cols, w, n, **over)
    disp, seg, roads = synth.make_batch(n, start=3, rows=rows, cols=cols, column_step=w)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(mode == "pairwise", n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    got = _objects(st, 0, n)
    want = _host(exe, tmp_path, *st.FetchBatchResults(n), rows, cols, w)
    _check_equal(got, want, n)
    _check_consistency(st, got, n, rows, cols, w)
    print(f"{case}: {len(want['objects'])} objects")
    st.Finish()


@pytest.mark.gpu
def test_objects_after_single_frame_compute_and_a_streamed_batch(tmp_path):
    exe = _build_harness(tmp_path)
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=11, rows=rows, cols=cols)
    st.SetDisparityImage(disp[2]); st.SetSegmentation(seg[2]); st.SetRoadParameters(**roads[2])
    data = st.Compute(True)
    rec = st.instance_records()
    want = _host(exe, tmp_path, data.sections[None], rec, np.array([0, len(rec)], np.int32), rows, cols, 8)
    _check_equal(_objects(st, 0, 1), want, 1)
    outs = [np.zeros((n, st.GetRealCols(), 200), dtype=L.SECTION_DTYPE) for _ in range(2)]
    st.SubmitBatch(True, disp, seg, roads, outs[0])
    st.SubmitBatch(True, disp[::-1].copy(), seg[::-1].copy(), roads[::-1], outs[1])
    st.WaitBatch()
    delivered = st.WaitBatch()
    want = _host(exe, tmp_path, *delivered, rows, cols, 8)
    got = _objects(st, 0, n)
    _check_equal(got, want, n)
    _check_consistency(st, got, n, rows, cols, 8)
    st.Finish()


@pytest.mark.gpu
def test_objects_after_a_batch_with_road_estimation(tmp_path):
    import torch
    exe = _build_harness(tmp_path)
    rows, cols, n = 256, 512, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    re = api.RoadEstimation()
    re.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], rows, cols, 128, 0.2, max_batch=n)
    disp, seg, _ = synth.make_batch(n, start=21, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDeviceRoad(re, True, n, d_disp.data_ptr(), d_seg.data_ptr(), FALLBACK)
    got = _objects(st, 0, n)
    want = _host(exe, tmp_path, *st.FetchBatchResults(n), rows, cols, 8)
    _check_equal(got, want, n)
    st.Finish()
    re.Finish()


@pytest.mark.gpu
def test_objects_are_deterministic_bounded_and_take_subranges():
    import torch
    rows, cols, n = 256, 512, 6
    st = _stixels("unary", rows, cols, 8, n, **DENSE)
    disp, seg, roads = synth.make_batch(n, start=20, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(False, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    a, b = _objects(st, 0, n), _objects(st, 0, n)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    fo, co = a["frame_offsets"].view(np.int32), a["class_offsets"].view(np.int32)
    total = int(fo[n])
    for k, size in (("objects", 48), ("extents", 24)):
        assert (a[k][total * size:] == FILL).all(), k
    # frames [2, 5): the matching slice, offsets rebased to 0
    s = _objects(st, 2, 3)
    lo, hi = int(fo[2]), int(fo[5])
    assert np.array_equal(s["frame_offsets"].view(np.int32), fo[2:6] - lo)
    assert np.array_equal(s["class_offsets"].view(np.int32), co[16:41] - lo)
    for k, size in (("objects", 48), ("extents", 24)):
        assert np.array_equal(s[k][:(hi - lo) * size], a[k][lo * size:hi * size]), k
        assert (s[k][(hi - lo) * size:] == FILL).all(), k
    # capacity that ends inside frame g (the first after frame 0 with two objects or more): frames before g written,
    # nothing else, offsets complete
    g = next(f for f in range(1, n) if fo[f + 1] - fo[f] >= 2)
    cap = int(fo[g]) + (int(fo[g + 1]) - int(fo[g])) // 2
    c = _objects(st, 0, n, capacity=cap)
    for k in ("frame_offsets", "class_offsets"):
        assert np.array_equal(c[k], a[k]), k
    end = int(fo[g])
    assert end > 0
    for k, size in (("objects", 48), ("extents", 24)):
        assert np.array_equal(c[k][:end * size], a[k][:end * size]), k
        assert (c[k][end * size:] == FILL).all(), k
    # capacity 0: offsets only
    z = _objects(st, 0, n, capacity=0)
    for k in ("frame_offsets", "class_offsets"):
        assert np.array_equal(z[k], a[k]), k
    assert (z["objects"] == FILL).all() and (z["extents"] == FILL).all()
    # without extents: the same objects
    e = _objects(st, 0, n, extents=False)
    assert np.array_equal(e["objects"], a["objects"]) and (e["extents"] == FILL).all()
    st.Finish()


@pytest.mark.gpu
def test_refused_object_exports_enqueue_nothing():
    import torch
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=40, rows=rows, cols=cols)
    sections, _, _ = st.ComputeBatch(True, disp, seg, roads)
    cap = n * st.GetRealCols() * 200
    b = _buffers(n, cap)
    torch.cuda.synchronize()
    lib = st._lib

    def out_of(**over):
        args = dict(objects=b["objects"].data_ptr(), frame_offsets=b["frame_offsets"].data_ptr(),
                    class_offsets=b["class_offsets"].data_ptr(), extents=b["extents"].data_ptr(), capacity=cap)
        args.update(over)
        return L.DeviceObjects(*(args[k] or None for k in ("objects", "frame_offsets", "class_offsets", "extents")),
                               args["capacity"], 0)

    def call(handle, first, nn, **over):
        return lib.isx_export_objects_device(handle._h, first, nn, C.byref(out_of(**over)))

    launches = lib.isx_kernel_launch_count()
    refusals = [call(st, -1, 1), call(st, 0, 0), call(st, 1, n), call(st, 0, n, frame_offsets=0),
                call(st, 0, n, objects=b["objects"].data_ptr() + 4), call(st, 0, n, capacity=-1)]
    assert lib.isx_kernel_launch_count() == launches
    # extents without the camera centre, on a handle configured without it
    nocam = _stixels("pairwise", rows, cols, 8, n, camera_center_x=-1.0)
    nocam.ComputeBatch(True, disp, seg, roads)
    launches = lib.isx_kernel_launch_count()
    refusals.append(call(nocam, 0, n))
    assert b"Camera parameters are not set" in lib.isx_last_error(nocam._h)
    assert lib.isx_kernel_launch_count() == launches
    nocam.Finish()
    # an uninitialised handle, refused as by the export
    raw = api.Stixels()
    launches = lib.isx_kernel_launch_count()
    rc = call(raw, 0, 1)
    res = L.DeviceResults(None, b["frame_offsets"].data_ptr(), None, None, None, None, 0, 0)
    assert rc == lib.isx_export_batch_device(raw._h, 0, 1, C.byref(res)) == -2
    assert lib.isx_kernel_launch_count() == launches
    # batches in flight
    st.SubmitBatch(True, disp, seg, roads, np.zeros_like(sections))
    launches = lib.isx_kernel_launch_count()
    refusals.append(call(st, 0, n))
    assert lib.isx_kernel_launch_count() == launches
    st.WaitBatch()
    assert refusals == [-1] * len(refusals)
    st.Synchronize()
    assert all((v.cpu().numpy() == FILL).all() for v in b.values())
    assert int(_objects(st, 0, n)["frame_offsets"].view(np.int32)[n]) > 0
    st.Finish()


@pytest.mark.gpu
def test_torch_path_with_objects_without_synchronize():
    import torch
    rows, cols, n = 256, 512, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=50, rows=rows, cols=cols)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):    # inputs produced on another stream, as a CNN runtime would
        d_disp = torch.from_numpy(disp).pin_memory().cuda(non_blocking=True)
        d_seg = torch.from_numpy(seg).pin_memory().cuda(non_blocking=True)
    torch.cuda.current_stream().wait_stream(side)
    out = st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_seg, vertices=True, objects=True)
    del d_disp, d_seg
    # consumers on the current stream
    ob = out.objects
    total = int(ob.frame_offsets[n].item())
    got = dict(objects=ob.data[:total].cpu().numpy(), frame_offsets=ob.frame_offsets.cpu().numpy(),
               class_offsets=ob.class_offsets.cpu().numpy(), extents=ob.extents[:total].cpu().numpy(),
               disparity_min=ob.disparity_min[:total].cpu().numpy(), x1=ob.x1[:total].cpu().numpy())
    assert ob.data.shape == (n * st.GetRealCols() * 200, 12) and ob.extents.shape == (ob.data.shape[0], 2, 3)
    ref = _objects(st, 0, n)
    assert np.array_equal(got["frame_offsets"].view(np.uint8), ref["frame_offsets"])
    assert np.array_equal(got["class_offsets"].view(np.uint8), ref["class_offsets"])
    assert np.array_equal(got["objects"].reshape(-1).view(np.uint8), ref["objects"][:total * 48])
    assert np.array_equal(got["extents"].reshape(-1).view(np.uint8), ref["extents"][:total * 24])
    obj = ref["objects"][:total * 48].view(L.OBJECT_DTYPE)
    assert np.array_equal(got["disparity_min"].view(np.uint32), obj["disparity_min"].view(np.uint32))
    assert np.array_equal(got["x1"], obj["x1"]) and total > 0
    # without vertices: objects, no extents
    out2 = st.ComputeBatchTensors(True, torch.from_numpy(disp).cuda(), roads, segmentation=torch.from_numpy(seg).cuda(),
                                  objects=True, object_capacity=total)
    assert out2.objects.extents is None and out2.objects.data.shape == (total, 12)
    assert np.array_equal(out2.objects.data.cpu().numpy().reshape(-1).view(np.uint8), ref["objects"][:total * 48])
    st.Finish()
