"""Bird's-eye-view grids on the device (isx_bev_grid_device, Stixels.ComputeBatchTensors(bev=)): equal byte for byte
to Stixels::GetBevGrid of the drop-in header run on the host results of the same frames, and consistent with the
stixel export, the objects and the tracker."""
import ctypes as C
import os

import numpy as np
import pytest

from instance_stixels_b200 import _lib as L
from instance_stixels_b200 import api, synth

from test_bev_host import ROAD_DTYPE, build_harness, run_host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILL = 0x5A
CAM = dict(focal=synth.CAMERA["focal"], baseline=synth.CAMERA["baseline"], cx=synth.CAMERA["camera_center_x"],
           cy=synth.CAMERA["camera_center_y"])
FALLBACK = dict(vhor=100, camera_tilt=0.0, camera_height=1.18, alpha_ground=0.177384)
GRIDS = {
    "default": dict(x_min=-20.0, z_min=0.0, cell=0.2, nx=200, nz=300),
    "fine": dict(x_min=-20.0, z_min=0.0, cell=0.05, nx=800, nz=1200),
    "offset": dict(x_min=-7.3, z_min=2.5, cell=0.3, nx=97, nz=150),
    "wider_than_view": dict(x_min=-150.0, z_min=-5.0, cell=1.0, nx=300, nz=90),
}


def _stixels(mode, rows, cols, w, max_batch, **over):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(over)
    return api.make_stixels(pre, max_batch=max_batch)


def _params(g):
    return api.BevParams(**g)


def _grid(st, first, n, g):
    """BevGridDevice into a buffer pre-filled with 0x5A; int32 [n][nz][nx][2]."""
    import torch
    buf = torch.full((n * g["nz"] * g["nx"] * 8,), FILL, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    st.BevGridDevice(first, n, _params(g), buf.data_ptr())
    st.Synchronize()
    return buf.cpu().numpy().view(np.int32).reshape(n, g["nz"], g["nx"], 2)


def _roads(rows, roads):
    """Road dicts (or isx_road records) -> the harness's {alpha_ground, flipped vhor}."""
    return np.array([(float(r["alpha_ground"]), rows - int(r["vhor"]) - 1) for r in roads], dtype=ROAD_DTYPE)


def _check_grids(st, exe, tmp_path, sections, roads, rows, w, grids=GRIDS):
    n = sections.shape[0]
    for name, g in grids.items():
        got = _grid(st, 0, n, g)
        want = run_host(exe, tmp_path, sections, _roads(rows, roads), rows, w, CAM, g)
        assert isinstance(want, np.ndarray), want
        assert np.array_equal(got, want), name
        states = np.bincount(got[..., 1].reshape(-1), minlength=3)
        print(f"{name}: unknown / free / occupied cells {states.tolist()}")
        if name != "offset":
            assert states[1] > 0 and states[2] > 0, name


DENSE = {"size_filter": 2, "min_pts": 2}
CASES = {
    "unary_1024x2048_chunks": ("unary", 1024, 2048, 8, 5, DENSE, "2"),
    "pairwise_1024x2048_chunks": ("pairwise", 1024, 2048, 8, 5, {}, "2"),
    "pairwise_w4": ("pairwise", 256, 512, 4, 3, {}, None),
    "median_join": ("pairwise", 256, 512, 8, 3, {"median_join": 1}, None),
    "tall_1208": ("pairwise", 1208, 512, 8, 2, {}, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_device_grid_equals_the_header(case, tmp_path, monkeypatch):
    import torch
    exe = build_harness(tmp_path)
    mode, rows, cols, w, n, over, chunk = CASES[case]
    if chunk:
        monkeypatch.setenv("ISX_CHUNK", chunk)
    st = _stixels(mode, rows, cols, w, n, **over)
    disp, seg, roads = synth.make_batch(n, start=3, rows=rows, cols=cols, column_step=w)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(mode == "pairwise", n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    sections = st.FetchBatchResults(n, want_instances=False)[0]
    grids = GRIDS if rows == 1024 else {k: GRIDS[k] for k in ("default", "offset")}
    _check_grids(st, exe, tmp_path, sections, roads, rows, w, grids)
    st.Finish()


@pytest.mark.gpu
def test_grid_after_single_frame_compute_and_a_streamed_batch(tmp_path):
    exe = build_harness(tmp_path)
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=11, rows=rows, cols=cols)
    st.SetDisparityImage(disp[2]); st.SetSegmentation(seg[2]); st.SetRoadParameters(**roads[2])
    data = st.Compute(True)
    _check_grids(st, exe, tmp_path, data.sections.reshape(1, st.GetRealCols(), 200), roads[2:], rows, 8)
    outs = [np.zeros((n, st.GetRealCols(), 200), dtype=L.SECTION_DTYPE) for _ in range(2)]
    st.SubmitBatch(True, disp, seg, roads, outs[0])
    st.SubmitBatch(True, disp[::-1].copy(), seg[::-1].copy(), roads[::-1], outs[1])
    st.WaitBatch()
    sections = st.WaitBatch()[0]
    _check_grids(st, exe, tmp_path, sections, roads[::-1], rows, 8)
    st.Finish()


@pytest.mark.gpu
def test_grid_after_a_batch_with_road_estimation(tmp_path):
    import torch
    exe = build_harness(tmp_path)
    rows, cols, n = 256, 512, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    re = api.RoadEstimation()
    re.Initialize(CAM["cy"], CAM["baseline"], CAM["focal"], rows, cols, 128, 0.2, max_batch=n)
    disp, seg, _ = synth.make_batch(n, start=21, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    d_roads = torch.empty((n, 4), dtype=torch.int32, device="cuda")
    st.ComputeBatchDeviceRoad(re, True, n, d_disp.data_ptr(), d_seg.data_ptr(), FALLBACK, d_roads=d_roads.data_ptr())
    st.Synchronize()
    r = d_roads.cpu().numpy()
    roads = [dict(vhor=int(x[0]), alpha_ground=float(x[3:4].view(np.float32)[0])) for x in r]
    sections = st.FetchBatchResults(n, want_instances=False)[0]
    _check_grids(st, exe, tmp_path, sections, roads, rows, 8, {k: GRIDS[k] for k in ("default", "offset")})
    st.Finish()
    re.Finish()


def _export(st, n):
    import torch
    C_ = st.GetRealCols()
    cap = n * C_ * 200
    b = dict(sections=torch.empty((cap, 8), dtype=torch.int32, device="cuda"),
             frame_offsets=torch.empty(n + 1, dtype=torch.int32, device="cuda"),
             labels=torch.empty(cap, dtype=torch.int32, device="cuda"),
             vertices=torch.empty((cap, 4, 3), dtype=torch.float32, device="cuda"))
    torch.cuda.synchronize()
    st.ExportBatchDevice(0, n, b["frame_offsets"].data_ptr(), sections=b["sections"].data_ptr(),
                         labels=b["labels"].data_ptr(), vertices=b["vertices"].data_ptr(), capacity=cap)
    st.Synchronize()
    return {k: v.cpu().numpy() for k, v in b.items()}


@pytest.mark.gpu
def test_grids_are_deterministic_take_subranges_and_index_object_stixels():
    import torch
    rows, cols, n = 1024, 2048, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=30, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(True, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    g = GRIDS["default"]
    a, b = _grid(st, 0, n, g), _grid(st, 0, n, g)
    assert np.array_equal(a, b)
    assert np.array_equal(_grid(st, 1, 2, g), a[1:3])
    assert np.array_equal(_grid(st, 3, 1, g), a[3:])
    ex = _export(st, n)
    fo = ex["frame_offsets"]
    sec = ex["sections"].reshape(-1).view(L.SECTION_DTYPE)
    for f in range(n):
        occ = a[f, ..., 1] == 2
        assert ((a[f, ..., 0] >= 0) == occ).all()
        iz, ix = np.nonzero(occ)
        i = a[f, iz, ix, 0]
        assert (i < fo[f + 1] - fo[f]).all()
        s = sec[fo[f] + i]
        assert (s["type"] == 1).all()
        z = ex["vertices"][fo[f] + i, 0, 2]
        # the vertex z lies in the cell's row
        assert np.array_equal(((z - np.float32(g["z_min"])) / np.float32(g["cell"])).astype(np.int32), iz)
    st.Finish()


@pytest.mark.gpu
def test_rectangles_of_the_synthetic_scene_are_occupied_at_their_depth():
    """Every object rectangle of the synthetic frames that is nearer than the grid's far edge, inside its width and
    visible over at least 3 stixel columns has occupied cells within 10 % (at least 2 cells) of its depth over its x
    range.  The bound is 0.9 of those rectangles; the measured fraction is printed."""
    import torch
    rows, cols, w, n = 1024, 2048, 8, 6
    st = _stixels("pairwise", rows, cols, w, n)
    disp, seg, roads = synth.make_batch(n, start=40, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(True, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    g = GRIDS["default"]
    grid = _grid(st, 0, n, g)
    bf = np.float32(CAM["baseline"]) * np.float32(CAM["focal"])
    zc = g["z_min"] + (np.arange(g["nz"]) + 0.5) * g["cell"]
    xc = g["x_min"] + (np.arange(g["nx"]) + 0.5) * g["cell"]
    hits = total = 0
    for f in range(n):
        rng = np.random.Generator(np.random.PCG64(synth.SEED0 + 40 + f))
        vhor, alpha = synth._horizon(rows, None)
        rects = synth._rectangles(rng, rows, cols, vhor)
        owner = np.full(cols, -1)
        for k in sorted(range(len(rects)), key=lambda k: rects[k]):   # nearer rectangles are drawn later
            owner[rects[k][2]:rects[k][2] + rects[k][3]] = k
        for k, (base, top, x0, rw, c) in enumerate(rects):
            z = float(bf / np.float32(alpha * (base - vhor)))
            visible = np.nonzero(owner == k)[0]
            cols_seen = len(set(visible // w))
            xs = (visible - CAM["cx"]) * z / CAM["focal"]
            if z >= g["z_min"] + g["nz"] * g["cell"] or cols_seen < 3 or xs.min() < g["x_min"] or \
                    xs.max() >= g["x_min"] + g["nx"] * g["cell"]:
                continue
            total += 1
            near = np.abs(zc - z) <= max(0.1 * z, 2 * g["cell"])
            across = (xc >= xs.min() - g["cell"]) & (xc <= xs.max() + g["cell"])
            hits += bool((grid[f][np.ix_(near, across)][..., 1] == 2).any())
    print(f"rectangles occupied at their depth: {hits} of {total} ({hits / total:.3f}; bound 0.9)")
    assert total >= 10 and hits >= 0.9 * total
    st.Finish()


@pytest.mark.gpu
def test_refused_grids_enqueue_nothing():
    import torch
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=40, rows=rows, cols=cols)
    sections, _, _ = st.ComputeBatch(True, disp, seg, roads)
    g = GRIDS["default"]
    buf = torch.full((n * g["nz"] * g["nx"] * 8 + 8,), FILL, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    lib = st._lib

    def call(handle, first, nn, ptr=None, **over):
        p = api.BevParams(**dict(g, **over))
        return lib.isx_bev_grid_device(handle._h, first, nn, C.byref(p), buf.data_ptr() if ptr is None else ptr)

    launches = lib.isx_kernel_launch_count()
    nan, inf = float("nan"), float("inf")
    refusals = [call(st, -1, 1), call(st, 0, 0), call(st, 1, n), call(st, 0, n, ptr=0),
                call(st, 0, n, ptr=buf.data_ptr() + 4), call(st, 0, n, cell=nan), call(st, 0, n, cell=inf),
                call(st, 0, n, cell=0.0009), call(st, 0, n, cell=1001.0), call(st, 0, n, nx=0),
                call(st, 0, n, nx=4097), call(st, 0, n, nz=0), call(st, 0, n, nz=4097), call(st, 0, n, x_min=nan),
                call(st, 0, n, x_min=-inf), call(st, 0, n, x_min=1.1e5), call(st, 0, n, z_min=-1.1e5),
                call(st, 0, n, reserved=1)]
    assert lib.isx_kernel_launch_count() == launches
    # a handle configured without the camera centre
    nocam = _stixels("pairwise", rows, cols, 8, n, camera_center_x=-1.0)
    nocam.ComputeBatch(True, disp, seg, roads)
    launches = lib.isx_kernel_launch_count()
    refusals.append(call(nocam, 0, n))
    assert lib.isx_last_error(nocam._h) == b"Camera parameters are not set."
    assert lib.isx_kernel_launch_count() == launches
    nocam.Finish()
    # an uninitialised handle, refused as by the export
    raw = api.Stixels()
    launches = lib.isx_kernel_launch_count()
    assert call(raw, 0, 1) == -2
    assert lib.isx_kernel_launch_count() == launches
    # batches in flight
    st.SubmitBatch(True, disp, seg, roads, np.zeros_like(sections))
    launches = lib.isx_kernel_launch_count()
    refusals.append(call(st, 0, n))
    assert lib.isx_kernel_launch_count() == launches
    st.WaitBatch()
    assert refusals == [-1] * len(refusals)
    st.Synchronize()
    assert (buf.cpu().numpy() == FILL).all()
    with pytest.raises(api.InvalidArgument):
        st.BevGridDevice(0, n, api.BevParams(reserved=1), buf.data_ptr())
    st.Finish()


@pytest.mark.gpu
def test_torch_path_with_bev_objects_and_tracker_without_synchronize():
    import torch
    rows, cols, n = 256, 512, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    tracker = api.ObjectTracker()
    disp, seg, roads = synth.make_moving_batch(n, rows=rows, cols=cols)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):    # inputs produced on another stream, as a CNN runtime would
        d_disp = torch.from_numpy(disp).pin_memory().cuda(non_blocking=True)
        d_seg = torch.from_numpy(seg).pin_memory().cuda(non_blocking=True)
    torch.cuda.current_stream().wait_stream(side)
    g = GRIDS["offset"]
    out = st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_seg, objects=True, tracker=tracker,
                                 bev=api.BevParams(**g))
    del d_disp, d_seg
    # consumers on the current stream: the gather cells -> labels -> objects -> track ids on the device
    bev, ob = out.bev, out.objects
    assert bev.cells.shape == (n, g["nz"], g["nx"], 2) and bev.cells.dtype == torch.int32
    assert bev.params.cell == np.float32(g["cell"]) and bev.params.nx == g["nx"]
    frame = torch.arange(n, device="cuda")[:, None, None].expand(n, g["nz"], g["nx"])
    occ = bev.state == 2
    f_occ = frame[occ]
    row = out.frame_offsets[f_occ].long() + bev.stixel[occ].long()
    label, cls = out.labels[row], out.semantic_class[row]
    is_obj = (label >= 0) & (cls >= 11) & (cls <= 18)
    obj = ob.class_offsets[(8 * f_occ + cls - 11).clamp(min=0)].long() + label.long()
    track = torch.where(is_obj, ob.track_ids[obj.clamp(min=0)], torch.full_like(ob.track_ids[:1], -5)[0])
    got = dict(cells=bev.cells.cpu().numpy(), track=track.cpu().numpy(), obj=obj.cpu().numpy(),
               is_obj=is_obj.cpu().numpy(), obj_cls=ob.semantic_class[obj.clamp(min=0)].cpu().numpy(),
               obj_label=ob.label[obj.clamp(min=0)].cpu().numpy(), ids=ob.track_ids.cpu().numpy())
    # the explicit call on the same batch
    assert np.array_equal(got["cells"], _grid(st, 0, n, g))
    # the host chain: the frame-local index -> (column, index) of the host results -> label of GetInstanceStixels ->
    # object (class_offsets restated from the records) -> its track id
    sections, inst, offs = st.FetchBatchResults(n)
    counts = np.zeros((n, 8), np.int64)
    for f in range(n):
        for r in inst[offs[f]:offs[f + 1]]:
            if r["label"] >= 0 and 11 <= r["semantic_class"] <= 18:
                counts[f, r["semantic_class"] - 11] = max(counts[f, r["semantic_class"] - 11], r["label"] + 1)
    co = np.concatenate([[0], np.cumsum(counts.reshape(-1))])
    want_track, want_obj = [], []
    cells = got["cells"]
    for f, iz, ix in zip(*np.nonzero(cells[..., 1] == 2)):
        i = int(cells[f, iz, ix, 0])
        ends = sections[f]["type"] == -1
        per_col = np.where(ends.any(axis=1), ends.argmax(axis=1), ends.shape[1])   # stixels before the terminator
        col = int(np.searchsorted(np.cumsum(per_col), i, side="right"))
        j = i - int(per_col[:col].sum())
        s = sections[f, col, j]
        label = {(int(r["column"]), int(r["index"])): int(r["label"]) for r in inst[offs[f]:offs[f + 1]]}.get((col, j), -2)
        if label >= 0 and 11 <= s["semantic_class"] <= 18:
            o = int(co[8 * f + s["semantic_class"] - 11] + label)
            want_obj.append(o)
            want_track.append(int(got["ids"][o]))
        else:
            want_obj.append(None)
            want_track.append(-5)
    assert np.array_equal(got["track"], want_track)
    assert [o for o, k in zip(got["obj"], got["is_obj"]) if k] == [o for o in want_obj if o is not None]
    linked = got["is_obj"]
    assert linked.sum() > 0 and (got["track"][linked] >= 0).all()
    assert (got["obj_cls"][linked] >= 11).all()
    print(f"occupied cells {len(want_track)}, linked to a tracked object {int(linked.sum())}")
    st.Finish()
