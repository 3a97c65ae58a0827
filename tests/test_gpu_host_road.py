"""Road estimation inside streamed host batches (isx_submit_batch_host_road / _u16_road) and the frame pool
(isx_pool_compute_host_road), and the batch runner's --road-on-device mode.  Everything must equal, byte for byte, a
composition of entry points that already exist: isx_road_compute_host per frame -> keep-last (or, for the pool, the
per-frame rule) -> isx_submit_batch_host{,_u16} / isx_pool_compute_host with those roads."""
import ctypes as C
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from instance_stixels_b200 import _lib as L  # noqa: E402
from instance_stixels_b200 import api, synth  # noqa: E402

CAM = dict(camera_center_y=512.0, baseline=0.209313, focal=2262.52)
FALLBACK = dict(vhor=100, camera_tilt=0.0, camera_height=1.18, alpha_ground=0.177384)
FILL = 0x5A
HARNESS = os.path.join(ROOT, "tests", "cpp", "host_road_harness.cpp")
APP = os.path.join(ROOT, "apps", "cityscapes_runner")


def _stixels(mode, rows, cols, w, max_batch, **over):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(over)
    return api.make_stixels(pre, max_batch=max_batch)


def _road(rows, cols, max_batch, max_dis=128, device=0):
    re_ = api.RoadEstimation(device)
    re_.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], rows, cols, max_dis, 0.2,
                   max_batch=max_batch)
    return re_


def _frames(n, rows, cols, w, zero=(0, 3), start=0):
    """Frames with horizons spread over the image (different Hough cells, different ground tables); the frames in
    `zero` have no disparity at all, so their estimation fails."""
    frames = [synth.make_frame(start + i, rows=rows, cols=cols, column_step=w,
                               vhor=int(rows * (0.3 + 0.1 * (i % 4)))) for i in range(n)]
    disp = np.stack([f.disparity for f in frames])
    seg = np.stack([f.segmentation for f in frames])
    for i in zero:
        if i < n:
            disp[i] = 0.0
    return np.ascontiguousarray(disp), np.ascontiguousarray(seg)


def _road_of(e):
    return dict(vhor=int(e.horizon_point), camera_tilt=e.pitch, camera_height=e.camera_height, alpha_ground=e.slope)


def _host_estimates(ref, disp):
    """isx_road_compute_host frame by frame."""
    est = (L.RoadEstimate * len(disp))()
    for f in range(len(disp)):
        img = np.ascontiguousarray(disp[f])
        assert ref._lib.isx_road_compute_host(ref.handle(), img.ctypes.data, img.size, C.byref(est[f])) == 0
    return est


def _keep_last(estimates, seed):
    out, cur = [], seed
    for e in estimates:
        if e.ok:
            cur = _road_of(e)
        out.append(cur)
    return out


def _poisoned(ctype, n):
    a = (ctype * n)()
    C.memset(a, FILL, C.sizeof(a))
    return a


def _sections(st, n):
    """A FILL-poisoned padded Section array: entries nobody writes must stay FILL in both paths."""
    C_ = st.GetRealCols()
    return np.frombuffer(bytes([FILL]) * (n * C_ * 200 * 32), dtype=L.SECTION_DTYPE).reshape(n, C_, 200).copy()


def _u8(nbytes):
    import torch
    return torch.full((nbytes,), FILL, dtype=torch.uint8, device="cuda")


def _export(st, n):
    """The full device export (Sections, offsets, labels, vertices, errors) of the last batch, as bytes."""
    import torch
    C_ = st.GetRealCols()
    cap = n * C_ * 200
    b = dict(sections=_u8(cap * 32), frame_offsets=_u8((n + 1) * 4), column_offsets=_u8((n * C_ + 1) * 4),
             labels=_u8(cap * 4), vertices=_u8(cap * 48), frame_errors=_u8(n * 4))
    st.ExportBatchDevice(0, n, b["frame_offsets"].data_ptr(), sections=b["sections"].data_ptr(),
                         column_offsets=b["column_offsets"].data_ptr(), labels=b["labels"].data_ptr(),
                         vertices=b["vertices"].data_ptr(), frame_errors=b["frame_errors"].data_ptr(), capacity=cap)
    st.Synchronize()
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in b.items()}


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


# mode, rows, cols, width, frames per batch, config overrides, ISX_CHUNK, failing frames of the three batches
CASES = {
    "unary_w8_chunks": ("unary", 256, 512, 8, 7, {}, "4", [(0, 3), (0, 3, 4), (6,)]),
    "pairwise_w8_chunks": ("pairwise", 256, 512, 8, 7, {}, "4", [(0, 3), (0, 3, 4), (6,)]),
    "unary_w4": ("unary", 256, 512, 4, 5, {}, None, [(0, 3), (0,), (2,)]),
    "pairwise_w4": ("pairwise", 256, 512, 4, 5, {}, None, [(0, 3), (0,), (2,)]),
    "median_join": ("pairwise", 256, 512, 8, 5, {"median_join": 1}, None, [(0, 3), (0,), (2,)]),
    "tall_1208": ("pairwise", 1208, 512, 8, 3, {}, None, [(0,), (0, 1), ()]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_submitted_batches_equal_the_composition(case, monkeypatch):
    """Three batches in flight, fallback on the first only: keep-last runs across chunk and batch boundaries."""
    mode, rows, cols, w, n, over, chunk, zeros = CASES[case]
    if chunk:
        monkeypatch.setenv("ISX_CHUNK", chunk)
    pairwise = mode == "pairwise"
    st = _stixels(mode, rows, cols, w, n, **over)
    st.ReserveInFlight(3)
    ref = _road(rows, cols, 1)
    batches = [_frames(n, rows, cols, w, zero=z, start=10 * b) for b, z in enumerate(zeros)]
    est = [_host_estimates(ref, d) for d, _ in batches]
    flat = [e for b in est for e in b]
    assert not flat[0].ok and sum(e.ok for e in flat) >= len(flat) - 6
    assert len({(e.horizon_point, e.rho, e.theta) for e in flat if e.ok}) >= 2, "frames should select different cells"
    roads = _keep_last(flat, FALLBACK)

    want = []
    for b, (d, s) in enumerate(batches):
        sec = _sections(st, n)
        st.SubmitBatch(pairwise, d, s, roads[b * n:(b + 1) * n], sec)
    for b in range(3):
        want.append(st.WaitBatch())
    want_export = _export(st, n)

    re_ = _road(rows, cols, n)
    outs = []
    for b, (d, s) in enumerate(batches):
        sec = _sections(st, n)
        outs.append(st.SubmitBatchRoad(re_, pairwise, d, s, FALLBACK if b == 0 else None, sec,
                                       estimates=_poisoned(L.RoadEstimate, n), roads_out=_poisoned(L.Road, n)))
    got = [st.WaitBatch() for _ in range(3)]
    got_export = _export(st, n)
    for b in range(3):
        g_est, g_roads = outs[b]
        assert bytes(g_est) == bytes(est[b]), b
        assert bytes(g_roads) == bytes(api._roads(roads[b * n:(b + 1) * n])), b
        (ws, wi, wo), (gs, gi, go) = want[b], got[b]
        assert _same(gs, ws), b
        assert _same(gi, wi) and np.array_equal(go, wo), b
    for k in want_export:
        assert _same(got_export[k], want_export[k]), k
    st.Finish()


def _narrow(disp, seg, rows):
    used = (rows + 7) // 8
    d16 = np.rint(disp * 256.0).astype(np.uint16)
    s16 = np.ascontiguousarray(seg[..., :used]).astype(np.int16)
    wide_d = (d16.astype(np.float32) / np.float32(256.0)).astype(np.float32)
    wide_s = np.zeros_like(seg)
    wide_s[..., :used] = s16
    return d16, s16, wide_d, wide_s


@pytest.mark.gpu
@pytest.mark.parametrize("pairwise", [0, 1])
def test_u16_equals_float_on_the_widened_image(pairwise, monkeypatch):
    monkeypatch.setenv("ISX_CHUNK", "4")
    rows, cols, w, n = 256, 512, 8, 6
    st = _stixels("pairwise" if pairwise else "unary", rows, cols, w, n)
    d16, s16, wide_d, wide_s = _narrow(*_frames(n, rows, cols, w, zero=(1, 4)), rows)
    results = []
    for narrow in (False, True):
        re_ = _road(rows, cols, n)
        outs = []
        for b in range(2):   # the second batch continues from the first
            sec = _sections(st, n)
            fb = FALLBACK if b == 0 else None
            if narrow:
                o = st.SubmitBatchU16Road(re_, bool(pairwise), d16, np.float32(1 / 256), s16, fb, sec)
            else:
                o = st.SubmitBatchRoad(re_, bool(pairwise), wide_d, wide_s, fb, sec)
            outs.append(o)
        waited = [st.WaitBatch() for _ in range(2)]
        results.append([(bytes(e), bytes(r), s, i, o) for (e, r), (s, i, o) in zip(outs, waited)])
    for (fe, fr, fs, fi, fo), (ue, ur, us, ui, uo) in zip(*results):
        assert fe == ue and fr == ur
        assert _same(fs, us) and _same(fi, ui) and np.array_equal(fo, uo)
    est = np.frombuffer(results[0][0][0], dtype=np.int32).reshape(n, 7)
    assert est[1, 0] == 0 and est[4, 0] == 0 and est[0, 0] == 1
    st.Finish()


def _pool_config(mode, rows, cols, w):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(CAM)
    return api.StixelConfig(**pre)


def _pool_devices():
    import torch
    g = torch.cuda.device_count()
    return {"one": ([0], 4), "two_workers_one_gpu": ([0, 0], 3), "all_gpus": (list(range(g)), 3),
            "one_frame_sub_batches": ([0, 0] if g == 1 else [0, 1], 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["one", "two_workers_one_gpu", "all_gpus", "one_frame_sub_batches"])
@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_pool_equals_the_per_frame_composition(layout, mode):
    rows, cols, w, n = 256, 512, 8, 11
    devices, max_batch = _pool_devices()[layout]
    pool = api.StixelsPool(_pool_config(mode, rows, cols, w), devices, max_batch=max_batch)
    disp, seg = _frames(n, rows, cols, w, zero=(0, 4, 5, 10))
    est = _host_estimates(_road(rows, cols, 1), disp)
    per_frame = [_road_of(e) if e.ok else FALLBACK for e in est]
    pairwise = mode == "pairwise"
    ws, wi, wo = pool.ComputeBatch(pairwise, disp, seg, per_frame)
    for _ in range(2):   # the second call: the road handles exist, nothing carries over from the first
        gs, gi, go, g_est, g_roads = pool.ComputeBatchRoad(pairwise, disp, seg, FALLBACK)
        assert bytes(g_est) == bytes(est)
        assert bytes(g_roads) == bytes(api._roads(per_frame))
        assert _same(gs, ws) and _same(gi, wi) and np.array_equal(go, wo)
        assert sum(pool.frames_by_worker()) == n
    pool.close()


@pytest.mark.gpu
def test_pool_requires_a_fallback():
    rows, cols, w, n = 256, 512, 8, 2
    pool = api.StixelsPool(_pool_config("unary", rows, cols, w), [0], max_batch=2)
    disp, seg = _frames(n, rows, cols, w, zero=())
    lib = pool._lib
    sec = np.zeros((n, pool.GetRealCols(), 200), L.SECTION_DTYPE)
    rc = lib.isx_pool_compute_host_road(pool._p, 0, n, disp.ctypes.data, seg.ctypes.data, None, None, None,
                                        sec.ctypes.data, None, 0, None)
    assert rc == -1
    pool.close()


@pytest.mark.gpu
def test_refusals_enqueue_and_copy_nothing():
    import torch
    rows, cols, w, n = 256, 512, 8, 8
    st = _stixels("unary", rows, cols, w, n)        # unary batches of 8 frames go in one chunk of 8
    disp, seg = _frames(n + 1, rows, cols, w, zero=())
    d16, s16, _, _ = _narrow(disp, seg, rows)
    lib = st._lib
    fb = C.byref(api._roads([FALLBACK])[0])
    est, rds = _poisoned(L.RoadEstimate, n + 1), _poisoned(L.Road, n + 1)
    sec = _sections(st, n + 1)

    def call(road_h, k, d=disp.ctypes.data, s=seg.ctypes.data, fallback=fb, u16=False):
        if u16:
            return lib.isx_submit_batch_host_u16_road(st._h, road_h, 0, k, d, np.float32(1 / 256), s, fallback, est,
                                                      rds, sec.ctypes.data)
        return lib.isx_submit_batch_host_road(st._h, road_h, 0, k, d, s, fallback, est, rds, sec.ctypes.data)

    good = _road(rows, cols, n)
    unset = api.RoadEstimation()
    other_rows = _road(rows // 2, cols, n)
    other_cols = _road(rows, cols // 2, n)
    other_dis = _road(rows, cols, n, max_dis=64)
    small = _road(rows, cols, n - 1)                # smaller than the chunk of 8
    fresh = _road(rows, cols, n)                    # never seeded
    other_device = _road(rows, cols, n, device=1) if torch.cuda.device_count() > 1 else None
    launches = lib.isx_kernel_launch_count()
    refusals = [
        (call(unset.handle(), n), -1), (call(other_rows.handle(), n), -1), (call(other_cols.handle(), n), -1),
        (call(other_dis.handle(), n), -1), (call(None, n), -1), (call(good.handle(), n, d=None), -1),
        (call(good.handle(), n, s=None), -1), (call(fresh.handle(), n, fallback=None), -1),
        (call(good.handle(), n, d=None, u16=True), -1), (call(small.handle(), n), -4),
        (call(small.handle(), n, d=d16.ctypes.data, s=s16.ctypes.data, u16=True), -4),
        (call(good.handle(), n + 1), -4), (call(good.handle(), 0), -4)]
    if other_device is not None:
        refusals.append((call(other_device.handle(), n), -1))
    assert [r for r, _ in refusals] == [c for _, c in refusals], refusals
    assert lib.isx_kernel_launch_count() == launches
    est_bytes, rds_bytes = bytes(est), bytes(rds)
    assert est_bytes == bytes([FILL]) * len(est_bytes) and rds_bytes == bytes([FILL]) * len(rds_bytes)
    assert _same(sec, _sections(st, n + 1))
    # a small batch fits the small road handle: only the chunk a batch is cut into counts
    assert call(small.handle(), 3) == 0
    assert lib.isx_kernel_launch_count() > launches
    assert lib.isx_wait_batch_host(st._h, None, 0, None) == 0
    # a fourth batch in flight
    for _ in range(3):
        assert call(good.handle(), n) == 0
    launches = lib.isx_kernel_launch_count()
    C.memset(est, FILL, C.sizeof(est))
    C.memset(rds, FILL, C.sizeof(rds))
    sec4 = _sections(st, n)
    assert lib.isx_submit_batch_host_road(st._h, good.handle(), 0, n, disp.ctypes.data, seg.ctypes.data, fb,
                                          est, rds, sec4.ctypes.data) == -4
    assert lib.isx_kernel_launch_count() == launches
    est4, rds4 = bytes(est), bytes(rds)
    assert est4 == bytes([FILL]) * len(est4) and rds4 == bytes([FILL]) * len(rds4)
    for _ in range(3):
        assert lib.isx_wait_batch_host(st._h, None, 0, None) == 0
    assert _same(sec4, _sections(st, n))
    st.Finish()


@pytest.mark.gpu
def test_refusals_leave_the_launch_count_alone():
    rows, cols, w, n = 256, 512, 8, 4
    st = _stixels("pairwise", rows, cols, w, n)
    disp, seg = _frames(n, rows, cols, w, zero=())
    lib = st._lib
    fb = C.byref(api._roads([FALLBACK])[0])
    unset, fresh, small = api.RoadEstimation(), _road(rows, cols, n), _road(rows, cols, n - 1)
    other = _road(rows, cols, n, max_dis=64)
    launches = lib.isx_kernel_launch_count()
    got = [lib.isx_submit_batch_host_road(st._h, r.handle(), 1, n, disp.ctypes.data, seg.ctypes.data, f, None, None,
                                          None) for r, f in ((unset, fb), (fresh, None), (small, fb), (other, fb))]
    assert got == [-1, -1, -4, -1]
    assert lib.isx_kernel_launch_count() == launches
    st.Finish()


def _cuda_home():
    nvcc = shutil.which("nvcc")
    return os.path.dirname(os.path.dirname(nvcc)) if nvcc else os.environ.get("CUDA_HOME", "/usr/local/cuda")


def _build_harness(tmp_path):
    exe = str(tmp_path / "host_road_harness")
    libdir = os.path.join(ROOT, "instance_stixels_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include", "InstanceStixels"), HARNESS,
           "-L" + libdir, "-linstance_stixels_b200", "-Wl,-rpath," + libdir, "-o", exe]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return exe


def test_host_road_harness_compiles(tmp_path):
    assert os.path.exists(_build_harness(tmp_path))


def test_host_road_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "host_road_bench.py"), "--help"],
                       capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout


def test_runner_accepts_the_flag_without_a_gpu_run(tmp_path):
    """--road-on-device is parsed as a flag, not as a positional argument (the usage line stays the reference's),
    and the one-frame loop refuses it instead of ignoring it."""
    subprocess.run(["make", "-C", os.path.join(ROOT, "apps")], check=True, capture_output=True, text=True)
    p = subprocess.run([APP, "--road-on-device", "--batch", "2"], capture_output=True, text=True)
    assert p.returncode != 0 and "Usage: stixels dir" in p.stderr
    args = [APP, str(tmp_path), "128", "1.0", "0.0", "1.0", "0", "8", "16.0", "2", "10"]
    p = subprocess.run(args + ["--road-on-device"], capture_output=True, text=True)
    assert p.returncode != 0 and "--road-on-device applies to the batched mode" in p.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("pairwise", [0, 1])
def test_cpp_overloads_equal_the_composition(tmp_path, pairwise):
    exe = _build_harness(tmp_path)
    rows, cols, w, n = 256, 512, 8, 5
    disp, seg = _frames(n, rows, cols, w, zero=(0, 2))
    disp.tofile(tmp_path / "d.f32")
    seg.tofile(tmp_path / "s.i32")
    p = subprocess.run([exe, str(tmp_path / "d.f32"), str(tmp_path / "s.i32"), str(n), str(rows), str(cols),
                        str(pairwise), str(tmp_path / "out")], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr + p.stdout
    fb = dict(FALLBACK)
    est = _host_estimates(_road(rows, cols, 1), disp)
    read = lambda ext: np.fromfile(tmp_path / f"out.{ext}", dtype=np.uint8)
    mode = "pairwise" if pairwise else "unary"
    # Stixels::SubmitBatch(..., RoadEstimation&, fallback): keep-last
    st = _stixels(mode, rows, cols, w, n)
    roads = _keep_last(est, fb)
    st.SubmitBatch(bool(pairwise), disp, seg, roads, np.zeros((n, st.GetRealCols(), 200), L.SECTION_DTYPE))
    sections, inst, offs = st.WaitBatch()
    assert read("stixels.estimates").tobytes() == bytes(est)
    assert read("stixels.roads").tobytes() == bytes(api._roads(roads))
    assert np.array_equal(read("stixels.sections"), sections.view(np.uint8).reshape(-1))
    maps = [sorted((int(r["column"]), int(r["index"]), int(r["label"])) for r in inst[offs[f]:offs[f + 1]])
            for f in range(n)]
    assert read("stixels.instances").view(np.int32).tolist() == [v for m in maps for t in m for v in t]
    assert np.array_equal(read("stixels.offsets").view(np.int32), offs)
    st.Finish()
    # StixelsPool::ComputeBatch(..., const Road& fallback, estimates, ...): per frame
    pool = api.StixelsPool(_pool_config(mode, rows, cols, w), [0], max_batch=n)
    per_frame = [_road_of(e) if e.ok else fb for e in est]
    sections, inst, offs = pool.ComputeBatch(bool(pairwise), disp, seg, per_frame)
    assert read("pool.estimates").tobytes() == bytes(est)
    assert read("pool.roads").tobytes() == bytes(api._roads(per_frame))
    assert np.array_equal(read("pool.sections"), sections.view(np.uint8).reshape(-1))
    assert np.array_equal(read("pool.instances"), inst.view(np.uint8).reshape(-1))
    assert np.array_equal(read("pool.offsets").view(np.int32), offs)
    pool.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pairwise", [0, 1])
def test_runner_road_on_device_writes_the_same_files(tmp_path, pairwise):
    """--road-on-device: road estimation inside the timed pool call; the same .stixels files as the one-frame loop,
    and a frame whose estimation fails gets no file and its message.

    The other discard branch, 'Invalid road estimation.' (an accepted estimate whose horizon, pitch, height and slope
    are all zero), has no input that reaches it: an accepted line has theta > 0 (theta = 0 puts the horizon at
    infinity and the pitch out of range), and with the horizon at row 0 its slope is close to -tan(theta), not zero.
    The runner keeps the check because the reference's loop makes it (apps/run_cityscapes.cu:401-405)."""
    cv2 = pytest.importorskip("cv2")
    import torch
    import write_h5
    subprocess.run(["make", "-C", os.path.join(ROOT, "apps")], check=True, capture_output=True, text=True)
    rows, cols, n = 256, 512, 7
    for d in ("disparities", "camera", "probs", "stixels"):
        (tmp_path / d).mkdir()
    cam = {"extrinsic": {"baseline": 0.209313}, "intrinsic": {"fx": 2262.52, "fy": 2262.52, "u0": 256.0, "v0": 128.0}}
    for i in range(n + 1):
        fr = synth.make_frame(50 + i, rows=rows, cols=cols)
        base = f"city_{i:06d}_000019"
        q = np.clip(np.rint(fr.disparity * 256.0), 0, 65535).astype(np.uint16)
        if i == n:
            base = "city_000003_000020"      # sorts into the middle of the others
            q[:] = 0
        cv2.imwrite(str(tmp_path / "disparities" / f"{base}_disparity.png"), q)
        (tmp_path / "camera" / f"{base}_camera.json").write_text(json.dumps(cam))
        write_h5.write_h5(str(tmp_path / "probs" / f"{base}_probs.h5"), "nlogprobs", fr.segmentation)
    pre = synth.preset("pairwise" if pairwise else "unary", rows, cols, 8)
    args = [APP, str(tmp_path), "128", repr(pre["segmentation_weight"]), repr(pre["instance_weight"]),
            repr(pre["disparity_weight"]), str(pairwise), "8", repr(pre["eps"]), str(pre["min_pts"]),
            str(pre["size_filter"])]
    p = subprocess.run(args, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:] + p.stdout[-2000:]
    assert "Road estimation failed." in p.stdout
    single = {f: open(tmp_path / "stixels" / f, "rb").read() for f in sorted(os.listdir(tmp_path / "stixels"))}
    assert len(single) == n and "city_000003_000020.stixels" not in single
    gpus = min(2, torch.cuda.device_count())
    for extra in (["--batch", "3"], ["--batch", "2", "--gpus", str(gpus)], ["--batch", "16"]):
        shutil.rmtree(tmp_path / "stixels")
        (tmp_path / "stixels").mkdir()
        p = subprocess.run(args + extra + ["--road-on-device"], capture_output=True, text=True)
        assert p.returncode == 0, p.stderr[-2000:] + p.stdout[-2000:]
        assert "city_000003_000020: Road estimation failed." in p.stdout, extra
        got = {f: open(tmp_path / "stixels" / f, "rb").read() for f in sorted(os.listdir(tmp_path / "stixels"))}
        assert got.keys() == single.keys(), extra
        for f in single:
            assert got[f] == single[f], (extra, f)
        time_line = [l for l in p.stdout.split("\n")[-3:] if l.startswith("It took an average")][0]
        assert re.search(r"([0-9]*\.[0-9]*) milliseconds", time_line) and time_line.rstrip().endswith("fps")
