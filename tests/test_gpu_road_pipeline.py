"""Road estimation inside device batches (isx_compute_batch_device_road): the road of every frame is estimated on
the device from its own disparity and the stixels follow in stream order.  Everything must equal, byte for byte,
the synchronous composition isx_road_compute_batch_device -> keep-last substitution -> isx_compute_batch_device."""
import ctypes as C
import os
import shutil
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from instance_stixels_b200 import _lib as L  # noqa: E402
from instance_stixels_b200 import api, synth  # noqa: E402

CAM = dict(camera_center_y=512.0, baseline=0.209313, focal=2262.52)
FALLBACK = dict(vhor=100, camera_tilt=0.0, camera_height=1.18, alpha_ground=0.177384)
FILL = 0x5A
HARNESS = os.path.join(ROOT, "tests", "cpp", "road_pipeline_harness.cpp")


def _stixels(mode, rows, cols, w, max_batch, **over):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(over)
    return api.make_stixels(pre, max_batch=max_batch)


def _road(rows, cols, max_batch, max_dis=128):
    re = api.RoadEstimation()
    re.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], rows, cols, max_dis, 0.2, max_batch=max_batch)
    return re


def _frames(n, rows, cols, w, zero=(0, 3), start=0):
    """Frames with horizons spread over the image (so that they select different Hough cells); the frames in `zero`
    have no disparity at all, so their estimation fails."""
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


def _keep_last(estimates, seed):
    out, cur = [], seed
    for e in estimates:
        if e.ok:
            cur = _road_of(e)
        out.append(cur)
    return out


def _host_estimates(re, n, d_disp):
    est = (L.RoadEstimate * n)()
    assert re._lib.isx_road_compute_batch_device(re.handle(), n, d_disp.data_ptr(), est) == 0
    return est


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


def _composition(st, re, pairwise, n, d_disp, d_seg, seed):
    est = _host_estimates(re, n, d_disp)
    roads = _keep_last(est, seed)
    st.ComputeBatchDevice(pairwise, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    return est, roads, st.FetchBatchResults(n), _export(st, n)


def _pipeline(st, re, pairwise, n, d_disp, d_seg, fallback):
    import torch
    d_est, d_roads = _u8(n * 28), _u8(n * 16)
    torch.cuda.synchronize()
    st.ComputeBatchDeviceRoad(re, pairwise, n, d_disp.data_ptr(), d_seg.data_ptr(), fallback, d_est.data_ptr(),
                              d_roads.data_ptr())
    fetched = st.FetchBatchResults(n)
    return d_est.cpu().numpy(), d_roads.cpu().numpy(), fetched, _export(st, n)


def _check_same(want, got):
    est, roads, (ws, wi, wo), wexp = want
    g_est, g_roads, (gs, gi, go), gexp = got
    assert g_est.tobytes() == bytes(est)
    assert g_roads.tobytes() == bytes(api._roads(roads))
    assert np.array_equal(gs.view(np.uint8), ws.view(np.uint8))
    assert np.array_equal(gi.view(np.uint8), wi.view(np.uint8)) and np.array_equal(go, wo)
    for k in wexp:
        assert np.array_equal(gexp[k], wexp[k]), k


CASES = {
    "unary_w8_chunks": ("unary", 256, 512, 8, 7, {}, "4"),
    "pairwise_w8_chunks": ("pairwise", 256, 512, 8, 7, {}, "4"),
    "unary_w4": ("unary", 256, 512, 4, 5, {}, None),
    "pairwise_w4": ("pairwise", 256, 512, 4, 5, {}, None),
    "median_join": ("pairwise", 256, 512, 8, 5, {"median_join": 1}, None),
    "tall_1208": ("pairwise", 1208, 512, 8, 3, {}, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_pipeline_equals_the_composition(case, monkeypatch):
    import torch
    mode, rows, cols, w, n, over, chunk = CASES[case]
    if chunk:
        monkeypatch.setenv("ISX_CHUNK", chunk)
    pairwise = mode == "pairwise"
    st = _stixels(mode, rows, cols, w, n, **over)
    re = _road(rows, cols, n)
    disp, seg = _frames(n, rows, cols, w, zero=(0, 3) if n > 3 else (0,))
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    want = _composition(st, re, pairwise, n, d_disp, d_seg, FALLBACK)
    est = want[0]
    assert not est[0].ok and sum(e.ok for e in est) >= n - 2
    assert len({(e.horizon_point, e.rho, e.theta) for e in est if e.ok}) >= 2, "frames should select different cells"
    got = _pipeline(st, re, pairwise, n, d_disp, d_seg, FALLBACK)
    _check_same(want, got)
    # the same again from the state the first call left (its last frame was accepted: the seed is not used)
    again = _pipeline(st, re, pairwise, n, d_disp, d_seg, None)
    want_again = _composition(st, re, pairwise, n, d_disp, d_seg, want[1][-1])
    _check_same(want_again, again)
    st.Finish()


@pytest.mark.gpu
def test_selection_agrees_with_the_oracle():
    import glob
    import torch
    import make_road_golden
    from oracle import road_cpu
    for path in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "road_*.npz"))):
        z = np.load(path)
        rows, cols = int(z["rows"]), int(z["cols"])
        frame = make_road_golden.frame_disparity(str(z["name"]), rows, cols, int(z["frame"]))
        disp = np.ascontiguousarray(np.stack([frame, np.zeros_like(frame), frame]))
        n = len(disp)
        st = _stixels("unary", rows, cols, 8, n)
        re = _road(rows, cols, n)
        d_disp = torch.from_numpy(disp).cuda()
        d_seg = torch.zeros(n * st.segmentation_elems(), dtype=torch.int32, device="cuda")
        d_est = _u8(n * 28)
        torch.cuda.synchronize()
        st.ComputeBatchDeviceRoad(re, False, n, d_disp.data_ptr(), d_seg.data_ptr(), FALLBACK, d_est.data_ptr())
        st.Synchronize()
        got = np.frombuffer(d_est.cpu().numpy().tobytes(), dtype=np.dtype(
            [("ok", "<i4"), ("horizon_point", "<i4"), ("f", "<f4", (5,))]))
        est, _ = road_cpu.estimate(frame, 128, *CAM.values())
        assert bool(est["ok"]) == bool(z["ok"]), path
        for f in (0, 2):
            assert bool(got[f]["ok"]) == bool(est["ok"]), path
            assert got[f]["horizon_point"] == (est["horizon_point"] if est["ok"] else 0), path
            want = np.array([est[k] for k in ("pitch", "camera_height", "slope", "rho", "theta")], np.float32)
            if not est["ok"]:
                want[:] = 0
            assert np.array_equal(got[f]["f"].view(np.int32), want.view(np.int32)), path
        assert not got[1]["ok"]
        if "tilted" in path:
            assert got[0]["f"][4] != 0.0      # the wall's vertical line (theta = 0) comes first and is skipped
        st.Finish()
        re.Finish()


@pytest.mark.gpu
def test_fallback_and_keep_last_across_calls():
    import torch
    rows, cols, w, n = 256, 512, 8, 5
    st = _stixels("unary", rows, cols, w, n)
    re = _road(rows, cols, n)
    disp, seg = _frames(n, rows, cols, w, zero=(0, 2, 4))
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    est = _host_estimates(re, n, d_disp)
    a, b = _road_of(est[1]), _road_of(est[3])
    assert est[1].ok and est[3].ok and a != b

    def roads_of(k, d, fallback):
        d_roads = _u8(k * 16)
        torch.cuda.synchronize()
        st.ComputeBatchDeviceRoad(re, False, k, d.data_ptr(), d_seg.data_ptr(), fallback, 0, d_roads.data_ptr())
        st.Synchronize()
        return d_roads.cpu().numpy().tobytes()

    # a failing first frame takes the seed, a failing frame mid-batch the previous accepted estimate
    assert roads_of(n, d_disp, FALLBACK) == bytes(api._roads([FALLBACK, a, a, b, b]))
    # fallback=None: the next call continues from b
    assert roads_of(1, d_disp[0:1].contiguous(), None) == bytes(api._roads([b]))
    assert roads_of(2, d_disp[0:2].contiguous(), None) == bytes(api._roads([b, a]))
    # a fallback given again resets the state
    other = dict(FALLBACK, vhor=90)
    assert roads_of(1, d_disp[0:1].contiguous(), other) == bytes(api._roads([other]))
    assert roads_of(1, d_disp[0:1].contiguous(), None) == bytes(api._roads([other]))
    st.Finish()


@pytest.mark.gpu
def test_refusals_enqueue_nothing():
    import torch
    rows, cols, w, n = 256, 512, 8, 3
    st = _stixels("pairwise", rows, cols, w, n)
    disp, seg = _frames(n + 1, rows, cols, w, zero=())
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    d_est = _u8((n + 1) * 28)
    torch.cuda.synchronize()
    lib = st._lib
    fb = C.byref(api._roads([FALLBACK])[0])

    def call(re_h, k, disp_ptr=d_disp.data_ptr(), seg_ptr=d_seg.data_ptr(), fallback=fb):
        return lib.isx_compute_batch_device_road(st._h, re_h, 1, k, disp_ptr, seg_ptr, fallback, d_est.data_ptr(),
                                                 None)

    good = _road(rows, cols, n + 1)
    unset = api.RoadEstimation()                   # never initialised
    other_rows = _road(rows // 2, cols, n)
    other_cols = _road(rows, cols // 2, n)
    other_dis = _road(rows, cols, n, max_dis=64)
    small = _road(rows, cols, n - 1)
    fresh = _road(rows, cols, n)                   # never seeded
    launches = lib.isx_kernel_launch_count()
    got = [call(unset.handle(), n), call(other_rows.handle(), n), call(other_cols.handle(), n),
           call(other_dis.handle(), n), call(None, n), call(good.handle(), n, disp_ptr=None),
           call(good.handle(), n, seg_ptr=None), call(fresh.handle(), n, fallback=None),
           call(good.handle(), n + 1), call(small.handle(), n), call(good.handle(), 0)]
    assert got == [-1] * 8 + [-4] * 3, got
    assert lib.isx_kernel_launch_count() == launches
    # batches in flight
    st.SubmitBatch(True, disp[:n], seg[:n], [FALLBACK] * n, np.zeros((n, st.GetRealCols(), 200), L.SECTION_DTYPE))
    launches = lib.isx_kernel_launch_count()
    assert call(good.handle(), n) == -1
    assert lib.isx_kernel_launch_count() == launches
    st.WaitBatch()
    torch.cuda.synchronize()
    assert (d_est.cpu().numpy() == FILL).all()
    assert call(good.handle(), n) == 0          # and the handle is usable afterwards
    st.Synchronize()
    st.Finish()


def _cnn_of(seg, rows):
    hs = rows // 8
    return np.ascontiguousarray(seg[:, :, :, :hs][:, :, :, ::-1].transpose(0, 2, 3, 1) / np.float32(8.0),
                                dtype=np.float32)


@pytest.mark.gpu
def test_torch_path_does_not_wait_for_the_device():
    import torch
    rows, cols, w, n = 256, 512, 8, 6
    st = _stixels("pairwise", rows, cols, w, n)
    re = _road(rows, cols, n)
    disp, seg = _frames(n, rows, cols, w, zero=(0, 4))
    # ComputeBatchTensors marks its inputs as used on isx_stream() (record_stream): they must be released while that
    # stream exists, i.e. before Finish(), also when an assertion fails
    inputs = dict(disp=torch.from_numpy(disp).cuda(), cnn=torch.from_numpy(_cnn_of(seg, rows)).cuda())
    try:
        # warm-up: the table of per-cell estimates and the result arrays are built on first use
        st.ComputeBatchTensors(True, inputs["disp"], road=re, cnn=inputs["cnn"], fallback=FALLBACK)
        torch.cuda.synchronize()
        cycles = 200_000_000
        t0 = time.perf_counter()
        torch.cuda._sleep(cycles)
        torch.cuda.synchronize()
        sleep_s = time.perf_counter() - t0
        torch.cuda._sleep(cycles)
        t0 = time.perf_counter()
        out = st.ComputeBatchTensors(True, inputs["disp"], road=re, cnn=inputs["cnn"], fallback=FALLBACK, vertices=True)
        call_s = time.perf_counter() - t0
        got = {k: getattr(out, k).cpu().numpy() for k in ("sections", "frame_offsets", "column_offsets", "labels",
                                                           "vertices", "frame_errors")}
        est, roads = out.road_estimates.data.cpu().numpy(), out.roads.data.cpu().numpy()
        ok, alpha = out.road_estimates.ok.cpu().tolist(), out.roads.alpha_ground.cpu().numpy()
        # the composition on the same stream
        host = _host_estimates(re, n, inputs["disp"])
        composed = _keep_last(host, FALLBACK)
        ref = st.ComputeBatchTensors(True, inputs["disp"], composed, cnn=inputs["cnn"], vertices=True)
        want = {k: getattr(ref, k).cpu().numpy() for k in got}
    finally:
        inputs.clear()
        torch.cuda.synchronize()
    st.Finish()
    assert call_s < 0.25 * sleep_s, (call_s, sleep_s)
    assert est.tobytes() == bytes(host) and roads.tobytes() == bytes(api._roads(composed))
    assert ok == [e.ok for e in host]
    assert alpha.tolist() == [np.float32(r["alpha_ground"]) for r in composed]
    total = int(want["frame_offsets"][n])
    for k in got:
        a, b = (got[k][:total], want[k][:total]) if k in ("sections", "labels", "vertices") else (got[k], want[k])
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), k


def _cuda_home():
    nvcc = shutil.which("nvcc")
    return os.path.dirname(os.path.dirname(nvcc)) if nvcc else os.environ.get("CUDA_HOME", "/usr/local/cuda")


def _build_harness(tmp_path):
    exe = str(tmp_path / "road_pipeline_harness")
    libdir = os.path.join(ROOT, "instance_stixels_b200")
    cuda = _cuda_home()
    cmd = ["g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include", "InstanceStixels"),
           "-I" + os.path.join(cuda, "include"), HARNESS, "-L" + libdir, "-linstance_stixels_b200",
           "-L" + os.path.join(cuda, "lib64"), "-lcudart", "-Wl,-rpath," + libdir,
           "-Wl,-rpath," + os.path.join(cuda, "lib64"), "-o", exe]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return exe


def test_road_pipeline_harness_compiles(tmp_path):
    assert os.path.exists(_build_harness(tmp_path))


def test_road_pipeline_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "road_pipeline_bench.py"), "--help"],
                       capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("pairwise", [0, 1])
def test_cpp_overload_equals_the_composition(tmp_path, pairwise):
    import torch
    exe = _build_harness(tmp_path)
    rows, cols, w, n = 256, 512, 8, 4
    disp, seg = _frames(n, rows, cols, w, zero=(0, 2))
    disp.tofile(tmp_path / "d.f32")
    seg.tofile(tmp_path / "s.i32")
    fb = dict(FALLBACK)
    p = subprocess.run([exe, str(tmp_path / "d.f32"), str(tmp_path / "s.i32"), str(n), str(rows), str(cols),
                        str(pairwise), str(fb["vhor"]), repr(fb["alpha_ground"]), str(tmp_path / "out")],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr + p.stdout
    fb["alpha_ground"] = float(np.float32(float(repr(fb["alpha_ground"]))))
    st = _stixels("pairwise" if pairwise else "unary", rows, cols, w, n)
    re = _road(rows, cols, n)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    est, roads, (sections, inst, offs), _ = _composition(st, re, bool(pairwise), n, d_disp, d_seg, fb)
    read = lambda ext: np.fromfile(tmp_path / f"out.{ext}", dtype=np.uint8)
    assert read("estimates").tobytes() == bytes(est)
    assert read("roads").tobytes() == bytes(api._roads(roads))
    assert np.array_equal(read("sections"), sections.view(np.uint8).reshape(-1))
    assert np.array_equal(read("instances"), inst.view(np.uint8).reshape(-1))
    assert np.array_equal(read("offsets").view(np.int32), offs)
    st.Finish()
