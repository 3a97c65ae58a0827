"""Device results (isx_export_batch_device, Stixels.ComputeBatchTensors): the stixels of a batch in caller device
buffers, frame-ordered, equal byte for byte to what the host entry points deliver."""
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


def _stixels(mode, rows, cols, w, max_batch, **over):
    pre = synth.preset(mode, rows, cols, w)
    pre.update(over)
    return api.make_stixels(pre, max_batch=max_batch)


def _expected(sections, inst, offs):
    """The host results ([n][C][200] Sections, packed instance records, per-frame offsets) in the export layout."""
    import parity
    n, C_ = sections.shape[:2]
    lens = np.stack([parity.column_lengths(sections[f]) for f in range(n)])         # [n][C]
    col_off = np.concatenate([[0], np.cumsum(lens.reshape(-1))]).astype(np.int32)
    frame_off = col_off[::C_].copy()
    packed = np.concatenate([sections[f, c, :lens[f, c]] for f in range(n) for c in range(C_)])
    labels = np.full(len(packed), -2, dtype=np.int32)
    for f in range(n):
        for r in inst[offs[f]:offs[f + 1]]:
            labels[col_off[f * C_ + r["column"]] + r["index"]] = r["label"]
    return dict(sections=packed, frame_offsets=frame_off, column_offsets=col_off, labels=labels)


def _buffers(n, C_, capacity):
    import torch
    u8 = lambda nbytes: torch.full((nbytes,), FILL, dtype=torch.uint8, device="cuda")
    return dict(sections=u8(capacity * 32), frame_offsets=u8((n + 1) * 4), column_offsets=u8((n * C_ + 1) * 4),
                labels=u8(capacity * 4), vertices=u8(capacity * 48), frame_errors=u8(n * 4))


def _export(st, first, n, capacity=None, vertices=True, **kw):
    """ExportBatchDevice into buffers pre-filled with 0x5A; returns their bytes as numpy arrays."""
    import torch
    C_ = st.GetRealCols()
    cap = n * C_ * 200 if capacity is None else capacity
    b = _buffers(n, C_, cap)
    if not vertices:
        b["vertices"] = b["vertices"][:0]
    torch.cuda.synchronize()
    st.ExportBatchDevice(first, n, b["frame_offsets"].data_ptr(), sections=b["sections"].data_ptr(),
                         column_offsets=b["column_offsets"].data_ptr(), labels=b["labels"].data_ptr(),
                         vertices=b["vertices"].data_ptr() if vertices else 0,
                         frame_errors=b["frame_errors"].data_ptr(), capacity=cap, **kw)
    st.Synchronize()
    return {k: v.cpu().numpy() for k, v in b.items()}


def _check_equal(got, want, n):
    fo = got["frame_offsets"].view(np.int32)
    assert np.array_equal(fo, want["frame_offsets"])
    assert np.array_equal(got["column_offsets"].view(np.int32), want["column_offsets"])
    total = int(fo[n])
    assert np.array_equal(got["sections"][:total * 32], want["sections"].view(np.uint8))
    assert np.array_equal(got["labels"].view(np.int32)[:total], want["labels"])
    assert np.array_equal(got["frame_errors"].view(np.int32), np.zeros(n, np.int32))
    assert (got["sections"][total * 32:] == FILL).all() and (got["labels"][total * 4:] == FILL).all()
    if got["vertices"].size:
        assert (got["vertices"][total * 48:] == FILL).all()


CASES = {
    "unary_w8_chunks": ("unary", 256, 512, 8, 6, {}, "4"),
    "pairwise_w8_chunks": ("pairwise", 256, 512, 8, 6, {}, "4"),
    "pairwise_w4": ("pairwise", 256, 512, 4, 3, {}, None),
    "median_join": ("pairwise", 256, 512, 8, 3, {"median_join": 1}, None),
    "tall_1208": ("pairwise", 1208, 512, 8, 1, {}, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_export_equals_the_host_results(case, monkeypatch):
    import torch
    mode, rows, cols, w, n, over, chunk = CASES[case]
    if chunk:
        monkeypatch.setenv("ISX_CHUNK", chunk)
    st = _stixels(mode, rows, cols, w, n, **over)
    disp, seg, roads = synth.make_batch(n, start=3, rows=rows, cols=cols, column_step=w)
    sections, inst, offs = st.ComputeBatch(mode == "pairwise", disp, seg, roads)
    want = _expected(sections, inst, offs)
    assert (want["labels"] >= -1).sum() == len(inst) > 0
    # after a device batch
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(mode == "pairwise", n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    _check_equal(_export(st, 0, n), want, n)
    # after a synchronous host batch
    st.ComputeBatch(mode == "pairwise", disp, seg, roads)
    _check_equal(_export(st, 0, n, vertices=False), want, n)
    st.Finish()


@pytest.mark.gpu
def test_export_after_single_frame_compute_and_a_streamed_batch():
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=11, rows=rows, cols=cols)
    sections, inst, offs = st.ComputeBatch(True, disp, seg, roads)
    want = _expected(sections, inst, offs)
    st.SetDisparityImage(disp[2]); st.SetSegmentation(seg[2]); st.SetRoadParameters(**roads[2])
    data = st.Compute(True)
    single = _expected(data.sections[None], st.instance_records(), np.array([0, len(st.instance_records())]))
    _check_equal(_export(st, 0, 1), single, 1)
    outs = [np.zeros_like(sections) for _ in range(2)]
    st.SubmitBatch(True, disp, seg, roads, outs[0])
    st.SubmitBatch(True, disp, seg, roads, outs[1])
    st.WaitBatch()
    st.WaitBatch()
    _check_equal(_export(st, 0, n), want, n)
    st.Finish()


@pytest.mark.gpu
def test_export_is_deterministic_bounded_and_takes_subranges():
    import torch
    rows, cols, n = 256, 512, 6
    st = _stixels("unary", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=20, rows=rows, cols=cols)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    st.ComputeBatchDevice(False, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    a, b = _export(st, 0, n), _export(st, 0, n)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    fo, co = a["frame_offsets"].view(np.int32), a["column_offsets"].view(np.int32)
    total, C_ = int(fo[n]), st.GetRealCols()
    for k, size in (("sections", 32), ("labels", 4), ("vertices", 48)):
        assert (a[k][total * size:] == FILL).all(), k
    # frames [2, 5): the matching slice, offsets rebased to 0
    s = _export(st, 2, 3)
    lo, hi = int(fo[2]), int(fo[5])
    assert np.array_equal(s["frame_offsets"].view(np.int32), fo[2:6] - lo)
    assert np.array_equal(s["column_offsets"].view(np.int32), co[2 * C_:5 * C_ + 1] - lo)
    for k, size in (("sections", 32), ("labels", 4), ("vertices", 48)):
        assert np.array_equal(s[k][:(hi - lo) * size], a[k][lo * size:hi * size]), k
    # capacity that ends inside frame 3: frames 0..2 written, nothing else, offsets complete
    cap = int(fo[3]) + (int(fo[4]) - int(fo[3])) // 2
    c = _export(st, 0, n, capacity=cap)
    assert np.array_equal(c["frame_offsets"], a["frame_offsets"])
    assert np.array_equal(c["column_offsets"], a["column_offsets"])
    assert np.array_equal(c["frame_errors"], a["frame_errors"])
    end = int(fo[3])
    for k, size in (("sections", 32), ("labels", 4), ("vertices", 48)):
        assert np.array_equal(c[k][:end * size], a[k][:end * size]), k
        assert (c[k][end * size:] == FILL).all(), k
    st.Finish()


def _build_vertices_harness(tmp_path):
    exe = str(tmp_path / "vertices_harness")
    libdir = os.path.join(ROOT, "instance_stixels_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include", "InstanceStixels"),
           os.path.join(ROOT, "tests", "cpp", "vertices_harness.cpp"), "-L" + libdir, "-linstance_stixels_b200",
           "-Wl,-rpath," + libdir, "-o", exe]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


def test_vertices_harness_compiles(tmp_path):
    assert os.path.exists(_build_vertices_harness(tmp_path))


def test_device_results_struct_is_56_bytes():
    assert C.sizeof(L.DeviceResults) == 56


def test_export_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "export_bench.py"), "--help"], capture_output=True,
                       text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout


@pytest.mark.gpu
def test_vertices_equal_the_header_bit_for_bit(tmp_path):
    import torch
    exe = _build_vertices_harness(tmp_path)
    rows, cols, n = 256, 512, 4
    # camera centre on a column boundary and an image row: with an infinite depth, corners there give NaN
    over = dict(camera_center_x=128.0, camera_center_y=100.0)
    st = _stixels("unary", rows, cols, 8, n, **over)
    disp, seg, roads = synth.make_batch(n, start=30, rows=rows, cols=cols)
    # A ground stixel always ends below the horizon here (vT < vhor), so the header's division by zero at
    # vT == vhor cannot be reached with a real road.  alpha_ground = 0 on frame 3 takes the same path instead:
    # every ground stixel of that frame lies at infinite depth.
    roads[3] = dict(roads[3], alpha_ground=0.0)
    sections, _, _ = st.ComputeBatch(False, disp, seg, roads)
    got = _export(st, 0, n)
    total = int(got["frame_offsets"].view(np.int32)[n])
    dev = got["vertices"][:total * 48].view(np.float32)
    pre = synth.preset("unary", rows, cols, 8)
    flipped = np.array([[np.float32(r["alpha_ground"]).view(np.int32), rows - r["vhor"] - 1] for r in roads],
                       dtype=np.int32)
    sections.tofile(tmp_path / "s.bin")
    flipped.tofile(tmp_path / "r.bin")
    p = subprocess.run([exe, str(tmp_path / "s.bin"), str(tmp_path / "r.bin"), str(n), str(rows), str(cols), "8",
                        repr(pre["focal"]), repr(pre["baseline"]), "128", "100", str(tmp_path / "v.f32")],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    host = np.fromfile(tmp_path / "v.f32", dtype=np.float32)
    assert host.size == dev.size == total * 12
    nan = np.isnan(host)
    assert np.array_equal(nan, np.isnan(dev))
    assert np.array_equal(host[~nan].view(np.int32), dev[~nan].view(np.int32))
    inf = np.isinf(host)
    print(f"compared {host.size} vertex values, {int(inf.sum())} inf, {int(nan.sum())} NaN")
    assert inf.sum() > 0 and nan.sum() > 0
    finite = dev[np.isfinite(dev)]
    assert not ((finite != 0) & (np.abs(finite) < np.finfo(np.float32).tiny)).any(), "subnormal vertex value"
    # ground stixels that end one row below the horizon (the farthest ground, the largest depth) are among the compared
    sec = got["sections"][:total * 32].view(L.SECTION_DTYPE)
    fo = got["frame_offsets"].view(np.int32)
    top_ground = [((sec[fo[f]:fo[f + 1]]["type"] == 0) & (sec[fo[f]:fo[f + 1]]["vT"] == flipped[f, 1] - 1)).sum()
                  for f in range(n)]
    assert sum(top_ground[:3]) > 0
    # without the camera centre the vertices are refused, like Get3DVertices
    st2 = _stixels("unary", rows, cols, 8, n, camera_center_x=-1.0)
    st2.ComputeBatch(False, disp, seg, roads)
    with pytest.raises(api.InvalidArgument, match="Camera parameters are not set"):
        _export(st2, 0, n)
    assert _export(st2, 0, n, vertices=False)["frame_offsets"].view(np.int32)[n] == total
    st2.Finish()
    st.Finish()


@pytest.mark.gpu
def test_frame_errors_belong_to_their_frame():
    rows, cols, n = 256, 128, 3
    st = _stixels("pairwise", rows, cols, 8, 4)
    disp, seg, roads = synth.make_batch(n, start=5, rows=rows, cols=cols)
    st.ComputeBatch(True, disp, seg, roads)
    clean = _export(st, 0, n)
    bad = seg.copy()
    bad[1, :, 20, :rows // 8] = 400000          # x offsets of 50 km: sum of the instance means >= 2^24
    with pytest.raises(api.StixelsError, match="frame 1"):
        st.ComputeBatch(True, disp, bad, roads)
    got = _export(st, 0, n)
    assert got["frame_errors"].view(np.int32).tolist() == [0, 2, 0]
    cf, gf = clean["frame_offsets"].view(np.int32), got["frame_offsets"].view(np.int32)
    for f in (0, 2):
        a = clean["sections"][cf[f] * 32:cf[f + 1] * 32]
        b = got["sections"][gf[f] * 32:gf[f + 1] * 32]
        assert np.array_equal(a, b), f
    st.Finish()


@pytest.mark.gpu
def test_refused_exports_enqueue_nothing():
    import torch
    rows, cols, n = 256, 512, 3
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=40, rows=rows, cols=cols)
    sections, inst, offs = st.ComputeBatch(True, disp, seg, roads)
    want = _expected(sections, inst, offs)
    C_, cap = st.GetRealCols(), n * st.GetRealCols() * 200
    b = _buffers(n, C_, cap)
    torch.cuda.synchronize()
    lib = st._lib

    def call(first, nn, **over):
        args = dict(sections=b["sections"].data_ptr(), frame_offsets=b["frame_offsets"].data_ptr(),
                    column_offsets=b["column_offsets"].data_ptr(), labels=b["labels"].data_ptr(),
                    vertices=b["vertices"].data_ptr(), frame_errors=b["frame_errors"].data_ptr(), capacity=cap)
        args.update(over)
        out = L.DeviceResults(*(args[k] or None for k in ("sections", "frame_offsets", "column_offsets", "labels",
                                                           "vertices", "frame_errors")), args["capacity"], 0)
        return lib.isx_export_batch_device(st._h, first, nn, C.byref(out))

    launches = lib.isx_kernel_launch_count()
    refusals = [call(-1, 1), call(0, 0), call(1, n), call(0, n, frame_offsets=0),
                call(0, n, sections=b["sections"].data_ptr() + 4), call(0, n, capacity=-1)]
    assert lib.isx_kernel_launch_count() == launches
    # vertices without the camera centre, on a handle configured without it
    nocam = _stixels("pairwise", rows, cols, 8, n, camera_center_x=-1.0)
    nocam.ComputeBatch(True, disp, seg, roads)
    launches = lib.isx_kernel_launch_count()
    out = L.DeviceResults(b["sections"].data_ptr(), b["frame_offsets"].data_ptr(), b["column_offsets"].data_ptr(),
                          b["labels"].data_ptr(), b["vertices"].data_ptr(), b["frame_errors"].data_ptr(), cap, 0)
    refusals.append(lib.isx_export_batch_device(nocam._h, 0, n, C.byref(out)))
    assert b"Camera parameters are not set" in lib.isx_last_error(nocam._h)
    assert lib.isx_kernel_launch_count() == launches
    nocam.Finish()
    st.SubmitBatch(True, disp, seg, roads, np.zeros_like(sections))
    launches = lib.isx_kernel_launch_count()
    refusals.append(call(0, n))
    assert lib.isx_kernel_launch_count() == launches
    st.WaitBatch()
    assert refusals == [-1] * len(refusals)
    st.Synchronize()
    assert all((v.cpu().numpy() == FILL).all() for v in b.values())
    _check_equal(_export(st, 0, n), want, n)
    st.Finish()


def _cnn_of(seg, rows):
    """The float CNN output [n][21][rows/8][cols/8] whose FlipAndPad is `seg` (column_step 8)."""
    hs = rows // 8
    return np.ascontiguousarray(seg[:, :, :, :hs][:, :, :, ::-1].transpose(0, 2, 3, 1) / np.float32(8.0),
                                dtype=np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["segmentation", "cnn"])
def test_torch_path_without_synchronize(source):
    import torch
    rows, cols, n = 256, 512, 4
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=50, rows=rows, cols=cols)
    cnn = _cnn_of(seg, rows)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):    # inputs produced on another stream, as a CNN runtime would
        d_disp = torch.from_numpy(disp).pin_memory().cuda(non_blocking=True)
        d_in = torch.from_numpy(cnn if source == "cnn" else seg).pin_memory().cuda(non_blocking=True)
    torch.cuda.current_stream().wait_stream(side)
    if source == "cnn":
        out = st.ComputeBatchTensors(True, d_disp, roads, cnn=d_in, vertices=True)
    else:
        out = st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_in, vertices=True)
    del d_disp, d_in
    # consumers on the current stream
    total = int(out.frame_offsets[n].item())
    sections = out.sections[:total].clone().cpu().numpy().reshape(-1).view(L.SECTION_DTYPE)
    got = dict(frame_offsets=out.frame_offsets.cpu().numpy(), column_offsets=out.column_offsets.cpu().numpy(),
               labels=out.labels[:total].cpu().numpy(), errors=out.frame_errors.cpu().numpy())
    if source == "cnn":
        # the reference input: FlipAndPadBatchDevice of a separate copy of the CNN tensor, after the outputs were read
        d_ref = torch.from_numpy(cnn).cuda()
        ingest = torch.empty(n * st.segmentation_elems(), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        st.FlipAndPadBatchDevice(n, d_ref.data_ptr(), rows // 8, cols // 8, ingest.data_ptr())
        st.Synchronize()
        seg = ingest.cpu().numpy().reshape(seg.shape)
    want = _expected(*st.ComputeBatch(True, disp, seg, roads))
    assert np.array_equal(got["frame_offsets"], want["frame_offsets"])
    assert np.array_equal(got["column_offsets"], want["column_offsets"])
    assert np.array_equal(sections.view(np.uint8), want["sections"].view(np.uint8))
    assert np.array_equal(got["labels"], want["labels"]) and not got["errors"].any()
    assert np.array_equal(out.disparity[:total].cpu().numpy(), want["sections"]["disparity"])
    assert np.array_equal(out.vT[:total].cpu().numpy(), want["sections"]["vT"])
    assert out.vertices.shape == (n * st.GetRealCols() * 200, 4, 3)
    st.Finish()


@pytest.mark.gpu
def test_torch_path_refuses_tensors_off_the_handles_device():
    import torch
    rows, cols, n = 256, 512, 2
    st = _stixels("pairwise", rows, cols, 8, n)
    disp, seg, roads = synth.make_batch(n, start=60, rows=rows, cols=cols)
    with pytest.raises(api.InvalidArgument):
        st.ComputeBatchTensors(True, torch.from_numpy(disp), roads, segmentation=torch.from_numpy(seg).cuda())
    with pytest.raises(api.InvalidArgument, match="device"):
        st.ComputeBatchTensors(True, torch.from_numpy(disp).cuda(), roads, segmentation=torch.from_numpy(seg))
    if torch.cuda.device_count() > 1:
        with pytest.raises(api.InvalidArgument, match="handle computes on cuda:0"):
            st.ComputeBatchTensors(True, torch.from_numpy(disp).to("cuda:1"), roads,
                                   segmentation=torch.from_numpy(seg).to("cuda:1"))
    st.Finish()
