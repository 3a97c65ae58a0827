"""Frames of 1025 to 2047 rows (ISX_MAX_ROWS): 1080-, 1200- and 1280-row cameras.

The reference stops at 1024 rows, so the CPU oracle (oracle/stixels_cpu.cpp, the reference restated for any height
and pinned to the reference build by the golden vectors) is the checker: its Blelloch scans run over
rows_power2 = 2048 like the reference's would, and up to 2047 rows rows_power2_segmentation stays 256.
  * tables bit for bit (object LUT, the four Blelloch-order prefixes), results with the criteria of
    test_gpu_parity.test_against_cpu_oracle_with_tables;
  * the pruning kernels against the exhaustive ones, byte for byte, on fixed shapes and a seeded fuzz;
  * the entry points against each other at 1208 rows; the limits; ingest, road estimation, raster and the runner."""
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

import parity
from instance_stixels_b200 import _lib as L, api, synth
from oracle import cpubind, ingest_cpu, raster_cpu, road_cpu

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# rows, cols, step, invalid_disparity, median_join
ORACLE_CASES = [
    (1025, 256, 8, 0.0, False),    # 33 tiles, the last one a single row
    (1208, 512, 8, 0.0, False),    # rows % 32 != 0
    (1280, 384, 8, -1.0, False),   # no invalid disparity
    (2047, 256, 8, 0.0, False),    # the tallest frame: 64 chunk carries per LUT row
    (1208, 256, 4, 0.0, False),    # width 4
    (1280, 256, 8, 0.0, True),     # median join
    (2040, 256, 8, 0.0, False),    # the tallest frame whose rows all have a defined reference result (below)
]
SHAPES = ORACLE_CASES[:4]


def _rows_with_reference_result(rows):
    """Rows v whose costs the reference defines.  Its class sums read the exclusive prefix of downsampled entry
    v // 8 + 1 (Cityscapes.h:28-42); when that is rows_power2_segmentation itself (rows 2041-2047: entry 256) the
    read lies one past the channel's prefix array, in the next channel (the CPU oracle restates that literally).  The
    library uses the sum of the caller's entries there, so only the rows below are compared with the oracle."""
    hs2 = 1 << (rows // 8).bit_length()
    return rows if (rows - 1) // 8 + 1 < hs2 else 8 * (hs2 - 1)
PS_TENSORS = (L.T_DISPARITY_PS, L.T_VALID_PS, L.T_GROUND_PS, L.T_SKY_PS)


@pytest.fixture(scope="module")
def oracle_prefix(tmp_path_factory):
    """(config, pairwise, disparity, segmentation, road) -> [C][4][rows+1] prefixes of disparity, valid, ground, sky:
    tests/cpp/oracle_prefix.cpp, the CPU oracle's source compiled unchanged with an entry point that returns them."""
    so = str(tmp_path_factory.mktemp("oracle_prefix") / "liboracle_prefix.so")
    cxx = "/usr/bin/g++" if os.access("/usr/bin/g++", os.X_OK) else "g++"
    subprocess.run([cxx, "-std=c++17", "-O2", "-mfma", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-o", so,
                    os.path.join(ROOT, "tests", "cpp", "oracle_prefix.cpp")], check=True, capture_output=True, text=True)
    lib = ctypes.CDLL(so)
    V = ctypes.c_void_p
    lib.orc_prefix_tables.argtypes = [ctypes.POINTER(L.Config), ctypes.c_int, V, V, ctypes.POINTER(L.Road),
                                      ctypes.c_int, V]

    def compute(config, pairwise, disparity, segmentation, road):
        C_ = (int(config.cols) - config.width_margin) // config.column_step
        out = np.zeros((C_, 4, int(config.rows) + 1), np.float32)
        d = np.ascontiguousarray(disparity, dtype=np.float32)
        s_ = np.ascontiguousarray(segmentation, dtype=np.int32)
        r = L.Road(int(road["vhor"]), road["camera_tilt"], road["camera_height"], road["alpha_ground"])
        lib.orc_prefix_tables(ctypes.byref(config), int(pairwise), d.ctypes.data, s_.ctypes.data, ctypes.byref(r), 0,
                              out.ctypes.data)
        return out
    return compute


def _case_id(c):
    return f"{c[0]}x{c[1]}w{c[2]}inv{c[3]:g}" + ("med" if c[4] else "")


def _preset(mode, rows, cols, step, invalid=0.0, median=False, **weights):
    pre = synth.preset(mode, rows, cols, step)
    pre["invalid_disparity"] = invalid
    pre["median_join"] = median
    pre.update(weights)
    return pre


def _compute(pre, pairwise, disp, seg, road):
    st = api.make_stixels(pre, max_batch=1)
    st.SetDisparityImage(disp)
    st.SetSegmentation(seg)
    st.SetRoadParameters(**road)
    data = st.Compute(pairwise)
    out = dict(sections=data.sections.copy(), inst=st.instance_records().copy(),
               cost=st.read_tensor(L.T_COST_TABLE).copy(), index=st.read_tensor(L.T_INDEX_TABLE).copy(),
               units=st.dp_units())
    return st, out


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
@pytest.mark.parametrize("case", ORACLE_CASES, ids=_case_id)
def test_against_cpu_oracle_with_tables(case, mode, oracle_prefix):
    rows, cols, step, invalid, median = case
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, step, invalid, median)
    fr = synth.make_frame(rows % 97, rows=rows, cols=cols, column_step=step)
    st, ours = _compute(pre, pairwise, fr.disparity, fr.segmentation, fr.road)
    osec, oinst, ex = cpubind.compute_frame(cpubind.default_config(**pre), pairwise, fr.disparity, fr.segmentation,
                                            fr.road, tables=True)
    prefix = oracle_prefix(cpubind.default_config(**pre), pairwise, fr.disparity, fr.segmentation, fr.road)
    C_ = cols // step
    # tables: pure fp32 adds in the reference's orders, bit for bit
    lut = st.read_tensor(L.T_OBJECT_LUT).reshape(C_, -1, rows + 1)
    assert np.array_equal(lut.view(np.int32), ex["object_lut"].view(np.int32))
    for i, t in enumerate(PS_TENSORS):
        if t == L.T_VALID_PS and invalid < 0:
            continue                      # not scanned by the reference without an invalid disparity
        ps = st.read_tensor(t).reshape(C_, rows + 1)
        assert np.array_equal(ps.view(np.int32), prefix[:, i].view(np.int32)), t
    j = st.read_tensor(L.T_JOINED_DISPARITY).reshape(C_, rows)
    assert np.allclose(j, ex["joined"], rtol=1e-6, atol=0)
    # results: the criteria of the CPU-oracle test at <= 1024 rows
    nrows = _rows_with_reference_result(rows)
    cost = ours["cost"].reshape(C_, rows, 3)[:, :nrows]
    index = ours["index"].reshape(C_, rows, 3)[:, :nrows]
    ocost, oindex = ex["cost_table"][:, :nrows], ex["index_table"][:, :nrows]
    fin = np.isfinite(ocost)
    assert np.array_equal(fin, np.isfinite(cost))
    rel = np.abs(cost[fin] - ocost[fin]) / np.maximum(np.abs(ocost[fin]), 1e-6)
    assert np.quantile(rel, 0.999) <= 1e-4
    assert (index == oindex)[fin].mean() >= 0.99
    if nrows == rows:   # Sections and instances are backtracked from the top row
        r = parity.compare_sections(ours["sections"], osec, rtol=1e-4)
        print(f"{_case_id(case)} {mode}: column-exact {r['exact']:.4f}, close {r['close']:.4f}, "
              f"{r['stixels_ours']} stixels")
        assert r["exact"] >= 0.99 and r["close"] >= 0.99, r
        if pairwise:
            assert parity.compare_instances(ours["inst"], oinst)["same_partition"]
    st.Finish()


EXHAUSTIVE = {"ISX_UNARY_EXHAUSTIVE": "1", "ISX_PAIRWISE_WALK": "0"}
PRUNING_SWITCHES = ("ISX_UNARY_EXHAUSTIVE", "ISX_PAIRWISE_WALK", "ISX_UNARY_PRUNE", "ISX_PAIRWISE_PRUNE")


def _pruned_and_exhaustive(pre, pairwise, disp, seg, road, monkeypatch):
    outs = {}
    for name, env in {"pruning": {}, "exhaustive": EXHAUSTIVE}.items():
        for k in PRUNING_SWITCHES:
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        st = None
        try:
            st, outs[name] = _compute(pre, pairwise, disp, seg, road)
        except api.StixelsError as e:     # e.g. > 199 stixels in a column: both kernels must agree on that too
            outs[name] = dict(error=str(e))
        if st is not None:
            st.Finish()
    return outs["pruning"], outs["exhaustive"]


def _assert_identical(a, b):
    assert ("error" in a) == ("error" in b), (a.get("error"), b.get("error"))
    if "error" in a:
        return
    assert np.array_equal(a["cost"].view(np.int32), b["cost"].view(np.int32))
    assert np.array_equal(a["index"], b["index"])
    assert np.array_equal(a["sections"].view(np.uint8), b["sections"].view(np.uint8))
    assert np.array_equal(a["inst"].view(np.uint8), b["inst"].view(np.uint8))


@pytest.mark.parametrize("dp_warps", ["4", "8"])
@pytest.mark.parametrize("mode", ["unary", "pairwise"])
@pytest.mark.parametrize("case", SHAPES, ids=_case_id)
def test_pruning_is_exact(case, mode, dp_warps, monkeypatch):
    """The pruning kernels (unary branch and bound, pairwise tile walk) return byte-identical (cost, argmin) tables,
    Sections and instance records to the exhaustive kernels; ISX_DP_WARPS also forces the walk for one frame."""
    rows, cols, step, invalid, median = case
    monkeypatch.setenv("ISX_DP_WARPS", dp_warps)
    pre = _preset(mode, rows, cols, step, invalid, median)
    fr = synth.make_frame(3 + rows % 11, rows=rows, cols=cols, column_step=step)
    a, b = _pruned_and_exhaustive(pre, mode == "pairwise", fr.disparity, fr.segmentation, fr.road, monkeypatch)
    _assert_identical(a, b)
    ev, tot = a["units"]
    assert b["units"][0] == tot and 0 < ev <= tot, (ev, tot)
    print(f"{_case_id(case)} {mode} dp{dp_warps}: {ev} of {tot} units evaluated")


def _fuzz_inputs(kind, rows, cols, step, rng):
    fr = synth.make_frame(int(rng.integers(0, 50)), rows=rows, cols=cols, column_step=step)
    disp, seg = fr.disparity.copy(), fr.segmentation.copy()
    used = (rows + 7) // 8
    if kind == "noise_costs":
        seg[:, :19, :used] = rng.integers(0, 60, size=seg[:, :19, :used].shape)
    elif kind == "sparse_costs":
        seg[:, :19, :used] = np.where(rng.random(seg[:, :19, :used].shape) < 0.03, 200, 0)
    elif kind == "zero_costs":
        seg[:, :19, :] = 0
    elif kind == "random_disparity":
        disp[:] = rng.uniform(0.0, 127.0, size=disp.shape).astype(np.float32)
    elif kind == "huge_offsets":
        seg[:, 19:21, :used] = rng.integers(-400, 400, size=seg[:, 19:21, :used].shape)
    return disp, seg, fr.road


FUZZ_WEIGHTS = [{}, dict(prior_weight=1.0, disparity_weight=1.0),
                dict(segmentation_weight=0.05, instance_weight=0.05, disparity_weight=0.5)]


@pytest.mark.parametrize("seed", range(8))
def test_pruning_fuzz_over_tall_heights(seed, monkeypatch):
    """Seeded heights in [1025, 2047], widths, input kinds and weights: pruning == exhaustive, byte for byte.  The
    data slack of the pruning bounds (kDataErrTall) is what this checks at heights the fixed shapes do not cover."""
    rng = np.random.default_rng(1000 + seed)
    rows = int(rng.integers(1025, 2048))
    cols = 8 * int(rng.integers(8, 33))
    mode = ("unary", "pairwise")[seed % 2]
    kind = ("synthetic", "noise_costs", "sparse_costs", "zero_costs", "random_disparity", "huge_offsets")[
        int(rng.integers(0, 6))]
    weights = FUZZ_WEIGHTS[int(rng.integers(0, len(FUZZ_WEIGHTS)))]
    if mode == "unary" and "instance_weight" in weights:
        weights = {}
    monkeypatch.setenv("ISX_DP_WARPS", "4")
    pre = _preset(mode, rows, cols, 8, 0.0, False, **weights)
    disp, seg, road = _fuzz_inputs(kind, rows, cols, 8, rng)
    a, b = _pruned_and_exhaustive(pre, mode == "pairwise", disp, seg, road, monkeypatch)
    print(f"seed {seed}: {rows}x{cols} {mode} {kind} {weights}: "
          f"{a['units'] if 'units' in a else a['error']}")
    _assert_identical(a, b)


# ---- entry points at 1208 rows ----
EP_ROWS, EP_COLS = 1208, 256


def _narrow(disp, seg, rows):
    used = (rows + 7) // 8
    d16 = np.rint(disp * 256.0).astype(np.uint16)
    s16 = np.ascontiguousarray(seg[..., :used]).astype(np.int16)
    wide_d = (d16.astype(np.float32) / np.float32(256.0)).astype(np.float32)
    wide_s = np.zeros_like(seg)
    wide_s[..., :used] = s16
    return d16, s16, wide_d, wide_s


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_entry_points_agree(mode, monkeypatch):
    """Batch == frame by frame; u16/int16 inputs == float inputs; device-resident == host; three batches in flight
    == synchronous calls; launches of 2 frames == the default chunks."""
    import torch
    rows, cols, n = EP_ROWS, EP_COLS, 5
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, 8)
    disp, seg, roads = synth.make_batch(n, start=60, rows=rows, cols=cols)
    roads[2] = dict(roads[2], vhor=roads[2]["vhor"] + 9)
    d16, s16, wide_d, wide_s = _narrow(disp, seg, rows)
    st = api.make_stixels(pre, max_batch=8)
    want, want_inst, want_offs = st.ComputeBatch(pairwise, wide_d, wide_s, roads)

    def same(sec, inst, offs):
        assert all(parity.same_used_sections(want[f], sec[f]) for f in range(n))
        assert np.array_equal(want_inst.view(np.uint8), inst.view(np.uint8)) and np.array_equal(want_offs, offs)

    for f in range(n):                                        # frame by frame
        st.SetDisparityImage(wide_d[f]); st.SetSegmentation(wide_s[f]); st.SetRoadParameters(**roads[f])
        data = st.Compute(pairwise)
        assert parity.same_used_sections(data.sections, want[f]), f
        assert np.array_equal(st.instance_records().view(np.uint8),
                              want_inst[want_offs[f]:want_offs[f + 1]].view(np.uint8)), f
    same(*st.ComputeBatchU16(pairwise, d16, 1.0 / 256.0, s16, roads))       # narrow inputs
    d_disp, d_seg = torch.from_numpy(wide_d).cuda(), torch.from_numpy(wide_s).cuda()
    st.ComputeBatchDevice(pairwise, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)   # device-resident inputs
    st.Synchronize()
    same(*st.FetchBatchResults(n))
    C_, S = st.GetRealCols(), st.GetMaxSections()
    outs = [np.zeros((n, C_, S), dtype=L.SECTION_DTYPE) for _ in range(3)]
    for i in range(3):                                        # three batches in flight, float and narrow
        if i == 1:
            st.SubmitBatchU16(pairwise, d16, 1.0 / 256.0, s16, roads, outs[i])
        else:
            st.SubmitBatch(pairwise, wide_d, wide_s, roads, outs[i])
    for _ in range(3):
        sec, inst, offs = st.WaitBatch()
        same(sec.copy(), inst, offs)
    st.Finish()
    monkeypatch.setenv("ISX_CHUNK", "2")                      # launch sizes
    st2 = api.make_stixels(pre, max_batch=8)
    monkeypatch.delenv("ISX_CHUNK")
    same(*st2.ComputeBatch(pairwise, wide_d, wide_s, roads))
    assert st2.chunk_frames() == 2
    st2.Finish()


def test_frame_pool_equals_one_context():
    rows, cols, n = EP_ROWS, EP_COLS, 5
    pre = _preset("pairwise", rows, cols, 8)
    disp, seg, roads = synth.make_batch(n, start=70, rows=rows, cols=cols)
    st = api.make_stixels(pre, max_batch=n)
    want, want_inst, want_offs = st.ComputeBatch(True, disp, seg, roads)
    st.Finish()
    pool = api.StixelsPool(api.StixelConfig(**pre), [0, 0], max_batch=2)
    sec, inst, offs = pool.ComputeBatch(True, disp, seg, roads)
    assert all(parity.same_used_sections(want[f], sec[f]) for f in range(n))
    assert np.array_equal(want_offs, offs) and np.array_equal(want_inst.view(np.uint8), inst.view(np.uint8))
    pool.close()


def test_frames_per_chunk_for_tall_frames():
    """Tall frames keep the 64 / 32 frames per launch while their chunk sets fit the footprint of 1024 x 2048 frames
    at width 4; 2047 x 1920 frames at width 4 do not, and get fewer frames per chunk."""
    st = api.make_stixels(_preset("pairwise", 1280, 1920, 8), max_batch=64)
    st.ComputeBatch(True, *synth.make_batch(1, start=0, rows=1280, cols=1920))
    assert st.chunk_frames() == 64
    st.Finish()
    st = api.make_stixels(_preset("pairwise", 2047, 1920, 4), max_batch=64)
    st.ComputeBatch(True, *synth.make_batch(1, start=0, rows=2047, cols=1920, column_step=4))
    assert 1 <= st.chunk_frames() < 64
    st.Finish()


# ---- limits ----
def test_row_limit():
    fr = synth.make_frame(4, rows=2047, cols=128)
    st = api.make_stixels(_preset("pairwise", 2047, 128, 8), max_batch=1)
    st.SetDisparityImage(fr.disparity); st.SetSegmentation(fr.segmentation); st.SetRoadParameters(**fr.road)
    assert parity.column_lengths(st.Compute(True).sections).min() >= 1
    st.Finish()
    st = api.Stixels()
    st.SetConfig(api.StixelConfig(**_preset("pairwise", 2048, 128, 8)))
    with pytest.raises(api.StixelsError, match="isx error -5"):   # ISX_ERR_UNSUPPORTED
        st.Initialize(1)


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_values_above_the_tall_guards_flag_their_columns(mode, monkeypatch):
    """Class values above 2^19 and squared offsets above 2^18 pass the guards of frames up to 1024 rows but could
    wrap the int32 sums of a 2047-row column: such columns are walked exhaustively, and the result still equals the
    exhaustive kernels."""
    rows, cols = 2047, 16                  # two columns, both flagged below
    pairwise = mode == "pairwise"
    monkeypatch.setenv("ISX_DP_WARPS", "4")
    pre = _preset(mode, rows, cols, 8)
    fr = synth.make_frame(9, rows=rows, cols=cols)
    seg = fr.segmentation.copy()
    seg[0, 5, 40] = (1 << 19) + 1          # a class value
    seg[1, 20, 100] = 600                  # an x offset: 600^2 > 2^18
    st, clean = _compute(pre, pairwise, fr.disparity, fr.segmentation, fr.road)
    st.Finish()
    a, b = _pruned_and_exhaustive(pre, pairwise, fr.disparity, seg, fr.road, monkeypatch)
    _assert_identical(a, b)
    assert clean["units"][0] < clean["units"][1]       # the clean columns are pruned
    assert a["units"][0] == a["units"][1]              # the flagged ones are walked completely


def test_offsets_beyond_the_exact_float_range_raise_the_frame_error():
    rows, cols, n = 1208, 128, 3
    pre = _preset("pairwise", rows, cols, 8)
    disp, seg, roads = synth.make_batch(n, start=5, rows=rows, cols=cols)
    st = api.make_stixels(pre, max_batch=4)
    want, _, _ = st.ComputeBatch(True, disp, seg, roads)
    bad = seg.copy()
    bad[1, :, 20, :rows // 8] = 20000       # sum of the instance means of a column >= 2^24
    out = np.zeros_like(want)
    with pytest.raises(api.StixelsError, match="frame 1"):
        st.ComputeBatch(True, disp, bad, roads, sections_out=out)
    assert parity.same_used_sections(want[0], out[0]) and parity.same_used_sections(want[2], out[2])
    st.Finish()


# ---- the steps either side ----
@pytest.mark.parametrize("rows,cols", [(1208, 512), (1280, 384)])
def test_device_ingest_matches_restatement(rows, cols):
    import torch
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_ingest_golden
    hs, ws, n = rows // 8, cols // 8, 2         # CNN outputs of 151 / 160 rows
    cnn = np.stack([make_ingest_golden.make_input(30 + i, hs, ws) for i in range(n)])
    cnn[:, :19] = np.minimum(cnn[:, :19], 30.0)
    cnn[:, 19:] = np.clip(np.rint(cnn[:, 19:]), -50, 50) / 8.0
    want = np.stack([ingest_cpu.flip_and_pad(cnn[i], 8) for i in range(n)])
    st = api.make_stixels(_preset("pairwise", rows, cols, 8), max_batch=2)
    assert want[0].size == st.segmentation_elems()
    d_cnn = torch.from_numpy(cnn).cuda()
    d_seg = torch.full(want.shape, -7, dtype=torch.int32, device="cuda")
    st.FlipAndPadBatchDevice(n, d_cnn.data_ptr(), hs, ws, d_seg.data_ptr())
    st.Synchronize()
    assert np.array_equal(d_seg.cpu().numpy(), want)
    st.Finish()


def test_road_estimation_matches_restatement():
    import torch
    rows, cols, n = 1208, 512, 3
    cam = dict(camera_center_y=604.0, baseline=0.209313, focal=2262.52)
    disp = np.stack([synth.make_frame(40 + i, rows=rows, cols=cols).disparity for i in range(n)])
    re = api.RoadEstimation()
    re.Initialize(cam["camera_center_y"], cam["baseline"], cam["focal"], rows, cols, 128, 0.2, max_batch=4)
    batch = re.ComputeBatchDevice(n, torch.from_numpy(disp).cuda().data_ptr())
    n_ok = 0
    for i in range(n):
        est, inter = road_cpu.estimate(disp[i], 128, *cam.values())
        assert batch[i]["ok"] == est["ok"]
        ok = re.Compute(disp[i])
        assert ok == est["ok"]
        assert np.array_equal(re.read_tensor(0), inter["vdisp"])
        assert np.array_equal(re.read_tensor(1), inter["binary"])
        assert np.array_equal(re.read_tensor(2), inter["accum"])
        if est["ok"]:
            n_ok += 1
            assert batch[i]["vhor"] == est["horizon_point"] == re.GetHorizonPoint()
            a = np.array([batch[i][k] for k in ("camera_tilt", "camera_height", "alpha_ground", "rho", "theta")],
                         np.float32)
            b = np.array([est[k] for k in ("pitch", "camera_height", "slope", "rho", "theta")], np.float32)
            assert np.array_equal(a.view(np.int32), b.view(np.int32)), (a, b)
    assert n_ok > 0
    re.Finish()


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_device_rasteriser_matches_restatement(mode):
    import torch
    rows, cols, n = 1208, 256, 2
    st = api.make_stixels(_preset(mode, rows, cols, 8), max_batch=2)
    sec, inst, offs = st.ComputeBatch(mode == "pairwise", *synth.make_batch(n, start=90, rows=rows, cols=cols))
    lab = torch.full((n, rows, cols), 255, dtype=torch.uint8, device="cuda")
    ins = torch.full((n, rows, cols), -5, dtype=torch.int32, device="cuda")
    dsp = torch.full((n, rows, cols), -1.0, dtype=torch.float32, device="cuda")
    st.RasterizeBatchDevice(0, n, lab.data_ptr(), ins.data_ptr(), dsp.data_ptr())
    st.Synchronize()
    for f in range(n):
        m = {(int(x["column"]), int(x["index"])): int(x["label"]) for x in inst[offs[f]:offs[f + 1]]}
        want = raster_cpu.draw(sec[f], m, rows, cols)
        assert np.array_equal(lab[f].cpu().numpy(), want[0])
        assert np.array_equal(ins[f].cpu().numpy(), want[1])
        assert np.array_equal(dsp[f].cpu().numpy().view(np.int32), want[2].view(np.int32))
    st.Finish()


def test_runner_admits_tall_frames_with_the_opt_in(tmp_path):
    """apps/cityscapes_runner refuses >= 1024 rows like the reference unless ISX_ALLOW_1024=1; then a directory of
    1208-row frames gives the same .stixels as the C ABI on the same inputs."""
    cv2 = pytest.importorskip("cv2")
    subprocess.run(["make", "-C", os.path.join(ROOT, "apps")], check=True, capture_output=True, text=True)
    app = os.path.join(ROOT, "apps", "cityscapes_runner")
    rows, cols = 1208, 512
    for d in ("disparities", "camera", "probs", "stixels"):
        (tmp_path / d).mkdir()
    cam = {"extrinsic": {"baseline": 0.209313}, "intrinsic": {"fx": 2262.52, "fy": 2262.52, "u0": 256.0, "v0": 604.0}}
    frames = {}
    for i in range(2):
        fr = synth.make_frame(70 + i, rows=rows, cols=cols)
        base = f"tall_{i:06d}_000019"
        q = np.clip(np.rint(fr.disparity * 256.0), 0, 65535).astype(np.uint16)
        cv2.imwrite(str(tmp_path / "disparities" / f"{base}_disparity.png"), q)
        (tmp_path / "camera" / f"{base}_camera.json").write_text(json.dumps(cam))
        np.save(tmp_path / "probs" / f"{base}_probs.npy", fr.segmentation)
        frames[base] = (q.astype(np.float32) / 256.0, fr.segmentation)
    pre = synth.preset("pairwise", rows, cols, 8)
    args = [app, str(tmp_path), "128", repr(pre["segmentation_weight"]), repr(pre["instance_weight"]),
            repr(pre["disparity_weight"]), "1", "8", repr(pre["eps"]), str(pre["min_pts"]), str(pre["size_filter"])]
    env = {k: v for k, v in os.environ.items() if k != "ISX_ALLOW_1024"}
    p = subprocess.run(args, capture_output=True, text=True, env=env)   # each frame is refused and skipped
    assert p.stderr.count("less than 1024") == 2 and not os.listdir(tmp_path / "stixels")
    p = subprocess.run(args, capture_output=True, text=True, env=dict(env, ISX_ALLOW_1024="1"))
    assert p.returncode == 0, p.stderr[-2000:] + p.stdout[-2000:]
    st = api.Stixels()
    st.SetConfig(api.StixelConfig(
        rows=rows, cols=cols, max_dis=128, column_step=8, invalid_disparity=0.0, n_semantic_classes=19,
        n_offset_channels=2, prior_weight=1.0, segmentation_weight=pre["segmentation_weight"],
        instance_weight=pre["instance_weight"], disparity_weight=pre["disparity_weight"], eps=pre["eps"],
        min_pts=pre["min_pts"], size_filter=pre["size_filter"], baseline=0.209313, focal=2262.52,
        camera_center_y=604.0))
    st.Initialize()
    road = api.RoadEstimation()
    road.Initialize(604.0, 0.209313, 2262.52, rows, cols, 128)
    for base, (disp, seg) in frames.items():
        assert road.Compute(disp)
        st.SetDisparityImage(disp)
        st.SetSegmentation(seg)
        st.SetRoadParameters(road.GetHorizonPoint(), road.GetPitch(), road.GetCameraHeight(), road.GetSlope())
        data = st.Compute(True)
        inst = st.GetInstanceStixels()
        got = [[item.split(",") for item in line.split(";") if item]
               for line in open(tmp_path / "stixels" / f"{base}.stixels").read().splitlines()
               if not line.startswith("groundplane")]
        assert len(got) == cols // 8
        for c, items in enumerate(got):
            for j, f in enumerate(items):
                s = data.sections[c, j]
                assert (int(f[0]), int(f[1]), int(f[2]), int(f[4])) == (s["type"], s["vB"], s["vT"], s["semantic_class"])
                assert np.isclose(float(f[3]), s["disparity"], rtol=1e-5) and np.isclose(float(f[5]), s["cost"], rtol=1e-5)
                assert (len(f) == 9) == ((c, j) in inst)
            assert data.sections[c, len(items)]["type"] == -1
    st.Finish()
    road.Finish()
