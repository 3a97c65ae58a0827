"""Parity of the CUDA product (through the C ABI) on a B200:
  * bit-for-bit against what the reference CUDA build computed on identical seeded inputs (stored under
    tests/golden/, see tools/make_reference_build_golden.py),
  * against the committed golden vectors (outputs of the reference itself),
  * against the CPU oracle (column-exact, floats within 1e-4 relative),
  * at BASELINE.json's full size through size-independent properties.
Bar: stixel boundaries / types / classes / instance partitions identical; DP costs and stixel
disparities bit-identical to the reference build (tolerance stated where the CPU oracle is the
checker: 1e-4 relative, the north-star tolerance)."""
import functools
import json
import os

import numpy as np
import pytest

import parity
from instance_stixels_b200 import _lib as L, api, synth
from oracle import cpubind, refbind

pytestmark = pytest.mark.gpu

CASES = [  # name, mode, rows, cols, step, frame, invalid_disparity, median
    ("small_unary", "unary", 256, 512, 8, 0, 0.0, False),
    ("small_pairwise", "pairwise", 256, 512, 8, 1, 0.0, False),
    ("small_pairwise_w4", "pairwise", 256, 512, 4, 2, 0.0, False),
    ("ragged_pairwise", "pairwise", 200, 328, 8, 3, 0.0, False),   # rows % 32 != 0, 41 columns
    ("ragged_unary_noinvalid", "unary", 200, 328, 8, 4, -1.0, False),
    ("median_pairwise", "pairwise", 128, 256, 8, 5, 0.0, True),
    ("short_rows", "pairwise", 136, 64, 8, 6, 0.0, False),         # four full 32-row tiles + a partial one
    ("crop_reference_size", "pairwise", 784, 1792, 8, 0, 0.0, False),  # the reference's own test size
]
# host tables and stage tensors the reference build computes bit for bit like the product
TABLES = ("T_OBJ_COST_LUT", "T_OBJECT_DISPARITY_RANGE", "T_GROUND_TABLES", "T_JOINED_DISPARITY", "T_OBJECT_LUT")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _preset(mode, rows, cols, step, invalid, median):
    pre = synth.preset(mode, rows, cols, step)
    pre["invalid_disparity"] = invalid
    pre["median_join"] = median
    return pre


def _run_ours(pre, pairwise, fr, max_batch=1):
    st = api.make_stixels(pre, max_batch=max_batch)
    st.SetDisparityImage(fr.disparity)
    st.SetSegmentation(fr.segmentation)
    st.SetRoadParameters(**fr.road)
    data = st.Compute(pairwise)
    inst = st.instance_records()
    return st, data, inst


@pytest.fixture(params=["4", "8"], ids=["dp4warps", "dp8warps"])
def dp_warps(request, monkeypatch):
    """Both DP kernel variants (throughput: 4 warps per column, latency: 8) on every case."""
    monkeypatch.setenv("ISX_DP_WARPS", request.param)
    return request.param


@pytest.fixture(params=["0", "1"], ids=["chunkmajor", "tilewalk"])
def pairwise_walk(request, monkeypatch):
    """Both pairwise DP kernels: chunk-major exhaustive, and the tile-major walk with exact pruning."""
    monkeypatch.setenv("ISX_PAIRWISE_WALK", request.param)
    return request.param


@functools.lru_cache(maxsize=None)
def _reference_build_digests():
    with open(os.path.join(GOLDEN, "reference_build", "digests.json")) as f:
        return json.load(f)


def _reference_build_results(name, frame, realcols):
    """[C][200] Sections and instance records of the reference CUDA build for a case: its own output where
    tests/golden/ holds one, otherwise the stored copy under tests/golden/reference_build/."""
    path = os.path.join(GOLDEN, f"{name}_f{frame}.npz")
    if not os.path.exists(path):
        path = os.path.join(GOLDEN, "reference_build", f"{name}_f{frame}.npz")
    z = np.load(path)
    sections = np.zeros((realcols, 200), dtype=L.SECTION_DTYPE)
    sections["type"] = -1
    sections[:, :z["sections"].shape[1]] = z["sections"]
    return sections, z["instances"]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_bit_exact_against_reference_cuda_build(case, dp_warps, pairwise_walk):
    name, mode, rows, cols, step, frame, invalid, median = case
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, step, invalid, median)
    fr = synth.make_frame(frame, rows=rows, cols=cols, column_step=step)
    want = _reference_build_digests()["cases"][name]
    rsec, rinst = _reference_build_results(name, frame, cols // step)
    st, data, inst = _run_ours(pre, pairwise, fr)
    # host tables and stage tensors (integer/byte/index work and these float tables: bit-exact)
    for t in TABLES:
        assert parity.array_digest(st.read_tensor(getattr(L, t)).view(np.int32)) == want["tables"][t], t
    r = parity.compare_sections(data.sections, rsec)
    assert r["exact"] == 1.0, r          # boundaries, types, classes on every column
    assert r["close"] == 1.0 and r["bitwise"] >= 0.995, r   # costs / disparities / instance means
    ri = parity.compare_instances(inst, rinst)
    assert ri["same_keys"] and ri["same_partition"], ri   # instance ids up to label permutation
    for n, _ in L.FrameMeta._fields_:
        assert getattr(data, n) == want["meta"][n], n
    st.Finish()


UNARY_WALKS = {  # how the unary DP visits the chunks of a tile
    "pruned": {},                                   # from the diagonal downwards until no chunk below can win
    "all_chunks": {"ISX_UNARY_PRUNE": "0"},         # the same walk without the bound test
    "exhaustive": {"ISX_UNARY_EXHAUSTIVE": "1"},    # chunk-major over every unit (the pairwise kernel's schedule)
}


@pytest.mark.parametrize("shape", [(256, 512, 8, -1.0), (200, 328, 8, 0.0), (784, 1792, 8, 0.0), (1024, 2048, 8, 0.0),
                                   (1024, 2048, 4, 0.0), (1024, 640, 8, -1.0)],
                         ids=lambda s: f"{s[0]}x{s[1]}w{s[2]}inv{s[3]:g}")
def test_unary_branch_and_bound_is_exact(shape, dp_warps, monkeypatch):
    """The pruned unary DP returns byte-identical Sections and instance records to the exhaustive scan (and to
    the reference CUDA build), and at full size it really skips most of the (tile, chunk) units."""
    rows, cols, step, invalid = shape
    pre = _preset("unary", rows, cols, step, invalid, False)
    frames = [synth.make_frame(f, rows=rows, cols=cols, column_step=step) for f in (0, 5)]
    results, work = {}, {}
    for walk, env in UNARY_WALKS.items():
        for k in ("ISX_UNARY_PRUNE", "ISX_UNARY_EXHAUSTIVE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        st = api.make_stixels(pre, max_batch=2)
        out = []
        for fr in frames:
            st.SetDisparityImage(fr.disparity)
            st.SetSegmentation(fr.segmentation)
            st.SetRoadParameters(**fr.road)
            data = st.Compute(False)
            out.append((data.sections.copy(), st.instance_records().copy(),
                        st.read_tensor(L.T_COST_TABLE).copy(), st.read_tensor(L.T_INDEX_TABLE).copy()))
        sec_b, inst_b, _ = st.ComputeBatch(False, np.stack([f.disparity for f in frames]),
                                           np.stack([f.segmentation for f in frames]), [f.road for f in frames])
        for i in range(len(frames)):
            assert parity.same_used_sections(sec_b[i], out[i][0])
        results[walk], work[walk] = out, st.dp_units()
        st.Finish()
    for walk in ("all_chunks", "exhaustive"):
        for (s0, i0, c0, x0), (s1, i1, c1, x1) in zip(results["pruned"], results[walk]):
            assert np.array_equal(s0.view(np.uint8), s1.view(np.uint8)), walk
            assert np.array_equal(i0.view(np.uint8), i1.view(np.uint8)), walk
            # the whole (cost, argmin) tables, not just the rows on the optimal path
            assert np.array_equal(c0.view(np.int32), c1.view(np.int32)), walk
            assert np.array_equal(x0, x1), walk
    ev, tot = work["pruned"]
    assert work["all_chunks"][0] == work["all_chunks"][1] == tot and work["exhaustive"][0] == tot
    assert 0 < ev <= tot
    if rows == 1024 and cols == 2048:
        assert ev < 0.5 * tot, (ev, tot)     # the synthetic Cityscapes-shaped frames: most units cannot win
    if refbind.available() and rows * cols <= 784 * 1792:
        ref = refbind.RefStixels(api.StixelConfig(**pre))
        for fr, (sec, inst, _, _) in zip(frames, results["pruned"]):
            rsec, rinst, _ = ref.compute(False, fr.disparity, fr.segmentation, fr.road)
            r = parity.compare_sections(sec, rsec)
            assert r["exact"] == 1.0 and r["close"] == 1.0 and r["bitwise"] >= 0.995, r
            assert parity.compare_instances(inst, rinst)["same_partition"]
        ref.close()


PAIRWISE_WALKS = {
    "tilewalk": {"ISX_PAIRWISE_WALK": "1"},                                   # tile-major, pruned
    "tilewalk_all": {"ISX_PAIRWISE_WALK": "1", "ISX_PAIRWISE_PRUNE": "0"},    # the same walk without the bound test
    "tilewalk_cta": {"ISX_PAIRWISE_WALK": "1", "ISX_WALK_WARPS": "4"},        # a 4-warp CTA per column instead of a warp
    "chunkmajor": {"ISX_PAIRWISE_WALK": "0"},                                 # exhaustive
}


@pytest.mark.parametrize("shape", [(256, 512, 8, -1.0), (200, 328, 8, 0.0), (784, 1792, 8, 0.0), (1024, 2048, 8, 0.0),
                                   (1024, 1024, 4, 0.0)],
                         ids=lambda s: f"{s[0]}x{s[1]}w{s[2]}inv{s[3]:g}")
def test_pairwise_tile_walk_is_exact(shape, dp_warps, monkeypatch):
    """The tile-major pairwise DP (with and without pruning) returns byte-identical Sections, instance records and
    full (cost, argmin) tables to the chunk-major exhaustive kernel."""
    rows, cols, step, invalid = shape
    pre = _preset("pairwise", rows, cols, step, invalid, False)
    frames = [synth.make_frame(f, rows=rows, cols=cols, column_step=step) for f in (1, 6)]
    results, work = {}, {}
    for walk, env in PAIRWISE_WALKS.items():
        for k in ("ISX_PAIRWISE_WALK", "ISX_PAIRWISE_PRUNE", "ISX_WALK_WARPS"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        st = api.make_stixels(pre, max_batch=2)
        out = []
        for fr in frames:
            st.SetDisparityImage(fr.disparity)
            st.SetSegmentation(fr.segmentation)
            st.SetRoadParameters(**fr.road)
            data = st.Compute(True)
            out.append((data.sections.copy(), st.instance_records().copy(),
                        st.read_tensor(L.T_COST_TABLE).copy(), st.read_tensor(L.T_INDEX_TABLE).copy()))
        sec_b, _, _ = st.ComputeBatch(True, np.stack([f.disparity for f in frames]),
                                      np.stack([f.segmentation for f in frames]), [f.road for f in frames])
        for i in range(len(frames)):
            assert parity.same_used_sections(sec_b[i], out[i][0])
        results[walk], work[walk] = out, st.dp_units()
        st.Finish()
    for walk in ("tilewalk", "tilewalk_all", "tilewalk_cta"):
        for (s0, i0, c0, x0), (s1, i1, c1, x1) in zip(results["chunkmajor"], results[walk]):
            assert np.array_equal(c0.view(np.int32), c1.view(np.int32)), walk
            assert np.array_equal(x0, x1), walk
            assert np.array_equal(s0.view(np.uint8), s1.view(np.uint8)), walk
            assert np.array_equal(i0.view(np.uint8), i1.view(np.uint8)), walk
    ev, tot = work["tilewalk"]
    assert work["tilewalk_all"][0] == tot and work["chunkmajor"][0] == tot and 0 < ev <= tot
    print(f"pairwise tile walk {rows}x{cols} w{step}: {ev} of {tot} units evaluated")


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_negative_class_values_disable_the_pruning_of_their_columns(mode, dp_warps, monkeypatch):
    """The bounds of the pruning kernels need non-negative class values; a column with a negative one (the
    reference just sums whatever it is given) is walked exhaustively -- results stay identical to the exhaustive
    kernels, and the evaluated units show that exactly those columns lost their pruning."""
    rows, cols = 512, 512
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, 8, 0.0, False)
    fr = synth.make_frame(2, rows=rows, cols=cols)
    seg = fr.segmentation.copy()
    bad_cols = [3, 17, 40]
    for c in bad_cols:
        seg[c, 5, 7] = -3          # one negative value of class 5 in each of three columns
    outs, units = {}, {}
    for name, env in {"pruning": {}, "exhaustive": {"ISX_UNARY_EXHAUSTIVE": "1", "ISX_PAIRWISE_WALK": "0"}}.items():
        for k in ("ISX_UNARY_EXHAUSTIVE", "ISX_PAIRWISE_WALK"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        res = []
        for s_ in (fr.segmentation, seg):
            st = api.make_stixels(pre, max_batch=1)
            st.SetDisparityImage(fr.disparity)
            st.SetSegmentation(s_)
            st.SetRoadParameters(**fr.road)
            data = st.Compute(pairwise)
            res.append((data.sections.copy(), st.read_tensor(L.T_COST_TABLE).copy(),
                        st.read_tensor(L.T_INDEX_TABLE).copy(), st.dp_units()))
            st.Finish()
        outs[name] = res
    for (s0, c0, x0, _), (s1, c1, x1, _) in zip(outs["pruning"], outs["exhaustive"]):
        assert np.array_equal(c0.view(np.int32), c1.view(np.int32)) and np.array_equal(x0, x1)
        assert np.array_equal(s0.view(np.uint8), s1.view(np.uint8))
    (ev_clean, tot), (ev_bad, _) = outs["pruning"][0][3], outs["pruning"][1][3]
    per_col = tot // (cols // 8)
    assert ev_clean < tot and ev_bad > ev_clean
    # the three flagged columns are evaluated completely, the others as before (+- what the changed values prune)
    assert ev_bad >= 3 * per_col


def _stress_inputs(kind, rows, cols, step, seed):
    """Inputs far from the synthetic street scenes, to stress the bounds of the pruning kernels."""
    rng = np.random.default_rng(seed)
    fr = synth.make_frame(seed % 7, rows=rows, cols=cols, column_step=step)
    disp, seg = fr.disparity.copy(), fr.segmentation.copy()
    used = (rows + 7) // 8
    if kind == "zero_costs":            # a CNN that is certain everywhere: every class sum is 0, only priors decide
        seg[:, :19, :] = 0
    elif kind == "noise_costs":         # no structure at all
        seg[:, :19, :used] = rng.integers(0, 60, size=seg[:, :19, :used].shape)
    elif kind == "sparse_costs":        # mostly zeros, a few expensive rows
        seg[:, :19, :used] = np.where(rng.random(seg[:, :19, :used].shape) < 0.03, 200, 0)
    elif kind == "all_invalid":         # no disparity measurement at all
        disp[:] = 0.0
    elif kind == "random_disparity":
        disp[:] = rng.uniform(0.0, 127.0, size=disp.shape).astype(np.float32)
    elif kind == "huge_offsets":        # instance offsets at the edge of the exact-float range
        seg[:, 19:21, :used] = rng.integers(-400, 400, size=seg[:, 19:21, :used].shape)
    return disp, seg, fr.road


@pytest.mark.parametrize("kind", ["zero_costs", "noise_costs", "sparse_costs", "all_invalid", "random_disparity",
                                  "huge_offsets"])
@pytest.mark.parametrize("mode,weights", [
    ("unary", {}), ("pairwise", {}),
    ("unary", dict(prior_weight=1.0, disparity_weight=1.0)),                 # the prior no longer dominates
    ("pairwise", dict(segmentation_weight=0.05, instance_weight=0.05, disparity_weight=0.5)),
])
def test_pruning_kernels_are_exact_on_unusual_inputs(kind, mode, weights, monkeypatch):
    rows, cols, step = 512, 256, 8
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, step, 0.0, False)
    pre.update(weights)
    disp, seg, road = _stress_inputs(kind, rows, cols, step, seed=len(kind) + len(weights))
    monkeypatch.setenv("ISX_DP_WARPS", "4")     # forces the walk variants even for one frame
    outs = {}
    for name, env in {"pruning": {}, "exhaustive": {"ISX_UNARY_EXHAUSTIVE": "1", "ISX_PAIRWISE_WALK": "0"}}.items():
        for k in ("ISX_UNARY_EXHAUSTIVE", "ISX_PAIRWISE_WALK"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        st = api.make_stixels(pre, max_batch=1)
        st.SetDisparityImage(disp)
        st.SetSegmentation(seg)
        st.SetRoadParameters(**road)
        try:
            data = st.Compute(pairwise)
        except api.StixelsError as e:       # e.g. > 199 stixels in a column: both kernels must agree on that too
            outs[name] = ("error", str(e))
            st.Finish()
            continue
        outs[name] = (data.sections.copy(), st.read_tensor(L.T_COST_TABLE).copy(),
                      st.read_tensor(L.T_INDEX_TABLE).copy())
        st.Finish()
    a, b = outs["pruning"], outs["exhaustive"]
    a_err, b_err = isinstance(a[0], str), isinstance(b[0], str)
    assert a_err == b_err, (a[1] if a_err else "ok", b[1] if b_err else "ok")
    if not a_err:
        assert np.array_equal(a[1].view(np.int32), b[1].view(np.int32))
        assert np.array_equal(a[2], b[2])
        assert np.array_equal(a[0].view(np.uint8), b[0].view(np.uint8))


def test_against_golden_vectors(golden_files):
    for path in golden_files:
        z = np.load(path)
        mode = str(z["mode"])
        rows, cols, step, frame = int(z["rows"]), int(z["cols"]), int(z["step"]), int(z["frame"])
        pre = _preset(mode, rows, cols, step, float(z["invalid"]), False)
        fr = synth.make_frame(frame, rows=rows, cols=cols, column_step=step)
        st, data, inst = _run_ours(pre, mode == "pairwise", fr)
        ref = np.zeros((cols // step, 200), dtype=L.SECTION_DTYPE)
        ref["type"] = -1
        ref[:, :z["sections"].shape[1]] = z["sections"]
        r = parity.compare_sections(data.sections, ref)
        assert r["exact"] == 1.0 and r["bitwise"] == 1.0, (path, r)
        assert parity.compare_instances(inst, z["instances"])["same_partition"], path
        st.Finish()


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_against_cpu_oracle_with_tables(mode):
    rows, cols = 160, 256
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, 8, 0.0, False)
    fr = synth.make_frame(11, rows=rows, cols=cols)
    st, data, inst = _run_ours(pre, pairwise, fr)
    osec, oinst, ex = cpubind.compute_frame(cpubind.default_config(**pre), pairwise, fr.disparity,
                                            fr.segmentation, fr.road, tables=True)
    r = parity.compare_sections(data.sections, osec, rtol=1e-4)
    assert r["exact"] >= 0.99 and r["close"] >= 0.99, r
    C_ = cols // 8
    cost = st.read_tensor(L.T_COST_TABLE).reshape(C_, rows, 3)
    index = st.read_tensor(L.T_INDEX_TABLE).reshape(C_, rows, 3)
    fin = np.isfinite(ex["cost_table"])
    assert np.array_equal(fin, np.isfinite(cost))
    rel = np.abs(cost[fin] - ex["cost_table"][fin]) / np.maximum(np.abs(ex["cost_table"][fin]), 1e-6)
    assert np.quantile(rel, 0.999) <= 1e-4    # DP costs: 1e-4 relative (north star)
    same = (index == ex["index_table"])[fin]
    assert same.mean() >= 0.99                # back-pointers (argmin vB and predecessor type)
    j = st.read_tensor(L.T_JOINED_DISPARITY).reshape(C_, rows)
    assert np.allclose(j, ex["joined"], rtol=1e-6, atol=0)
    lut = st.read_tensor(L.T_OBJECT_LUT).reshape(C_, -1, rows + 1)
    assert np.array_equal(lut.view(np.int32), ex["object_lut"].view(np.int32))  # pure fp32 adds: bit-exact
    st.Finish()


def test_batch_equals_single_frame_and_is_deterministic():
    rows, cols, n = 256, 512, 5
    pre = _preset("pairwise", rows, cols, 8, 0.0, False)
    disp, seg, roads = synth.make_batch(n, start=20, rows=rows, cols=cols)
    roads[2] = dict(roads[2], vhor=roads[2]["vhor"] + 9, camera_tilt=0.01)   # per-frame road parameters
    st = api.make_stixels(pre, max_batch=8)
    sec1, inst1, offs1 = st.ComputeBatch(True, disp, seg, roads)
    sec2, inst2, offs2 = st.ComputeBatch(True, disp, seg, roads)
    assert np.array_equal(sec1.view(np.uint8), sec2.view(np.uint8))
    assert np.array_equal(inst1.view(np.uint8), inst2.view(np.uint8)) and np.array_equal(offs1, offs2)
    for f in range(n):
        st.SetDisparityImage(disp[f])
        st.SetSegmentation(seg[f])
        st.SetRoadParameters(**roads[f])
        data = st.Compute(True)
        assert parity.same_used_sections(data.sections, sec1[f]), f
        assert np.array_equal(st.instance_records().view(np.uint8), inst1[offs1[f]:offs1[f + 1]].view(np.uint8))
    # the padding of the segmentation tensor (entries >= rows/8 of every channel row) is never read: the host
    # batch path does not even copy it
    seg_junk = seg.copy()
    seg_junk[..., (rows + 7) // 8:] = np.random.default_rng(3).integers(-1000, 1000, seg_junk[..., (rows + 7) // 8:].shape)
    sec4, inst4, offs4 = st.ComputeBatch(True, disp, seg_junk, roads)
    assert all(parity.same_used_sections(sec1[f], sec4[f]) for f in range(n))   # (entries behind a terminator are stale)
    assert np.array_equal(inst1.view(np.uint8), inst4.view(np.uint8)) and np.array_equal(offs1, offs4)
    st.SetDisparityImage(disp[1]); st.SetSegmentation(seg_junk[1]); st.SetRoadParameters(**roads[1])
    assert parity.same_used_sections(st.Compute(True).sections, sec1[1])
    st.Finish()
    # chunked execution (ISX_CHUNK) does not change results
    import os
    os.environ["ISX_CHUNK"] = "2"
    try:
        st2 = api.make_stixels(pre, max_batch=8)
        sec3, inst3, offs3 = st2.ComputeBatch(True, disp, seg, roads)
        st2.Finish()
    finally:
        del os.environ["ISX_CHUNK"]
    assert all(parity.same_used_sections(sec1[f], sec3[f]) for f in range(n)) and np.array_equal(offs1, offs3)
    assert np.array_equal(inst1.view(np.uint8), inst3.view(np.uint8))


def test_device_resident_entry_point_matches_host_entry_point():
    import torch
    rows, cols, n = 128, 256, 3
    pre = _preset("unary", rows, cols, 8, 0.0, False)
    disp, seg, roads = synth.make_batch(n, start=3, rows=rows, cols=cols)
    st = api.make_stixels(pre, max_batch=4)
    sec_h, inst_h, offs_h = st.ComputeBatch(False, disp, seg, roads)
    d_disp, d_seg = torch.from_numpy(disp).cuda(), torch.from_numpy(seg).cuda()
    before = seg.copy()
    st.ComputeBatchDevice(False, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    st.Synchronize()
    sec_d, inst_d, offs_d = st.FetchBatchResults(n)
    assert all(parity.same_used_sections(sec_h[f], sec_d[f]) for f in range(n))
    assert np.array_equal(inst_h.view(np.uint8), inst_d.view(np.uint8))
    # unlike the reference (StixelsKernels.cu:411-416, 462-469) the borrowed tensor is not modified
    assert np.array_equal(d_seg.cpu().numpy(), before)
    # back-to-back device batches (the emission stream is joined lazily): the results fetched afterwards are
    # those of the LAST batch, whichever entry point touches them first (fetch / flush + own stream work)
    disp2, seg2, roads2 = synth.make_batch(n, start=11, rows=rows, cols=cols)
    sec_h2, inst_h2, _ = st.ComputeBatch(False, disp2, seg2, roads2)
    d_disp2, d_seg2 = torch.from_numpy(disp2).cuda(), torch.from_numpy(seg2).cuda()
    for _ in range(3):
        st.ComputeBatchDevice(False, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
        st.ComputeBatchDevice(False, n, d_disp2.data_ptr(), d_seg2.data_ptr(), roads2)
    sec_d2, inst_d2, _ = st.FetchBatchResults(n)
    assert all(parity.same_used_sections(sec_h2[f], sec_d2[f]) for f in range(n))
    assert np.array_equal(inst_h2.view(np.uint8), inst_d2.view(np.uint8))
    st.ComputeBatchDevice(False, n, d_disp.data_ptr(), d_seg.data_ptr(), roads)
    st.Flush()
    stream = torch.cuda.ExternalStream(st.stream())
    with torch.cuda.stream(stream):
        marker = torch.zeros(1, device="cuda") + 1   # caller's own work on isx_stream(), ordered after the results
    stream.synchronize()
    sec_d3, inst_d3, _ = st.FetchBatchResults(n)
    assert all(parity.same_used_sections(sec_h[f], sec_d3[f]) for f in range(n)) and float(marker.item()) == 1.0
    assert np.array_equal(inst_h.view(np.uint8), inst_d3.view(np.uint8))
    st.Finish()


def test_submit_wait_pipeline_equals_synchronous_batches():
    """isx_submit_batch_host / isx_wait_batch_host: two and three batches in flight, results in submission order and
    identical to the synchronous entry point; misuse is refused."""
    rows, cols, n = 128, 256, 5
    pre = _preset("pairwise", rows, cols, 8, 0.0, False)
    import os
    os.environ["ISX_CHUNK"] = "2"      # several chunks per batch, short first chunk logic aside
    try:
        st = api.make_stixels(pre, max_batch=8)
    finally:
        del os.environ["ISX_CHUNK"]
    batches = [synth.make_batch(n, start=s0, rows=rows, cols=cols) for s0 in (0, 7, 14, 21)]
    want = []
    for disp, seg, roads in batches:
        sec, inst, offs = st.ComputeBatch(True, disp, seg, roads)
        want.append((sec.copy(), inst.copy(), offs.copy()))
    C_, S = st.GetRealCols(), st.GetMaxSections()
    outs = [np.zeros((n, C_, S), dtype=api.L.SECTION_DTYPE) for _ in batches]
    got = []
    with pytest.raises(api.InvalidArgument):
        st.WaitBatch()
    for rep, depth in enumerate((2, 3, 3, 2)):    # the later rounds reuse the result sets
        got.clear()
        for o in outs:
            o[:] = 0
        for i, (disp, seg, roads) in enumerate(batches):
            st.SubmitBatch(True, disp, seg, roads, outs[i])
            if i == 2 and depth == 3:
                with pytest.raises(api.StixelsError):   # a fourth batch in flight
                    st.SubmitBatch(True, disp, seg, roads, outs[i])
                with pytest.raises(api.InvalidArgument):  # synchronous call while batches are in flight
                    st.ComputeBatch(True, disp, seg, roads)
            if i >= depth - 1:
                sec, inst, offs = st.WaitBatch()
                got.append((sec.copy(), inst, offs))
        for _ in range(depth - 1):
            sec, inst, offs = st.WaitBatch()
            got.append((sec.copy(), inst, offs))
        assert len(got) == len(batches)
        for i, ((ws, wi, wo), (gs, gi, go)) in enumerate(zip(want, got)):
            assert all(parity.same_used_sections(ws[f], gs[f]) for f in range(n)), (rep, i)
            assert np.array_equal(wo, go) and np.array_equal(wi.view(np.uint8), gi.view(np.uint8)), (rep, i)
    # back to the synchronous calls once nothing is in flight
    sec, inst, offs = st.ComputeBatch(True, *batches[2])
    assert np.array_equal(inst.view(np.uint8), want[2][1].view(np.uint8))
    st.SetDisparityImage(batches[0][0][0]); st.SetSegmentation(batches[0][1][0]); st.SetRoadParameters(**batches[0][2][0])
    assert parity.same_used_sections(st.Compute(True).sections, want[0][0][0])
    st.Finish()


def test_fewer_rows_than_disparities_against_cpu_oracle():
    """rows < max_dis: the reference kernel only fills object_disparity_range[0..rows) of its shared
    copy (StixelsKernels.cu:378-380, one thread per row), so its own results depend on uninitialised
    shared memory there; the CPU oracle (full table) is the checker for such sizes."""
    rows, cols = 40, 64
    pre = _preset("pairwise", rows, cols, 8, 0.0, False)
    fr = synth.make_frame(6, rows=rows, cols=cols)
    st, data, inst = _run_ours(pre, True, fr)
    osec, oinst, _ = cpubind.compute_frame(cpubind.default_config(**pre), True, fr.disparity, fr.segmentation,
                                           fr.road)
    r = parity.compare_sections(data.sections, osec, rtol=1e-4)
    assert r["exact"] == 1.0 and r["close"] == 1.0, r
    st.Finish()


def test_edge_inputs():
    rows, cols = 64, 64
    pre = _preset("pairwise", rows, cols, 8, 0.0, False)
    fr = synth.make_frame(1, rows=rows, cols=cols)
    cfg = cpubind.default_config(**pre)
    st = api.make_stixels(pre)
    for disp, seg in ((np.zeros_like(fr.disparity), fr.segmentation),          # every pixel invalid
                      (fr.disparity, np.zeros_like(fr.segmentation)),          # empty CNN output
                      (np.full_like(fr.disparity, 127.5), fr.segmentation)):   # maximum disparity everywhere
        st.SetDisparityImage(disp)
        st.SetSegmentation(seg)
        st.SetRoadParameters(**fr.road)
        data = st.Compute(True)
        osec, oinst, _ = cpubind.compute_frame(cfg, True, disp, seg, fr.road)
        r = parity.compare_sections(data.sections, osec, rtol=1e-4)
        assert r["exact"] == 1.0 and r["close"] == 1.0, r
        assert parity.compare_instances(st.instance_records(), oinst)["same_partition"]
    st.Finish()


@pytest.mark.parametrize("mode,step", [("unary", 8), ("pairwise", 8), ("pairwise", 4)])
def test_full_size_properties(mode, step):
    """BASELINE.json sizes (1024x2048): every column is tiled bottom to top without gaps or overlaps,
    stixel costs are the table minima, frames of a batch do not interact, and the result equals the
    reference CUDA build when it is available."""
    rows, cols, n = 1024, 2048, 3
    pairwise = mode == "pairwise"
    pre = _preset(mode, rows, cols, step, 0.0, False)
    disp, seg, roads = synth.make_batch(n, start=100, rows=rows, cols=cols, column_step=step)
    st = api.make_stixels(pre, max_batch=4)
    sec, inst, offs = st.ComputeBatch(pairwise, disp, seg, roads)
    for f in range(n):
        ln = parity.column_lengths(sec[f])
        assert ln.min() >= 1 and ln.max() < 199
        idx = np.arange(sec.shape[1])
        assert np.all(sec[f]["vT"][idx, 0] == rows - 1)
        assert np.all(sec[f]["vB"][idx, ln - 1] == 0)
        for c in range(0, sec.shape[1], 7):
            s = sec[f][c, :ln[c]]
            assert np.all(s["vB"][:-1] == s["vT"][1:] + 1) and np.all(s["vT"] >= s["vB"])
            assert np.all((s["type"] >= 0) & (s["type"] <= 2)) and np.all(np.isfinite(s["cost"]))
            assert np.all((s["semantic_class"] >= 0) & (s["semantic_class"] < 19))
    # permuting the frames of the batch permutes the results (no cross-frame state)
    perm = [2, 0, 1]
    sec_p, inst_p, offs_p = st.ComputeBatch(pairwise, disp[perm], seg[perm], [roads[i] for i in perm])
    for k, f in enumerate(perm):
        assert parity.same_used_sections(sec_p[k], sec[f])
    if refbind.available():
        ref = refbind.RefStixels(api.StixelConfig(**pre))
        rsec, rinst, _ = ref.compute(pairwise, disp[0], seg[0], roads[0])
        ref.close()
        r = parity.compare_sections(sec[0], rsec)
        assert r["exact"] >= 0.999 and r["close"] >= 0.999, r
        assert parity.compare_instances(inst[offs[0]:offs[1]], rinst)["same_keys"]
    st.Finish()
