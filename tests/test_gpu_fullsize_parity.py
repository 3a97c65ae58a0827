"""Parity at BASELINE.json's size ON THE FRAMES THE BENCH TIMES: all 64 frames of unary_b64, pairwise_b64 and
pairwise_w4_b64 (1024 x 2048) through the batched host entry point against what the reference CUDA build computed
for them, frame by frame (per-frame digests in tests/golden/reference_build/digests.json, see
tools/make_reference_build_golden.py).  Bar: boundaries / types / classes / instance partitions identical on every
column and every float field of every stixel bit-identical.

Plus a seeded fuzz of the two pruning DP kernels against the exhaustive ones (full cost / argmin tables) over random
small shapes, weights and horizons."""
import json
import os

import numpy as np
import pytest

import parity
from instance_stixels_b200 import _lib as L, api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DIGESTS = os.path.join(ROOT, "tests", "golden", "reference_build", "digests.json")
FULL_ROWS, FULL_COLS = 1024, 2048
# the bench's workloads (bench.py WORKLOADS): mode, column_step
BENCH_WORKLOADS = {"unary_b64": ("unary", 8), "pairwise_b64": ("pairwise", 8), "pairwise_w4_b64": ("pairwise", 4)}

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("workload", list(BENCH_WORKLOADS))
def test_all_bench_frames_against_reference_cuda_build(workload):
    mode, step = BENCH_WORKLOADS[workload]
    with open(DIGESTS) as f:
        want = json.load(f)["fullsize"][workload]
    pre = synth.preset(mode, FULL_ROWS, FULL_COLS, step)
    disp, seg, roads = synth.make_batch(64, rows=FULL_ROWS, cols=FULL_COLS, column_step=step)
    st = api.make_stixels(pre, max_batch=64)
    sec, inst, offs = st.ComputeBatch(mode == "pairwise", disp, seg, roads)
    ev, tot = st.dp_units()
    st.Finish()
    assert sec.shape[:2] == (64, FULL_COLS // step)
    assert [int(parity.column_lengths(s).sum()) for s in sec] == want["stixels"]
    # stixel boundaries, types and classes identical and every float field of every stixel bit-identical, on EVERY
    # column of every frame (profiles/r2_fullsize_parity.json: 2.8 million stixels, no differing bit).  The kernels
    # spell every float operation in the order of the reference's SASS.
    differing = [f for f in range(64) if parity.sections_digest(sec[f]) != want["sections"][f]]
    assert not differing, differing
    # instance ids up to label permutation (same candidates AND same partition), frame by frame
    differing = [f for f in range(64) if parity.partition_digest(inst[offs[f]:offs[f + 1]]) != want["instances"][f]]
    assert not differing, differing
    if workload == "unary_b64":
        assert ev / tot < 0.5


def _fuzz_case(rng, mode):
    step = int(rng.choice([4, 8]))
    rows = int(rng.integers(33, 417))
    cols = step * int(rng.integers(4, 25))
    pre = synth.preset(mode, rows, cols, step)
    # random non-negative weights around (and far from) the tuned ones
    pre["prior_weight"] = float(10.0 ** rng.uniform(-1.0, 4.3)) if mode == "unary" else float(10.0 ** rng.uniform(-1.0, 1.0))
    pre["segmentation_weight"] = float(10.0 ** rng.uniform(-2.0, 1.5))
    pre["instance_weight"] = float(10.0 ** rng.uniform(-4.0, -1.0)) * rng.integers(0, 2)
    pre["disparity_weight"] = float(10.0 ** rng.uniform(-4.0, 0.5))
    pre["invalid_disparity"] = float(rng.choice([0.0, -1.0]))
    pre["max_dis"] = int(rng.choice([64, 128]))
    vhor = int(rng.integers(0, rows - 12))            # anywhere, including the top border
    fr = synth.make_frame(int(rng.integers(0, 1000)), rows=rows, cols=cols, column_step=step, max_dis=pre["max_dis"],
                          vhor=vhor)
    seg = fr.segmentation.copy()
    kind = int(rng.integers(0, 4))
    used = (rows + 7) // 8
    if kind == 1:      # confident CNN: many zero costs, ties everywhere
        seg[:, :19, :used] = np.where(rng.random(seg[:, :19, :used].shape) < 0.7, 0, seg[:, :19, :used])
    elif kind == 2:    # structureless
        seg[:, :19, :used] = rng.integers(0, 80, size=seg[:, :19, :used].shape)
    return pre, fr.disparity, seg, fr.road


@pytest.mark.parametrize("mode", ["unary", "pairwise"])
def test_pruning_fuzz_against_exhaustive_tables(mode, monkeypatch):
    """>= 200 random (shape, weights, horizon, input statistics) cases per mode: the pruning kernel's full
    (cost, argmin) tables and Sections are byte-identical to the exhaustive kernel's."""
    pairwise = mode == "pairwise"
    rng = np.random.default_rng(0xF0221 + (1 if pairwise else 0))
    monkeypatch.setenv("ISX_DP_WARPS", "4")      # the walk variants even for a single small frame
    envs = {"pruning": {}, "exhaustive": {"ISX_UNARY_EXHAUSTIVE": "1", "ISX_PAIRWISE_WALK": "0"}}
    pruned_units = total_units = 0
    n_cases = 200
    for case in range(n_cases):
        pre, disp, seg, road = _fuzz_case(rng, mode)
        outs = {}
        for name, env in envs.items():
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
                outs[name] = (data.sections.copy(), st.read_tensor(L.T_COST_TABLE).copy(),
                              st.read_tensor(L.T_INDEX_TABLE).copy())
            except api.StixelsError as e:     # >= 200 stixels in a column: both kernels must agree on that too
                outs[name] = ("error", str(e))
            if name == "pruning":
                ev, tot = st.dp_units()
                pruned_units += ev
                total_units += tot
            st.Finish()
        a, b = outs["pruning"], outs["exhaustive"]
        ctx = (case, {k: pre[k] for k in ("rows", "cols", "column_step", "prior_weight", "segmentation_weight",
                                          "instance_weight", "disparity_weight", "invalid_disparity", "max_dis")}, road)
        assert isinstance(a[0], str) == isinstance(b[0], str), ctx
        if isinstance(a[0], str):
            continue
        assert np.array_equal(a[1].view(np.int32), b[1].view(np.int32)), ctx
        assert np.array_equal(a[2], b[2]), ctx
        assert parity.same_used_sections(a[0], b[0]), ctx
    assert 0 < pruned_units < total_units      # the bounds did fire somewhere
    print(f"fuzz {mode}: {n_cases} cases, {pruned_units} of {total_units} units evaluated")
