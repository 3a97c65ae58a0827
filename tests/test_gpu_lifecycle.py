"""Lifetime of an initialised handle: a failed Initialize leaves the handle uninitialised and holding nothing, Finish
releases everything (also with batches in flight), and a handle may be initialised again after either."""
import os

import numpy as np
import pytest

from instance_stixels_b200 import api, synth

pytestmark = pytest.mark.gpu

# A result set for this many frames is tens of TB (an estimator's arrays too): the allocation fails at once with
# cudaErrorMemoryAllocation and takes no memory from anything else on the device.
TOO_MANY = 1 << 30
CAM = {k: synth.CAMERA[k] for k in ("camera_center_y", "baseline", "focal")}


def _compute(st, pairwise, n, start=0, rows=64, cols=64, column_step=8):
    disp, seg, roads = synth.make_batch(n, start=start, rows=rows, cols=cols, column_step=column_step)
    sec, inst, offs = st.ComputeBatch(pairwise, disp, seg, roads)
    return sec.view(np.uint8).copy(), inst.view(np.uint8).copy(), offs.copy()


def _same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


def _fresh(pre, n, pairwise, **kw):
    st = api.make_stixels(pre, max_batch=n)
    out = _compute(st, pairwise, n, **kw)
    st.Finish()
    return out


def _road_estimates(re, frames):
    out = []
    for fr in frames:
        re.Compute(fr.disparity)
        out.append((re.GetHorizonPoint(), re.GetPitch(), re.GetCameraHeight(), re.GetSlope(), re.line()))
    return out


def test_failed_initialize_then_a_working_one():
    pre = synth.preset("pairwise", rows=64, cols=64)
    st = api.Stixels()
    st.SetConfig(api.StixelConfig(**pre))
    with pytest.raises(api.StixelsError):
        st.Initialize(TOO_MANY)
    assert not st.IsInitialized()
    st.Initialize(3)
    for pairwise in (False, True):
        assert _same(_compute(st, pairwise, 3), _fresh(pre, 3, pairwise))
    st.Finish()

    frames = [synth.make_frame(i, rows=64, cols=64) for i in range(3)]
    re = api.RoadEstimation()
    with pytest.raises(api.StixelsError):
        re.Initialize(*CAM.values(), 64, 64, 128, 0.2, max_batch=TOO_MANY)
    assert not re.IsInitialized()
    re.Initialize(*CAM.values(), 64, 64, 128)
    fresh = api.RoadEstimation()
    fresh.Initialize(*CAM.values(), 64, 64, 128)
    assert _road_estimates(re, frames) == _road_estimates(fresh, frames)


def test_finish_with_batches_in_flight():
    st = api.make_stixels(synth.preset("pairwise", rows=64, cols=64), max_batch=2)
    kept = []
    for start in (0, 2):
        disp, seg, roads = synth.make_batch(2, start=start, rows=64, cols=64)
        out = np.zeros((2, st.GetRealCols(), st.GetMaxSections()), dtype=api.L.SECTION_DTYPE)
        st.SubmitBatch(True, disp, seg, roads, out)
        kept.append((disp, seg, out))
    st.Finish()
    assert not st.IsInitialized()
    pre4 = synth.preset("pairwise", rows=64, cols=64, column_step=4)
    st.SetConfig(api.StixelConfig(**pre4))
    st.Initialize(2)
    assert st.GetRealCols() == 16
    assert _same(_compute(st, True, 2, column_step=4), _fresh(pre4, 2, True, column_step=4))
    st.Finish()


def _process_gpu_bytes():
    """This process's memory on the GPUs by NVML's per-process query, or None when NVML does not list the process
    (a PID namespace)."""
    import pynvml
    pynvml.nvmlInit()
    try:
        total, seen = 0, False
        for i in range(pynvml.nvmlDeviceGetCount()):
            for p in pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i)):
                if p.pid == os.getpid() and p.usedGpuMemory is not None:
                    total, seen = total + p.usedGpuMemory, True
        return total if seen else None
    finally:
        pynvml.nvmlShutdown()


def _lifecycle_round(large, small):
    """Every way a handle is left: failed Initialize + destroy, Finish after profiled work, a failing frame pool, a
    failed road Initialize + destroy."""
    os.environ["ISX_CHUNK"] = "1"   # a few hundred MB of chunk buffers before the result set fails
    try:
        st = api.Stixels()
        st.SetConfig(api.StixelConfig(**large))
        with pytest.raises(api.StixelsError):
            st.Initialize(TOO_MANY)
        st.__del__()
        with pytest.raises(api.StixelsError):
            api.StixelsPool(api.StixelConfig(**large), [0], max_batch=TOO_MANY)
    finally:
        del os.environ["ISX_CHUNK"]
    st = api.make_stixels(small, max_batch=2)
    st.set_profiling(True)
    disp, seg, roads = synth.make_batch(2, rows=64, cols=64)
    out = np.zeros((2, st.GetRealCols(), st.GetMaxSections()), dtype=api.L.SECTION_DTYPE)
    st.SubmitBatch(True, disp, seg, roads, out)
    st.WaitBatch()
    st.stage_times()
    st.Finish()
    st.__del__()
    re = api.RoadEstimation()
    with pytest.raises(api.StixelsError):
        re.Initialize(*CAM.values(), 1024, 2048, 128, 0.2, max_batch=TOO_MANY)
    re.__del__()


def test_memory_is_released():
    import torch
    large = synth.preset("pairwise", rows=1024, cols=2048)
    small = synth.preset("pairwise", rows=64, cols=64)
    torch.cuda.init()
    _lifecycle_round(large, small)   # warm-up: lazy module loading allocates on the first launch of every kernel
    torch.cuda.synchronize()

    def used():
        b = _process_gpu_bytes()
        return b if b is not None else -torch.cuda.mem_get_info(0)[0]

    before = used()
    for _ in range(3):
        _lifecycle_round(large, small)
    growth = used() - before
    assert growth < 64 << 20, f"GPU memory grew by {growth / 2**20:.0f} MiB over three rounds"
