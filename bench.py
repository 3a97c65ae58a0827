#!/usr/bin/env python
"""Benchmark of the stixel hot path (BASELINE.json metric: stixel frames/sec @1024x2048).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload unary_b64|pairwise_b64|pairwise_w4_b64|...]
  python bench.py --impl reference ...      # the reference's own implementation, same workload
  python bench.py ... --dump-outputs DIR    # also write the results of the last timed step as DIR/*.npy

A "step" is one pass of the whole path (column join -> tables -> DP -> backtracking -> instance
grouping -> result packing) over one batch of synthetic Cityscapes-shaped frames per GPU.  Frames are
independent, so N GPUs run N shards with no collective in the data path (weak scaling).

  value : frames/s with inputs already resident in HBM (isx_compute_batch_device), timed with CUDA
          events on the stream the kernels are launched on, max over ranks.
  e2e   : the same batches through the host-buffer entry points (isx_submit_batch_host /
          isx_wait_batch_host, three batches in flight): pinned host inputs -> H2D -> kernels -> the device
          writes the used Sections into the caller's pinned [C][200] array and packs counts / instance records
          into pinned host memory, every step.
  e2e_u16: the same with the narrow host inputs (uint16 disparity, unpadded int16 segmentation).

The line's top-level keys describe --workload (default unary_b64 = BASELINE.json configs[1]); `workloads`
carries the other BASELINE configurations measured in the same process (configs[2] pairwise_b64, configs[3]
pairwise_w4_b64, configs[4] pairwise_stream_b256 = the 4096-frame stream in batches of 256 per GPU), each
with value / e2e / roofline / latency_ms_batch1 / value_no_prune.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # BASELINE.json configs[1]: unary model, batch of 64 frames on 1 B200
    "unary_b64": dict(mode="unary", step=8, batch=64),
    # configs[2]: pairwise model + instance grouping, batch 64
    "pairwise_b64": dict(mode="pairwise", step=8, batch=64),
    # configs[3]: pairwise at stixel width 4
    "pairwise_w4_b64": dict(mode="pairwise", step=4, batch=64),
    # configs[4]: the 4096-frame stream at the largest batch; --steps 4096 / (256 * N) covers the stream
    "pairwise_stream_b256": dict(mode="pairwise", step=8, batch=256),
}
ROWS, COLS = 1024, 2048
RECORD_WORDS_PER_ROW = 32   # prefix records: one 128-byte row per image row and column (common.cuh kRecBWords)
OPS_PER_CELL = {"unary": 103, "pairwise": 128}  # SURVEY.md 8d minimal op budget
NCU_SOURCE = "profiles/r2d_*.txt"
DUMP_BYTES = 64 * 2**20 - 2**16   # --dump-outputs: at most 64 MB, .npy headers included
DUMP_SEED = 0x5717E1
# dram__bytes_read.sum + dram__bytes_write.sum per launch, from the `ncu --set full` captures summarised in
# profiles/r2d_{unary,pairwise}.txt (width 8; unary launches carry 32 frames, pairwise launches 64; no capture for
# width 4).  "tables" = join_columns + (frame_tables) + column_tables + object_lut kernels.
NCU_TRAFFIC = {
    ("unary", 8): dict(chunk=32, dp=(1.4432 + 0.1301) * 1e9,     # dp_unary_pruned_kernel
                       tables=(0.2685 + 0.0270 + 0.1440 + 1.0158 + 0.0337 + 4.2360) * 1e9),
    ("pairwise", 8): dict(chunk=64, dp=(3.2113 + 1.1235) * 1e9,  # dp_pairwise_walk_kernel
                          tables=(0.5369 + 0.0601 + 0.0003 + 0.2880 + 2.0902 + 0.0674 + 8.5304) * 1e9),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm_gbs=d.get("hbm_gbs", 6650.0), sm_max_mhz=d.get("sm_max_mhz", 1965.0), source="measured")
    return dict(hbm_gbs=6650.0, sm_max_mhz=1965.0, source="fallback")


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line):
    NVML in-process every 10 ms, nvidia-smi as the fallback."""

    _REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index = index
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.mem_mhz = None
        self.power_w = None
        self.source = "nvml"
        self._stop = threading.Event()
        self._t = None
        self._h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
                self._h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nv = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None
            self.source = "nvidia-smi"

    def _sample_nvml(self):
        nv = self._nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
        if self.mem_mhz is None:
            try:
                self.mem_mhz = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_MEM))
                self.power_w = nv.nvmlDeviceGetPowerUsage(self._h) / 1000.0
            except Exception:
                self.mem_mhz = 0.0
        try:
            bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
        except Exception:
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        for bit, name in self._REASONS.items():
            if bits & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout
        parts = [x.strip() for x in out.strip().split(",")]
        if len(parts) >= 6:
            self.sm.append(float(parts[0]))
            self.sm_max = float(parts[1])
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], parts[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(name)

    def _loop(self):
        while not self._stop.is_set():
            try:
                if self._h is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.01 if self._h is not None else 0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.sm:
            return dict(sm_mhz=None, sm_max_mhz=self.sm_max, reasons=["unavailable"], samples=0, source=self.source)
        sm = sorted(self.sm)
        return dict(sm_mhz=sm[len(sm) // 2], sm_min_mhz=sm[0], sm_max_mhz=self.sm_max, reasons=sorted(self.reasons),
                    samples=len(sm), source=self.source)


def cpu_baseline(wl, nframes=1):
    """The oracle port on the host cores, bounded sample of the same workload."""
    from instance_stixels_b200 import synth
    from oracle import cpubind
    pre = synth.preset(wl["mode"], ROWS, COLS, wl["step"])
    cfg = cpubind.default_config(**pre)
    lib = cpubind.load()
    cores = lib.orc_max_threads()
    frames = [synth.make_frame(i, rows=ROWS, cols=COLS, column_step=wl["step"]) for i in range(nframes)]
    t0 = time.perf_counter()
    for fr in frames:
        cpubind.compute_frame(cfg, wl["mode"] == "pairwise", fr.disparity, fr.segmentation, fr.road)
    dt = time.perf_counter() - t0
    return dict(value=nframes / dt, unit="frames/s", cores=cores, kind="port",
                sample=f"{nframes} frame(s) of the workload, oracle/stixels_cpu.cpp, OpenMP over columns")


def workload_config(name, wl, **extra):
    """The `config` object both arms print (same keys, same values: the driver compares them)."""
    return dict(workload=name, rows=ROWS, cols=COLS, column_step=wl["step"], mode=wl["mode"],
                frames_per_step=wl["batch"], **extra)


def synth_batch(wl, rank):
    """`batch` frames of this rank's shard of the synthetic stream.  At most 64 distinct frames are generated
    (0.12 s each on one host core); larger batches repeat them."""
    from instance_stixels_b200 import synth
    B = wl["batch"]
    distinct = min(B, 64)
    disp, seg, roads = synth.make_batch(distinct, start=rank * B, rows=ROWS, cols=COLS, column_step=wl["step"])
    if distinct < B:
        reps = B // distinct
        disp, seg, roads = np.concatenate([disp] * reps), np.concatenate([seg] * reps), roads * reps
    return disp, seg, roads, distinct


def run_reference(args, name, wl, rank, world):
    """--impl reference: the reference's own implementation of the path.  The reference has no CPU
    path (all stages are __global__ kernels): its implementation IS the CUDA build, compiled
    unmodified for sm_100a into oracle/_ref and driven one frame per Compute() like
    apps/run_cityscapes.cu:346-431.  Falls back to the CPU port when oracle/_ref cannot be used.
    Nothing of the product is loaded in this process: the config comes from the reference's own
    StixelConfig defaults (ref_config_init) + the preset fields."""
    if rank != 0:
        return
    import ctypes
    from instance_stixels_b200 import synth            # numpy only
    from instance_stixels_b200 import _lib as L        # ctypes struct layouts only (the .so is not loaded)
    from oracle import refbind
    pairwise = wl["mode"] == "pairwise"
    line = dict(impl="reference", metric="stixel frames/sec @1024x2048", unit="frames/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", config=workload_config(name, wl))
    B = min(wl["batch"], 64)     # frames actually pushed through per step (the stream workload repeats 64 anyway)
    try:
        import torch
        if not (refbind.available() and torch.cuda.is_available()):
            raise RuntimeError("oracle/_ref or CUDA device not available")
        disp, seg, roads, _ = synth_batch(dict(wl, batch=B), 0)
        cfg = L.Config()
        refbind.load().ref_config_init(ctypes.byref(cfg))
        for k, v in synth.preset(wl["mode"], ROWS, COLS, wl["step"]).items():
            setattr(cfg, k, int(v) if isinstance(v, bool) else v)
        ref = refbind.RefStixels(cfg)
        for _ in range(max(args.warmup, 1)):
            ref.time_frames(pairwise, disp[:2], seg[:2], roads[0])
        t = 0.0
        for _ in range(args.steps):
            t += ref.time_frames(pairwise, disp, seg, roads[0])
        sp = ref.time_frames_split(pairwise, disp, seg, roads[0])      # one more pass, host clock around every call
        ref.close()
        fps = B * args.steps / t
        per = 1e3 / sp["frames"]
        split = dict(set_inputs_h2d_ms=sp["set_inputs"] * per, compute_ms=sp["compute"] * per,
                     get_instance_stixels_ms=sp["get_instance_stixels"] * per,
                     dbscan_standin_ms=sp["dbscan_standin"] * per,
                     kernels_and_section_copy_ms=(sp["compute"] - sp["dbscan_standin"]) * per,
                     total_ms=sp["total"] * per,
                     note="per frame, host clock around the blocking calls of one extra pass; dbscan_standin = the "
                          "builder's host DBSCAN (3 blocking copies + O(n^2) loop) that replaces the cuML fork the "
                          "reference links (not available): reference time without it = total_ms - dbscan_standin_ms")
        line.update(value=fps, ms_per_step=1e3 * t / args.steps * (wl["batch"] / B), split_ms_per_frame=split,
                    value_without_dbscan_standin=1e3 / max(split["total_ms"] - split["dbscan_standin_ms"], 1e-9),
                    product_library_loaded=L._lib is not None,
                    cpu_baseline=dict(value=fps, unit="frames/s", cores=0, kind="reference",
                                      sample=f"{B} frames per timed pass through the reference CUDA build "
                                             "(oracle/_ref, sm_100a) on GPU 0, one frame per Compute()"))
    except Exception as e:  # no GPU / no _ref: time the CPU port instead
        cb = cpu_baseline(wl, 1)
        line.update(value=cb["value"], ms_per_step=1e3 * wl["batch"] / cb["value"], cpu_baseline=cb,
                    note=f"reference CUDA build unusable: {e!r}")
    line["e2e"] = dict(value=line["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    print(json.dumps(line), flush=True)


class Env:
    """Rank / world plumbing shared by the measurements."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))

    def barrier(self):
        import torch
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, obj):
        """`obj` of every rank, in rank order (the per-rank step times and clocks of a multi-GPU line)."""
        if self.world == 1:
            return [obj]
        import torch.distributed as dist
        out = [None] * self.world
        dist.all_gather_object(out, obj)
        return out


def narrow_inputs(disp, seg):
    """The same frames as a caller with 16-bit data holds them: disparity u16 = round(d * 256) (a 16-bit disparity
    PNG, apps/run_cityscapes.cu:141-147), segmentation int16 without the padding."""
    used = (ROWS + 7) // 8
    d16 = np.rint(disp * 256.0).astype(np.uint16)
    s16 = np.ascontiguousarray(seg[..., :used]).astype(np.int16)
    return d16, s16


def dump_outputs(out_dir, sections, instances, offsets):
    """What the timed path delivers for its last batch (isx_fetch_batch_results), as float32 .npy files so that two
    builds can be compared output for output: the stixels of every column of every frame, top to bottom, one file
    per Section field (section_<field>.npy), stixels_per_column.npy [frames][C], and the instance records, one file
    per field (instance_<field>.npy) with instances_per_frame.npy.  Every value is an integer below 2**24 or a
    float32, so float32 holds it exactly.  When the whole batch does not fit in DUMP_BYTES, frames are taken in a
    seeded random order until the next one would not fit; frames.npy lists the frames written, in batch order."""
    S = sections.shape[2]
    term = sections["type"] == -1
    lengths = np.where(term.any(axis=2), term.argmax(axis=2), S)
    inst_counts = np.diff(offsets)
    frame_bytes = (lengths.sum(axis=1) * len(sections.dtype.names) + lengths.shape[1]) * 4 + \
        inst_counts * len(instances.dtype.names) * 4 + 8
    order = np.random.default_rng(DUMP_SEED).permutation(len(sections))
    k = int(np.searchsorted(np.cumsum(frame_bytes[order]), DUMP_BYTES, side="right"))
    frames = np.sort(order[:k])
    used = np.arange(S)[None, None, :] < lengths[frames][:, :, None]
    stixels = sections[frames][used]
    inst = np.concatenate([instances[offsets[f]:offsets[f + 1]] for f in frames]) if k else instances[:0]
    os.makedirs(out_dir, exist_ok=True)
    arrays = {f"section_{n}": stixels[n] for n in sections.dtype.names}
    arrays.update({f"instance_{n}": inst[n] for n in instances.dtype.names})
    arrays.update(stixels_per_column=lengths[frames], instances_per_frame=inst_counts[frames], frames=frames)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def time_device(env, st, step, steps, stream):
    """`steps` device-resident batches between two CUDA events on the library's stream, max over ranks (ms)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    e0.record(stream)
    for _ in range(steps):
        step()
    st.Flush()  # the emission stream's last results are ordered before the closing event
    e1.record(stream)
    st.Synchronize()
    env.barrier()
    local = e0.elapsed_time(e1)
    return env.max_over_ranks(local), local


def measure(env, name, wl, steps, warmup, primary, extras=True, dump_dir=None):
    """One workload on this rank's GPU: the same dict on every rank (rank 0 prints it)."""
    import torch
    from instance_stixels_b200 import api, synth
    B = wl["batch"]
    world = env.world
    pairwise = wl["mode"] == "pairwise"
    pre = synth.preset(wl["mode"], ROWS, COLS, wl["step"])
    st = api.make_stixels(pre, max_batch=B, device=env.local)
    C_ = st.GetRealCols()
    disp, seg, roads, distinct = synth_batch(wl, env.rank)
    h_disp = torch.from_numpy(disp).pin_memory()
    h_seg = torch.from_numpy(seg).pin_memory()
    d_disp = h_disp.cuda(non_blocking=True)
    d_seg = h_seg.cuda(non_blocking=True)
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(st.stream(), device=env.local)

    def device_step():
        st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), roads)

    # ---- value: inputs resident in HBM ----
    for _ in range(max(warmup, 3)):
        device_step()
    st.Synchronize()
    st.set_profiling(True)
    st.stage_times(reset=True)
    launches0 = st._lib.isx_kernel_launch_count()
    units0 = st.dp_units()
    with ClockSampler(env.local) as clk:
        ms_max, ms_local = time_device(env, st, device_step, steps, stream)
    per_rank = env.gather(dict(ms_per_step=round(ms_local / steps, 3), sm_mhz=clk.summary().get("sm_mhz"),
                               mem_mhz=clk.mem_mhz, reasons=clk.summary().get("reasons"))) if primary else None
    launches = st._lib.isx_kernel_launch_count() - launches0
    units1 = st.dp_units()
    units_eval, units_total = units1[0] - units0[0], units1[1] - units0[1]
    stages = st.stage_times(reset=True)
    st.set_profiling(False)
    if dump_dir:   # before the e2e runs below overwrite the results of the timed steps
        dump_outputs(dump_dir, *st.FetchBatchResults(B))

    # ---- e2e: host buffers through the public batch API, copies inside the timed region ----
    # One host thread, one context, the streaming form of the batch call: isx_submit_batch_host enqueues a batch
    # (H2D of its inputs from pinned memory, kernels, results packed by the device into pinned host memory) and
    # isx_wait_batch_host delivers the oldest one into the caller's [C][200] Section array + instance records; three
    # batches are in flight (the input copies of batch k+2 are queued while batch k still computes: with two, the copy
    # engine waited for the host thread to come back from the wait).  Every step moves its own inputs and reads its
    # own results back.
    DEPTH = 3
    sections_host = [torch.empty((B, C_, 200, 32), dtype=torch.uint8).pin_memory() for _ in range(DEPTH)]
    sec_np = [t.numpy().view(api.L.SECTION_DTYPE).reshape(B, C_, 200) for t in sections_host]
    d16, s16 = narrow_inputs(disp, seg)
    h_d16, h_s16 = torch.from_numpy(d16).pin_memory(), torch.from_numpy(s16).pin_memory()
    seen = dict(inst=0)

    def run_e2e(kind, nsteps):
        def submit(i):
            if kind == "u16":
                st.SubmitBatchU16(pairwise, h_d16.numpy(), 1.0 / 256.0, h_s16.numpy(), roads, sec_np[i % DEPTH])
            else:
                st.SubmitBatch(pairwise, h_disp.numpy(), h_seg.numpy(), roads, sec_np[i % DEPTH])
        for w in range(DEPTH + 1):  # warm-up of the path that is timed (result sets are allocated on first use)
            if kind == "single":
                st.ComputeBatch(pairwise, h_disp.numpy(), h_seg.numpy(), roads, sections_out=sec_np[0])
            else:
                submit(w)
                if w >= DEPTH - 1:
                    st.WaitBatch()
        if kind != "single":
            for _ in range(DEPTH - 1):
                st.WaitBatch()
        env.barrier()
        t0 = time.perf_counter()
        if kind == "single":
            for _ in range(nsteps):
                _, inst, _ = st.ComputeBatch(pairwise, h_disp.numpy(), h_seg.numpy(), roads, sections_out=sec_np[0])
        else:
            for i in range(nsteps):
                submit(i)
                if i >= DEPTH - 1:
                    _, inst, _ = st.WaitBatch()
            for _ in range(min(DEPTH - 1, nsteps)):
                _, inst, _ = st.WaitBatch()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        seen["inst"] = len(inst)
        return env.max_over_ranks(dt) / nsteps

    e2e_s = run_e2e("float", steps)
    e2e_u16_s = run_e2e("u16", steps)
    e2e_single_s = run_e2e("single", max(2, steps // 2)) if primary else None
    # what the device wrote into host memory for one batch: the used Sections and the terminator of every column
    # (straight into the caller's pinned padded array) + per-column counts + instance records + one descriptor per frame
    n_stixels = int((sec_np[0]["type"] == -1).argmax(axis=2).sum())
    d2h_bytes = (n_stixels + B * C_) * 32 + B * C_ * 4 + seen["inst"] * 16 + B * 32
    h2d_float = int(h_disp.numel() * 4 + h_seg.numel() * 4 * ((ROWS + 7) // 8) // h_seg.shape[-1] + B * 3 * ROWS * 4)
    h2d_u16 = int(h_d16.numel() * 2 + h_s16.numel() * 2 + B * 3 * ROWS * 4)

    out = dict(name=name)
    H = ROWS
    peaks = measured_peaks()
    cells_per_frame = C_ * H * (H + 1) // 2
    dp_ms, dp_launches = stages["dp"]
    chunk = st.chunk_frames()
    # The DP kernels prune (tile, chunk) units that provably cannot win (exact branch and bound), so the roofline is
    # taken over the cells the kernel EVALUATED: 32 x 32 per off-diagonal unit, 32 * 33 / 2 live cells per diagonal
    # unit (every tile's diagonal unit is always evaluated; its other half lies above the diagonal, vB > vT).
    nt = (H + 31) // 32
    diag_units = B * steps * C_ * nt
    eval_frac = units_eval / max(units_total, 1)
    cells_eval = (units_eval - diag_units) * 1024 + diag_units * 528
    cells_eval_per_launch = cells_eval / max(dp_launches, 1)
    ops_per_launch = cells_eval_per_launch * OPS_PER_CELL[wl["mode"]]
    dp_avg_s = dp_ms * 1e-3 / max(dp_launches, 1)
    achieved = ops_per_launch / dp_avg_s / 1e12
    peak = 148 * 128 * peaks["sm_max_mhz"] * 1e6 / 1e12
    # table build (join + column tables + object LUT).  Bytes the three kernels must move per frame in this design:
    # the inputs (SURVEY.md 8d: disparity + unpadded segmentation), the joined disparity (written once, read by two
    # kernels), and the tables the DP consumes (prefix records, object LUT).
    seg_bytes = C_ * 21 * (H // 8) * 4
    in_bytes = H * COLS * 4 + seg_bytes
    rec_stride = 1056  # kRecStride (common.cuh)
    rec_words = RECORD_WORDS_PER_ROW
    table_bytes = C_ * H * 4 * 3 + C_ * rec_words * rec_stride * 4 + C_ * 128 * H * 4
    tab_bytes = (in_bytes + table_bytes) * chunk
    tab_ms = stages["join"][0] + stages["column_tables"][0]
    tab_launches = max(stages["join"][1], 1)
    tab_avg_s = tab_ms * 1e-3 / tab_launches
    ncu = NCU_TRAFFIC.get((wl["mode"], wl["step"]))
    if ncu and ncu["chunk"] != chunk:
        ncu = None
    dp_alg_bytes = (C_ * 128 * H * 4 + C_ * rec_words * rec_stride * 4 + C_ * H * 16) * chunk
    fps = world * B / (ms_max * 1e-3 / steps)
    out.update(
        value=fps, ms_per_step=ms_max / steps, steps=steps,
        config=workload_config(name, wl, frames_per_step_per_gpu=B, distinct_frames=distinct, chunk_frames=chunk,
                               l2="inputs (%d MB/step) and tables (>2 GB/chunk) exceed the 126 MB L2" % (B * 13.9)),
        e2e=dict(value=world * B / e2e_s, unit="frames/s", h2d_bytes_per_step=h2d_float, d2h_bytes_per_step=d2h_bytes,
                 pipeline="1 host thread, isx_submit_batch_host / isx_wait_batch_host, 3 batches in flight; float "
                          "disparity + int32 segmentation (the reference's types); the device writes the used "
                          "Sections straight into the caller's pinned [C][200] array and packs counts and instance "
                          "records into pinned host memory",
                 h2d_gbs_per_gpu=h2d_float / e2e_s / 1e9),
        e2e_u16=dict(value=world * B / e2e_u16_s, unit="frames/s", h2d_bytes_per_step=h2d_u16,
                     d2h_bytes_per_step=d2h_bytes, h2d_gbs_per_gpu=h2d_u16 / e2e_u16_s / 1e9,
                     pipeline="the same with isx_submit_batch_host_u16: uint16 disparity (x 1/256) + unpadded int16 "
                              "segmentation, widened on the device"),
        gpu_launches=int(launches),
        clocks=clk.summary(),
        **(dict(ranks=per_rank) if per_rank and env.world > 1 else {}),
        roofline=dict(bound="alu", kernel="dp_pairwise_walk_kernel" if pairwise else "dp_unary_pruned_kernel",
                      achieved=achieved, peak=peak, unit="Tlane-op/s", frac=achieved / peak,
                      traffic=ncu["dp"] if ncu else None,
                      traffic_note=f"DRAM bytes per launch (ncu, {NCU_SOURCE}); the tables one launch reads "
                                   f"once are {dp_alg_bytes} bytes",
                      units_evaluated_frac=eval_frac, live_cells_evaluated_frac=cells_eval / max(cells_per_frame * B * steps, 1),
                      note=f"over evaluated cells: {OPS_PER_CELL[wl['mode']]} lane-ops per DP cell (SURVEY 8d) x "
                           f"{cells_eval_per_launch:.0f} live cells evaluated per launch "
                           f"({100 * eval_frac:.1f} % of the (tile, chunk) units of the exhaustive scan; the dead half of "
                           f"the diagonal units is not counted) / {dp_avg_s * 1e3:.2f} ms avg launch (CUDA events, "
                           f"{dp_launches} launches); peak = 148 SM x 128 lanes x {peaks['sm_max_mhz']:.0f} MHz "
                           f"({peaks['source']}); the pruned cells are not work the kernel claims"),
        roofline_tables=dict(bound="hbm", kernel="join_columns+column_tables+object_lut",
                             achieved=tab_bytes / tab_avg_s / 1e9, peak=peaks["hbm_gbs"], unit="GB/s",
                             frac=tab_bytes / tab_avg_s / 1e9 / peaks["hbm_gbs"],
                             traffic=ncu["tables"] if ncu else None,
                             algorithmic_input_bytes=in_bytes * chunk,
                             traffic_over_algorithmic_input=(ncu["tables"] / (in_bytes * chunk)) if ncu else None,
                             design_bytes_over_algorithmic_input=tab_bytes / (in_bytes * chunk),
                             note=f"bytes per launch {tab_bytes}; per frame: inputs {in_bytes} + joined/records/object LUT "
                                  f"{table_bytes}; inputs alone are {in_bytes * chunk / tab_avg_s / 1e9:.0f} GB/s"),
        stage_ms_per_step={k: v[0] / steps for k, v in stages.items()},
    )
    if e2e_single_s is not None:
        out["e2e_single"] = dict(value=world * B / e2e_single_s, unit="frames/s",
                                 pipeline="1 host thread, 1 context, synchronous isx_compute_batch_host")
    if extras:
        # p50 / p99 latency of one frame through the reference call sequence (host in -> host out), with the
        # caller's buffers in pinned memory and -- like the reference's callers -- in pageable memory
        fr = synth.make_frame(0, rows=ROWS, cols=COLS, column_step=wl["step"])
        pin = [torch.from_numpy(fr.disparity).pin_memory(), torch.from_numpy(fr.segmentation).pin_memory(),
               torch.empty(C_ * 200 * 32, dtype=torch.uint8).pin_memory()]

        def one_frame(d, s_, o):
            t0 = time.perf_counter()
            st.SetDisparityImage(d)
            st.SetSegmentation(s_)
            st.SetRoadParameters(**fr.road)
            st.Compute(pairwise, sections_out=o)
            st.GetInstanceStixels()
            return 1e3 * (time.perf_counter() - t0)

        torch.cuda.synchronize()
        lat = sorted([one_frame(pin[0].numpy(), pin[1].numpy(), pin[2].numpy().view(api.L.SECTION_DTYPE))
                      for _ in range(240)][40:])   # 40 warm-up frames: clocks and caches settle after the batches
        lat_pageable = sorted([one_frame(fr.disparity, fr.segmentation, None) for _ in range(50)][10:])
        out["latency_ms_batch1"] = dict(p50=lat[len(lat) // 2], p99=lat[int(len(lat) * 0.99)], max=lat[-1],
                                        frames=len(lat), buffers="pinned",
                                        p50_pageable=lat_pageable[len(lat_pageable) // 2])
    st.Finish()
    del st
    if extras:
        # worst case of the data-dependent pruning: the same kernels walking every unit (ISX_*_PRUNE=0)
        key = "ISX_PAIRWISE_PRUNE" if pairwise else "ISX_UNARY_PRUNE"
        os.environ[key] = "0"
        try:
            st2 = api.make_stixels(pre, max_batch=B, device=env.local)
        finally:
            del os.environ[key]
        stream2 = torch.cuda.ExternalStream(st2.stream(), device=env.local)

        def step2():
            st2.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), roads)
        step2()
        st2.Synchronize()
        n2 = max(2, steps // 4)
        ms2, _ = time_device(env, st2, step2, n2, stream2)
        out["value_no_prune"] = dict(value=world * B / (ms2 * 1e-3 / n2), unit="frames/s",
                                     note="every (tile, chunk) unit evaluated: the floor of the data-dependent pruning")
        st2.Finish()
        del st2
        # The table kernels on their own: in the pipeline above their CTAs wait for places the DP of the chunk before
        # vacates, so the stage times around them contain that wait.  ISX_OVERLAP_TABLES=0 runs one kernel at a time.
        os.environ["ISX_OVERLAP_TABLES"] = "0"
        try:
            st3 = api.make_stixels(pre, max_batch=B, device=env.local)
        finally:
            del os.environ["ISX_OVERLAP_TABLES"]

        def step3():
            st3.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), roads)
        step3()
        st3.Synchronize()
        st3.set_profiling(True)
        st3.stage_times(reset=True)
        n3 = max(2, steps // 4)
        for _ in range(n3):
            step3()
        st3.Synchronize()
        stages3 = st3.stage_times(reset=True)
        st3.Finish()
        alone_s = (stages3["join"][0] + stages3["column_tables"][0]) * 1e-3 / max(stages3["join"][1], 1)
        rt = out["roofline_tables"]
        rt["achieved_alone"] = tab_bytes / alone_s / 1e9
        rt["frac_alone"] = rt["achieved_alone"] / peaks["hbm_gbs"]
        rt["note_alone"] = (f"the same kernels with nothing beside them (ISX_OVERLAP_TABLES=0, {stages3['join'][1]} launches, "
                            f"{alone_s * 1e3:.2f} ms per launch); `achieved` is from the pipelined run, where the stage "
                            f"events also see the wait for the DP's CTAs to retire")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="unary_b64", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="only --workload: no other configurations, latency or no-prune runs")
    ap.add_argument("--extra-workloads", default="pairwise_b64,pairwise_w4_b64,pairwise_stream_b256")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of --workload computed as DIR/<name>.npy (float32, at most "
                         "64 MB; with several ranks DIR/rank<k>/)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of --impl ours")
    wl = WORKLOADS[args.workload]
    env = Env()

    if args.impl == "reference":
        run_reference(args, args.workload, wl, env.rank, env.world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the stixel path has no CPU fallback")
    torch.cuda.set_device(env.local)
    # Bind this process to the CPUs next to its GPU before any host buffer is allocated or pinned: the host <-> device
    # copies of the e2e arm then stay on the local NUMA node (what a multi-GPU launcher does per rank).
    host_cpus = None
    if not os.environ.get("ISX_BENCH_NO_AFFINITY"):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                nvh = pynvml.nvmlDeviceGetHandleByUUID("GPU-" + str(torch.cuda.get_device_properties(env.local).uuid))
            except Exception:
                nvh = pynvml.nvmlDeviceGetHandleByIndex(env.local)
            pynvml.nvmlDeviceSetCpuAffinity(nvh)
            host_cpus = len(os.sched_getaffinity(0))
        except Exception:
            host_cpus = None
    if env.world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", env.local))

    t_start = time.perf_counter()
    dump_dir = args.dump_outputs
    if dump_dir and env.world > 1:
        dump_dir = os.path.join(dump_dir, f"rank{env.rank}")
    main_res = measure(env, args.workload, wl, args.steps, args.warmup, primary=True, extras=not args.no_extra,
                       dump_dir=dump_dir)
    others = {}
    if not args.no_extra:
        for name in [n for n in args.extra_workloads.split(",") if n and n != args.workload]:
            w2 = WORKLOADS[name]
            if name == "pairwise_stream_b256":
                steps2 = max(2, 4096 // (w2["batch"] * env.world))     # the 4096-frame stream over the whole box
            else:
                steps2 = max(4, args.steps // 2)
            r = measure(env, name, w2, steps2, args.warmup, primary=False, extras=True)
            if name == "pairwise_stream_b256":
                r["stream_frames"] = steps2 * w2["batch"] * env.world
            others[name] = r

    if env.rank == 0:
        line = dict(metric="stixel frames/sec @1024x2048", value=main_res.pop("value"), unit="frames/s",
                    n_gpus=env.world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=main_res.pop("ms_per_step"), higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="f32", data="synthetic")
        main_res.pop("name")
        main_res.pop("steps")
        line.update(main_res)
        line["host"] = dict(cpus_bound_to_gpu=host_cpus)
        if others:
            for r in others.values():
                r.pop("name")
            line["workloads"] = others
        if not args.no_cpu_baseline and env.world == 1:
            try:   # the CPU baseline gets every core of the box again
                os.sched_setaffinity(0, range(os.cpu_count()))
            except Exception:
                pass
            line["cpu_baseline"] = cpu_baseline(wl, 24)
        line["bench_wall_s"] = time.perf_counter() - t_start
        print(json.dumps(line), flush=True)
    if env.world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
