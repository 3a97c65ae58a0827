"""Road estimation inside device batches (isx_compute_batch_device_road) against the synchronous composition, on one
GPU.

Workloads: bench.py's unary_b64 and pairwise_b64 (1024 x 2048, width 8, synth.make_batch(64), inputs resident in
HBM).  Three step kinds are timed in alternating windows of --steps back-to-back steps each (host clock around the
window, which ends in isx_synchronize), --rounds windows per kind:
  given       isx_compute_batch_device with the roads given
  composed    isx_road_compute_batch_device (blocks: candidates to the host), keep-last substitution in Python,
              then isx_compute_batch_device
  pipeline    isx_compute_batch_device_road: road kernels, device line selection, ground tables by a host function
              per chunk, stixels -- all in stream order
For every kind: frames/s, step time and the host time spent inside the calls of a step.  The road step on its own
(isx_road_compute_batch_device, blocking) is timed too.  The results of the last pipeline step are compared with the
composition byte for byte.  The device name and power limit are read in the same run.  One JSON line per workload
goes to stdout and to --out (default profiles/r5_road_pipeline_bench_n1.jsonl).

    python tools/road_pipeline_bench.py [--steps 20] [--rounds 3] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from tall_bench import device_info  # noqa: E402

WORKLOADS = ("unary_b64", "pairwise_b64")
CAM = dict(camera_center_y=512.0, baseline=0.209313, focal=2262.52)


def keep_last(estimates, seed):
    out, cur = [], seed
    for e in estimates:
        if e["ok"]:
            cur = dict(vhor=e["vhor"], camera_tilt=e["camera_tilt"], camera_height=e["camera_height"],
                       alpha_ground=e["alpha_ground"])
        out.append(cur)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window (at least 10)")
    ap.add_argument("--rounds", type=int, default=3, help="windows per step kind, alternating")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_road_pipeline_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 10:
        ap.error("--steps must be at least 10")
    import torch
    from instance_stixels_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("road_pipeline_bench.py measures on a GPU; none is visible")
    env = bench.Env()
    lines = []
    for name in args.workloads.split(","):
        wl = bench.WORKLOADS[name]
        B, pairwise = wl["batch"], wl["mode"] == "pairwise"
        st = api.make_stixels(synth.preset(wl["mode"], bench.ROWS, bench.COLS, wl["step"]), max_batch=B,
                              device=env.local)
        road = api.RoadEstimation(env.local)
        road.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], bench.ROWS, bench.COLS, 128, 0.2,
                        max_batch=B)
        disp, seg, roads, _ = bench.synth_batch(wl, 0)
        seed = roads[0]
        d_disp = torch.from_numpy(disp).cuda()
        d_seg = torch.from_numpy(seg).cuda()
        torch.cuda.synchronize()
        estimates = road.ComputeBatchDevice(B, d_disp.data_ptr())
        given = keep_last(estimates, seed)
        host_s = {}

        def timed(kind, fn):
            t0 = time.perf_counter()
            fn()
            host_s[kind] = host_s.get(kind, 0.0) + time.perf_counter() - t0

        def step_given():
            timed("given", lambda: st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), given))

        def step_composed():
            def run():
                est = road.ComputeBatchDevice(B, d_disp.data_ptr())
                st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), keep_last(est, seed))
            timed("composed", run)

        def step_pipeline():
            timed("pipeline", lambda: st.ComputeBatchDeviceRoad(road, pairwise, B, d_disp.data_ptr(),
                                                                d_seg.data_ptr(), seed))

        kinds = {"given": step_given, "composed": step_composed, "pipeline": step_pipeline}

        def window(step, steps):
            st.Synchronize()
            host_s.clear()
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            st.Synchronize()
            return (time.perf_counter() - t0) * 1e3 / steps, sum(host_s.values()) * 1e3 / steps

        for step in kinds.values():
            window(step, args.warmup)
        ms = {k: [] for k in kinds}
        host_ms = {k: [] for k in kinds}
        with bench.ClockSampler(env.local) as clk:
            for _ in range(args.rounds):
                for k, step in kinds.items():
                    t, h = window(step, args.steps)
                    ms[k].append(t)
                    host_ms[k].append(h)
            road_alone = []
            for _ in range(args.steps):
                t0 = time.perf_counter()
                road.ComputeBatchDevice(B, d_disp.data_ptr())
                road_alone.append((time.perf_counter() - t0) * 1e3)
        # the last pipeline step against the composition
        st.ComputeBatchDeviceRoad(road, pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), seed)
        got = st.FetchBatchResults(B)
        st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), given)
        want = st.FetchBatchResults(B)
        equal = all(np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
                    for a, b in zip(got, want))
        st.Finish()
        road.Finish()
        med = {k: statistics.median(v) for k, v in ms.items()}
        out = dict(name=name, config=bench.workload_config(name, wl), steps_per_window=args.steps,
                   rounds=args.rounds, ms_per_step={k: [round(x, 4) for x in v] for k, v in ms.items()},
                   ms_per_step_median={k: round(v, 4) for k, v in med.items()},
                   frames_per_s={k: round(B / (v * 1e-3), 1) for k, v in med.items()},
                   host_ms_in_calls_per_step={k: round(statistics.median(v), 4) for k, v in host_ms.items()},
                   road_step_alone_ms=round(statistics.median(road_alone), 4),
                   accepted_frames=sum(1 for e in estimates if e["ok"]),
                   pipeline_equals_composition=bool(equal))
        out["device"] = dict(device_info(env.local), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
        line = json.dumps(out)
        print(line, flush=True)
        lines.append(line)
        del d_disp, d_seg
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not all(json.loads(x)["pipeline_equals_composition"] for x in lines):
        raise SystemExit("the pipeline's results differ from the composition")


if __name__ == "__main__":
    main()
