"""Cost of the device tracker (isx_tracker_update_device, api.ObjectTracker) on one GPU.

Records, each with CUDA events on the stream the work runs on:
  moving        tracker device time per 64-frame batch on the objects of a moving pairwise scene (1024 x 2048, width 8,
                synth.make_moving_batch), the same batch fed --repeats times after --warmup updates
  dense         the same on a dense record stream: 300 objects per class and frame, about 900 live tracks per class
                (test_gpu_tracking.dense_frames)
  one_frame     a one-frame update of the moving scene, one at a time: device time between events around the update
                and host time from before the enqueue to after the synchronise (medians over --repeats)
  step          ComputeBatchTensors(objects=True) on the moving scene with and without tracker=, in alternating windows
                of --steps steps, --rounds windows per kind
The device name, power limit and SM clock are read in the same run.  One JSON line goes to stdout and to --out
(default profiles/r8_track_bench_n1.jsonl).

    python tools/track_bench.py [--steps 20] [--rounds 3] [--repeats 50] [--out PATH]
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

B = 64


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window (at least 10)")
    ap.add_argument("--rounds", type=int, default=3, help="windows per step kind, alternating")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=50, help="tracker updates timed on their own")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_track_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 10:
        ap.error("--steps must be at least 10")
    import torch
    from instance_stixels_b200 import api, synth
    from test_gpu_tracking import DeviceStream, dense_frames
    if not torch.cuda.is_available():
        raise SystemExit("track_bench.py measures on a GPU; none is visible")
    env = bench.Env()
    dev = torch.device("cuda", env.local)
    torch.cuda.set_device(dev)
    st = api.make_stixels(synth.preset("pairwise", bench.ROWS, bench.COLS, 8), max_batch=B, device=env.local)
    disp, seg, roads = synth.make_moving_batch(B, rows=bench.ROWS, cols=bench.COLS, column_step=8)
    d_disp, d_seg = torch.from_numpy(disp).to(dev), torch.from_numpy(seg).to(dev)
    stream = torch.cuda.current_stream(dev)

    def events_ms(fn, count):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(count):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / count

    def tracker_alone(objects, n):
        t = api.ObjectTracker(env.local)
        events_ms(lambda: t.update(objects, n), args.warmup)
        ms = events_ms(lambda: t.update(objects, n), args.repeats)
        live = len(t.state()[0])
        return ms, live

    out = dict(name="track_bench", batch=B, rows=bench.ROWS, cols=bench.COLS, column_step=8, mode="pairwise",
               repeats=args.repeats, steps_per_window=args.steps, rounds=args.rounds)
    with bench.ClockSampler(env.local) as clk:
        res = st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_seg, objects=True)
        moving = res.objects
        fo = moving.frame_offsets.cpu().numpy()
        ms, live = tracker_alone(moving, B)
        out["moving"] = dict(ms_per_batch=round(ms, 4), objects_per_frame=round(float(np.diff(fo).mean()), 2),
                             live_tracks_after=live)
        dense = DeviceStream(dense_frames(np.random.default_rng(1), B))
        dense_objects = dense.call(0, B)[0]
        ms, live = tracker_alone(dense_objects, B)
        out["dense"] = dict(ms_per_batch=round(ms, 4), objects_per_frame=int(dense.fo[1]),
                            live_tracks_after=live, live_tracks_per_class=round(live / 8, 1))
        # one frame: the first frame of the moving batch (its offsets are a prefix of the batch's)
        one = api.DeviceObjects(data=moving.data, frame_offsets=moving.frame_offsets[:2],
                                class_offsets=moving.class_offsets[:9])
        t = api.ObjectTracker(env.local)
        events_ms(lambda: t.update(one, 1), args.warmup)
        dev_ms, host_ms = [], []
        for _ in range(args.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(stream)
            t.update(one, 1)
            e1.record(stream)
            torch.cuda.synchronize()
            host_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(e0.elapsed_time(e1))
        out["one_frame"] = dict(device_ms_median=round(statistics.median(dev_ms), 4),
                                host_ms_median=round(statistics.median(host_ms), 4))
        # the step with and without the tracker
        tracker = api.ObjectTracker(env.local)
        kinds = {"objects": lambda: st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_seg, objects=True),
                 "objects_tracker": lambda: st.ComputeBatchTensors(True, d_disp, roads, segmentation=d_seg,
                                                                   objects=True, tracker=tracker)}
        for fn in kinds.values():
            events_ms(fn, args.warmup)
        ms = {k: [] for k in kinds}
        for _ in range(args.rounds):
            for k, fn in kinds.items():
                ms[k].append(round(events_ms(fn, args.steps), 4))
        med = {k: statistics.median(v) for k, v in ms.items()}
        out["step"] = dict(ms_per_step=ms, ms_per_step_median={k: round(v, 4) for k, v in med.items()},
                           tracker_overhead_frac=round(med["objects_tracker"] / med["objects"] - 1.0, 4))
    out["device"] = dict(device_info(env.local), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
    # the inputs were handed to the library's stream (record_stream): free them while that stream exists
    del kinds, d_disp, d_seg
    torch.cuda.synchronize()
    st.Finish()
    line = json.dumps(out)
    print(line, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
