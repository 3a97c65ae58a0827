"""Road estimation inside streamed host batches (isx_submit_batch_host_road / _u16_road) against the two ways a
host caller had before, on one GPU.

Setup: 64-frame batches of 1024 x 2048 frames, width 8, from pinned host memory, three batches in flight.  Three
different batches (192 frames, horizons spread over rows 256 .. 665) are streamed in turn, so that the ground-table
cache of the library (64 roads) does not hide the cost of the host function.  Modes unary and pairwise, inputs float
(isx_submit_batch_host*) and u16 (isx_submit_batch_host_u16*, value = u16 / 256).  Arms:
  given     the roads are known: isx_submit_batch_host{,_u16} with them
  host      what apps/cityscapes_runner's batched mode does: isx_road_compute_host frame by frame (blocking), keep-last,
            then isx_submit_batch_host{,_u16}
  device    isx_submit_batch_host{,_u16}_road: the road step in the pipeline
Per arm: frames/s over --steps batches (host clock, the window ends with the last wait), the host milliseconds per
batch inside the submit calls (road estimation included for `host`) and inside the waits, and a chunk trace of a
separate profiled window: the copy engine's idle time between the input copies of consecutive chunks, and for
`device` the host time of the ground-table host function per chunk.  The results of the `device` arm are compared
with the `host` arm byte for byte.  The device name, power limit and SM clock are read in the same run.  One JSON line
per (mode, input) goes to stdout and to --out (default profiles/r6_host_road_bench_n1.jsonl).

    python tools/host_road_bench.py [--steps 12] [--rounds 2] [--modes unary,pairwise] [--inputs float,u16]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

ROWS, COLS, WIDTH, B, DEPTH, SETS = 1024, 2048, 8, 64, 3, 3
CAM = dict(camera_center_y=512.0, baseline=0.209313, focal=2262.52)
FALLBACK = dict(vhor=512, camera_tilt=0.0, camera_height=1.2, alpha_ground=0.209313 / 1.2)


def make_sets(synth):
    sets = []
    for s in range(SETS):
        frames = [synth.make_frame(s * B + i, rows=ROWS, cols=COLS, column_step=WIDTH,
                                   vhor=256 + ((s * B + i) * 41) % 410) for i in range(B)]
        sets.append((np.stack([f.disparity for f in frames]), np.stack([f.segmentation for f in frames])))
    return sets


def keep_last(est, seed):
    out, cur = [], seed
    for e in est:
        if e.ok:
            cur = dict(vhor=int(e.horizon_point), camera_tilt=e.pitch, camera_height=e.camera_height,
                       alpha_ground=e.slope)
        out.append(cur)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=12, help="batches per timed window (at least 6)")
    ap.add_argument("--rounds", type=int, default=2, help="windows per arm, alternating")
    ap.add_argument("--modes", default="unary,pairwise")
    ap.add_argument("--inputs", default="float,u16")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_host_road_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 6:
        ap.error("--steps must be at least 6")
    import torch
    import bench
    from instance_stixels_b200 import _lib as L
    from instance_stixels_b200 import api, synth
    from tall_bench import device_info
    if not torch.cuda.is_available():
        raise SystemExit("host_road_bench.py measures on a GPU; none is visible")
    t0 = time.perf_counter()
    raw = make_sets(synth)
    print(f"{SETS * B} frames made in {time.perf_counter() - t0:.1f} s", file=sys.stderr, flush=True)
    used = (ROWS + 7) // 8
    pinned = []
    for disp, seg in raw:
        d16 = np.rint(disp * 256.0).astype(np.uint16)
        wide = (d16.astype(np.float32) / np.float32(256.0)).astype(np.float32)
        pinned.append(dict(
            float=(torch.from_numpy(disp).pin_memory().numpy(), torch.from_numpy(seg).pin_memory().numpy()),
            u16=(torch.from_numpy(d16).pin_memory().numpy(),
                 torch.from_numpy(np.ascontiguousarray(seg[..., :used]).astype(np.int16)).pin_memory().numpy()),
            road_image=dict(float=disp, u16=wide)))
    del raw
    ref = api.RoadEstimation()
    ref.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], ROWS, COLS, 128, 0.2, max_batch=1)
    lines = []
    for mode in args.modes.split(","):
        pairwise = mode == "pairwise"
        st = api.make_stixels(synth.preset(mode, ROWS, COLS, WIDTH), max_batch=B)
        st.ReserveInFlight(DEPTH)
        road = api.RoadEstimation()
        road.Initialize(CAM["camera_center_y"], CAM["baseline"], CAM["focal"], ROWS, COLS, 128, 0.2, max_batch=B)
        C_ = st.GetRealCols()
        outs = [torch.empty((B, C_, 200, 32), dtype=torch.uint8).pin_memory().numpy().view(L.SECTION_DTYPE)
                .reshape(B, C_, 200) for _ in range(DEPTH)]
        for kind in args.inputs.split(","):
            host_s = dict(submit=0.0, wait=0.0)
            state = dict(first=True)

            def host_estimates(i):
                img = pinned[i % SETS]["road_image"][kind]
                est = (L.RoadEstimate * B)()
                for f in range(B):
                    a = np.ascontiguousarray(img[f])
                    rc = ref._lib.isx_road_compute_host(ref.handle(), a.ctypes.data, a.size, C.byref(est[f]))
                    assert rc == 0
                return est

            def submit_given(i, roads):
                d, s = pinned[i % SETS][kind]
                if kind == "u16":
                    st.SubmitBatchU16(pairwise, d, 1.0 / 256.0, s, roads, outs[i % DEPTH])
                else:
                    st.SubmitBatch(pairwise, d, s, roads, outs[i % DEPTH])

            given_roads = [keep_last(host_estimates(i), FALLBACK) for i in range(SETS)]

            def arm_given(i):
                submit_given(i, given_roads[i % SETS])

            def arm_host(i):
                roads = keep_last(host_estimates(i), state["seed"])   # keep-last across batches, like the device
                state["seed"] = roads[-1]
                submit_given(i, roads)

            def arm_device(i):
                d, s = pinned[i % SETS][kind]
                fb = FALLBACK if state["first"] else None
                state["first"] = False
                if kind == "u16":
                    return st.SubmitBatchU16Road(road, pairwise, d, 1.0 / 256.0, s, fb, outs[i % DEPTH])
                return st.SubmitBatchRoad(road, pairwise, d, s, fb, outs[i % DEPTH])

            arms = dict(given=arm_given, host=arm_host, device=arm_device)

            def window(arm, steps, keep=None):
                host_s.update(submit=0.0, wait=0.0)
                state["first"] = True
                state["seed"] = FALLBACK
                t_start = time.perf_counter()
                for i in range(steps):
                    a = time.perf_counter()
                    arm(i)
                    host_s["submit"] += time.perf_counter() - a
                    if i >= DEPTH - 1:
                        a = time.perf_counter()
                        r = st.WaitBatch(want_instances=keep is not None)
                        host_s["wait"] += time.perf_counter() - a
                        if keep is not None:
                            keep.append(tuple(np.array(x, copy=True) for x in r))
                for _ in range(min(DEPTH - 1, steps)):
                    a = time.perf_counter()
                    r = st.WaitBatch(want_instances=keep is not None)
                    host_s["wait"] += time.perf_counter() - a
                    if keep is not None:
                        keep.append(tuple(np.array(x, copy=True) for x in r))
                wall = time.perf_counter() - t_start
                return (B * steps / wall, host_s["submit"] * 1e3 / steps, host_s["wait"] * 1e3 / steps)

            for arm in arms.values():
                window(arm, DEPTH + 1)
            fps = {k: [] for k in arms}
            sub = {k: [] for k in arms}
            wai = {k: [] for k in arms}
            with bench.ClockSampler(0) as clk:
                for _ in range(args.rounds):
                    for k, arm in arms.items():
                        f, s_, w_ = window(arm, args.steps)
                        fps[k].append(f)
                        sub[k].append(s_)
                        wai[k].append(w_)
            # byte identity of the device arm with the host arm (SETS batches, the road stream continuing)
            want, got = [], []
            window(arm_host, SETS, keep=want)
            window(arm_device, SETS, keep=got)
            equal = all(all(np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))
                            for a, b in zip(x, y)) for x, y in zip(want, got))
            # profiled window per arm: the chunk trace and the host function's time
            traces = {}
            for k, arm in arms.items():
                st.stage_times(reset=True)
                st.set_profiling(True)
                window(arm, 2 * DEPTH)
                buf = (C.c_double * (11 * 256))()
                nch = st._lib.isx_get_chunk_trace(st._h, buf, 256)
                fill_ms, fill_calls = C.c_double(0), C.c_long(0)
                st._lib.isx_get_road_fill_time(st._h, C.byref(fill_ms), C.byref(fill_calls), 1)
                st.stage_times(reset=True)
                st.set_profiling(False)
                rows_ = [[round(buf[c * 11 + j], 3) for j in range(11)] for c in range(nch)]
                gaps = [rows_[c + 1][0] - rows_[c][1] for c in range(nch - 1)]
                traces[k] = dict(chunks=nch, h2d_ms_median=round(statistics.median(r[1] - r[0] for r in rows_), 3),
                                 copy_gap_ms_median=round(statistics.median(gaps), 3) if gaps else None,
                                 copy_gap_ms_max=round(max(gaps), 3) if gaps else None,
                                 copy_gap_ms_total=round(sum(gaps), 3),
                                 span_ms=round(rows_[-1][10] - rows_[0][0], 3) if rows_ else None,
                                 host_function_ms_per_chunk=(round(fill_ms.value / fill_calls.value, 4)
                                                             if fill_calls.value else None),
                                 host_function_calls=int(fill_calls.value),
                                 first_chunks=rows_[:6])
            med = {k: statistics.median(v) for k, v in fps.items()}
            out = dict(name=f"{mode}_b{B}_{kind}", mode=mode, input=kind, batch=B, rows=ROWS, cols=COLS,
                       width=WIDTH, in_flight=DEPTH, distinct_batches=SETS, steps_per_window=args.steps,
                       rounds=args.rounds, frames_per_s={k: [round(x, 1) for x in v] for k, v in fps.items()},
                       frames_per_s_median={k: round(v, 1) for k, v in med.items()},
                       device_vs_given=round(med["device"] / med["given"], 4),
                       host_ms_in_submit_per_batch={k: round(statistics.median(v), 3) for k, v in sub.items()},
                       host_ms_in_wait_per_batch={k: round(statistics.median(v), 3) for k, v in wai.items()},
                       trace=traces, device_equals_host=bool(equal))
            out["device"] = dict(device_info(0), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
            line = json.dumps(out)
            print(line, flush=True)
            lines.append(line)
        st.Finish()
        road.Finish()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not all(json.loads(x)["device_equals_host"] for x in lines):
        raise SystemExit("the in-stream road path differs from the host composition")


if __name__ == "__main__":
    main()
