"""Cost of handing a batch's instances to device consumers as objects (isx_export_objects_device) on one GPU.

Workloads: bench.py's unary_b64 and pairwise_b64 (1024 x 2048, width 8, synth.make_batch(64), inputs resident in
HBM).  Two step kinds are timed in alternating windows of --steps back-to-back steps each (CUDA events on
isx_stream(), isx_flush before the closing event), --rounds windows per kind:
  compute_export          isx_compute_batch_device + isx_export_batch_device of all 64 frames (Sections, offsets,
                          labels, errors)
  compute_export_objects  the same + isx_export_objects_device of all 64 frames (objects, offsets, extents)
The object export on its own is timed with CUDA events over --repeats calls on the same batch, with and without
extents.  Objects and members (labelled instance records) per frame are counted from the exported offsets.  The
device name, power limit and SM clock are read in the same run.  One JSON line per workload goes to stdout and to
--out (default profiles/r7_objects_bench_n1.jsonl).

    python tools/objects_bench.py [--steps 20] [--rounds 3] [--repeats 200] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from tall_bench import device_info  # noqa: E402

WORKLOADS = ("unary_b64", "pairwise_b64")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window (at least 20)")
    ap.add_argument("--rounds", type=int, default=3, help="windows per step kind, alternating")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=200, help="object exports timed on their own")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_objects_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 20:
        ap.error("--steps must be at least 20")
    import torch
    from instance_stixels_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("objects_bench.py measures on a GPU; none is visible")
    env = bench.Env()
    lines = []
    for name in args.workloads.split(","):
        wl = bench.WORKLOADS[name]
        B, pairwise = wl["batch"], wl["mode"] == "pairwise"
        st = api.make_stixels(synth.preset(wl["mode"], bench.ROWS, bench.COLS, wl["step"]), max_batch=B,
                              device=env.local)
        C_ = st.GetRealCols()
        disp, seg, roads, _ = bench.synth_batch(wl, 0)
        d_disp = torch.from_numpy(disp).cuda()
        d_seg = torch.from_numpy(seg).cuda()
        cap = B * C_ * 200
        dev = dict(device="cuda")
        buf = dict(sections=torch.empty((cap, 8), dtype=torch.int32, **dev),
                   frame_offsets=torch.empty(B + 1, dtype=torch.int32, **dev),
                   column_offsets=torch.empty(B * C_ + 1, dtype=torch.int32, **dev),
                   labels=torch.empty(cap, dtype=torch.int32, **dev),
                   frame_errors=torch.empty(B, dtype=torch.int32, **dev),
                   objects=torch.empty((cap, 12), dtype=torch.int32, **dev),
                   object_frame_offsets=torch.empty(B + 1, dtype=torch.int32, **dev),
                   class_offsets=torch.empty(B * 8 + 1, dtype=torch.int32, **dev),
                   extents=torch.empty((cap, 2, 3), dtype=torch.float32, **dev))
        torch.cuda.synchronize()
        stream = torch.cuda.ExternalStream(st.stream(), device=env.local)

        def export():
            st.ExportBatchDevice(0, B, buf["frame_offsets"].data_ptr(), sections=buf["sections"].data_ptr(),
                                 column_offsets=buf["column_offsets"].data_ptr(), labels=buf["labels"].data_ptr(),
                                 frame_errors=buf["frame_errors"].data_ptr(), capacity=cap)

        def objects(extents):
            st.ExportObjectsDevice(0, B, buf["object_frame_offsets"].data_ptr(), objects=buf["objects"].data_ptr(),
                                   class_offsets=buf["class_offsets"].data_ptr(),
                                   extents=buf["extents"].data_ptr() if extents else 0, capacity=cap)

        def compute():
            st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), roads)

        kinds = {"compute_export": lambda: (compute(), export()),
                 "compute_export_objects": lambda: (compute(), export(), objects(True))}

        def window(step, steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(steps):
                step()
            st.Flush()
            e1.record(stream)
            st.Synchronize()
            return e0.elapsed_time(e1) / steps

        for step in kinds.values():
            window(step, args.warmup)
        ms = {k: [] for k in kinds}
        with bench.ClockSampler(env.local) as clk:
            for _ in range(args.rounds):
                for k, step in kinds.items():
                    ms[k].append(window(step, args.steps))
            # the object export on its own, on the batch the last window computed
            alone = {}
            for extents in (False, True):
                objects(extents)
                st.Synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.repeats):
                    objects(extents)
                e1.record(stream)
                st.Synchronize()
                alone["extents" if extents else "no_extents"] = round(e0.elapsed_time(e1) / args.repeats, 4)
        export()
        st.Synchronize()
        fo = buf["object_frame_offsets"].cpu().numpy()
        per_frame_objects = np.diff(fo)
        total = int(fo[B])
        stixels_per_object = buf["objects"][:total, 2].cpu().numpy()
        efo = buf["frame_offsets"].cpu().numpy()
        labels = buf["labels"][:int(efo[B])].cpu().numpy()
        per_frame_members = np.array([(labels[efo[f]:efo[f + 1]] >= 0).sum() for f in range(B)])
        members_ok = bool(np.array_equal(per_frame_members,
                                          [stixels_per_object[fo[f]:fo[f + 1]].sum() for f in range(B)]))
        st.Finish()
        med = {k: statistics.median(v) for k, v in ms.items()}
        out = dict(name=name, config=bench.workload_config(name, wl), steps_per_window=args.steps,
                   rounds=args.rounds, ms_per_step={k: [round(x, 4) for x in v] for k, v in ms.items()},
                   ms_per_step_median={k: round(v, 4) for k, v in med.items()},
                   objects_overhead_frac=round(med["compute_export_objects"] / med["compute_export"] - 1.0, 4),
                   objects_repeats=args.repeats, objects_alone_ms=alone,
                   objects_per_frame=dict(mean=round(float(per_frame_objects.mean()), 2),
                                          min=int(per_frame_objects.min()), max=int(per_frame_objects.max())),
                   members_per_frame=dict(mean=round(float(per_frame_members.mean()), 2),
                                          min=int(per_frame_members.min()), max=int(per_frame_members.max())),
                   members_equal_labelled_stixels=members_ok)
        out["device"] = dict(device_info(env.local), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
        line = json.dumps(out)
        print(line, flush=True)
        lines.append(line)
        del d_disp, d_seg, buf
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not all(json.loads(x)["members_equal_labelled_stixels"] for x in lines):
        raise SystemExit("object members differ from the labelled stixels of the export")


if __name__ == "__main__":
    main()
