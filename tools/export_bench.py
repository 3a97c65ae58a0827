"""Cost of handing a batch's stixels to device consumers (isx_export_batch_device) on one GPU.

Workloads: bench.py's unary_b64 and pairwise_b64 (1024 x 2048, width 8, synth.make_batch(64), inputs resident in
HBM).  Four step kinds are timed in alternating windows of --steps back-to-back steps each (CUDA events on
isx_stream(), isx_flush before the closing event), --rounds windows per kind:
  compute          isx_compute_batch_device
  compute_flush    + isx_flush (the results ordered on isx_stream(), what the export does before it reads them)
  compute_export   + isx_export_batch_device of all 64 frames: Sections, offsets, labels, errors
  compute_export_vertices  the same with the 3D vertices
The export on its own is timed with CUDA events over --repeats calls on the same batch.  Bytes moved follow from the
exported offsets (bytes_model below); the rate is set against the 6547.5 GB/s device copy rate DESIGN.md 4 uses.
The device name, power limit and SM clock are read in the same run.  One JSON line per workload goes to stdout and
to --out (default profiles/r4_export_bench_n1.jsonl).

    python tools/export_bench.py [--steps 20] [--rounds 3] [--repeats 200] [--out PATH]
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
COPY_GBS = 6547.5   # device-to-device copy rate of one B200 (DESIGN.md 4)


def bytes_model(n, C_, stixels, records, vertices):
    """DRAM bytes one export moves: the column scan reads the counts and writes the frame-relative offsets; the
    stixel pass reads counts, offsets and the used Sections, writes Sections, labels, column offsets (and
    vertices), then reads the instance records and scatters their labels."""
    scan = n * C_ * 4 * 2
    stix = n * C_ * 4 * 2 + stixels * 32 + stixels * (32 + 4) + (n * C_ + 1) * 4 + records * (16 + 4)
    return scan + stix + (stixels * 48 if vertices else 0)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window (at least 20)")
    ap.add_argument("--rounds", type=int, default=3, help="windows per step kind, alternating")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=200, help="exports timed on their own")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_export_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 20:
        ap.error("--steps must be at least 20")
    import torch
    import parity
    from instance_stixels_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("export_bench.py measures on a GPU; none is visible")
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
        buf = dict(sections=torch.empty((cap, 8), dtype=torch.int32, device="cuda"),
                   frame_offsets=torch.empty(B + 1, dtype=torch.int32, device="cuda"),
                   column_offsets=torch.empty(B * C_ + 1, dtype=torch.int32, device="cuda"),
                   labels=torch.empty(cap, dtype=torch.int32, device="cuda"),
                   vertices=torch.empty((cap, 4, 3), dtype=torch.float32, device="cuda"),
                   frame_errors=torch.empty(B, dtype=torch.int32, device="cuda"))
        torch.cuda.synchronize()
        stream = torch.cuda.ExternalStream(st.stream(), device=env.local)

        def export(vertices):
            st.ExportBatchDevice(0, B, buf["frame_offsets"].data_ptr(), sections=buf["sections"].data_ptr(),
                                 column_offsets=buf["column_offsets"].data_ptr(), labels=buf["labels"].data_ptr(),
                                 vertices=buf["vertices"].data_ptr() if vertices else 0,
                                 frame_errors=buf["frame_errors"].data_ptr(), capacity=cap)

        def compute():
            st.ComputeBatchDevice(pairwise, B, d_disp.data_ptr(), d_seg.data_ptr(), roads)

        # compute_flush: each batch's results ordered on isx_stream(), as the export orders them before it reads
        kinds = {"compute": compute,
                 "compute_flush": lambda: (compute(), st.Flush()),
                 "compute_export": lambda: (compute(), export(False)),
                 "compute_export_vertices": lambda: (compute(), export(True))}

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
            # the export on its own, on the batch the last window computed
            alone = {}
            for vertices in (False, True):
                export(vertices)
                st.Synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.repeats):
                    export(vertices)
                e1.record(stream)
                st.Synchronize()
                alone["vertices" if vertices else "no_vertices"] = e0.elapsed_time(e1) / args.repeats
        fo = buf["frame_offsets"].cpu().numpy()
        errors = buf["frame_errors"].cpu().numpy()
        stixels = int(fo[B])
        # the exported offsets against the host fetch of the same batch
        sections, inst, _ = st.FetchBatchResults(B)
        lens = np.stack([parity.column_lengths(sections[f]) for f in range(B)]).reshape(-1)
        offsets_ok = bool(np.array_equal(buf["column_offsets"].cpu().numpy(),
                                         np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)))
        st.Finish()
        med = {k: statistics.median(v) for k, v in ms.items()}
        out = dict(name=name, config=bench.workload_config(name, wl), steps_per_window=args.steps,
                   rounds=args.rounds, ms_per_step={k: [round(x, 4) for x in v] for k, v in ms.items()},
                   ms_per_step_median={k: round(v, 4) for k, v in med.items()},
                   export_overhead_frac={k: round(med[k] / med["compute"] - 1.0, 4)
                                         for k in ("compute_flush", "compute_export", "compute_export_vertices")},
                   stixels=stixels, instance_records=int(len(inst)), frame_errors=int(errors.any()),
                   offsets_equal_host=offsets_ok, export_repeats=args.repeats, export_alone={})
        for k, t in alone.items():
            nbytes = bytes_model(B, C_, stixels, len(inst), k == "vertices")
            gbs = nbytes / (t * 1e-3) / 1e9
            out["export_alone"][k] = dict(ms=round(t, 4), bytes=int(nbytes), gbs=round(gbs, 1),
                                          frac_of_copy_rate=round(gbs / COPY_GBS, 4))
        out["copy_rate_gbs"] = COPY_GBS
        out["device"] = dict(device_info(env.local), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
        line = json.dumps(out)
        print(line, flush=True)
        lines.append(line)
        del d_disp, d_seg, buf
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not all(json.loads(x)["offsets_equal_host"] for x in lines):
        raise SystemExit("exported offsets differ from the host results")


if __name__ == "__main__":
    main()
