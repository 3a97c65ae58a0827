"""Cost of the bird's-eye-view grid (isx_bev_grid_device) on one GPU.

Workloads: bench.py's unary_b64 and pairwise_b64 (1024 x 2048, width 8, synth.make_batch(64), inputs resident in
HBM).  Per workload:
  bev_alone_ms   the BEV call on its own on the computed batch, CUDA events on isx_stream() over --repeats calls, for
                 the default grid (0.2 m, 200 x 300 cells) and a fine grid (0.05 m, 800 x 1200 cells)
  ms_per_step    Stixels.ComputeBatchTensors steps without and with bev= (default grid), in alternating windows of
                 --steps back-to-back steps each (CUDA events on the current torch stream), --rounds windows per kind
The share of unknown / free / occupied cells of the last grid, the device name, power limit and SM clock are read in the
same run.  One JSON line per workload goes to stdout and to --out (default profiles/r9_bev_bench_n1.jsonl).

    python tools/bev_bench.py [--steps 20] [--rounds 3] [--repeats 200] [--out PATH]
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
GRIDS = {"default": {}, "fine": dict(cell=0.05, nx=800, nz=1200)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed window (at least 20)")
    ap.add_argument("--rounds", type=int, default=3, help="windows per step kind, alternating")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=200, help="BEV calls timed on their own")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_bev_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 20:
        ap.error("--steps must be at least 20")
    import torch
    from instance_stixels_b200 import api, synth
    if not torch.cuda.is_available():
        raise SystemExit("bev_bench.py measures on a GPU; none is visible")
    env = bench.Env()
    lines = []
    for name in args.workloads.split(","):
        wl = bench.WORKLOADS[name]
        B, pairwise = wl["batch"], wl["mode"] == "pairwise"
        st = api.make_stixels(synth.preset(wl["mode"], bench.ROWS, bench.COLS, wl["step"]), max_batch=B,
                              device=env.local)
        disp, seg, roads, _ = bench.synth_batch(wl, 0)
        d_disp = torch.from_numpy(disp).cuda()
        d_seg = torch.from_numpy(seg).cuda()
        params = {k: api.BevParams(**g) for k, g in GRIDS.items()}
        cells = {k: torch.empty((B, p.nz, p.nx, 2), dtype=torch.int32, device="cuda") for k, p in params.items()}
        stream = torch.cuda.ExternalStream(st.stream(), device=env.local)
        current = torch.cuda.current_stream()

        def step(bev):
            return st.ComputeBatchTensors(pairwise, d_disp, roads, segmentation=d_seg,
                                          bev=params["default"] if bev else None)

        kinds = {"compute_tensors": lambda: step(False), "compute_tensors_bev": lambda: step(True)}

        def window(fn, steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(current)
            for _ in range(steps):
                fn()
            e1.record(current)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / steps

        for fn in kinds.values():
            window(fn, args.warmup)
        ms = {k: [] for k in kinds}
        alone = {}
        with bench.ClockSampler(env.local) as clk:
            for _ in range(args.rounds):
                for k, fn in kinds.items():
                    ms[k].append(window(fn, args.steps))
            # the BEV call on its own, on the batch the last window computed
            for k, p in params.items():
                st.BevGridDevice(0, B, p, cells[k].data_ptr())
                st.Synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(args.repeats):
                    st.BevGridDevice(0, B, p, cells[k].data_ptr())
                e1.record(stream)
                st.Synchronize()
                alone[k] = round(e0.elapsed_time(e1) / args.repeats, 4)
        share = {}
        for k in params:
            counts = np.bincount(cells[k][..., 1].reshape(-1).cpu().numpy(), minlength=3)
            share[k] = dict(zip(("unknown", "free", "occupied"), (round(float(c / counts.sum()), 4) for c in counts)))
        # the inputs were recorded on the library's stream: release them before Finish destroys it
        del d_disp, d_seg, cells
        torch.cuda.synchronize()
        st.Finish()
        med = {k: statistics.median(v) for k, v in ms.items()}
        out = dict(name=name, config=bench.workload_config(name, wl), steps_per_window=args.steps,
                   rounds=args.rounds, ms_per_step={k: [round(x, 4) for x in v] for k, v in ms.items()},
                   ms_per_step_median={k: round(v, 4) for k, v in med.items()},
                   bev_overhead_frac=round(med["compute_tensors_bev"] / med["compute_tensors"] - 1.0, 4),
                   bev_repeats=args.repeats, bev_alone_ms=alone,
                   grids={k: dict(cell=round(p.cell, 4), nx=p.nx, nz=p.nz, cells_per_batch=B * p.nx * p.nz)
                          for k, p in params.items()},
                   cell_share=share)
        out["device"] = dict(device_info(env.local), sm_mhz_during_timing=clk.summary().get("sm_mhz"))
        line = json.dumps(out)
        print(line, flush=True)
        lines.append(line)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
