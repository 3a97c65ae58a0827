"""Throughput of frames taller than 1024 rows on one GPU (bench.py measures the 1024 x 2048 workloads only).

Workloads: 1280 x 1920 unary and pairwise, 2047 x 1920 pairwise; batch 64, stixel width 8.  Each one runs
bench.measure() at its own frame size (inputs resident in HBM: isx_compute_batch_device between CUDA events on
isx_stream() with isx_flush before the closing event; end to end with float and u16 inputs from pinned buffers,
three batches in flight; the ALU roofline over the live cells evaluated, with units_evaluated_frac), and adds the
device memory isx_initialize takes, the device name, power limit and SM clocks read in the same run, and a check of
a seeded sample of the timed frames against the CPU oracle with the criteria of tests/test_gpu_tall_frames.py.
One JSON line per workload goes to stdout and to --out (default profiles/r3_tall_bench_n1.jsonl).

    python tools/tall_bench.py [--steps 20] [--warmup 3] [--check-frames 4] [--out PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402

WORKLOADS = {
    "unary_1280x1920_b64": dict(rows=1280, cols=1920, mode="unary", step=8, batch=64),
    "pairwise_1280x1920_b64": dict(rows=1280, cols=1920, mode="pairwise", step=8, batch=64),
    "pairwise_2047x1920_b64": dict(rows=2047, cols=1920, mode="pairwise", step=8, batch=64),
}
CHECK_SEED = 0x7A11


def device_info(index=0):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(index)],
                         capture_output=True, text=True).stdout.strip()
    parts = [x.strip() for x in out.split(",")]
    if len(parts) != 4:
        return dict(raw=out)
    return dict(name=parts[0], power_limit_w=float(parts[1]), sm_mhz_idle=float(parts[2]), sm_max_mhz=float(parts[3]))


def init_memory_bytes(pre, batch):
    """Device memory isx_initialize allocates for `batch` frames (free memory before and after)."""
    import torch
    from instance_stixels_b200 import api
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    st = api.make_stixels(pre, max_batch=batch)
    torch.cuda.synchronize()
    free1, _ = torch.cuda.mem_get_info()
    return st, free0 - free1


def oracle_check(st, pre, wl, nframes):
    """A seeded sample of the timed frames, one at a time through the C ABI, against the CPU oracle."""
    import parity
    from instance_stixels_b200 import _lib as L
    from oracle import cpubind
    pairwise = wl["mode"] == "pairwise"
    disp, seg, roads, distinct = bench.synth_batch(wl, 0)
    frames = sorted(np.random.default_rng(CHECK_SEED).choice(distinct, size=min(nframes, distinct), replace=False))
    C_ = st.GetRealCols()
    rows = wl["rows"]
    # rows 2041-2047: the reference's class sums of the top rows read past their prefix array, and so does the oracle
    # (tests/test_gpu_tall_frames.py, _rows_with_reference_result): there only the rows below are compared
    hs2 = 1 << (rows // 8).bit_length()
    nrows = rows if (rows - 1) // 8 + 1 < hs2 else 8 * (hs2 - 1)
    res = []
    for f in frames:
        st.SetDisparityImage(disp[f]); st.SetSegmentation(seg[f]); st.SetRoadParameters(**roads[f])
        data = st.Compute(pairwise)
        inst = st.instance_records()
        cost = st.read_tensor(L.T_COST_TABLE).reshape(C_, rows, 3)[:, :nrows]
        index = st.read_tensor(L.T_INDEX_TABLE).reshape(C_, rows, 3)[:, :nrows]
        osec, oinst, ex = cpubind.compute_frame(cpubind.default_config(**pre), pairwise, disp[f], seg[f], roads[f],
                                                tables=True)
        ocost, oindex = ex["cost_table"][:, :nrows], ex["index_table"][:, :nrows]
        fin = np.isfinite(ocost)
        rel = np.abs(cost[fin] - ocost[fin]) / np.maximum(np.abs(ocost[fin]), 1e-6)
        item = dict(frame=int(f), rows_compared=nrows,
                    finite_pattern_equal=bool(np.array_equal(fin, np.isfinite(cost))),
                    cost_rel_q999=float(np.quantile(rel, 0.999)),
                    backpointers_equal=float((index == oindex)[fin].mean()))
        ok = item["finite_pattern_equal"] and item["cost_rel_q999"] <= 1e-4 and item["backpointers_equal"] >= 0.99
        if nrows == rows:   # Sections and instances are backtracked from the top row
            r = parity.compare_sections(data.sections, osec, rtol=1e-4)
            item.update(exact=r["exact"], close=r["close"])
            ok = ok and r["exact"] >= 0.99 and r["close"] >= 0.99
            if pairwise:
                item["same_partition"] = bool(parity.compare_instances(inst, oinst)["same_partition"])
                ok = ok and item["same_partition"]
        item["ok"] = bool(ok)
        res.append(item)
    return dict(frames=res, ok=all(x["ok"] for x in res))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--check-frames", type=int, default=4)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_tall_bench_n1.jsonl"))
    args = ap.parse_args()
    if args.steps < 20:
        ap.error("--steps must be at least 20")
    import torch
    from instance_stixels_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit("tall_bench.py measures on a GPU; none is visible")
    env = bench.Env()
    # bench.py's DRAM captures are of 1024-row launches: not attached to these workloads
    bench.NCU_TRAFFIC = {}
    lines = []
    for name in args.workloads.split(","):
        wl = WORKLOADS[name]
        bench.ROWS, bench.COLS = wl["rows"], wl["cols"]
        pre = synth.preset(wl["mode"], wl["rows"], wl["cols"], wl["step"])
        st, init_bytes = init_memory_bytes(pre, wl["batch"])
        st.Finish()
        dev = device_info(env.local)
        out = bench.measure(env, name, wl, args.steps, args.warmup, primary=True, extras=False)
        # measure()'s table-build roofline assumes the record stride of <= 1024 rows; the ALU roofline is row-generic
        out.pop("roofline_tables", None)
        out["config"].update(rows=wl["rows"], cols=wl["cols"])
        out["config"].pop("l2", None)
        out["device"] = dict(dev, sm_mhz_during_timing=out.get("clocks", {}).get("sm_mhz"))
        out["isx_initialize_device_bytes"] = int(init_bytes)
        from instance_stixels_b200 import api
        st = api.make_stixels(pre, max_batch=1)
        out["oracle_check"] = oracle_check(st, pre, wl, args.check_frames)
        st.Finish()
        line = json.dumps(out)
        print(line, flush=True)
        lines.append(line)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not all(json.loads(x)["oracle_check"]["ok"] for x in lines):
        raise SystemExit("oracle check failed")


if __name__ == "__main__":
    main()
