"""Golden data for the parity tests against the reference CUDA build (GPU box):
  python tools/make_reference_build_golden.py [--out tests/golden/reference_build]

The reference's sources are not part of this repository, so tests/test_gpu_parity.py and
tests/test_gpu_fullsize_parity.py compare with stored results instead of running oracle/_ref.  This tool wrote them
with the library at the commit where both tests last passed against oracle/_ref (profiles/r2_pytest_gpu.log; full
size: profiles/r2_fullsize_parity.json, no differing bit), so they hold what the reference build computed:
  * <case>_f<frame>.npz   Sections and instance records of the CASES of test_gpu_parity.py that tests/golden/ does
                          not already hold as outputs of the reference itself (same layout as those files);
  * digests.json          per case the FrameMeta and SHA-256 digests of the five tables the test compares bit for
                          bit; per bench workload and frame, digests of the Sections and of the instance partition
                          (tests/parity.py: sections_digest, partition_digest).
Where tests/golden/ holds the reference's own output of a case, this tool first checks that the library
reproduces it bit for bit."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from instance_stixels_b200 import _lib as L, api, synth  # noqa: E402
import parity  # noqa: E402
from test_gpu_parity import CASES, TABLES, _preset, _run_ours  # noqa: E402
from test_gpu_fullsize_parity import BENCH_WORKLOADS, FULL_ROWS, FULL_COLS  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden", "reference_build"))
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    digests = dict(cases={}, fullsize={})
    for name, mode, rows, cols, step, frame, invalid, median in CASES:
        pairwise = mode == "pairwise"
        pre = _preset(mode, rows, cols, step, invalid, median)
        fr = synth.make_frame(frame, rows=rows, cols=cols, column_step=step)
        st, data, inst = _run_ours(pre, pairwise, fr)
        sec = data.sections
        lengths = parity.column_lengths(sec)
        reference_own = os.path.join(ROOT, "tests", "golden", f"{name}_f{frame}.npz")
        if os.path.exists(reference_own):
            z = np.load(reference_own)
            ref = np.zeros_like(sec)
            ref["type"] = -1
            ref[:, :z["sections"].shape[1]] = z["sections"]
            r = parity.compare_sections(sec, ref)
            assert r["exact"] == 1.0 and r["bitwise"] == 1.0, (name, r)
            assert parity.compare_instances(inst, z["instances"])["same_partition"], name
        else:
            np.savez_compressed(os.path.join(args.out, f"{name}_f{frame}.npz"),
                                sections=sec[:, :int(lengths.max()) + 1].copy(), lengths=lengths, instances=inst,
                                rows=rows, cols=cols, step=step, mode=mode, frame=frame, invalid=invalid,
                                median=median)
        digests["cases"][name] = dict(
            meta={n: getattr(data, n) for n, _ in L.FrameMeta._fields_},
            tables={t: parity.array_digest(st.read_tensor(getattr(L, t)).view(np.int32)) for t in TABLES})
        st.Finish()
        print(name, int(lengths.sum()), "stixels", len(inst), "instance stixels", flush=True)
    for name, (mode, step) in BENCH_WORKLOADS.items():
        pre = synth.preset(mode, FULL_ROWS, FULL_COLS, step)
        disp, seg, roads = synth.make_batch(64, rows=FULL_ROWS, cols=FULL_COLS, column_step=step)
        st = api.make_stixels(pre, max_batch=64)
        sec, inst, offs = st.ComputeBatch(mode == "pairwise", disp, seg, roads)
        st.Finish()
        digests["fullsize"][name] = dict(
            stixels=[int(parity.column_lengths(s).sum()) for s in sec],
            sections=[parity.sections_digest(s) for s in sec],
            instances=[parity.partition_digest(inst[offs[f]:offs[f + 1]]) for f in range(len(sec))])
        print(name, sum(digests["fullsize"][name]["stixels"]), "stixels", flush=True)
    with open(os.path.join(args.out, "digests.json"), "w") as f:
        json.dump(digests, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
