"""apps/cityscapes_runner --batch B --gpus G on a synthetic Cityscapes-shaped dataset directory at 1024 x 2048
(16-bit disparity PNGs, camera JSON, nlogprobs HDF5 files), built on the GPU box: the reference-style CLI's own
"It took an average of ... fps" line beside bench.py's e2e number.  ISX_ALLOW_1024=1 lifts the reference's
rows < 1024 guard of the loader (apps/run_cityscapes.cu:129-134) for the BASELINE size.

  python tools/runner_bench.py [--frames 128] [--mode unary|pairwise] [--batch 64] [--gpus 1] [--road-on-device]
"""
import argparse, json, os, re, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
import cv2
import write_h5
from instance_stixels_b200 import synth

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=64)
ap.add_argument("--replicate", type=int, default=10, help="the timed call streams the loaded frames this many times")
ap.add_argument("--mode", default="unary")
ap.add_argument("--batch", type=int, default=64)
ap.add_argument("--gpus", type=int, default=1)
ap.add_argument("--road-on-device", action="store_true", help="estimate the roads inside the timed pool call")
a = ap.parse_args()
rows, cols = 1024, 2048
d = tempfile.mkdtemp(prefix="isx_ds_")
for sub in ("disparities", "camera", "probs", "stixels"):
    os.makedirs(os.path.join(d, sub))
cam = {"extrinsic": {"baseline": 0.209313}, "intrinsic": {"fx": 2262.52, "fy": 2262.52, "u0": 1024.0, "v0": 512.0}}
t0 = time.time()
for i in range(a.frames):
    fr = synth.make_frame(i % 32, rows=rows, cols=cols)
    base = f"synth_{i:06d}_000019"
    cv2.imwrite(os.path.join(d, "disparities", base + "_disparity.png"), np.clip(np.rint(fr.disparity * 256.0), 0, 65535).astype(np.uint16),
                [cv2.IMWRITE_PNG_COMPRESSION, 1])
    open(os.path.join(d, "camera", base + "_camera.json"), "w").write(json.dumps(cam))
    write_h5.write_h5(os.path.join(d, "probs", base + "_probs.h5"), "nlogprobs", fr.segmentation)
print("dataset of %d frames written in %.1f s" % (a.frames, time.time() - t0), file=sys.stderr)
pre = synth.preset(a.mode, rows, cols, 8)
pairwise = int(a.mode == "pairwise")
args = [os.path.join(ROOT, "apps", "cityscapes_runner"), d, "128", repr(pre["segmentation_weight"]), repr(pre["instance_weight"]),
        repr(pre["disparity_weight"]), str(pairwise), "8", repr(pre["eps"]), str(pre["min_pts"]), str(pre["size_filter"]),
        "--batch", str(a.batch), "--gpus", str(a.gpus), "--replicate", str(a.replicate)] + \
       (["--road-on-device"] if a.road_on_device else [])
env = dict(os.environ, ISX_ALLOW_1024="1")
p = subprocess.run(args, capture_output=True, text=True, env=env)
line = [l for l in p.stdout.splitlines() if l.startswith("It took an average")]
done = [l for l in p.stdout.splitlines() if l.startswith("Done.")]
m = re.search(r"([0-9.]+) milliseconds, ([0-9.]+) fps", line[0]) if line else None
print(json.dumps(dict(mode=a.mode, road_on_device=a.road_on_device, frames=a.frames, replicate=a.replicate, batch=a.batch, gpus=a.gpus, runner_fps=float(m.group(2)) if m else None,
                      runner_ms_per_frame=float(m.group(1)) if m else None, done_line=done[-1] if done else None,
                      stixels_files=len(os.listdir(os.path.join(d, "stixels"))), rc=p.returncode, stderr=p.stderr[-300:])))
subprocess.run(["rm", "-rf", d])
