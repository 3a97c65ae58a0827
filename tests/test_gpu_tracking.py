"""Device tracker (isx_tracker_*, api.ObjectTracker, ComputeBatchTensors(tracker=)): byte for byte the host definition
HostObjectTracker of include/InstanceStixels/ObjectTracker.hpp, on random record streams and end to end on a moving
scene; call splits, resets, two trackers, two streams, refusals and destroy with updates in flight."""
import ctypes as C
import os

import numpy as np
import pytest

from instance_stixels_b200 import _lib as L
from instance_stixels_b200 import api, synth
from test_tracking_host import Bits, build_harness, frame, run_host, stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILL = 0x5A
PARAMS = {
    "defaults": dict(iou_min_permille=300, max_age=2, disparity_margin=2.0, max_tracks=1024),
    "tight": dict(iou_min_permille=100, max_age=0, disparity_margin=0.0, max_tracks=40),
    "no_gate": dict(iou_min_permille=500, max_age=4, disparity_margin=float("inf"), max_tracks=300),
}


def fuzz_frames(seed, n, big=(), dense_class=13):
    """n frames of moving boxes in three classes with near-tied and duplicated boxes, NaN, -0.0, +-inf and subnormal
    disparities; frames in `big` hold 300 small near-tied boxes in `dense_class`."""
    rng = np.random.default_rng(seed)
    pool = [0.0, -0.0, Bits(1), Bits(2), Bits(3), Bits(0x80000001), float("nan"), float("inf"), float("-inf"), 1.0,
            2.5, 3.0, 40.0, 41.5]
    world = []
    for _ in range(24):
        w, h = int(rng.integers(8, 200)), int(rng.integers(8, 200))
        world.append([int(rng.choice([11, 13, 18])), float(rng.integers(0, 1800)), float(rng.integers(0, 800)), w, h,
                      float(rng.normal(0, 3)), float(rng.normal(0, 1))])
    frames = []
    for f in range(n):
        objs = []
        for o in world:
            o[1] += o[5]
            o[2] += o[6]
            if rng.random() < 0.2:
                continue
            x, y = int(o[1]) + int(rng.integers(-1, 2)), int(o[2]) + int(rng.integers(-1, 2))
            box = (x, y, x + o[3] - 1, y + o[4] - 1)
            d = rng.choice(len(pool), 2)
            dmin, dmax = pool[d[0]], pool[d[1]]
            if rng.random() < 0.5:
                base = float(rng.uniform(0, 60))
                dmin, dmax = base, base + float(rng.uniform(0, 3))
            objs.append((o[0], box, dmin, dmax))
            if rng.random() < 0.15:   # an exact or one-pixel duplicate: IoU ties
                s = int(rng.integers(0, 2))
                objs.append((o[0], (box[0] + s, box[1], box[2] + s, box[3]), dmin, dmax))
        if rng.random() < 0.1:
            world[int(rng.integers(0, len(world)))][1] = float(rng.integers(0, 1800))   # a jump: a new track
        if f in big:
            for i in range(300):
                x, y = 4 * (i % 30) + int(rng.integers(0, 2)), 8 * (i // 30)
                objs.append((dense_class, (x, y, x + 7, y + 7), 5.0, 5.0 + float(i % 3)))
        frames.append(frame(*objs) if objs else np.zeros(0, L.OBJECT_DTYPE))
    return frames


class DeviceStream:
    """A record stream on the device, one call at a time: objects, rebased offsets and capacity like the export's."""

    def __init__(self, frames):
        self.objects, self.fo, self.co = stream(frames)

    def call(self, f0, n, capacity=None):
        import torch
        lo, hi = int(self.fo[f0]), int(self.fo[f0 + n])
        cap = hi - lo if capacity is None else capacity
        rows = max(cap, 1)              # the buffer holds `capacity` records, like the export's
        data = np.full(rows * 48, FILL, np.uint8)
        m = min(cap, hi - lo)
        data[:m * 48] = self.objects[lo:lo + m].view(np.uint8)
        ob = api.DeviceObjects(data=torch.from_numpy(data.view(np.int32).reshape(rows, 12)).cuda(),
                               frame_offsets=torch.from_numpy(self.fo[f0:f0 + n + 1] - lo).cuda(),
                               class_offsets=torch.from_numpy(self.co[8 * f0:8 * (f0 + n) + 1] - lo).cuda())
        return ob, cap, lo


def device_run(tracker, ds, calls, torch_stream=None):
    """calls = [(n, capacity or None, reset)] -> ids, hits (aligned with the stream, FILL where not written), flags."""
    import torch
    total, frames = len(ds.objects), len(ds.fo) - 1
    ids = np.full(max(total, 1) * 8, FILL, np.uint8)
    hits = np.full(max(total, 1) * 4, FILL, np.uint8)
    flags = np.zeros(frames, np.int32)
    f0 = 0
    for n, capacity, reset in calls:
        if reset:
            tracker.reset()
        ob, cap, lo = ds.call(f0, n, capacity)
        rows = ob.data.shape[0]
        d_ids = torch.full((rows * 8,), FILL, dtype=torch.uint8, device="cuda")
        d_hits = torch.full((rows * 4,), FILL, dtype=torch.uint8, device="cuda")
        d_flags = torch.full((n * 4,), FILL, dtype=torch.uint8, device="cuda")
        s = torch_stream or torch.cuda.current_stream()
        tracker._enqueue(s.cuda_stream, n, ob, d_ids, d_hits, d_flags)
        torch.cuda.synchronize()
        ends = ds.fo[f0 + 1:f0 + n + 1] - lo
        m = int(ends[ends <= cap].max(initial=0))   # objects of the written frames (fo[f+1] <= capacity)
        ids[lo * 8:(lo + m) * 8] = d_ids.cpu().numpy()[:m * 8]
        hits[lo * 4:(lo + m) * 4] = d_hits.cpu().numpy()[:m * 4]
        assert (d_ids.cpu().numpy()[m * 8:] == FILL).all() and (d_hits.cpu().numpy()[m * 4:] == FILL).all()
        flags[f0:f0 + n] = d_flags.cpu().numpy().view(np.int32)
        f0 += n
    return ids[:total * 8].view(np.int64), hits[:total * 4].view(np.int32), flags


def host_calls(calls, ds):
    out, f0 = [], 0
    for n, capacity, reset in calls:
        out.append((n, int(ds.fo[f0 + n] - ds.fo[f0]) if capacity is None else capacity, reset))
        f0 += n
    return out


def assert_same(dev, host, tracker):
    ids, hits, flags = dev
    assert np.array_equal(ids.view(np.uint8), host["ids"].view(np.uint8))
    assert np.array_equal(hits.view(np.uint8), host["hits"].view(np.uint8))
    assert np.array_equal(flags, host["flags"])
    state, next_id = tracker.state()
    assert next_id == host["next_id"]
    assert np.array_equal(state.view(np.uint8), host["state"].view(np.uint8))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_harness(tmp_path_factory.mktemp("tracker"))


@pytest.mark.gpu
@pytest.mark.parametrize("params", sorted(PARAMS))
def test_fuzz_streams_equal_the_host_definition(params, exe, tmp_path):
    p = PARAMS[params]
    frames = fuzz_frames(7 + len(params), 300, big=(40, 41, 42, 200))
    ds = DeviceStream(frames)
    # calls of 64, 7 and 1 frames; two of them with a capacity that ends inside a frame
    calls, f0 = [], 0
    for i, n in enumerate([64, 7, 1, 64, 64, 7, 1, 64, 28]):
        cap = None
        if i in (3, 6):
            lo = int(ds.fo[f0])
            cap = int(ds.fo[f0 + n // 2]) - lo + 1
        calls.append((n, cap, 0))
        f0 += n
    assert f0 == 300
    t = api.ObjectTracker(**p)
    dev = device_run(t, ds, calls)
    host = run_host(exe, tmp_path, ds.objects, ds.fo, host_calls(calls, ds), **p)
    assert_same(dev, host, t)
    # the streams cover what they are meant to
    per_class = np.diff(ds.co).reshape(-1, 8)
    assert per_class.max() > 256
    d = ds.objects[["disparity_min", "disparity_max"]]
    bits = np.concatenate([d["disparity_min"].view(np.uint32), d["disparity_max"].view(np.uint32)])
    assert (bits == 0x80000000).any() and ((bits > 0) & (bits < 0x800000)).any() and np.isnan(d["disparity_min"]).any()
    assert (host["flags"] & 2).sum() >= 2 and len(set(host["ids"][host["ids"] >= 0].tolist())) > 50
    if params == "tight":
        assert (host["flags"] & 1).any()
    print(f"{params}: {host['next_id']} ids, {len(host['state'])} live tracks")


@pytest.mark.gpu
def test_call_splits_reset_and_two_trackers(exe, tmp_path):
    frames = fuzz_frames(3, 128, big=(5,))
    ds = DeviceStream(frames)
    want = run_host(exe, tmp_path, ds.objects, ds.fo, [(128, len(ds.objects), 0)])
    for split in ([128], [1] * 128, [7] * 18 + [2], [64, 64]):
        t = api.ObjectTracker()
        assert_same(device_run(t, ds, [(n, None, 0) for n in split]), want, t)
    # reset restarts at id 0: the second pass gives the bytes of the first
    t = api.ObjectTracker()
    device_run(t, ds, [(64, None, 0), (64, None, 0)])
    again = device_run(t, ds, [(64, None, 1), (64, None, 0)])
    assert_same(again, want, t)
    # two trackers, updates interleaved on one stream, each on its own sequence
    other = fuzz_frames(4, 128)
    ds2 = DeviceStream(other)
    want2 = run_host(exe, tmp_path, ds2.objects, ds2.fo, [(128, len(ds2.objects), 0)])
    a, b = api.ObjectTracker(), api.ObjectTracker()
    got_a, got_b = [], []
    for f0 in range(0, 128, 32):
        got_a.append(device_run_slice(a, ds, f0, 32))
        got_b.append(device_run_slice(b, ds2, f0, 32))
    for got, w, t in ((got_a, want, a), (got_b, want2, b)):
        ids = np.concatenate([g[0] for g in got])
        hits = np.concatenate([g[1] for g in got])
        flags = np.concatenate([g[2] for g in got])
        assert_same((ids, hits, flags), w, t)


def device_run_slice(tracker, ds, f0, n):
    """One call of frames [f0, f0 + n) with all records written: ids, hits, flags of those frames."""
    import torch
    ob, cap, lo = ds.call(f0, n)
    ids, hits, flags = tracker.update(ob, n)
    torch.cuda.synchronize()
    return ids.cpu().numpy()[:cap], hits.cpu().numpy()[:cap], flags.cpu().numpy()


@pytest.mark.gpu
def test_calls_on_two_streams_are_applied_in_call_order(exe, tmp_path):
    import torch
    frames = fuzz_frames(5, 64)
    ds = DeviceStream(frames)
    want = run_host(exe, tmp_path, ds.objects, ds.fo, [(64, len(ds.objects), 0)])
    t = api.ObjectTracker()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    inputs = [ds.call(f0, 16) for f0 in range(0, 64, 16)]
    torch.cuda.synchronize()
    for i, (ob, cap, lo) in enumerate(inputs):
        s = s1 if i % 2 == 0 else s2
        with torch.cuda.stream(s):
            if i % 2 == 0:
                torch.cuda._sleep(50_000_000)   # s1 lags far behind s2: only the tracker's event orders the calls
            rows = ob.data.shape[0]
            o = (torch.full((rows,), -7, dtype=torch.int64, device="cuda"),
                 torch.full((rows,), -7, dtype=torch.int32, device="cuda"),
                 torch.full((16,), -7, dtype=torch.int32, device="cuda"))
            t._enqueue(s.cuda_stream, 16, ob, *o)
            outs.append((o, cap))
    torch.cuda.synchronize()
    ids = np.concatenate([o[0].cpu().numpy()[:cap] for o, cap in outs])
    hits = np.concatenate([o[1].cpu().numpy()[:cap] for o, cap in outs])
    flags = np.concatenate([o[2].cpu().numpy() for o, cap in outs])
    assert_same((ids, hits, flags), want, t)


@pytest.mark.gpu
def test_refusals_enqueue_nothing_and_leave_the_state_alone():
    import torch
    lib = L.load()
    ds = DeviceStream(fuzz_frames(9, 8))
    t = api.ObjectTracker()
    t.update(ds.call(0, 4)[0], 4)
    before = t.state()
    ob, cap, _ = ds.call(4, 4)
    rows = ob.data.shape[0]
    ids = torch.full((rows * 8 + 8,), FILL, dtype=torch.uint8, device="cuda")
    hits = torch.full((rows * 4,), FILL, dtype=torch.uint8, device="cuda")
    flags = torch.full((16,), FILL, dtype=torch.uint8, device="cuda")
    host_ids = np.zeros(rows, np.int64)
    torch.cuda.synchronize()

    def call(n=4, objects=ob.data.data_ptr(), fo=ob.frame_offsets.data_ptr(), co=ob.class_offsets.data_ptr(),
             capacity=cap, d_ids=ids.data_ptr(), d_hits=hits.data_ptr(), d_flags=flags.data_ptr()):
        d = L.DeviceObjects(objects or None, fo or None, co or None, None, capacity, 0)
        return lib.isx_tracker_update_device(t.handle(), torch.cuda.current_stream().cuda_stream, n, C.byref(d),
                                             d_ids or None, d_hits or None, d_flags or None)

    launches = lib.isx_kernel_launch_count()
    rcs = [call(n=0), call(n=4097), call(objects=0), call(fo=0), call(co=0), call(d_ids=0),
           call(objects=ob.data.data_ptr() + 8), call(d_ids=ids.data_ptr() + 4), call(d_hits=hits.data_ptr() + 2),
           call(d_flags=flags.data_ptr() + 1), call(capacity=-1), call(d_ids=host_ids.ctypes.data)]
    assert rcs == [-1] * len(rcs)
    assert lib.isx_kernel_launch_count() == launches
    torch.cuda.synchronize()
    assert all((x.cpu().numpy() == FILL).all() for x in (ids, hits, flags))
    after = t.state()
    assert after[1] == before[1] and np.array_equal(after[0].view(np.uint8), before[0].view(np.uint8))
    assert call() == 0   # the same arguments, accepted
    # parameters
    with pytest.raises(api.InvalidArgument):
        api.ObjectTracker(iou_min_permille=0)
    with pytest.raises(api.InvalidArgument):
        api.ObjectTracker(disparity_margin=float("nan"))
    with pytest.raises(api.StixelsError, match="-5"):
        api.ObjectTracker(max_tracks=1025)
    # tracker= without objects=True
    st = api.make_stixels(synth.preset("pairwise", 256, 512, 8), max_batch=1)
    d, s, r = synth.make_batch(1, rows=256, cols=512)
    with pytest.raises(api.InvalidArgument, match="objects=True"):
        st.ComputeBatchTensors(True, torch.from_numpy(d).cuda(), r, segmentation=torch.from_numpy(s).cuda(), tracker=t)
    st.Finish()


@pytest.mark.gpu
def test_destroy_with_updates_in_flight_is_clean():
    import torch
    ds = DeviceStream(dense_frames(np.random.default_rng(1), 64))
    ob, cap, _ = ds.call(0, 64)
    t = api.ObjectTracker()
    outs = [t.update(ob, 64) for _ in range(4)]
    del t                      # isx_tracker_destroy waits for the four updates
    torch.cuda.synchronize()
    assert all(int(o[0][:cap].min().item()) >= -1 for o in outs)
    t2 = api.ObjectTracker()
    ids, hits, flags = t2.update(ob, 64)
    assert int(ids[0].item()) == 0 and t2.state()[1] > 0


def dense_frames(rng, n, per_class=300):
    """n frames with `per_class` 10 x 10 boxes in every class, on a grid in one of three disjoint bands (frame f uses
    band f % 3), x jittered by a pixel: hundreds of objects per class, and with max_age 2 every track is matched every
    third frame, so about 900 tracks per class stay live (the benchmark's dense case)."""
    frames = []
    for f in range(n):
        objs = []
        for c in range(11, 19):
            for i in range(per_class):
                x = 12 * (i % 150) + int(rng.integers(-1, 2))
                y = 12 * (i // 150) + 24 * (f % 3) + 80 * (c - 11)
                objs.append((c, (x, y, x + 9, y + 9), 5.0, 6.0))
        frames.append(frame(*objs))
    return frames


# ---- end to end: a moving scene through ComputeBatchTensors(objects=True, tracker=) ----

@pytest.mark.gpu
def test_moving_scene_end_to_end_equals_the_host_chain(exe, tmp_path):
    import torch
    from test_gpu_objects import _build_harness as build_objects_harness, _host as host_objects
    rows, cols, w, B = 1024, 2048, 8, 6
    objects_exe = build_objects_harness(tmp_path)
    st = api.make_stixels(synth.preset("pairwise", rows, cols, w), max_batch=B)
    t = api.ObjectTracker()
    dev_ids, dev_hits, dev_flags, host_objects_all, host_fo = [], [], [], [], [0]
    for b in range(2):
        disp, seg, roads = synth.make_moving_batch(B, start=b * B, rows=rows, cols=cols, column_step=w)
        out = st.ComputeBatchTensors(True, torch.from_numpy(disp).cuda(), roads, segmentation=torch.from_numpy(seg).cuda(),
                                     objects=True, tracker=t)
        ob = out.objects
        total = int(ob.frame_offsets[B].item())
        dev_ids.append(ob.track_ids[:total].cpu().numpy())
        dev_hits.append(ob.track_hits[:total].cpu().numpy())
        dev_flags.append(ob.track_flags.cpu().numpy())
        # the host chain: ComputeBatch -> GetInstanceObjects -> HostObjectTracker
        sections, inst, offs = st.ComputeBatch(True, disp, seg, roads)
        h = host_objects(objects_exe, tmp_path, sections, inst, offs, rows, cols, w)
        assert np.array_equal(h["objects"].view(np.uint8), ob.data[:total].cpu().numpy().reshape(-1).view(np.uint8))
        host_objects_all.append(h["objects"])
        host_fo.extend((h["frame_offsets"][1:] + host_fo[-1]).tolist())
    objects = np.concatenate(host_objects_all)
    fo = np.array(host_fo, np.int32)
    host = run_host(exe, tmp_path, objects, fo, [(B, int(fo[B]), 0), (B, int(fo[2 * B] - fo[B]), 0)])
    assert_same((np.concatenate(dev_ids), np.concatenate(dev_hits), np.concatenate(dev_flags)), host, t)
    later = host["hits"][fo[1]:]
    continued = float((later > 1).mean())
    print(f"moving scene: {len(objects)} objects in {2 * B} frames, {host['next_id']} ids, "
          f"{continued:.3f} of the objects after the first frame continue a track")
    assert continued >= 0.9   # 1.000 observed on a B200 (60 objects in 12 frames)
    st.Finish()
