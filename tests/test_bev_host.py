"""The bird's-eye-view grid definition (Stixels::GetBevGrid in include/InstanceStixels/Stixels.hpp) against a numpy
float32 statement of it on hand-made frames, through tests/cpp/bev_harness.cpp.  No device."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

from instance_stixels_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GROUND, OBJECT, SKY = 0, 1, 2
ROAD_DTYPE = np.dtype([("alpha_ground", "<f4"), ("vhor", "<i4")])
f32 = np.float32


def build_harness(tmp_path):
    exe = str(tmp_path / "bev_harness")
    libdir = os.path.join(ROOT, "instance_stixels_b200")
    cmd = ["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-I" + os.path.join(ROOT, "include", "InstanceStixels"),
           os.path.join(ROOT, "tests", "cpp", "bev_harness.cpp"), "-L" + libdir, "-linstance_stixels_b200",
           "-Wl,-rpath," + libdir, "-o", exe]
    subprocess.run(cmd, check=True, capture_output=True, text=True)
    return exe


def _arg(x):
    return repr(float(f32(x)))


def run_host(exe, tmp_path, sections, roads, rows, w, cam, grid):
    """GetBevGrid of the header over the frames: int32 [n][nz][nx][2] cells, or the refusal text."""
    n, realcols = sections.shape[0], sections.shape[1]
    np.ascontiguousarray(sections).tofile(tmp_path / "s.bin")
    np.ascontiguousarray(roads, dtype=ROAD_DTYPE).tofile(tmp_path / "r.bin")
    p = subprocess.run([exe, str(tmp_path / "s.bin"), str(tmp_path / "r.bin"), str(n), str(rows), str(realcols),
                        str(w), _arg(cam["focal"]), _arg(cam["baseline"]), _arg(cam["cx"]), _arg(cam["cy"]),
                        _arg(grid["x_min"]), _arg(grid["z_min"]), _arg(grid["cell"]), str(grid["nx"]),
                        str(grid["nz"]), str(tmp_path / "cells.bin")], capture_output=True, text=True)
    assert p.returncode == 0, p.stdout + p.stderr
    if p.stdout.startswith("refused"):
        return p.stdout
    return np.fromfile(tmp_path / "cells.bin", dtype=np.int32).reshape(n, grid["nz"], grid["nx"], 2)


def restate(sections, roads, rows, w, cam, grid):
    """The definition in numpy float32, one rounding per operation.  Returns the cells [n][nz][nx][2] and, per cell,
    why it has its state (occupied, zc, fov, below, above, column, object, sky, ground) plus the occupancy candidates."""
    n, realcols = sections.shape[0], sections.shape[1]
    nx, nz = grid["nx"], grid["nz"]
    x_min, z_min, cell = f32(grid["x_min"]), f32(grid["z_min"]), f32(grid["cell"])
    focal, cx = f32(cam["focal"]), f32(cam["cx"])
    bf = f32(cam["baseline"]) * focal
    cells = np.zeros((n, nz, nx, 2), np.int32)
    cells[..., 0] = -1
    why = np.empty((n, nz, nx), object)
    cand = [dict() for _ in range(n)]
    for f in range(n):
        alpha, vhor = f32(roads[f]["alpha_ground"]), int(roads[f]["vhor"])
        best = {}
        i = 0
        for col in range(realcols):
            for j in range(sections.shape[2]):
                s = sections[f, col, j]
                if s["type"] == -1:
                    break
                if s["type"] == OBJECT:
                    z = bf / f32(s["disparity"])
                    q = -z / focal
                    xl = f32(col * w)
                    xr = xl + f32(w)
                    vl, vr = q * (cx - xl), q * (cx - xr)
                    a = (z - z_min) / cell
                    if a >= 0 and a < nz:
                        l, r = (vl - x_min) / cell, (vr - x_min) / cell
                        if r >= 0 and l < nx:
                            for ix in range(0 if l < 0 else int(l), (nx - 1 if r >= nx else int(r)) + 1):
                                k = (int(a), ix)
                                cand[f].setdefault(k, []).append((i, z, col, float(l), float(r)))
                                if k not in best or z < best[k][1]:
                                    best[k] = (i, z)
                i += 1
        for iz in range(nz):
            for ix in range(nx):
                if (iz, ix) in best:
                    cells[f, iz, ix] = (best[(iz, ix)][0], 2)
                    why[f, iz, ix] = "occupied"
                    continue
                xc = x_min + (f32(ix) + f32(0.5)) * cell
                zc = z_min + (f32(iz) + f32(0.5)) * cell
                if not zc > 0:
                    why[f, iz, ix] = "zc"
                    continue
                u = cx + focal * (xc / zc)
                if not (u >= 0 and u < realcols * w):
                    why[f, iz, ix] = "fov"
                    continue
                c = int(u) // w
                t = bf / (alpha * zc)
                vf = f32(vhor) - t
                if not (t > 0 and vf >= 0 and vf < rows):
                    why[f, iz, ix] = "below" if t > 0 and vf < 0 else ("above" if t > 0 and vf >= rows else "road")
                    continue
                v = int(vf)
                hit = next((s for s in sections[f, c] if s["type"] == -1 or s["vB"] <= v), None)
                if hit is None or hit["type"] == -1 or v > hit["vT"]:
                    why[f, iz, ix] = "column"
                elif hit["type"] == GROUND:
                    cells[f, iz, ix, 1] = 1
                    why[f, iz, ix] = "ground"
                else:
                    why[f, iz, ix] = "object" if hit["type"] == OBJECT else "sky"
    return cells, why, cand


def empty_sections(n, realcols):
    sec = np.zeros((n, realcols, 200), dtype=L.SECTION_DTYPE)
    sec["type"] = -1
    return sec


def put(sec, f, col, stixels):
    """stixels top to bottom: (type, vB, vT, disparity)."""
    for j, (t, vB, vT, dis) in enumerate(stixels):
        sec[f, col, j] = (t, vB, vT, dis, 13 if t == OBJECT else (0 if t == GROUND else 10), 0.0, 0.0, 0.0)


def small_frames():
    """Three 64 x 64 frames, width 8, with the same stixels and three roads: alpha 0.5 (horizon row 40), 0 and -0.5.
    Column 0 and 7: objects at z = 15 reaching past the grid's left / right edge.  Columns 3 and 4: objects at z = 5
    whose corners meet on the cell edge x = 0 (equal z: the lower index wins).  Column 5: two objects in one cell row
    (z = 5.2 above z = 5.0: the nearer one wins).  Column 6: a NaN-disparity object, one at infinite depth and one past
    the far edge.  Column 1: sky from row 30 down to the ground.  Every column ends with ground."""
    rows, w, realcols = 64, 8, 8
    sec = empty_sections(3, realcols)
    for f in range(3):
        put(sec, f, 0, [(SKY, 46, 63, 0.0), (OBJECT, 30, 45, 50.0 / 15.0), (GROUND, 0, 29, 0.0)])
        put(sec, f, 1, [(SKY, 30, 63, 0.0), (GROUND, 0, 29, 0.0)])
        put(sec, f, 2, [(SKY, 50, 63, 0.0), (GROUND, 0, 49, 0.0)])
        put(sec, f, 3, [(SKY, 46, 63, 0.0), (OBJECT, 30, 45, 10.0), (GROUND, 0, 29, 0.0)])
        put(sec, f, 4, [(SKY, 46, 63, 0.0), (OBJECT, 30, 45, 10.0), (GROUND, 0, 29, 0.0)])
        put(sec, f, 5, [(SKY, 50, 63, 0.0), (OBJECT, 40, 49, float(f32(50.0) / f32(5.2))), (OBJECT, 32, 39, 10.0),
                        (GROUND, 0, 31, 0.0)])
        put(sec, f, 6, [(SKY, 54, 63, 0.0), (OBJECT, 48, 53, float("nan")), (OBJECT, 44, 47, 0.0),
                        (OBJECT, 40, 43, 1.0), (GROUND, 0, 39, 0.0)])
        put(sec, f, 7, [(SKY, 46, 63, 0.0), (OBJECT, 30, 45, 50.0 / 15.0), (GROUND, 0, 29, 0.0)])
    roads = np.array([(0.5, 40), (0.0, 40), (-0.5, 40)], dtype=ROAD_DTYPE)
    return sec, roads, rows, w


CAM = dict(focal=100.0, baseline=0.5, cx=32.0, cy=30.0)
GRID = dict(x_min=-4.0, z_min=0.0, cell=0.5, nx=16, nz=40)


def check(exe, tmp_path, sec, roads, rows, w, cam, grid):
    got = run_host(exe, tmp_path, sec, roads, rows, w, cam, grid)
    with np.errstate(all="ignore"):     # divisions by 0, NaN and inf disparities are part of the cases
        want, why, cand = restate(sec, roads, rows, w, cam, grid)
    assert isinstance(got, np.ndarray), got
    assert np.array_equal(got, want)
    return got, why, cand


def test_header_grid_equals_a_numpy_statement(tmp_path):
    exe = build_harness(tmp_path)
    sec, roads, rows, w = small_frames()
    got, why, cand = check(exe, tmp_path, sec, roads, rows, w, CAM, GRID)
    occ = got[..., 1] == 2
    # objects occupy the same cells whatever the road; the states are all three and nothing else
    assert (occ == occ[0]).all() and set(np.unique(got[..., 1])) == {0, 1, 2}
    assert ((got[..., 0] >= 0) == occ).all()
    c0 = cand[0]
    # stixels straddling cell edges and the grid's left and right edges
    spans = [(e[2], e[3], e[4]) for v in c0.values() for e in v]
    assert any(col == 0 and l < 0 for col, l, r in spans) and any(col == 7 and r >= 16 for col, l, r in spans)
    assert any(col == 3 and r == 8.0 for col, l, r in spans)
    # two occupants in one cell: equal z goes to the lower index, else the nearer one wins
    ties = [v for v in c0.values() if len(v) >= 2 and len({e[1] for e in v}) < len(v)]
    nearer = [v for v in c0.values() if len({e[1] for e in v}) >= 2]
    assert ties and nearer
    for (iz, ix), v in c0.items():
        assert got[0, iz, ix, 0] == min(v, key=lambda e: (e[1], e[0]))[0]
    assert any(got[0, iz, ix, 0] != min(e[0] for e in v) for (iz, ix), v in c0.items())
    # the NaN, infinite-depth and far objects of column 6 occupy nothing
    i6 = [int(sum((sec[0, c]["type"] != -1).sum() for c in range(6))) + j for j in (1, 2, 3)]
    assert not np.isin(got[0, ..., 0], i6).any()
    # frame 0: visible ground is free; ground behind an object, sky, outside the field of view and below the image
    # are unknown
    for reason in ("ground", "object", "sky", "fov", "below"):
        assert (why[0] == reason).any(), reason
    assert ((why[0] == "ground") == (got[0, ..., 1] == 1)).all()
    # alpha_ground 0 and negative: nothing is free
    assert (got[1:, ..., 1] != 1).all()


def test_header_grid_with_a_negative_z_min_and_a_fine_grid(tmp_path):
    exe = build_harness(tmp_path)
    sec, roads, rows, w = small_frames()
    got, why, _ = check(exe, tmp_path, sec, roads, rows, w, CAM, dict(x_min=-3.3, z_min=-2.0, cell=0.05, nx=140,
                                                                       nz=400))
    assert (why[0] == "zc").any() and (got[0, ..., 1] == 1).any() and (got[0, ..., 1] == 2).any()


def tall_frames(rng, n, rows, realcols):
    """Random well-formed columns: ground, then up to three objects (some NaN or zero disparity), then sky."""
    sec = empty_sections(n, realcols)
    for f in range(n):
        for col in range(realcols):
            cuts = sorted(rng.choice(np.arange(1, rows - 1), size=int(rng.integers(1, 5)), replace=False))
            bounds = [0] + list(cuts) + [rows]
            st = []
            for k in range(len(bounds) - 1):
                vB, vT = bounds[k], bounds[k + 1] - 1
                t = GROUND if k == 0 else (SKY if k == len(bounds) - 2 and k > 1 else OBJECT)
                d = float(rng.choice([rng.uniform(0.5, 60.0), np.nan, 0.0], p=[0.9, 0.05, 0.05]))
                st.append((t, vB, vT, d if t == OBJECT else 0.0))
            put(sec, f, col, st[::-1])
    return sec


def test_header_grid_with_width_4_a_width_margin_and_1208_rows(tmp_path):
    exe = build_harness(tmp_path)
    rng = np.random.default_rng(7)
    rows, w, realcols, cols = 1208, 4, 40, 164   # width margin: 4 columns of pixels without stixels
    sec = tall_frames(rng, 2, rows, realcols)
    roads = np.array([(0.177, 700), (0.2, 650)], dtype=ROAD_DTYPE)
    cam = dict(focal=200.0, baseline=0.2, cx=cols / 2.0, cy=600.0)
    got, why, _ = check(exe, tmp_path, sec, roads, rows, w, cam, dict(x_min=-10.0, z_min=0.0, cell=0.1, nx=200,
                                                                       nz=300))
    for reason in ("ground", "object", "fov", "below", "occupied"):
        assert (why == reason).any(), reason
    # centres that project into the margin (realcols * w <= u < cols) are outside the field of view
    x = f32(-10.0) + (np.arange(200, dtype=f32) + f32(0.5)) * f32(0.1)
    z = (np.arange(300, dtype=f32) + f32(0.5)) * f32(0.1)
    u = f32(cam["cx"]) + f32(200.0) * (x[None, :] / z[:, None])
    margin = (u >= realcols * w) & (u < cols)
    assert margin.any() and (why[0][margin & (got[0, ..., 1] != 2)] == "fov").all()


def test_header_refuses_without_camera_centre_or_with_bad_parameters(tmp_path):
    exe = build_harness(tmp_path)
    sec, roads, rows, w = small_frames()
    out = run_host(exe, tmp_path, sec, roads, rows, w, dict(CAM, cx=-1.0, cy=-1.0), GRID)
    assert out.startswith("refused: Camera parameters are not set.")
    for bad in (dict(cell=0.0), dict(cell=float("inf")), dict(cell=2e3), dict(nx=0), dict(nz=4097),
                dict(x_min=float("nan")), dict(z_min=-2e5)):
        assert run_host(exe, tmp_path, sec, roads, rows, w, CAM, dict(GRID, **bad)).startswith("refused"), bad


def test_bev_structs_and_defaults():
    assert C.sizeof(L.BevParams) == 24 and C.sizeof(L.BevCell) == 8
    p = L.BevParams()
    L.load().isx_bev_params_init(C.byref(p))
    assert (p.x_min, p.z_min, p.nx, p.nz, p.reserved) == (-20.0, 0.0, 200, 300, 0) and p.cell == f32(0.2)
    from instance_stixels_b200 import api
    q = api.BevParams(cell=0.05, nx=800, nz=1200)
    assert (q.x_min, q.nx, q.nz) == (-20.0, 800, 1200) and q.cell == f32(0.05)
    try:
        api.BevParams(size=3)
    except api.InvalidArgument:
        pass
    else:
        raise AssertionError("unknown field accepted")


def test_bev_bench_help_runs_without_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bev_bench.py"), "--help"],
                       capture_output=True, text=True, cwd=ROOT)
    assert p.returncode == 0 and "--steps" in p.stdout
