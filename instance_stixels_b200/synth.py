"""Deterministic synthetic Cityscapes-shaped frames and the reference's parameter presets.

The CNN, its weights and the dataset are not available offline, so every test
and benchmark feeds the hot path with frames built here (SURVEY.md 8d).  The
same bytes go to the CUDA product, the CPU oracle and the reference build.

Input formats (what `Stixels::SetDisparityImage` / `SetSegmentation` take):
  * disparity  float32 [H][W], top-left origin, values in [0, max_dis)
    (apps/run_cityscapes.cu:109-152); `invalid_disparity` (0) marks holes.
  * segmentation int32 [C][19+2][Hs2], C = W / column_step, rows bottom-up and
    zero padded from H/8 to Hs2 = 2**ceil(log2(H/8+1)); channels 0..18 =
    trunc(8 * -log_softmax), 19 = y-offset, 20 = x-offset in pixels
    (tools/CNN_training/models/wrappers.py:35-61, kernel indexing
    InstanceStixels/src/StixelsKernels.cu:393-405).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

SEED0 = 0x5717E1
N_CLASSES = 19
N_OFFSETS = 2
ROAD, SIDEWALK, SKY_CLASS = 0, 1, 10
OBJECT_CLASSES = [2, 3, 4, 5, 6, 7, 8, 9, 11, 12, 13, 14, 15, 16, 17, 18]

# Cityscapes-like camera / road scalars (types.h:78-82 comments; SURVEY.md 8d).
CAMERA = dict(focal=2262.52, baseline=0.209313, camera_center_x=1024.0, camera_center_y=512.0)
ROAD_PARAMS = dict(vhor=400, camera_tilt=0.0, camera_height=1.18, alpha_ground=0.209313 / 1.18)

# cfg/drn_d_22_unary_cfg.yaml (unrounded: apps/stixels_wrapper.cu:35-40)
UNARY_PRESET = dict(
    pairwise=False, prior_weight=1e4, segmentation_weight=11.241965032069425,
    instance_weight=0.0017313017435431333, disparity_weight=0.0069935800364145494,
    eps=23.89408062110343, min_pts=4, size_filter=42,
)
# cfg/drn_d_38_pairwise_cfg.yaml (unrounded: tests/run_test.sh:84-87)
PAIRWISE_PRESET = dict(
    pairwise=True, prior_weight=1.0, segmentation_weight=4.709500548254913,
    instance_weight=0.0031312903639774976, disparity_weight=0.0001,
    eps=18.82232269133926, min_pts=3, size_filter=25,
)
# both YAMLs: pground = pobject = psky = 0.33 (the struct default is 1/3)
COMMON_PRESET = dict(pground=0.33, pobject=0.33, psky=0.33, invalid_disparity=0.0, max_dis=128,
                     n_semantic_classes=N_CLASSES, n_offset_channels=N_OFFSETS)


def rows_power2_segmentation(rows: int) -> int:
    """Stixels.cu:132-133."""
    return 2 ** math.ceil(math.log2(rows // 8 + 1))


@dataclass
class Frame:
    disparity: np.ndarray      # float32 [H][W]
    segmentation: np.ndarray   # int32 [C][21][Hs2]
    road: dict                 # SetRoadParameters arguments


def make_frame(index: int, rows: int = 1024, cols: int = 2048, column_step: int = 8,
               max_dis: int = 128, vhor: int | None = None) -> Frame:
    """Frame `index` of the synthetic stream (seed = SEED0 + index)."""
    rng = np.random.Generator(np.random.PCG64(SEED0 + index))
    vhor, alpha = _horizon(rows, vhor)
    return _render(rng, _rectangles(rng, rows, cols, vhor), rows, cols, column_step, max_dis, vhor, alpha)


def make_moving_batch(n: int, start: int = 0, rows: int = 1024, cols: int = 2048, column_step: int = 8,
                      max_dis: int = 128, seed: int = 0):
    """A moving scene: the rectangles of scene `seed`, each shifted sideways by its own 1..4 pixels per frame (bouncing
    off the image borders), over the same road.  Frames start..start+n-1 as make_batch returns them; the noise and the
    CNN output of frame i are drawn afresh (seed and i)."""
    rng = np.random.Generator(np.random.PCG64([SEED0, seed]))
    vhor, alpha = _horizon(rows, None)
    rects = _rectangles(rng, rows, cols, vhor)
    speed = rng.integers(1, 5, size=len(rects)) * rng.choice([-1, 1], size=len(rects))
    frames = []
    for i in range(start, start + n):
        moved = []
        for (base, top, x0, rw, c), v in zip(rects, speed):
            span = cols - rw
            x = (x0 + i * int(v)) % (2 * span)          # bounce between 0 and cols - rw
            moved.append((base, top, x if x <= span else 2 * span - x, rw, c))
        frame_rng = np.random.Generator(np.random.PCG64([SEED0, seed, i]))
        frames.append(_render(frame_rng, moved, rows, cols, column_step, max_dis, vhor, alpha))
    return (np.stack([f.disparity for f in frames]), np.stack([f.segmentation for f in frames]),
            [f.road for f in frames])


def _horizon(rows: int, vhor: int | None):
    if vhor is None:
        vhor = int(round(ROAD_PARAMS["vhor"] * rows / 1024.0))
    alpha = ROAD_PARAMS["alpha_ground"] * 1024.0 / rows  # keep bottom-row disparity ~110 < max_dis - epsilon
    return vhor, alpha


def _rectangles(rng, rows: int, cols: int, vhor: int):
    """6..14 object rectangles (base row, top row, x0, width, class)."""
    H, W = rows, cols
    n_rect = int(rng.integers(6, 15))
    rects = []
    for _ in range(n_rect):
        rw = int(rng.integers(max(8, 40 * W // 2048), max(9, 400 * W // 2048) + 1))
        rh = int(rng.integers(max(8, 60 * H // 1024), max(9, 500 * H // 1024) + 1))
        x0 = int(rng.integers(0, W - rw))
        base = int(rng.integers(vhor + max(2, 20 * H // 1024), H))  # image row of the base
        top = max(0, base - rh)
        c = int(OBJECT_CLASSES[int(rng.integers(0, len(OBJECT_CLASSES)))])
        rects.append((base, top, x0, rw, c))
    return rects


def _render(rng, rects, rows: int, cols: int, column_step: int, max_dis: int, vhor: int, alpha: float) -> Frame:
    H, W, w = rows, cols, column_step
    Hs, C = H // 8, W // w
    Hs2 = rows_power2_segmentation(H)

    y = np.arange(H, dtype=np.float32)[:, None]
    disp = np.where(y > vhor, alpha * (y - vhor), 0.0).astype(np.float32)
    disp = np.broadcast_to(disp, (H, W)).copy()
    # class / instance-centre maps at full resolution, downsampled below
    cls = np.where(np.arange(H)[:, None] > vhor, ROAD, SKY_CLASS).astype(np.int32)
    cls = np.broadcast_to(cls, (H, W)).copy()
    x_idx = np.arange(W)
    cls[:, (x_idx < W // 6) | (x_idx >= W - W // 6)] = np.where(
        np.arange(H)[:, None] > vhor, SIDEWALK, SKY_CLASS)
    cx = np.full((H, W), np.nan, dtype=np.float32)
    cy = np.full((H, W), np.nan, dtype=np.float32)

    # far objects first so nearer ones (larger base row) occlude them
    for base, top, x0, rw, c in sorted(rects):
        d = alpha * (base - vhor)
        disp[top:base + 1, x0:x0 + rw] = d
        cls[top:base + 1, x0:x0 + rw] = c
        if c >= 11:
            cx[top:base + 1, x0:x0 + rw] = x0 + 0.5 * (rw - 1)
            cy[top:base + 1, x0:x0 + rw] = 0.5 * (top + base)
        else:
            cx[top:base + 1, x0:x0 + rw] = np.nan
            cy[top:base + 1, x0:x0 + rw] = np.nan

    disp += rng.normal(0.0, 0.5, size=(H, W)).astype(np.float32)
    disp[rng.random(size=(H, W)) < 0.05] = 0.0
    np.clip(disp, 0.0, max_dis - 0.5, out=disp)
    disp = disp.astype(np.float32)

    # ---- CNN-like output at 1/8 vertical resolution, one column per stixel ----
    ys = np.arange(Hs) * 8 + 4
    xs = np.arange(C) * w + w // 2
    cls_s = cls[np.ix_(ys, xs)]                  # [Hs][C]
    logits = rng.normal(0.0, 1.0, size=(Hs, C, N_CLASSES)).astype(np.float32)
    np.put_along_axis(logits, cls_s[..., None], np.take_along_axis(logits, cls_s[..., None], 2) + 4.0, 2)
    m = logits.max(axis=2, keepdims=True)
    lse = m + np.log(np.exp(logits - m).sum(axis=2, keepdims=True))
    nlogp = np.trunc(8.0 * (lse - logits)).astype(np.int32)       # >= 0
    offx = np.rint(rng.normal(0.0, 2.0, size=(Hs, C))).astype(np.int32)
    offy = np.rint(rng.normal(0.0, 2.0, size=(Hs, C))).astype(np.int32)
    cx_s, cy_s = cx[np.ix_(ys, xs)], cy[np.ix_(ys, xs)]
    inst = ~np.isnan(cx_s)
    offx[inst] = np.rint(cx_s[inst] - np.broadcast_to(xs[None, :], (Hs, C))[inst]).astype(np.int32)
    offy[inst] = np.rint(cy_s[inst] - np.broadcast_to(ys[:, None], (Hs, C))[inst]).astype(np.int32)
    np.clip(offx, -400, 400, out=offx)
    np.clip(offy, -400, 400, out=offy)

    seg = np.zeros((C, N_CLASSES + N_OFFSETS, Hs2), dtype=np.int32)
    # flip rows: index 0 = bottom of the image
    seg[:, :N_CLASSES, :Hs] = nlogp[::-1].transpose(1, 2, 0)
    seg[:, N_CLASSES, :Hs] = offy[::-1].T
    seg[:, N_CLASSES + 1, :Hs] = offx[::-1].T

    road = dict(vhor=vhor, camera_tilt=ROAD_PARAMS["camera_tilt"],
                camera_height=ROAD_PARAMS["camera_height"], alpha_ground=float(np.float32(alpha)))
    return Frame(np.ascontiguousarray(disp), np.ascontiguousarray(seg), road)


def make_batch(n: int, start: int = 0, **kw):
    """(disparity [n][H][W], segmentation [n][C][21][Hs2], roads list) for frames start..start+n-1."""
    frames = [make_frame(start + i, **kw) for i in range(n)]
    return (np.stack([f.disparity for f in frames]), np.stack([f.segmentation for f in frames]),
            [f.road for f in frames])


def preset(name: str, rows: int = 1024, cols: int = 2048, column_step: int = 8) -> dict:
    """Full StixelConfig field dict for 'unary' (drn_d_22) or 'pairwise' (drn_d_38)."""
    base = dict(UNARY_PRESET if name == "unary" else PAIRWISE_PRESET)
    base.update(COMMON_PRESET)
    base.update(CAMERA)
    base.update(rows=float(rows), cols=float(cols), column_step=column_step)
    return base
