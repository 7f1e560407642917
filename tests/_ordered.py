"""Shared helpers for the Reduction.sum / mean / prod tests (csrc/dm_ordered.cu and the paths that reach it).

orth_project_ordered restates maps._orth_project_composed with the oracle's primitives, in the same order and with
the same point counts, so that the GPU's composed path can be compared with it bit for bit.  sum_bound_violations is
the plain float64 cross-check of a sum: it does not depend on the order of the hits, so it catches lost or
duplicated hits even where the oracle and the kernel could share an ordering mistake.
"""
import math

import numpy as np

from dungeon_maps_b200 import synth
from oracle import dm_oracle as orc

REDUCTIONS = ("sum", "mean", "prod")
HFOV = math.radians(70)
PITCH = math.radians(-10)
U32 = 2.0 ** -24  # unit roundoff of float32


def one_hot(label_map, num_classes):
  """(b, 1, h, w) integer class ids → (b, C, h, w) float32 planes; ids outside [0, C) give no plane."""
  ids = np.asarray(label_map).astype(np.int64)[:, 0]
  return (np.arange(num_classes).reshape(1, -1, 1, 1) == ids[:, None]).astype(np.float32)


def ordered_cells(depth, valid_map, cam_pose, width_offset, height_offset, cam_pitch, cam_height, map_res, map_height,
                  focal_x, focal_y, center_x, center_y, trunc_depth_min, trunc_depth_max, trunc_height_max, clip_border,
                  to_global, flip_h=True):
  """The points of maps._orth_project_composed up to the scatter: depth_to_points, border clip, camera → local
  (→ global) with the point count of the whole sample (it selects the rotation path, oracle.dm_oracle.fused_for),
  trunc_height_max on the local heights, map_quantize.  Returns coords (b, dc, H*W, 2) = [row, col], the local
  heights (b, dc, H*W) and the valid points (b, dc, H*W)."""
  depth = np.ascontiguousarray(depth, np.float32)
  b, dc, H, W = depth.shape
  Mh = int(map_height)
  pts, ok = orc.depth_to_points(depth, valid_map, focal_x, focal_y, center_x, center_y, flip_h, trunc_depth_min,
                                trunc_depth_max)                                            # (b, dc, H, W, 3)
  if clip_border is not None and clip_border > 0:
    k = int(clip_border)
    border = np.zeros((H, W), bool)
    border[k:H - k, k:W - k] = True
    ok = ok & border
  n = dc * H * W  # points per sample that each transform sees
  pts = pts.reshape(b, n, 3)
  pose = np.asarray(cam_pose, np.float32).reshape(-1, 3)
  if pose.shape[0] == 1 and b > 1:
    pose = np.repeat(pose, b, 0)
  pts = orc.transform_points(pts, [orc.to_local_steps(orc._vec(cam_pitch, b), orc._vec(cam_height, b), n)])
  ok = ok.reshape(b, n)
  if trunc_height_max is not None:
    ok = ok & (pts[..., 1] <= np.float32(trunc_height_max))
  if to_global:
    pts = orc.transform_points(pts, [orc.to_global_steps(pose, n)])
  xb, zb = orc.map_quantize(pts[..., 0], pts[..., 2], orc._vec(width_offset, b), orc._vec(height_offset, b), map_res,
                            Mh, flip_h)
  coords = np.stack((zb, xb), -1).reshape(b, dc, H * W, 2)
  return coords, pts[..., 1].reshape(b, dc, H * W), ok.reshape(b, dc, H * W)


def orth_project_ordered(depth, value_map, valid_map, cam_pose, width_offset, height_offset, cam_pitch, cam_height,
                         map_res, map_width, map_height, focal_x, focal_y, center_x, center_y, trunc_depth_min,
                         trunc_depth_max, trunc_height_max, clip_border, to_global, flip_h=True, fill_value=None,
                         reduction=None, get_height_map=False, label_map=None, num_classes=None):
  """orth_project for sum / mean / prod as maps._orth_project_composed computes it (maps.py:259-351): the points of
  ordered_cells, one ordered scatter of the values and one max scatter of the heights."""
  b, dc, H, W = np.shape(depth)
  Mh, Mw = int(map_height), int(map_width)
  if label_map is not None:
    value_map = one_hot(label_map, int(num_classes))
  coords, heights, flat_ok = ordered_cells(depth, valid_map, cam_pose, width_offset, height_offset, cam_pitch,
                                           cam_height, map_res, Mh, focal_x, focal_y, center_x, center_y,
                                           trunc_depth_min, trunc_depth_max, trunc_height_max, clip_border, to_global,
                                           flip_h)
  values = heights if value_map is None else np.asarray(value_map, np.float32).reshape(b, -1, H * W)
  canvas = np.zeros(values.shape[:-1] + (Mh, Mw), np.float32)
  top, mask = orc.scatter(values, coords, flat_ok, canvas, fill_value, reduction)
  if not get_height_map:
    return top, mask
  if value_map is None:
    return top, mask, top
  hgt, _ = orc.scatter(heights, coords, flat_ok, np.zeros((b, dc, Mh, Mw), np.float32), orc.NINF, None)
  return top, mask, np.broadcast_to(hgt, top.shape)


def sum_bound_violations(got, values, coords, valid, canvas):
  """Cells of a scatter-sum result `got` (B..., Mh, Mw) farther from the float64 sum than the a-priori bound of
  recursive float32 summation, |got - S| <= gamma_n * (|canvas| + sum |v_i|) with n = hits + 1 terms.  Order-free:
  it holds for any order of the hits, and fails where a hit is lost or counted twice.  Cells whose float64 sum is not
  finite are skipped.  Returns the number of violating cells."""
  got = np.asarray(got, np.float32)
  Mh, Mw = got.shape[-2:]
  M = Mh * Mw
  values = np.asarray(values, np.float32)
  rows = int(np.prod(values.shape[:-1]))
  N = values.shape[-1]
  coords = np.broadcast_to(coords, values.shape + (2,)).reshape(rows, N, 2)
  ok = np.ones((rows, N), bool) if valid is None else np.broadcast_to(valid, values.shape).reshape(rows, N).astype(bool)
  r, c = coords[..., 0], coords[..., 1]
  ok = ok & (r >= 0) & (r < Mh) & (c >= 0) & (c < Mw)
  key = (np.arange(rows).reshape(-1, 1) * M + np.where(ok, r * Mw + c, 0))[ok]
  v = values.reshape(rows, N)[ok].astype(np.float64)
  base = np.broadcast_to(canvas, values.shape[:-1] + (Mh, Mw)).reshape(-1).astype(np.float64)
  s = base + np.bincount(key, weights=v, minlength=rows * M)
  a = np.abs(base) + np.bincount(key, weights=np.abs(v), minlength=rows * M)
  n = np.bincount(key, minlength=rows * M) + 1.0
  gamma = n * U32 / (1.0 - n * U32)
  err = np.abs(got.reshape(-1).astype(np.float64) - s)
  fin = np.isfinite(s) & np.isfinite(a)
  return int(np.count_nonzero(fin & ~(err <= gamma * a)))


def fill_for(reduction, rng):
  """A fill value that suits the reduction: its neutral element, None (the caller's canvas), or an edge value."""
  neutral = 1.0 if reduction == "prod" else 0.0
  return [neutral, neutral, None, -np.inf, np.nan][int(rng.integers(0, 5))]


def special_values(shape, seed, lo=-3.0, hi=3.0, rate=0.0):
  """Uniform values in [lo, hi) with a fraction `rate` replaced by NaN, +-inf, -0.0 and 0.0."""
  v = synth.uniform(shape, seed, lo, hi).numpy()
  if rate > 0:
    rng = np.random.default_rng(seed)
    flat = v.reshape(-1)
    pick = rng.random(flat.size) < rate
    flat[pick] = rng.choice(np.asarray([np.nan, np.inf, -np.inf, -0.0, 0.0], np.float32), int(pick.sum()))
  return v


def scatter_case(seed, max_n=200_000):
  """A random project()/scatter case: batch shape, points, canvas size, out-of-range coordinates, masks, special
  values; reduction drawn from sum / mean / prod with a fill that suits it."""
  rng = np.random.default_rng(seed)
  batch = [(1,), (2,), (3, 2), (40,), (5,), (1, 7)][int(rng.integers(0, 6))]
  Mh, Mw = [(1, 1), (2, 3), (9, 11), (31, 33), (64, 64), (300, 300), (1, 257)][int(rng.integers(0, 7))]
  N = int(rng.integers(1, max_n // int(np.prod(batch)) + 2))
  red = REDUCTIONS[int(rng.integers(0, 3))]
  lo, hi = (0.5, 1.5) if red == "prod" else (-3.0, 3.0)  # products of many values stay finite and non-zero
  values = special_values(batch + (N,), seed + 1, lo, hi, rate=float(rng.choice([0.0, 0.0, 0.01])))
  rows = rng.integers(-2, Mh + 2, size=batch + (N,))
  cols = rng.integers(-2, Mw + 2, size=batch + (N,))
  coords = np.stack((rows, cols), -1).astype(np.int64)
  valid = rng.random(batch + (N,)) > 0.2 if rng.random() < 0.6 else None
  canvas = synth.uniform(batch + (Mh, Mw), seed + 2, -1.0, 1.0).numpy()
  return values, coords, valid, canvas, fill_for(red, rng), red


def orth_case(seed):
  """A random orth_project case for the composed path, modelled on test_gpu_parity._random_case."""
  rng = np.random.default_rng(seed)
  H = int(rng.integers(5, 60)); W = int(rng.integers(5, 80))
  b = int(rng.integers(1, 7))
  C = int(rng.choice([0, 1, 3, 16, 17, 40]))
  Mh = int(rng.integers(3, 70)); Mw = int(rng.integers(3, 70))
  red = REDUCTIONS[int(rng.integers(0, 3))]
  intr = orc.intrinsics(W, H, HFOV, None if rng.random() < 0.5 else math.radians(50))
  kw = dict(map_res=float(rng.choice([0.05, 0.1, 0.25, 0.5])), map_width=Mw, map_height=Mh, focal_x=intr["fx"],
            focal_y=intr["fy"], center_x=intr["cx"], center_y=intr["cy"],
            trunc_depth_min=None if rng.random() < 0.3 else 0.15,
            trunc_depth_max=None if rng.random() < 0.3 else 5.05,
            trunc_height_max=None if rng.random() < 0.6 else 1.2,
            clip_border=None if rng.random() < 0.3 else int(rng.integers(0, 4)),
            to_global=bool(rng.random() < 0.5), flip_h=bool(rng.random() < 0.7),
            fill_value=fill_for(red, rng), reduction=red, get_height_map=bool(rng.random() < 0.7))
  dc = 1
  if C == 0 and rng.random() < 0.3:
    dc = int(rng.integers(2, 4))  # several depth channels: one index set per channel
  depth = synth.iid_depth(b * dc, H, W, seed=seed).numpy().reshape(b, dc, H, W)
  if rng.random() < 0.3:
    depth.reshape(-1)[::13] = np.nan
  values, labels = None, None
  if C > 0:
    lo, hi = (0.5, 1.5) if red == "prod" else (-2.0, 2.0)
    if rng.random() < 0.3:
      labels = rng.integers(-2, C + 3, size=(b, 1, H, W)).astype(np.int64)  # some ids out of range: no plane
    elif rng.random() < 0.5:
      values = synth.block_onehot(b, C, H, W, seed=seed, block=3).numpy()
    else:
      values = synth.uniform((b, C, H, W), seed + 7, lo, hi).numpy()
  valid = (synth.uniform((b, 1, H, W), seed + 9).numpy() > 0.3) if rng.random() < 0.4 else None
  pose = synth.poses(b, seed).numpy()
  woff = (Mw / 2 + rng.normal(size=b)).astype(np.float32)
  hoff = rng.normal(size=b).astype(np.float32) + (Mh / 2 if kw["to_global"] else 0)
  pitch = np.full(b, PITCH, np.float32) + rng.normal(size=b).astype(np.float32) * 0.05
  camh = np.full(b, 0.88, np.float32)
  if labels is not None:
    kw.update(label_map=labels, num_classes=C)
  return depth, values, valid, pose, woff, hoff, pitch, camh, kw
