"""numpy oracle of visible_cells / count_visible (dm_line_of_sight_u8): the definition in the maps.py docstring, one
origin at a time, vectorised over the targets of its window, one loop iteration per line step i.

For origin o and target t = o + (dx, dz), with ax = |dx|, az = |dz|, m = max(ax, az): the line is
p_i = (ox + sx * i, oz + sz * floor((2 * i * az + m) / (2 * m))) for ax >= az, the axes swapped otherwise.  t is visible
when dx^2 + dz^2 <= r^2, t is inside the map, no p_i with 0 < i < m blocks, and no diagonal step p_i -> p_i+1 has both
side cells (x_i+1, z_i) and (x_i, z_i+1) blocking."""
import numpy as np


def visible_window(block, ox, oz, r):
  """(2r+1, 2r+1) bool: window[r + dz, r + dx] is True iff (ox + dx, oz + dz) is visible from (ox, oz) on the (H, W)
  bool map `block`."""
  H, W = block.shape
  side = 2 * r + 1
  out = np.zeros((side, side), bool)
  if not (0 <= ox < W and 0 <= oz < H):
    return out
  dz, dx = np.mgrid[-r:r + 1, -r:r + 1]
  cand = (dx * dx + dz * dz <= r * r) & (ox + dx >= 0) & (ox + dx < W) & (oz + dz >= 0) & (oz + dz < H)
  rows, cols = np.nonzero(cand)
  dx, dz = dx[rows, cols].astype(np.int64), dz[rows, cols].astype(np.int64)
  ax, az = np.abs(dx), np.abs(dz)
  m, mn = np.maximum(ax, az), np.minimum(ax, az)
  sx, sz = np.where(dx < 0, -1, 1), np.where(dz < 0, -1, 1)
  xmajor = ax >= az
  ok = np.ones(len(dx), bool)
  px, pz = np.full(len(dx), ox, np.int64), np.full(len(dx), oz, np.int64)
  alive = np.nonzero(m >= 1)[0]        # targets whose line still has steps to check
  for i in range(1, r + 1):
    alive = alive[(m[alive] >= i) & ok[alive]]
    if len(alive) == 0:
      break
    a_m = m[alive]
    q = (2 * i * mn[alive] + a_m) // (2 * a_m)
    cx = ox + np.where(xmajor[alive], sx[alive] * i, sx[alive] * q)
    cz = oz + np.where(xmajor[alive], sz[alive] * q, sz[alive] * i)
    x0, z0 = px[alive], pz[alive]
    diag = (cx != x0) & (cz != z0)
    leak = diag & block[z0, cx] & block[cz, x0]    # side cells lie in the box of o and t: inside the map
    mid = (i < a_m) & block[cz, cx]
    ok[alive] &= ~(leak | mid)
    px[alive], pz[alive] = cx, cz
  out[rows, cols] = ok
  return out


def visible_cells(blocking, origins, r):
  """blocking (b, H, W) bool, origins (b, n, 2) int [x, z] -> (b, n, 2r+1, 2r+1) bool."""
  b, n = origins.shape[:2]
  side = 2 * r + 1
  out = np.zeros((b, n, side, side), bool)
  for i in range(b):
    for k in range(n):
      out[i, k] = visible_window(blocking[i], int(origins[i, k, 0]), int(origins[i, k, 1]), r)
  return out


def target_windows(targets, origins, r):
  """targets (b, C, H, W) bool, origins (b, n, 2) -> (b, C, n, 2r+1, 2r+1): the target cells under each window, False
  outside the map."""
  b, C, H, W = targets.shape
  n = origins.shape[1]
  side = 2 * r + 1
  pad = np.zeros((b, C, H + 2 * side, W + 2 * side), bool)
  pad[:, :, side:side + H, side:side + W] = targets
  out = np.zeros((b, C, n, side, side), bool)
  for i in range(b):
    for k in range(n):
      x, z = int(origins[i, k, 0]), int(origins[i, k, 1])
      if -side <= x - r and x + r < W + side and -side <= z - r and z + r < H + side:
        out[i, :, k] = pad[i, :, z - r + side:z + r + 1 + side, x - r + side:x + r + 1 + side]
  return out


def count_visible(blocking, targets, origins, r):
  """blocking (b, H, W), targets (b, C, H, W), origins (b, n, 2) -> int32 (b, C, n)."""
  vis = visible_cells(blocking, origins, r)
  return (vis[:, None] & target_windows(targets, origins, r)).sum(axis=(3, 4)).astype(np.int32)
