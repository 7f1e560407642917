"""The definition of geodesic_path, restated without the library: a plain-Python walk per start, and a certificate
that checks a path against the field without depending on the order in which ties are broken.

For start s of environment i, with D = dist[i] and T = traversable[i]: if s lies outside the map or D[s] < 0 the path
is empty.  Otherwise p_0 = s; while D[p_k] > 0 and k + 1 < max_cells, p_k+1 is the first neighbour q = p_k + (dx, dz)
in ORDER inside the map with D[q] >= 0, D[q] == D[p_k] - c (c = 5 orthogonal, 7 diagonal) and an edge q -> p_k under
geodesic_distance's rule.  The walk stops at D == 0, when no neighbour qualifies, or at max_cells cells."""
import numpy as np

from tests._geodesic import edge_ok

# (dx, dz, cost) in the order the definition tries the neighbours
ORDER = [(1, 0, 5), (0, 1, 5), (-1, 0, 5), (0, -1, 5), (1, 1, 7), (-1, 1, 7), (-1, -1, 7), (1, -1, 7)]


def walk(trav, dist, x, z, max_cells):
  """(H, W) bool and int32 grids, a start [x, z] -> the path as a list of (x, z)."""
  H, W = dist.shape
  if not (0 <= x < W and 0 <= z < H) or dist[z, x] < 0:
    return []
  path = [(x, z)]
  while dist[z, x] > 0 and len(path) < max_cells:
    d = int(dist[z, x])
    for dx, dz, c in ORDER:
      qx, qz = x + dx, z + dz
      # the edge q -> p: from (row qz, column qx) by (-dz, -dx)
      if 0 <= qx < W and 0 <= qz < H and dist[qz, qx] >= 0 and dist[qz, qx] == d - c and \
          edge_ok(trav, qz, qx, -dz, -dx):
        x, z = qx, qz
        path.append((x, z))
        break
    else:
      break
  return path


def oracle(trav, dist, starts, max_cells):
  """(b, H, W) bool, (b, H, W) int32, (b, n, 2) int [x, z] -> cells int32 (b, n, max_cells, 2), lengths int32 (b, n)."""
  b, n = starts.shape[:2]
  cells = np.full((b, n, max_cells, 2), -1, np.int32)
  lengths = np.zeros((b, n), np.int32)
  for i in range(b):
    for k in range(n):
      p = walk(trav[i], dist[i], int(starts[i, k, 0]), int(starts[i, k, 1]), max_cells)
      lengths[i, k] = len(p)
      if p:
        cells[i, k, :len(p)] = p
  return cells, lengths


def certificate(trav, dist, start, path) -> bool:
  """True iff `path` ((L, 2) [x, z], L >= 1) is a shortest path from `start` to a source of the field `dist` over
  `trav` ((H, W) each): it starts at `start`, consecutive cells are 8-neighbours, every step p_k -> p_k+1 runs along
  an edge p_k+1 -> p_k of geodesic_distance's graph, the step costs sum to D[start], and D is 0 at the last cell.
  Which of several equally short paths was taken does not matter."""
  H, W = dist.shape
  p = np.asarray(path, np.int64).reshape(-1, 2)
  if len(p) == 0 or tuple(p[0]) != tuple(start):
    return False
  x, z = p[:, 0], p[:, 1]
  if (x < 0).any() or (x >= W).any() or (z < 0).any() or (z >= H).any():
    return False
  step = np.diff(p, axis=0)
  ax, az = np.abs(step[:, 0]), np.abs(step[:, 1])
  if (ax > 1).any() or (az > 1).any() or ((ax == 0) & (az == 0)).any():
    return False
  diag = (ax == 1) & (az == 1)
  # edge q -> p_k with q = p_k+1: T[p_k], and for a diagonal step T[(q.x, p_k.z)] and T[(p_k.x, q.z)]
  ok = trav[z[:-1], x[:-1]] & (~diag | (trav[z[:-1], x[1:]] & trav[z[1:], x[:-1]]))
  cost = np.where(diag, 7, 5).sum()
  return bool(ok.all() and cost == int(dist[z[0], x[0]]) and dist[z[-1], x[-1]] == 0)
