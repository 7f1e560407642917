"""The definition of geodesic_distance, restated without the library: a plain-Python heapq Dijkstra for small grids,
and a vectorised certificate that proves a distance field exact at any size.

Graph: the cells of an H x W grid.  An edge runs from u to an 8-neighbour v when T[v] holds and the step is orthogonal,
or diagonal with both cells that share an edge with u and with v traversable.  Orthogonal steps cost 5, diagonal ones 7.
dist = 0 on sources, else the least path cost from a source, -1 without a path."""
import heapq

import numpy as np

# (dr, dc, cost) of a step u -> v = u + (dr, dc)
STEPS = [(-1, 0, 5), (1, 0, 5), (0, -1, 5), (0, 1, 5), (-1, -1, 7), (-1, 1, 7), (1, -1, 7), (1, 1, 7)]


def edge_ok(trav, r, c, dr, dc) -> bool:
  """The edge from (r, c) to (r + dr, c + dc), the destination inside the grid."""
  if not trav[r + dr, c + dc]:
    return False
  return dr == 0 or dc == 0 or (trav[r + dr, c] and trav[r, c + dc])


def cells_to_mask(cells, H: int, W: int) -> np.ndarray:
  """(b, n, 2) [x, z] cells -> (b, H, W) bool; cells outside the map are dropped."""
  cells = np.asarray(cells, dtype=np.int64).reshape(len(cells), -1, 2)
  mask = np.zeros((len(cells), H, W), bool)
  for i, env in enumerate(cells):
    for x, z in env:
      if 0 <= x < W and 0 <= z < H:
        mask[i, z, x] = True
  return mask


def dijkstra(trav: np.ndarray, src: np.ndarray) -> np.ndarray:
  """(H, W) bool grids -> (H, W) int32 distances."""
  H, W = trav.shape
  dist = np.full((H, W), -1, np.int64)
  heap = [(0, int(r), int(c)) for r, c in zip(*np.nonzero(src))]
  for _, r, c in heap:
    dist[r, c] = 0
  heapq.heapify(heap)
  while heap:
    d, r, c = heapq.heappop(heap)
    if d > dist[r, c]:
      continue
    for dr, dc, w in STEPS:
      rr, cc = r + dr, c + dc
      if 0 <= rr < H and 0 <= cc < W and edge_ok(trav, r, c, dr, dc):
        nd = d + w
        if dist[rr, cc] < 0 or nd < dist[rr, cc]:
          dist[rr, cc] = nd
          heapq.heappush(heap, (nd, rr, cc))
  return dist.astype(np.int32)


def oracle(trav: np.ndarray, src: np.ndarray) -> np.ndarray:
  """(b, H, W) bool grids -> (b, H, W) int32."""
  return np.stack([dijkstra(t, s) for t, s in zip(trav, src)])


def certificate(trav: np.ndarray, src: np.ndarray, dist: np.ndarray) -> bool:
  """True iff `dist` ((b, H, W) int32) is the distance field of (trav, src).  With -1 read as infinity, the field is
  the unique solution of: d = 0 on sources, and for every other cell v, d(v) = min over the edges u -> v of
  d(u) + cost (infinity without a finite one).  Unique because the costs are positive: a set of unreachable cells with
  finite values would contain a smallest one, which no in-neighbour could explain."""
  if dist.dtype != np.int32 or dist.shape != trav.shape or (dist < -1).any():
    return False
  inf = np.int64(1) << 40
  d = np.where(dist < 0, inf, dist.astype(np.int64))
  b, H, W = trav.shape
  dp = np.full((b, H + 2, W + 2), inf, np.int64)
  dp[:, 1:-1, 1:-1] = d
  tp = np.zeros((b, H + 2, W + 2), bool)
  tp[:, 1:-1, 1:-1] = trav
  best = np.full((b, H, W), inf, np.int64)
  for dr, dc, w in STEPS:      # v = u + (dr, dc): u = v - (dr, dc)
    du = dp[:, 1 - dr:1 - dr + H, 1 - dc:1 - dc + W]
    ok = trav.copy()
    if dr and dc:              # the cells (u.r, v.c) = (v.r - dr, v.c) and (v.r, u.c) = (v.r, v.c - dc)
      ok &= tp[:, 1 - dr:1 - dr + H, 1:1 + W] & tp[:, 1:1 + H, 1 - dc:1 - dc + W]
    best = np.minimum(best, np.where(ok & (du < inf), du + w, inf))
  want = np.where(src, 0, best)
  return bool(np.array_equal(d, want))


def spiral_maze(H: int, W: int) -> np.ndarray:
  """(H, W) bool: a one-cell corridor winding inwards from the corner (0, 0) between one-cell walls, about half the
  cells on one path: the worst case for the number of rounds."""
  free = np.zeros((H, W), bool)
  free[0, 0] = True
  r = c = 0
  top, bottom, left, right = 0, H - 1, 0, W - 1
  dirs = [(0, 1), (1, 0), (0, -1), (-1, 0)]
  stuck = 0
  for d in range(4 * (H + W)):
    dr, dc = dirs[d % 4]
    moved = False
    # each walk checks only the bound ahead of it; the bound behind the corridor moves in by 2 after the walk
    while (c + dc <= right if dc > 0 else c + dc >= left) if dc else (r + dr <= bottom if dr > 0 else r + dr >= top):
      r, c = r + dr, c + dc
      free[r, c] = moved = True
    stuck = 0 if moved else stuck + 1
    if stuck == 2:
      break
    if d % 4 == 0:
      top += 2
    elif d % 4 == 1:
      right -= 2
    elif d % 4 == 2:
      bottom -= 2
    else:
      left += 2
  return free
