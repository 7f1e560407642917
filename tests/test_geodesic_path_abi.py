"""geodesic_path without a device: dm_geodesic_path_i32 refuses bad arguments before any CUDA call, the Python
functions refuse bad calls before any device work, they are exported, the plain-Python oracle (tests/_geodesic_path.py)
gives the expected paths on hand-made grids, and the certificate accepts every oracle path on random grids."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._geodesic import cells_to_mask, dijkstra, oracle as field_oracle
from tests._geodesic_path import certificate, oracle, walk

# never dereferenced: every call below is refused before the first launch
TRAV, DIST, STARTS, CELLS, LENGTHS = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000
REFUSALS = ["traversable", "dist", "starts", "cells", "lengths", "b=0", "H=0", "W=-1", "n=0", "max_cells=0",
            "max_cells=H*W+1", "H * W of 2^31", "b * n of 2^31"]


def _call(a):
  return nat.lib().dm_geodesic_path_i32(a["traversable"], a["dist"], a["b"], a["H"], a["W"], a["starts"], a["n"],
                                        a["max_cells"], a["cells"], a["lengths"], None)


def _args(**kw):
  a = dict(traversable=TRAV, dist=DIST, b=2, H=40, W=30, starts=STARTS, n=5, max_cells=64, cells=CELLS,
           lengths=LENGTHS)
  a.update(kw)
  return a


@pytest.mark.parametrize("case", REFUSALS)
def test_geodesic_path_refuses_bad_arguments(case):
  a = _args()
  if case in ("traversable", "dist", "starts", "cells", "lengths"):
    a[case] = None
  elif case == "max_cells=H*W+1":
    a["max_cells"] = 40 * 30 + 1
  elif case == "H * W of 2^31":
    a["H"], a["W"] = 1 << 16, 1 << 15
  elif case == "b * n of 2^31":
    a["b"], a["n"] = 1 << 16, 1 << 15
  else:
    name, value = case.split("=")
    a[name] = int(value)
  assert _call(a) == -1


@pytest.mark.skipif(torch.cuda.is_available(), reason="shows the limits by a call that passes validation and fails "
                    "at the launch, which needs a machine without a CUDA device")
def test_limits_are_exclusive():
  """One below each 2^31 limit, and max_cells at 1 and at H * W, pass validation: without a device the call then fails
  at the launch with a CUDA error code, not DM_EINVAL."""
  for kw in (dict(H=(1 << 16) - 1, W=1 << 15, max_cells=((1 << 16) - 1) << 15), dict(b=1 << 16, n=(1 << 15) - 1),
             dict(max_cells=1), dict(max_cells=40 * 30)):
    rc = _call(_args(**kw))
    assert rc not in (0, -1), kw


def test_exported():
  assert dmap.geodesic_path is dmap.maps.geodesic_path
  assert "geodesic_path" in dmap.maps.__all__
  assert callable(dmap.TopdownMap.geodesic_path)


def _big(shape, dtype=torch.bool):
  return torch.ones((1,) * len(shape), dtype=dtype).expand(*shape)


VALUE_ERRORS = {
  "traversable not a tensor": "bool tensor", "traversable uint8": "bool tensor", "traversable 2-D": r"\(b, H, W\)",
  "traversable two channels": r"\(b, H, W\)", "traversable empty": "empty", "traversable 7HW overflow": "int32",
  "dist not a tensor": "dist must be an int32", "dist int64": "dist must be an int32",
  "dist batch": "dist must be an int32", "dist grid": "dist must be an int32", "dist two channels": "dist must be",
  "float starts": "integers", "bool starts": "integers", "starts batch": r"\(2, n, 2\)",
  "starts last dim": r"\(2, n, 2\)", "zero starts": r"\(2, n, 2\)", "starts rank": r"\(2, n, 2\)",
  "starts list shape": r"\(2, n, 2\)", "max_cells 0": "max_cells", "max_cells H*W+1": "max_cells",
  "max_cells float": "max_cells", "max_cells bool": "max_cells", "max_cells tensor": "max_cells",
  "b * n": "2\\^31", "traversable on the host": "CUDA",
}
TRAVERSABLE = tuple(c for c in VALUE_ERRORS if c.startswith("traversable"))


@pytest.mark.parametrize("case", list(VALUE_ERRORS))
def test_value_errors_before_any_device_work(case):
  trav = torch.ones((2, 5, 6), dtype=torch.bool)
  dist = torch.zeros((2, 5, 6), dtype=torch.int32)
  starts, max_cells = [[1, 2], [3, 4]], 7
  if case == "traversable not a tensor":
    trav = np.ones((2, 5, 6), bool)
  elif case == "traversable uint8":
    trav = trav.to(torch.uint8)
  elif case == "traversable 2-D":
    trav = trav[0]
  elif case == "traversable two channels":
    trav = torch.ones((2, 2, 5, 6), dtype=torch.bool)
  elif case == "traversable empty":
    trav = trav[:, :0]
  elif case == "traversable 7HW overflow":
    trav = _big((2, 17516, 17515))
  elif case == "dist not a tensor":
    dist = dist.numpy()
  elif case == "dist int64":
    dist = dist.long()
  elif case == "dist batch":
    dist = dist[:1]
  elif case == "dist grid":
    dist = dist[:, :, 1:]
  elif case == "dist two channels":
    dist = torch.zeros((2, 2, 5, 6), dtype=torch.int32)
  elif case == "float starts":
    starts = torch.zeros((2, 2))
  elif case == "bool starts":
    starts = [[True, False], [False, True]]
  elif case == "starts batch":
    starts = torch.zeros((3, 2), dtype=torch.int64)
  elif case == "starts last dim":
    starts = torch.zeros((2, 4, 3), dtype=torch.int64)
  elif case == "zero starts":
    starts = torch.zeros((2, 0, 2), dtype=torch.int64)
  elif case == "starts rank":
    starts = torch.zeros((2, 1, 1, 2), dtype=torch.int64)
  elif case == "starts list shape":
    starts = [[1, 2, 3], [3, 4, 5]]
  elif case.startswith("max_cells"):
    max_cells = {"max_cells 0": 0, "max_cells H*W+1": 31, "max_cells float": 7.0, "max_cells bool": True,
                 "max_cells tensor": torch.tensor(7)}[case]
  elif case == "b * n":
    starts = torch.zeros((1, 1, 2), dtype=torch.int64).expand(2, 2 ** 30, 2)
  match = VALUE_ERRORS[case]
  m = dmap.TopdownMap(topdown_map=torch.zeros((2, 1, 5, 6)), mask=torch.zeros((2, 1, 5, 6), dtype=torch.bool),
                      height_map=torch.zeros((2, 1, 5, 6)), is_height_map=True,
                      map_projector=dmap.MapProjector(width=8, height=6, hfov=1.2, map_res=0.05, map_width=6,
                                                      map_height=5, width_offset=3., height_offset=2.))
  with pytest.raises(ValueError, match=match):
    dmap.geodesic_path(trav, dist, starts, max_cells)
  with pytest.raises(ValueError, match=match):
    m.geodesic_path(trav, dist, max_cells, starts)
  if "starts" not in case and case != "b * n":
    with pytest.raises(ValueError, match=match):   # the default start needs the batch of a valid grid first
      m.geodesic_path(trav, dist, max_cells)


def test_b_times_n_limit_is_exclusive():
  """b * n = 2^31 - 1 passes the size check: the call is refused next, for the traversable on the host."""
  trav = torch.ones((1, 1, 1), dtype=torch.bool)
  starts = torch.zeros((1, 1, 2), dtype=torch.int64).expand(1, 2 ** 31 - 1, 2)
  with pytest.raises(ValueError, match="CUDA"):
    dmap.geodesic_path(trav, torch.zeros((1, 1, 1), dtype=torch.int32), starts, 1)
  with pytest.raises(ValueError, match="CUDA"):     # max_cells = H * W is inside the range; (b, 1, H, W) dist too
    dmap.geodesic_path(torch.ones((2, 3, 4), dtype=torch.bool), torch.zeros((2, 1, 3, 4), dtype=torch.int32),
                       np.zeros((2, 2), np.int64), 12)


# ---- the oracle on hand-made grids ---------------------------------------------------------------------------------

def _field(trav, goals):
  """(H, W) bool grid, goal cells [x, z] -> the int32 field of geodesic_distance."""
  src = cells_to_mask(np.asarray(goals)[None], *trav.shape)[0]
  return dijkstra(trav, src)


def test_open_grid():
  trav = np.ones((5, 6), bool)
  dist = _field(trav, [(4, 3)])
  path = walk(trav, dist, 0, 0, 30)
  # the orthogonal step comes first in the order and is on a shortest path here; then three diagonal steps
  assert path == [(0, 0), (1, 0), (2, 1), (3, 2), (4, 3)]
  assert dist[0, 0] == 26 and certificate(trav, dist, (0, 0), path)


def test_l_shaped_corridor():
  trav = np.zeros((5, 5), bool)
  trav[0, :] = True                       # row z = 0
  trav[:, 4] = True                       # column x = 4
  dist = _field(trav, [(4, 4)])
  path = walk(trav, dist, 0, 0, 25)
  assert path == [(x, 0) for x in range(5)] + [(4, z) for z in range(1, 5)]
  assert certificate(trav, dist, (0, 0), path)


def test_diagonal_gap_is_gone_around():
  """Blocked cells (2, 1) and (1, 2) touch at a corner between start (1, 1) and goal (2, 2): no step through it."""
  trav = np.ones((4, 4), bool)
  trav[1, 2] = trav[2, 1] = False
  dist = _field(trav, [(2, 2)])
  assert dist[1, 1] == 30
  path = walk(trav, dist, 1, 1, 16)
  assert path == [(1, 1), (0, 1), (0, 2), (0, 3), (1, 3), (2, 3), (2, 2)]
  assert certificate(trav, dist, (1, 1), path)
  assert not certificate(trav, dist, (1, 1), [(1, 1), (2, 2)])     # the corner cut is not an edge


def test_start_on_a_goal_unreachable_and_outside():
  trav = np.ones((6, 7), bool)
  trav[:, 3] = False                      # a wall: the right half is not reached from the goal
  dist = _field(trav, [(1, 2)])
  assert walk(trav, dist, 1, 2, 10) == [(1, 2)]
  assert walk(trav, dist, 5, 2, 10) == []  # D = -1
  assert walk(trav, dist, 3, 0, 10) == []  # on the wall: D = -1
  for x, z in ((-1, 2), (7, 2), (1, -1), (1, 6)):
    assert walk(trav, dist, x, z, 10) == []
  starts = np.array([[[1, 2], [5, 2], [-1, 2], [0, 0]]])
  cells, lengths = oracle(trav[None], dist[None], starts, 5)
  assert lengths.tolist() == [[1, 0, 0, 3]]
  assert (cells[0, 1:3] == -1).all() and (cells[0, 3, 3:] == -1).all() and (cells[0, 0, 0] == (1, 2)).all()


def test_goal_on_an_obstacle():
  trav = np.ones((1, 6), bool)
  trav[0, 5] = False                      # the goal, an object's cell, is not traversable
  dist = _field(trav, [(5, 0)])
  path = walk(trav, dist, 0, 0, 6)
  assert path == [(x, 0) for x in range(6)] and not trav[0, 5]
  assert all(trav[z, x] for x, z in path[:-1]) and certificate(trav, dist, (0, 0), path)


def test_truncation_at_max_cells():
  trav = np.ones((5, 6), bool)
  dist = _field(trav, [(4, 3)])
  full = walk(trav, dist, 0, 0, 30)
  assert walk(trav, dist, 0, 0, 1) == full[:1]
  assert walk(trav, dist, 0, 0, 3) == full[:3]
  assert walk(trav, dist, 0, 0, len(full)) == full
  cells, lengths = oracle(trav[None], dist[None], np.array([[[0, 0]]]), 3)
  assert lengths[0, 0] == 3 and cells[0, 0].tolist() == [list(c) for c in full[:3]]


@pytest.mark.parametrize("seed", range(6))
def test_a_dist_that_is_not_a_field_terminates(seed):
  """Random int32 values: D strictly decreases along every walk, the cells are distinct and at most D[s] / 5 + 1."""
  rng = np.random.default_rng(seed)
  H, W = 12, 15
  trav = rng.random((H, W)) > 0.2
  dist = rng.integers(-1, 60, size=(H, W)).astype(np.int32)
  dist[0, :3] = [np.iinfo(np.int32).max, np.iinfo(np.int32).min, 0]
  dist[1, 0] = np.iinfo(np.int32).max - 5        # reachable from the int32 maximum by one step
  trav[1, 0] = trav[0, 0] = True
  early = 0
  for z in range(H):
    for x in range(W):
      path = walk(trav, dist, x, z, H * W)
      if dist[z, x] < 0:
        assert path == []
        continue
      d = [int(dist[pz, px]) for px, pz in path]
      assert len(set(path)) == len(path) and len(path) <= d[0] // 5 + 1
      assert all(a > b for a, b in zip(d, d[1:]))
      early += d[-1] != 0
  assert early > 0                                 # some walks stop before reaching 0
  assert walk(trav, dist, 0, 0, 10)[:2] == [(0, 0), (0, 1)]
  assert walk(trav, dist, 1, 0, 10) == []


@pytest.mark.parametrize("seed", range(8))
def test_certificate_accepts_every_oracle_path(seed):
  rng = np.random.default_rng(100 + seed)
  b, H, W = 2, int(rng.integers(1, 20)), int(rng.integers(1, 20))
  trav = rng.random((b, H, W)) > rng.choice([0.0, 0.2, 0.4])
  goals = rng.random((b, H, W)) < 0.03
  goals[:, rng.integers(H), rng.integers(W)] = True
  dist = field_oracle(trav, goals)
  zz, xx = np.mgrid[0:H, 0:W]
  starts = np.broadcast_to(np.stack([xx.ravel(), zz.ravel()], -1), (b, H * W, 2))
  cells, lengths = oracle(trav, dist, starts, H * W)
  for i in range(b):
    for k in range(H * W):
      x, z = starts[i, k]
      if dist[i, z, x] < 0:
        assert lengths[i, k] == 0
        continue
      path = cells[i, k, :lengths[i, k]]
      assert certificate(trav[i], dist[i], (x, z), path)
      assert (cells[i, k, lengths[i, k]:] == -1).all()
      if len(path) > 1:   # a wrong step, a step dropped or a path cut short is rejected
        assert not certificate(trav[i], dist[i], (x, z), path[:-1])
        assert not certificate(trav[i], dist[i], (x, z), np.concatenate([path[:1], path[2:]]))
