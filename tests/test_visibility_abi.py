"""visible_cells / count_visible without a device: dm_line_of_sight_u8 refuses bad arguments before any CUDA call, the
Python functions refuse bad calls before any device work, they are exported, and the numpy oracle (tests/_visibility.py)
gives the expected answer on hand-made maps."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._visibility import visible_window

# never dereferenced: every call below is refused before the first launch
BLOCK, ORIGINS, VISIBLE, TARGETS, COUNTS = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000
REFUSALS = ["blocking", "origins", "both outputs", "neither output", "targets without counts",
            "counts without targets", "counts with C=0", "visible with C=1", "b=0", "H=0", "W=-1", "n=0",
            "radius=-1", "radius=513", "b * n of 2^31", "H * W of 2^31", "b * C * H * W of 2^31"]


def _call(a):
  return nat.lib().dm_line_of_sight_u8(a["blocking"], a["b"], a["H"], a["W"], a["origins"], a["n"], a["radius"],
                                       a["visible"], a["targets"], a["C"], a["counts"], None)


@pytest.mark.parametrize("case", REFUSALS)
def test_line_of_sight_refuses_bad_arguments(case):
  a = dict(blocking=BLOCK, b=2, H=40, W=30, origins=ORIGINS, n=5, radius=7, visible=None, targets=TARGETS, C=3,
           counts=COUNTS)
  if case in ("blocking", "origins"):
    a[case] = None
  elif case == "both outputs":
    a["visible"] = VISIBLE
  elif case == "neither output":
    a["counts"] = None
  elif case == "targets without counts":
    a["counts"], a["visible"] = None, VISIBLE
  elif case == "counts without targets":
    a["targets"] = None
  elif case == "counts with C=0":
    a["C"] = 0
  elif case == "visible with C=1":
    a.update(visible=VISIBLE, targets=None, counts=None, C=1)
  elif case == "b * n of 2^31":
    a["b"], a["n"] = 1 << 16, 1 << 15
  elif case == "H * W of 2^31":
    a["H"], a["W"] = 1 << 16, 1 << 15
  elif case == "b * C * H * W of 2^31":
    a["b"], a["C"], a["H"], a["W"] = 4, 2, 1 << 14, 1 << 14
  else:
    name, value = case.split("=")
    a[name] = int(value)
  assert _call(a) == -1


def test_limits_are_exclusive():
  """One below each 2^31 limit is not refused for its size: the same call with no origins is what refuses it."""
  for b, n, H, W, C in ((1 << 16, (1 << 15) - 1, 4, 4, 1), (1, 1, (1 << 16) - 1, 1 << 15, 1),
                        (1, 1, (1 << 15) - 1, 1 << 16, 1), (2, 1, 1 << 14, (1 << 15) - 1, 2)):
    a = dict(blocking=BLOCK, b=b, H=H, W=W, origins=None, n=n, radius=512, visible=None, targets=TARGETS, C=C,
             counts=COUNTS)
    assert _call(a) == -1
  # and a valid call is refused only for the null origins: radius 0 and 512 are inside the range
  for radius in (0, 512):
    a = dict(blocking=BLOCK, b=2, H=40, W=30, origins=None, n=5, radius=radius, visible=VISIBLE, targets=None, C=0,
             counts=None)
    assert _call(a) == -1


def test_exported():
  assert dmap.visible_cells is dmap.maps.visible_cells
  assert dmap.count_visible is dmap.maps.count_visible
  assert "visible_cells" in dmap.maps.__all__ and "count_visible" in dmap.maps.__all__
  assert callable(dmap.TopdownMap.visible_cells) and callable(dmap.TopdownMap.count_visible)


def _big(shape):
  return torch.ones((1,) * len(shape), dtype=torch.bool).expand(*shape)


VALUE_ERRORS = {
  "blocking not a tensor": "bool tensor", "blocking uint8": "bool tensor", "blocking 2-D": r"\(b, H, W\)",
  "blocking two channels": r"\(b, H, W\)", "blocking empty": "empty", "radius -1": "radius", "radius 513": "radius",
  "radius float": "radius", "radius bool": "radius", "float origins": "integers", "origins batch": r"\(2, n, 2\)",
  "origins last dim": r"\(2, n, 2\)", "zero origins": r"\(2, n, 2\)", "origins rank": r"\(2, n, 2\)",
  "origins list shape": r"\(2, n, 2\)", "targets not a tensor": "bool tensor", "targets float": "bool tensor",
  "targets 2-D": r"\(b, C, H, W\)", "targets 5-D": r"\(b, C, H, W\)", "targets batch": "like blocking",
  "targets grid": "like blocking", "targets no plane": "like blocking", "b * n": "2\\^31", "H * W": "2\\^31",
  "b * C * H * W": "2\\^31", "blocking on the host": "CUDA",
}
COUNT_ONLY = ("targets not a tensor", "targets float", "targets 2-D", "targets 5-D", "targets batch", "targets grid",
              "targets no plane", "b * C * H * W")


@pytest.mark.parametrize("case", list(VALUE_ERRORS))
def test_value_errors_before_any_device_work(case):
  blocking = torch.zeros((2, 5, 6), dtype=torch.bool)
  targets = torch.zeros((2, 3, 5, 6), dtype=torch.bool)
  origins, radius = [[1, 2], [3, 4]], 3
  if case == "blocking not a tensor":
    blocking = np.zeros((2, 5, 6), bool)
  elif case == "blocking uint8":
    blocking = blocking.to(torch.uint8)
  elif case == "blocking 2-D":
    blocking = blocking[0]
  elif case == "blocking two channels":
    blocking = torch.zeros((2, 2, 5, 6), dtype=torch.bool)
  elif case == "blocking empty":
    blocking = blocking[:, :0]
  elif case.startswith("radius"):
    radius = {"radius -1": -1, "radius 513": 513, "radius float": 3.0, "radius bool": True}[case]
  elif case == "float origins":
    origins = torch.zeros((2, 2))
  elif case == "origins batch":
    origins = torch.zeros((3, 2), dtype=torch.int64)
  elif case == "origins last dim":
    origins = torch.zeros((2, 4, 3), dtype=torch.int64)
  elif case == "zero origins":
    origins = torch.zeros((2, 0, 2), dtype=torch.int64)
  elif case == "origins rank":
    origins = torch.zeros((2, 1, 1, 2), dtype=torch.int64)
  elif case == "origins list shape":
    origins = [[1, 2, 3], [3, 4, 5]]
  elif case == "targets not a tensor":
    targets = targets.numpy()
  elif case == "targets float":
    targets = targets.float()
  elif case == "targets 2-D":
    targets = targets[0, 0]
  elif case == "targets 5-D":
    targets = targets[None]
  elif case == "targets batch":
    targets = targets[:1]
  elif case == "targets grid":
    targets = targets[:, :, :, 1:]
  elif case == "targets no plane":
    targets = targets[:, :0]
  elif case == "b * n":
    origins = torch.zeros((1, 1, 2), dtype=torch.int64).expand(2, 2 ** 30, 2)
  elif case == "H * W":
    blocking, targets = _big((2, 1 << 16, 1 << 15)), _big((2, 1, 1 << 16, 1 << 15))
  elif case == "b * C * H * W":
    blocking, targets = _big((2, 1 << 14, 1 << 14)), _big((2, 4, 1 << 14, 1 << 14))
  match = VALUE_ERRORS[case]
  m = dmap.TopdownMap(topdown_map=torch.zeros((2, 1, 5, 6)), mask=torch.zeros((2, 1, 5, 6), dtype=torch.bool),
                      height_map=torch.zeros((2, 1, 5, 6)), is_height_map=True,
                      map_projector=dmap.MapProjector(width=8, height=6, hfov=1.2, map_res=0.05, map_width=6,
                                                      map_height=5, width_offset=3., height_offset=2.))
  with pytest.raises(ValueError, match=match):
    dmap.count_visible(blocking, targets, origins, radius)
  with pytest.raises(ValueError, match=match):
    m.count_visible(blocking, targets, radius, origins)
  if case not in COUNT_ONLY:
    with pytest.raises(ValueError, match=match):
      dmap.visible_cells(blocking, origins, radius)
    with pytest.raises(ValueError, match=match):
      m.visible_cells(blocking, radius, origins)
  if case.startswith("blocking") or case.startswith("radius") or case in COUNT_ONLY or case == "H * W":
    with pytest.raises(ValueError, match=match):   # the default origin needs the batch of a valid grid first
      m.count_visible(blocking, targets, radius)


# ---- the oracle on hand-made maps ----------------------------------------------------------------------------------

def _disk(r):
  dz, dx = np.mgrid[-r:r + 1, -r:r + 1]
  return dx * dx + dz * dz <= r * r


def test_open_map_sees_the_integer_disk():
  for r in (0, 1, 2, 7, 12):
    v = visible_window(np.zeros((40, 40), bool), 20, 19, r)
    assert np.array_equal(v, _disk(r))


def test_radius_zero_sees_only_the_origin():
  block = np.ones((5, 6), bool)
  v = visible_window(block, 2, 3, 0)
  assert v.shape == (1, 1) and v[0, 0]


def test_straight_wall_hides_what_is_behind_it_and_is_itself_visible():
  block = np.zeros((21, 21), bool)
  block[:, 14] = True                       # a column wall at x = 14
  r = 12
  v = visible_window(block, 5, 10, r)
  cols = np.arange(-r, r + 1) + 5
  rows = np.arange(-r, r + 1) + 10
  inside = (rows[:, None] >= 0) & (rows[:, None] < 21) & (cols[None] >= 0) & (cols[None] < 21)
  assert not v[:, cols > 14].any()
  wall = _disk(r) & inside & (cols[None] == 14)
  assert wall.any() and np.array_equal(v[:, cols == 14], wall[:, cols == 14])
  assert np.array_equal(v[:, cols < 14], (_disk(r) & inside)[:, cols < 14])


def test_staircase_blocks():
  """A 45-degree wall x + z = 14 whose cells touch only at corners: nothing beyond it is visible."""
  block = np.zeros((21, 21), bool)
  for x in range(15):
    block[14 - x, x] = True
  r = 12
  v = visible_window(block, 5, 5, r)
  dz, dx = np.mgrid[-r:r + 1, -r:r + 1]
  x, z = dx + 5, dz + 5
  beyond = (x + z > 14) & _disk(r) & (x < 21) & (z < 21)
  assert beyond.any() and not v[beyond].any()
  assert v[r + 2, r + 2] and v[r - 3, r + 4]            # wall cells (7, 7) and (9, 2) themselves


def test_random_8_connected_walls_leak_nothing():
  rng = np.random.default_rng(0)
  for _ in range(40):
    H = W = 31
    block = np.zeros((H, W), bool)
    x, cols = 15, []
    for z in range(H):
      x = int(np.clip(x + rng.integers(-1, 2), 8, 22))
      block[z, x] = True
      cols.append(x)
    r = 40
    v = visible_window(block, 2, 15, r)
    for z in range(H):
      assert not v[z - 15 + r, cols[z] + 1 - 2 + r:W - 2 + r].any()


def test_a_single_diagonal_gap_lets_sight_through():
  """Only one side cell of a diagonal step blocks: the step is allowed."""
  block = np.zeros((5, 5), bool)
  block[1, 2] = True                        # the side cell (x_1, z_0) of the step (1, 1) -> (2, 2)
  v = visible_window(block, 1, 1, 2)
  assert v[2 + 1, 2 + 1]                    # target (2, 2) = o + (1, 1)
  block[2, 1] = True                        # now both side cells block
  v = visible_window(block, 1, 1, 2)
  assert not v[2 + 1, 2 + 1] and v[2 + 1, 2 + 0] and v[2 + 0, 2 + 1]   # the two side cells stay visible


def test_origin_on_a_blocking_cell_sees_its_neighbours():
  block = np.zeros((9, 9), bool)
  block[4, 4] = True
  v = visible_window(block, 4, 4, 3)
  assert np.array_equal(v, _disk(3))


def test_origin_outside_the_map_sees_nothing():
  block = np.zeros((9, 9), bool)
  for ox, oz in ((-1, 4), (4, -1), (9, 4), (4, 9)):
    assert not visible_window(block, ox, oz, 3).any()
