"""dm_fuse_clear_envs_f32 (MapBuilder.reset_envs) without a device: the argument checks refuse bad calls before any CUDA
call, and the Python layer refuses a bad `done` before touching the library."""
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat

# never dereferenced: every call below is refused before the first launch
TOP, HEIGHT, MASK, DONE, PLANES, BOX = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000, 0x60000


def _map(fill=float("-inf"), reduction=0):
  t = nat.DmFuseTarget()
  t.Mh, t.Mw, t.flip_h, t.map_res = 40, 30, 1, 0.05
  t.width_offset, t.height_offset, t.fill_value, t.reduction = 15., 20., fill, reduction
  return t


@pytest.mark.parametrize("case", ["topdown", "mask", "done", "map", "b=0", "C=0", "Mh=0", "box without plane_box",
                                  "box with NaN fill", "box with sum", "box with prod", "reduction 5",
                                  "unaligned plane_box"])
def test_clear_envs_refuses_bad_arguments(case):
  args = dict(topdown=TOP, height=HEIGHT, mask=MASK, b=2, C=3, done=DONE, map=_map(), plane_box=PLANES, box=BOX)
  if case in ("topdown", "mask", "done", "map"):
    args[case] = None
  elif case == "b=0":
    args["b"] = 0
  elif case == "C=0":
    args["C"] = 0
  elif case == "Mh=0":
    args["map"].Mh = 0
  elif case == "box without plane_box":
    args["plane_box"] = None
  elif case == "box with NaN fill":
    args["map"] = _map(fill=float("nan"))
  elif case == "box with sum":
    args["map"] = _map(fill=0., reduction=2)
  elif case == "box with prod":
    args["map"] = _map(fill=0., reduction=4)
  elif case == "reduction 5":
    args["map"] = _map(reduction=5)
  elif case == "unaligned plane_box":
    args["plane_box"] = PLANES + 4
  a = args
  rc = nat.lib().dm_fuse_clear_envs_f32(a["topdown"], a["height"], a["mask"], a["b"], a["C"], a["done"], a["map"],
                                        a["plane_box"], a["box"], None)
  assert rc == -1


def test_done_flags_are_checked_before_any_device_work():
  flags = dmap.MapBuilder._done_flags
  dev = torch.device("cuda", 0)
  for bad in ([True, False], [1, 0, 1], torch.ones(3, dtype=torch.uint8), torch.ones((3, 1), dtype=torch.bool),
              torch.ones(2, dtype=torch.bool), [[True], [False], [True]]):
    with pytest.raises(ValueError):
      flags(bad, 3, dev)


def test_no_world_map_is_a_no_op():
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=0.05, map_width=10, map_height=10)
  builder = dmap.MapBuilder(map_projector=proj)
  builder.reset_envs([True, False])
  assert builder.world_map.is_empty
