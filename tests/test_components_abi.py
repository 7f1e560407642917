"""connected_components without a device: dm_connected_components_i32 refuses bad arguments before any CUDA call, the
Python function refuses bad calls before any device work, and the scipy oracle numbers components the way the
contract says (raster order of each component's first cell), so a change in scipy fails here."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._components import STRUCTURES, checkerboard, oracle, spiral_maze

# never dereferenced: every call below is refused before the first launch
MASK, LABELS, COUNTS, SIZES = 0x10000, 0x20000, 0x30000, 0x40000
REFUSALS = ["mask", "labels", "counts", "n_planes=0", "H=0", "W=-1", "connectivity=6", "connectivity=0",
            "cells over INT32_MAX"]


@pytest.mark.parametrize("case", REFUSALS)
def test_components_refuse_bad_arguments(case):
  a = dict(mask=MASK, n_planes=2, H=40, W=30, connectivity=8, labels=LABELS, counts=COUNTS, sizes=SIZES)
  if case in ("mask", "labels", "counts"):
    a[case] = None
  else:
    name, value = case.split("=") if "=" in case else ("", "")
    if name:
      a[name] = int(value)
    else:
      a["n_planes"], a["H"], a["W"] = 2, 32768, 32768   # 2^31 cells; one cell fewer would be accepted
  rc = nat.lib().dm_connected_components_i32(a["mask"], a["n_planes"], a["H"], a["W"], a["connectivity"], a["labels"],
                                             a["counts"], a["sizes"], None)
  assert rc == -1


@pytest.mark.parametrize("case", ["not a tensor", "uint8", "2-D", "5-D", "empty batch", "empty width", "too many cells",
                                  "on the host", "connectivity 6", "connectivity True", "connectivity 4.5"])
def test_value_errors_before_any_device_work(case):
  mask, conn, match = torch.ones((2, 5, 6), dtype=torch.bool), 8, None
  if case == "not a tensor":
    mask, match = np.ones((2, 5, 6), bool), "bool tensor"
  elif case == "uint8":
    mask, match = mask.to(torch.uint8), "bool tensor"
  elif case == "2-D":
    mask, match = mask[0], r"\(b, H, W\)"
  elif case == "5-D":
    mask, match = mask[None, None], r"\(b, H, W\)"
  elif case == "empty batch":
    mask, match = torch.ones((0, 5, 6), dtype=torch.bool), "empty"
  elif case == "empty width":
    mask, match = torch.ones((2, 3, 5, 0), dtype=torch.bool), "empty"
  elif case == "too many cells":
    mask, match = torch.ones((1, 1, 1), dtype=torch.bool).expand(2, 32768, 32768), "too large"
  elif case == "on the host":
    match = "CUDA"
  else:
    conn, match = {"connectivity 6": 6, "connectivity True": True, "connectivity 4.5": 4.5}[case], "connectivity"
  with pytest.raises(ValueError, match=match):
    dmap.connected_components(mask, conn)
  with pytest.raises(ValueError, match=match):
    dmap.connected_components(mask, conn, return_sizes=True)


def _raster_numbered(labels: np.ndarray) -> bool:
  """Components numbered 1..K in raster order of their first cell."""
  flat = labels.ravel()
  ids, first = np.unique(flat, return_index=True)
  order = ids[ids > 0][np.argsort(first[ids > 0])]
  return bool(np.array_equal(order, np.arange(1, len(order) + 1)))


@pytest.mark.parametrize("connectivity", [4, 8])
@pytest.mark.parametrize("seed", range(8))
def test_scipy_numbers_components_in_raster_order(seed, connectivity):
  from scipy import ndimage
  rng = np.random.default_rng(seed)
  H, W = rng.integers(1, 90, size=2)
  for density in (0.1, 0.41, 0.59, 0.9):
    mask = rng.random((H, W)) < density
    labels, k = ndimage.label(mask, STRUCTURES[connectivity])
    assert labels.max() == k and (labels[~mask] == 0).all() and (labels[mask] > 0).all()
    assert _raster_numbered(labels)


def test_oracle_on_known_masks():
  cb = checkerboard(7, 9)
  for conn, k in ((8, 1), (4, 32)):
    labels, counts, sizes = oracle(cb[None], conn)
    assert counts.tolist() == [k] and labels.max() == k
  labels, counts, sizes = oracle(cb[None], 4)
  assert (sizes[0][cb] == 1).all() and (sizes[0][~cb] == 0).all()
  spiral = spiral_maze(20, 23)
  labels, counts, sizes = oracle(np.stack([spiral, ~spiral]), 4)
  assert counts[0] == 1 and (sizes[0][spiral] == spiral.sum()).all()
  # a corner contact joins under 8-connectivity only
  diag = np.eye(4, dtype=bool)[None, None]
  assert oracle(diag, 8)[1].tolist() == [[1]] and oracle(diag, 4)[1].tolist() == [[4]]
