"""distance_transform without a device: dm_distance_transform_f32 refuses bad arguments before any CUDA call, the
Python function refuses bad calls before any device work, scipy's distances equal a brute-force minimum (so a change
in scipy fails here), scipy's own indices pass the tie-independent `nearest` check, and planes without a False cell are
pinned: scipy's phantom-cell output, and the library's defined +inf / -1."""
import numpy as np
import pytest
import torch
from scipy import ndimage

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._components import pattern
from tests._distance import brute_force, check_nearest, oracle, scipy_nearest, sqrtf_plane

# never dereferenced: every call below is refused before the first launch
MASK, DIST, NEAREST = 0x10000, 0x20000, 0x30000
REFUSALS = ["mask", "dist", "n_planes=0", "H=0", "W=-1", "H=32769", "W=32769", "cells over INT32_MAX"]


@pytest.mark.parametrize("case", REFUSALS)
def test_distance_refuses_bad_arguments(case):
  a = dict(mask=MASK, n_planes=2, H=40, W=30, dist=DIST, nearest=NEAREST)
  if case in ("mask", "dist"):
    a[case] = None
  elif "=" in case:
    name, value = case.split("=")
    a[name] = int(value)
  else:
    a["n_planes"], a["H"], a["W"] = 2, 32768, 32768   # 2^31 cells; one cell fewer would be accepted
  for nearest in (a["nearest"], None):
    rc = nat.lib().dm_distance_transform_f32(a["mask"], a["n_planes"], a["H"], a["W"], a["dist"], nearest, None)
    assert rc == -1


@pytest.mark.parametrize("case", ["not a tensor", "uint8", "float", "2-D", "5-D", "empty batch", "empty width",
                                  "H over 32768", "W over 32768", "too many cells", "on the host"])
def test_value_errors_before_any_device_work(case):
  mask, match = torch.ones((2, 5, 6), dtype=torch.bool), None
  if case == "not a tensor":
    mask, match = np.ones((2, 5, 6), bool), "bool tensor"
  elif case == "uint8":
    mask, match = mask.to(torch.uint8), "bool tensor"
  elif case == "float":
    mask, match = mask.float(), "bool tensor"
  elif case == "2-D":
    mask, match = mask[0], r"\(b, H, W\)"
  elif case == "5-D":
    mask, match = mask[None, None], r"\(b, H, W\)"
  elif case == "empty batch":
    mask, match = torch.ones((0, 5, 6), dtype=torch.bool), "empty"
  elif case == "empty width":
    mask, match = torch.ones((2, 3, 5, 0), dtype=torch.bool), "empty"
  elif case == "H over 32768":
    mask, match = torch.ones((1, 1, 1), dtype=torch.bool).expand(1, 32769, 2), "32768"
  elif case == "W over 32768":
    mask, match = torch.ones((1, 1, 1, 1), dtype=torch.bool).expand(1, 1, 1, 32769), "32768"
  elif case == "too many cells":
    mask, match = torch.ones((1, 1, 1), dtype=torch.bool).expand(2, 32768, 32768), "too large"
  else:
    match = "CUDA"
  with pytest.raises(ValueError, match=match):
    dmap.distance_transform(mask)
  with pytest.raises(ValueError, match=match):
    dmap.distance_transform(mask, return_indices=True)


def test_exported_from_the_package():
  assert "distance_transform" in dmap.maps.__all__ and dmap.distance_transform is dmap.maps.distance_transform


@pytest.mark.parametrize("seed", range(8))
def test_scipy_equals_brute_force(seed):
  rng = np.random.default_rng(seed)
  H, W = rng.integers(1, 60, size=2)
  for density in (0.01, 0.3, 0.9, 0.995):
    plane = rng.random((H, W)) < density
    plane.flat[rng.integers(plane.size)] = False        # at least one False cell
    assert np.array_equal(oracle(plane[None])[0], brute_force(plane))


@pytest.mark.parametrize("kind", ["random 0.001", "random 0.5", "random 0.999", "spiral", "checkerboard",
                                  "vertical stripes", "horizontal stripes", "rooms"])
def test_scipy_indices_pass_the_nearest_check(kind):
  rng = np.random.default_rng(len(kind))
  for H, W in ((1, 1), (7, 1), (1, 9), (37, 41), (80, 64)):
    plane = pattern(kind, H, W, rng)
    if plane.all():
      plane[H // 2, W // 2] = False
    check_nearest(plane[None], oracle(plane[None]), scipy_nearest(plane)[None])


def test_the_nearest_check_accepts_any_tie_choice():
  """Two opposite corners of a 5 x 5 plane: the cells of the anti-diagonal are as near to one corner as to the other.
  Pointing each of them at either corner passes the check; a False cell farther than the distance does not."""
  plane = np.ones((5, 5), bool)
  plane[0, 0] = plane[4, 4] = False
  d = oracle(plane[None])
  near = scipy_nearest(plane)
  check_nearest(plane[None], d, near[None])
  for corner in ((0, 0), (4, 4)):
    other = near.copy()
    for r in range(5):
      if plane[r, 4 - r]:
        other[r, 4 - r] = corner
    check_nearest(plane[None], d, other[None])
  bad = near.copy()
  bad[1, 0] = (4, 4)
  with pytest.raises(AssertionError):
    check_nearest(plane[None], d, bad[None])


@pytest.mark.parametrize("shape", [(1, 1), (3, 4), (1, 7)])
def test_planes_without_a_false_cell(shape):
  plane = np.ones(shape, bool)
  # scipy measures to a phantom feature at (row -1, column 0) and reports indices -1 / 0
  d, idx = ndimage.distance_transform_edt(plane, return_indices=True)
  r, c = np.indices(shape)
  assert np.array_equal(d, np.sqrt(((r + 1) ** 2 + c ** 2).astype(np.float64)))
  assert (idx[0] == -1).all() and (idx[1] == 0).all()
  # this library defines it instead
  assert np.isposinf(oracle(plane[None])).all()
  check_nearest(plane[None], oracle(plane[None]), np.full(shape + (2,), -1, np.int32)[None])
  with pytest.raises(AssertionError):
    check_nearest(plane[None], oracle(plane[None]), np.zeros(shape + (2,), np.int32)[None])


def test_sqrtf_differs_from_scipys_rounding_above_2_pow_24():
  """Why dist rounds through float64: up to d2 = 2^24 the float32 sqrt of float32(d2) equals scipy's float64 sqrt cast
  to float32, above it not always.  sqrtf_plane(), which the GPU tests run, has cells where the two differ."""
  d2 = np.arange(2 ** 24 - 4096, 2 ** 24 + 2 ** 16, dtype=np.int64)
  want = np.sqrt(d2.astype(np.float64)).astype(np.float32)
  f32 = np.sqrt(d2.astype(np.float32))
  low = d2 <= 2 ** 24
  assert np.array_equal(want[low], f32[low])
  assert (want[~low] != f32[~low]).any()
  plane = sqrtf_plane()
  d = oracle(plane[None])[0]
  r, c = np.indices(plane.shape)
  d2 = (r ** 2 + c ** 2).astype(np.int64)
  assert np.array_equal(d, brute_force(plane))
  assert (np.sqrt(d2.astype(np.float32)) != d).sum() > 1000
