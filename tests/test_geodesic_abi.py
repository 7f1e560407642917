"""geodesic_distance without a device: dm_geodesic_distance_i32 refuses bad arguments before any CUDA call, the Python
function refuses bad calls before any device work, and the oracle (tests/_geodesic.py) agrees with scipy's Dijkstra."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._geodesic import STEPS, certificate, dijkstra, edge_ok, oracle, spiral_maze

# never dereferenced: every call below is refused before the first launch
TRAV, MASK, CELLS, DIST = 0x10000, 0x20000, 0x30000, 0x40000
REFUSALS = ["traversable", "dist", "b=0", "H=0", "W=-1", "both forms", "neither form", "cells with n=0",
            "mask with n=1", "7HW overflow", "2^31 tiles"]


@pytest.mark.parametrize("case", REFUSALS)
def test_geodesic_refuses_bad_arguments(case):
  a = dict(traversable=TRAV, mask=None, cells=CELLS, n=3, b=2, H=40, W=30, dist=DIST)
  if case in ("traversable", "dist"):
    a[case] = None
  elif case in ("b=0", "H=0", "W=-1"):
    name, value = case.split("=")
    a[name] = int(value)
  elif case == "both forms":
    a["mask"] = MASK
  elif case == "neither form":
    a["cells"] = None
  elif case == "cells with n=0":
    a["n"] = 0
  elif case == "mask with n=1":
    a["mask"], a["cells"], a["n"] = MASK, None, 1
  elif case == "7HW overflow":
    a["H"], a["W"] = 17516, 17515      # 7 * H * W = 2147600115; at 17515 x 17515 it would fit
  elif case == "2^31 tiles":
    a["b"], a["H"], a["W"] = 1 << 29, 64, 64 * 2   # 8 tiles of 32 x 32 per environment
  rc = nat.lib().dm_geodesic_distance_i32(a["traversable"], a["mask"], a["cells"], a["n"], a["b"], a["H"], a["W"],
                                          a["dist"], None)
  assert rc == -1


def _trav(shape=(2, 5, 6)):
  return torch.ones(shape, dtype=torch.bool)


@pytest.mark.parametrize("case", ["not a tensor", "uint8", "2-D", "two channels", "empty", "7HW overflow",
                                  "mask shape", "float cells", "bool cells list", "cells batch", "cells last dim",
                                  "zero cells", "cells rank", "traversable on the host"])
def test_value_errors_before_any_device_work(case):
  trav, src = _trav(), [[1, 2], [3, 4]]
  match = None
  if case == "not a tensor":
    trav, match = np.ones((2, 5, 6), bool), "bool tensor"
  elif case == "uint8":
    trav, match = trav.to(torch.uint8), "bool tensor"
  elif case == "2-D":
    trav, match = trav[0], r"\(b, H, W\)"
  elif case == "two channels":
    trav, match = _trav((2, 2, 5, 6)), r"\(b, H, W\)"
  elif case == "empty":
    trav, match = _trav((0, 5, 6)), "empty"
  elif case == "7HW overflow":
    trav, match = torch.ones((1, 1, 1), dtype=torch.bool).expand(1, 17516, 17515), "int32"
  elif case == "mask shape":
    src, match = torch.zeros((2, 1, 5, 6), dtype=torch.bool), "shape"
  elif case == "float cells":
    src, match = torch.zeros((2, 2)), "integers"
  elif case == "bool cells list":
    src, match = [[True, False], [False, True]], "integers"
  elif case == "cells batch":
    src, match = torch.zeros((3, 2), dtype=torch.int64), r"\(2, n, 2\)"
  elif case == "cells last dim":
    src, match = torch.zeros((2, 4, 3), dtype=torch.int64), r"\(2, n, 2\)"
  elif case == "zero cells":
    src, match = torch.zeros((2, 0, 2), dtype=torch.int64), r"\(2, n, 2\)"
  elif case == "cells rank":
    src, match = torch.zeros((2, 1, 1, 2), dtype=torch.int64), r"\(2, n, 2\)"
  elif case == "traversable on the host":
    match = "CUDA"
  with pytest.raises(ValueError, match=match):
    dmap.geodesic_distance(trav, src)
  m = dmap.TopdownMap(topdown_map=torch.zeros((2, 1, 5, 6)), mask=torch.zeros((2, 1, 5, 6), dtype=torch.bool),
                      height_map=torch.zeros((2, 1, 5, 6)), is_height_map=True,
                      map_projector=dmap.MapProjector(width=8, height=6, hfov=1.2, map_res=0.05, map_width=6,
                                                      map_height=5, width_offset=3., height_offset=2.))
  with pytest.raises(ValueError, match=match):
    m.geodesic_distance(trav, src)
  if case in ("not a tensor", "uint8", "2-D", "two channels", "empty", "7HW overflow", "traversable on the host"):
    with pytest.raises(ValueError, match=match):
      m.geodesic_distance(trav)   # the default source needs the batch of a valid grid first


def _scipy(trav, src):
  sp = pytest.importorskip("scipy.sparse")
  csgraph = pytest.importorskip("scipy.sparse.csgraph")
  H, W = trav.shape
  rows, cols, costs = [], [], []
  for r in range(H):
    for c in range(W):
      for dr, dc, w in STEPS:
        if 0 <= r + dr < H and 0 <= c + dc < W and edge_ok(trav, r, c, dr, dc):
          rows.append(r * W + c)
          cols.append((r + dr) * W + c + dc)
          costs.append(w)
  g = sp.csr_matrix((np.array(costs, np.float64), (rows, cols)), shape=(H * W, H * W))
  starts = np.flatnonzero(src)
  if len(starts) == 0:
    return np.full((H, W), -1, np.int32)
  d = csgraph.dijkstra(g, directed=True, indices=starts, min_only=True)
  return np.where(np.isinf(d), -1, d).astype(np.int32).reshape(H, W)


@pytest.mark.parametrize("seed", range(12))
def test_oracle_matches_scipy(seed):
  rng = np.random.default_rng(seed)
  H, W = rng.integers(1, 24, size=2)
  trav = rng.random((H, W)) > rng.choice([0., 0.2, 0.4, 0.6])
  src = rng.random((H, W)) < rng.choice([0., 0.01, 0.05])
  if seed % 3 == 0:
    src[rng.integers(H), rng.integers(W)] = True   # possibly on an obstacle
  want = _scipy(trav, src)
  got = dijkstra(trav, src)
  assert np.array_equal(got, want)
  assert certificate(trav[None], src[None], got[None])


def test_oracle_on_a_spiral_and_certificate_rejects_wrong_fields():
  trav = spiral_maze(15, 17)
  src = np.zeros_like(trav)
  src[0, 0] = True
  d = dijkstra(trav, src)
  assert np.array_equal(d, _scipy(trav, src))
  assert (d[trav] > 0).sum() == trav.sum() - 1     # one corridor: every free cell is reachable
  assert certificate(trav[None], src[None], d[None])
  for bad in (d + (d > 0), np.where(d == d.max(), -1, d), np.where(d < 0, -2, d), d.astype(np.int64)):
    assert not certificate(trav[None], src[None], bad[None])
  assert np.array_equal(oracle(np.zeros((2, 3, 4), bool), np.ones((2, 3, 4), bool)), np.zeros((2, 3, 4), np.int32))
