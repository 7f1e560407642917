"""distance_transform (dm_distance_transform_f32) against scipy.ndimage.distance_transform_edt: dist bit for bit, and
nearest by the tie-independent check of tests/_distance.py, with and without return_indices.  Shapes around the
kernels' 32-cell row chunks, 4-row and 128-column CTAs (1 x 1 to 400 x 400, b = 1 and 32, and 2400 x 2400), random
masks at densities 0.001, 0.5 and 0.999, spirals, checkerboards, stripes, rooms, a single False cell, full and empty
planes, (b, C, H, W) input, views, a batch mixing planes with and without a False cell, squared distances above 2^24,
MapBuilder world maps (obstacle and free masks, growing and fixed canvas, the class planes of a semantic map) and both
docstring recipes.  Also: determinism, no host sync, one launch per call on a side stream, inputs never written, and
capture in a CUDA graph."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._components import pattern
from tests._distance import check_nearest, oracle, sqrtf_plane
from tests.test_gpu_components import _world
from tests._geodesic import cells_to_mask, certificate

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (1, 31), (1, 33), (31, 1), (33, 2), (4, 32), (5, 64), (32, 129), (97, 40), (128, 200)]
KINDS = ["random 0.001", "random 0.5", "random 0.999", "spiral", "checkerboard", "vertical stripes",
         "horizontal stripes", "rooms", "single False", "all true", "all false"]


def make(kind: str, H: int, W: int, rng) -> np.ndarray:
  if kind == "single False":
    plane = np.ones((H, W), bool)
    plane[rng.integers(H), rng.integers(W)] = False
    return plane
  return pattern(kind, H, W, rng)


def _check(mask: torch.Tensor):
  """Runs both forms of the call and compares them with the oracle."""
  dist, nearest = dmap.distance_transform(mask, return_indices=True)
  dist2 = dmap.distance_transform(mask)
  assert dist.dtype == torch.float32 and nearest.dtype == torch.int32
  assert dist.shape == mask.shape and nearest.shape == (*mask.shape, 2) and dist.is_cuda and nearest.is_cuda
  assert torch.equal(dist, dist2)
  m = mask.cpu().numpy()
  got = dist.cpu().numpy()
  want = oracle(m)
  assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "dist differs from scipy"
  check_nearest(m, got, nearest.cpu().numpy())
  return dist, nearest


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("H,W", SHAPES)
def test_matches_oracle(H, W, kind):
  rng = np.random.default_rng(H * 1000 + W + 7 * len(kind))
  _check(torch.from_numpy(np.stack([make(kind, H, W, rng) for _ in range(3)])).cuda())


@pytest.mark.parametrize("b", [1, 32])
@pytest.mark.parametrize("H,W", [(400, 400), (129, 257), (257, 33)])
def test_batches(b, H, W):
  rng = np.random.default_rng(b + H + W)
  _check(torch.from_numpy(np.stack([make((KINDS * 4)[i], H, W, rng) for i in range(b)])).cuda())


def test_mixed_batch_and_views():
  rng = np.random.default_rng(3)
  planes = [make(k, 70, 90, rng) for k in ("random 0.5", "all true", "single False", "all true", "random 0.999")]
  mask = torch.from_numpy(np.stack(planes)).cuda()
  dist, nearest = _check(mask)
  assert torch.isinf(dist[1]).all() and (nearest[1] == -1).all() and torch.isfinite(dist[2]).all()
  for i in range(5):                       # a plane's result does not depend on the others
    d, n = dmap.distance_transform(mask[i:i + 1], return_indices=True)
    assert torch.equal(d, dist[i:i + 1]) and torch.equal(n, nearest[i:i + 1])


def test_4d_equals_planes():
  rng = np.random.default_rng(4)
  mask = torch.from_numpy(rng.random((3, 5, 70, 90)) < 0.97).cuda()
  mask[1, 2] = True                        # one plane without a False cell
  dist, nearest = _check(mask)
  for c in range(5):
    d, n = dmap.distance_transform(mask[:, c], return_indices=True)   # a non-contiguous view
    assert torch.equal(d, dist[:, c]) and torch.equal(n, nearest[:, c])
  expanded = mask[:, :1].expand(3, 4, 70, 90)
  d, n = dmap.distance_transform(expanded, return_indices=True)
  assert torch.equal(d, dist[:, :1].expand(3, 4, 70, 90)) and torch.equal(n, nearest[:, :1].expand(3, 4, 70, 90, 2))
  t = mask.transpose(2, 3)                 # (3, 5, 90, 70), not contiguous
  _check(t)


def test_2400():
  rng = np.random.default_rng(24)
  mask = np.stack([pattern("rooms", 2400, 2400, rng), pattern("random 0.999", 2400, 2400, rng),
                   pattern("random 0.5", 2400, 2400, rng)])
  _check(torch.from_numpy(mask).cuda())


def test_squared_distances_above_2_pow_24():
  """One False cell at (0, 0) of an 8 x 6000 plane, its transpose and a 2 x 6000 plane: d2 up to 5999^2 + 7^2."""
  plane = sqrtf_plane()
  wide = np.ones((2, 6000), bool)
  wide[0, 0] = False
  for p in (plane, plane.T.copy(), wide):
    _check(torch.from_numpy(p)[None].cuda())
  r, c = np.indices(plane.shape)
  d2 = (r ** 2 + c ** 2).astype(np.int64)
  assert d2.max() > 2 ** 24
  dist = dmap.distance_transform(torch.from_numpy(plane)[None].cuda())[0].cpu().numpy()
  assert (np.sqrt(d2.astype(np.float32)) != dist).sum() > 1000   # sqrtf would have given other bits


def test_determinism():
  rng = np.random.default_rng(8)
  mask = np.stack([pattern("checkerboard", 301, 299, rng), make("single False", 301, 299, rng),
                   pattern("rooms", 301, 299, rng), rng.random((301, 299)) < 0.995])
  mask[1, 0, 0] = mask[1, -1, -1] = False   # many ties between two far corners
  m = torch.from_numpy(mask).cuda()
  d0, n0 = dmap.distance_transform(m, return_indices=True)
  for _ in range(5):
    d, n = dmap.distance_transform(m, return_indices=True)
    assert torch.equal(d, d0) and torch.equal(n, n0)


def _obstacle_free(world):
  seen = world.mask[:, 0]
  obstacle = seen & (world.height_map[:, 0] > 0.2)
  return seen, obstacle, seen & ~obstacle


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_builder_world_maps(fixed):
  world = _world(fixed)
  seen, obstacle, free = _obstacle_free(world)
  assert obstacle.any() and free.any()
  for mask in (~obstacle, ~free, free, seen):
    _check(mask)


def test_semantic_class_planes():
  world = _world(kind="labels", C=16, b=4)
  planes = world.topdown_map > 0.5          # (b, C, H, W): the cells each class was seen on
  assert planes.dim() == 4 and planes.shape[1] == 16 and planes.any()
  _check(planes)
  _check(~planes)


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_inflation_recipe(fixed):
  """The docstring's obstacle inflation: the geodesic field over the cells more than r metres from every obstacle
  equals the one over the thresholded oracle."""
  world = _world(fixed)
  seen, obstacle, free = _obstacle_free(world)
  r, map_res = 0.18, world.proj.map_res
  traversable = free & (dmap.distance_transform(~obstacle) * map_res > r)
  field = world.geodesic_distance(traversable)
  want_trav = free.cpu().numpy() & (oracle((~obstacle).cpu().numpy()) * np.float32(map_res) > r)
  assert np.array_equal(traversable.cpu().numpy(), want_trav)
  assert traversable.sum() < free.sum()     # the inflation removed cells
  want = dmap.geodesic_distance(torch.from_numpy(want_trav).cuda(), world.get_camera())
  assert torch.equal(field, want)
  src = cells_to_mask(world.get_camera().cpu().numpy()[:, None], *want_trav.shape[-2:])
  assert certificate(want_trav, src, field.cpu().numpy())


def test_goal_snapping_recipe():
  world = _world(None)
  seen, obstacle, free = _obstacle_free(world)
  d, nearest = dmap.distance_transform(~free, return_indices=True)
  fr = free.cpu().numpy()
  near = nearest.cpu().numpy()
  check_nearest(~fr, d.cpu().numpy(), near)
  ob = obstacle.cpu().numpy()
  for i in range(fr.shape[0]):
    zs, xs = np.nonzero(ob[i])               # goals on obstacles
    for z, x in list(zip(zs, xs))[:50]:
      x_free, z_free = near[i, z, x]
      assert fr[i, z_free, x_free]
      best = np.min((np.nonzero(fr[i])[0] - z) ** 2 + (np.nonzero(fr[i])[1] - x) ** 2)
      assert (z_free - z) ** 2 + (x_free - x) ** 2 == best


def test_no_sync_one_launch_side_stream_inputs_untouched():
  rng = np.random.default_rng(5)
  mask = torch.from_numpy(rng.random((4, 3, 300, 260)) < 0.95).cuda()
  view = mask[:, 1]
  keep = mask.clone()
  want = [dmap.distance_transform(mask, return_indices=True), (dmap.distance_transform(view),)]
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    with torch.cuda.stream(side):
      got = [dmap.distance_transform(mask, return_indices=True)]
      assert nat.launch_count() - before == 1
      got.append((dmap.distance_transform(view),))
      assert nat.launch_count() - before == 2
  finally:
    torch.cuda.set_sync_debug_mode(0)
  torch.cuda.current_stream().wait_stream(side)
  for g, w in zip(got, want):
    assert all(torch.equal(x, y) for x, y in zip(g, w))
  assert torch.equal(mask, keep)
  torch.cuda.synchronize()
  nat.device_status()


def test_cuda_graph_replay_sees_new_contents():
  rng = np.random.default_rng(9)
  first, second = (rng.random((2, 2, 150, 170)) < 0.98 for _ in range(2))
  second[1, 0] = True                       # a plane without a False cell in the second contents
  mask = torch.from_numpy(first).cuda()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    dmap.distance_transform(mask, return_indices=True)   # warm up off the capture
  torch.cuda.current_stream().wait_stream(side)
  torch.cuda.synchronize()
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    dist, nearest = dmap.distance_transform(mask, return_indices=True)
  for contents in (second, first):
    mask.copy_(torch.from_numpy(contents))
    graph.replay()
    torch.cuda.synchronize()
    got = dist.cpu().numpy()
    assert np.array_equal(got, oracle(contents))
    check_nearest(contents, got, nearest.cpu().numpy())
  nat.device_status()
