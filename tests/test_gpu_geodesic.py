"""geodesic_distance (dm_geodesic_distance_i32) against its definition, bit for bit: the heapq oracle of
tests/_geodesic.py on grids from 1 x 1 to 400 x 400 (random obstacles at several densities, open rooms, a spiral
maze, all blocked, no source, sources on obstacles, disconnected components; both source forms, cells outside the
map; b = 1 and 32), and the certificate at 2400 x 2400 and on MapBuilder world maps.  Also: TopdownMap's default
source against get_camera(), no host sync, a fixed launch count on the current stream, and inputs never written."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._geodesic import cells_to_mask, certificate, oracle, spiral_maze
from tests.test_gpu_semantic_builder import LOCAL, _builder, _depth, _walk

pytestmark = pytest.mark.gpu


def _grid(kind, b, H, W, rng):
  if kind.startswith("random"):
    return rng.random((b, H, W)) >= float(kind.split()[1])
  if kind == "rooms":      # open rooms: walls every 37 rows / 29 columns with doors
    t = np.ones((b, H, W), bool)
    t[:, 36::37, :] = False
    t[:, :, 28::29] = False
    t[:, 36::37, 5::29] = True
    t[:, 10::37, 28::29] = True
    return t
  if kind == "spiral":
    return np.broadcast_to(spiral_maze(H, W), (b, H, W)).copy()
  if kind == "blocked":
    return np.zeros((b, H, W), bool)
  if kind == "components":   # a wall through the middle column: the right half is never reached from the left
    t = rng.random((b, H, W)) >= 0.1
    t[:, :, W // 2] = False
    return t
  raise ValueError(kind)


def _run_both_forms(trav, cells):
  """The field from the cells and from their mask; they must agree."""
  b, H, W = trav.shape
  t = torch.from_numpy(trav).cuda()
  by_cells = dmap.geodesic_distance(t, torch.from_numpy(cells).cuda())
  by_host_cells = dmap.geodesic_distance(t, cells)
  by_mask = dmap.geodesic_distance(t, torch.from_numpy(cells_to_mask(cells, H, W)).cuda())
  assert torch.equal(by_cells, by_mask) and torch.equal(by_cells, by_host_cells)
  return by_cells.cpu().numpy()


SHAPES = [(1, 1), (1, 57), (45, 1), (32, 32), (33, 65), (97, 40), (128, 200)]
KINDS = ["random 0.0", "random 0.2", "random 0.45", "rooms", "spiral", "blocked", "components"]


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("kind", KINDS)
def test_matches_oracle(kind, H, W):
  rng = np.random.default_rng(H * 1000 + W + len(kind))
  b = 4
  trav = _grid(kind, b, H, W, rng)
  # a few cells per environment, some outside the map, some on obstacles
  cells = np.stack([rng.integers(-2, W + 2, size=(b, 5)), rng.integers(-2, H + 2, size=(b, 5))], axis=-1)
  cells[:, 0] = (0, 0)
  got = _run_both_forms(trav, cells)
  want = oracle(trav, cells_to_mask(cells, H, W))
  assert np.array_equal(got, want)


@pytest.mark.parametrize("b", [1, 32])
def test_batch_and_400(b):
  rng = np.random.default_rng(b)
  H, W = (400, 400) if b == 1 else (123, 77)
  trav = np.concatenate([_grid(k, 1, H, W, rng) for k in (KINDS * 5)[:b]])
  cells = np.stack([rng.integers(0, W, size=(b, 3)), rng.integers(0, H, size=(b, 3))], axis=-1)
  got = _run_both_forms(trav, cells)
  src = cells_to_mask(cells, H, W)
  assert np.array_equal(got, oracle(trav, src))


def test_no_source_and_sources_on_obstacles():
  rng = np.random.default_rng(3)
  trav = _grid("random 0.3", 3, 50, 70, rng)
  t = torch.from_numpy(trav).cuda()
  none = dmap.geodesic_distance(t, torch.zeros_like(t))
  assert (none == -1).all()
  src = ~trav & (rng.random(trav.shape) < 0.05)      # only obstacles as goals, as an object's class plane
  got = dmap.geodesic_distance(t, torch.from_numpy(src).cuda()).cpu().numpy()
  assert np.array_equal(got, oracle(trav, src))
  assert (got[src] == 0).all() and (got[~trav & ~src] == -1).all()
  # (b, 1, H, W) inputs and a (b, 2) cell
  got4 = dmap.geodesic_distance(t[:, None], torch.from_numpy(src).cuda()[:, None])
  assert torch.equal(got4.cpu(), torch.from_numpy(got))
  one = dmap.geodesic_distance(t, torch.tensor([[3, 4], [70, 2], [0, 0]], dtype=torch.int32))
  want = oracle(trav, cells_to_mask(np.array([[[3, 4]], [[70, 2]], [[0, 0]]]), 50, 70))
  assert np.array_equal(one.cpu().numpy(), want)


def test_certificate_2400():
  rng = np.random.default_rng(11)
  H = W = 2400
  trav = np.concatenate([_grid("rooms", 1, H, W, rng), _grid("random 0.25", 1, H, W, rng)])
  src = np.zeros_like(trav)
  src[0, 1200, 1200] = src[1, 5, 7] = src[1, 2000, 300] = True
  got = dmap.geodesic_distance(torch.from_numpy(trav).cuda(), torch.from_numpy(src).cuda()).cpu().numpy()
  assert certificate(trav, src, got)
  assert got[0].max() > 5 * 1200


def _world(b=8, T=12, fixed=None):
  poses = _walk(b, T, seed=21)
  nb = _builder(True, fixed=fixed)
  for t in range(T):
    nb.step(_depth(b, poses[t], 21), cam_pose=poses[t], **LOCAL)
  return nb.world_map


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_builder_world_maps(fixed):
  world = _world(fixed=fixed)
  hm, mask = world.height_map[:, 0], world.mask[:, 0]
  for unknown_free in (False, True):
    free = mask & (hm <= 0.2)
    if unknown_free:
      free = free | ~mask
    got = world.geodesic_distance(free)
    want = dmap.geodesic_distance(free, world.get_camera())
    assert torch.equal(got, want)
    src = cells_to_mask(world.get_camera().cpu().numpy()[:, None], *free.shape[-2:])
    assert certificate(free.cpu().numpy(), src, got.cpu().numpy())
    assert (got >= 0).any()


def test_default_source_is_get_camera():
  from dungeon_maps_b200.maps import _camera_cells
  world = _world(b=4, T=5)
  b = world.mask.shape[0]
  assert torch.equal(_camera_cells(world.proj, b), world.get_camera().cpu())
  win = world.select_egocentric(96, 80)
  cam = win.get_camera().cpu().expand(b, 2)   # one row when the window's offsets are scalars
  assert torch.equal(_camera_cells(win.proj, b), cam)
  free = win.mask[:, 0] | True
  got = win.geodesic_distance(free)
  assert torch.equal(got, dmap.geodesic_distance(free, cam))
  assert (got[torch.arange(b), cam[:, 1], cam[:, 0]] == 0).all()


def test_no_sync_fixed_launches_current_stream_inputs_untouched():
  rng = np.random.default_rng(5)
  trav = torch.from_numpy(_grid("rooms", 6, 300, 260, rng)).cuda()
  src = torch.from_numpy(rng.random((6, 300, 260)) < 0.001).cuda()
  cells_dev = torch.tensor(rng.integers(0, 260, size=(6, 4, 2)), device="cuda")
  cells_host = rng.integers(0, 260, size=(6, 4, 2))
  keep = [trav.clone(), src.clone(), cells_dev.clone()]
  world = _world(b=4, T=3)
  free = world.mask[:, 0] | True
  want = [dmap.geodesic_distance(trav, x) for x in (src, cells_dev, cells_host)]
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    with torch.cuda.stream(side):
      outs = [dmap.geodesic_distance(trav, x) for x in (src, cells_dev, cells_host)]
      outs.append(world.geodesic_distance(free))
  finally:
    torch.cuda.set_sync_debug_mode(0)
  assert nat.launch_count() - before == 4
  torch.cuda.current_stream().wait_stream(side)
  for o, w in zip(outs, want):
    assert torch.equal(o, w)
  assert torch.equal(trav, keep[0]) and torch.equal(src, keep[1]) and torch.equal(cells_dev, keep[2])
  nat.device_status()


def test_spiral_worst_case():
  trav = spiral_maze(300, 300)[None]
  src = np.zeros_like(trav)
  src[0, 0, 0] = True
  got = dmap.geodesic_distance(torch.from_numpy(trav).cuda(), torch.from_numpy(src).cuda()).cpu().numpy()
  assert np.array_equal(got, oracle(trav, src))
  nat.device_status()


def test_device_mismatch_is_a_value_error():
  t = torch.ones((2, 5, 6), dtype=torch.bool, device="cuda")
  with pytest.raises(ValueError, match="source mask"):
    dmap.geodesic_distance(t, torch.ones((2, 5, 6), dtype=torch.bool))
