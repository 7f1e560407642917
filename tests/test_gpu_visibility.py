"""visible_cells / count_visible (dm_line_of_sight_u8) against the numpy oracle of tests/_visibility.py, bit for bit:
random maps at blocking densities 0, 5 %, 30 % and 100 %, H != W and maps smaller than the window, origins at corners,
on borders, on blocking cells and outside the map, radii 0 to 512, b up to 8 and n up to 16, C = 1 and 16 target
planes, (b, 1, H, W) blocking and non-contiguous views.  count_visible equals the visible windows ANDed with the target
windows on every case.  Also: MapBuilder world maps with TopdownMap's default origin, a window output above 2^31
elements, no host sync, one launch per call on the current stream, inputs never written."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._visibility import count_visible, target_windows, visible_cells
from tests.test_gpu_semantic_builder import LOCAL, _builder, _depth, _walk

pytestmark = pytest.mark.gpu


def _origins(rng, b, n, H, W):
  """Random cells plus the corners, border cells and cells just outside the map."""
  special = [(0, 0), (W - 1, H - 1), (W - 1, 0), (0, H - 1), (W // 2, 0), (0, H // 2), (-1, H // 2), (W, 0),
             (W // 2, H), (-5, -5)]
  o = np.stack([rng.integers(0, W, size=(b, n)), rng.integers(0, H, size=(b, n))], axis=-1)
  for k in range(min(n, len(special))):
    o[:, (k * 3 + 1) % n] = special[k]
  return o.astype(np.int64)


def _check(blocking, targets, origins, r, views=False):
  """Both entries against the oracle, and against each other."""
  bt = torch.from_numpy(blocking).cuda()
  tt = torch.from_numpy(targets).cuda()
  if views:        # (b, 1, H, W) blocking, a channel-strided view of the targets
    bt = bt[:, None]
    tt = torch.stack([tt, tt], dim=2)[:, :, 1]
    assert not tt.is_contiguous()
  vis = dmap.visible_cells(bt, torch.from_numpy(origins).cuda(), r)
  cnt = dmap.count_visible(bt, tt, origins, r)            # host origins
  want = visible_cells(blocking, origins, r)
  assert np.array_equal(vis.cpu().numpy(), want)
  assert np.array_equal(cnt.cpu().numpy(), count_visible(blocking, targets, origins, r))
  tw = torch.from_numpy(target_windows(targets, origins, r)).cuda()
  assert torch.equal(cnt, (vis[:, None] & tw).sum(dim=(3, 4), dtype=torch.int32))
  return want


CASES = [  # (density, b, n, H, W, r, C)
  (0.0, 2, 5, 40, 57, 7, 1), (0.05, 3, 16, 64, 48, 33, 1), (0.3, 8, 4, 33, 70, 7, 16), (1.0, 2, 6, 20, 25, 2, 1),
  (0.05, 2, 3, 30, 19, 1, 16), (0.3, 1, 16, 9, 13, 0, 1), (0.0, 1, 4, 300, 260, 166, 1),
  (0.05, 2, 3, 150, 170, 166, 16), (0.3, 4, 8, 200, 90, 33, 1), (0.05, 2, 4, 5, 3, 7, 1), (1.0, 1, 3, 1, 1, 33, 1),
]


@pytest.mark.parametrize("density,b,n,H,W,r,C", CASES)
def test_matches_oracle(density, b, n, H, W, r, C):
  rng = np.random.default_rng(int(density * 100) + b * 7 + n * 13 + H + W * 3 + r + C)
  blocking = rng.random((b, H, W)) < density
  targets = rng.random((b, C, H, W)) < 0.4
  origins = _origins(rng, b, n, H, W)
  want = _check(blocking, targets, origins, r, views=(C == 16))
  if density == 0.0:     # an open map: every window is the disk clipped to the map
    assert want.any()


@pytest.mark.parametrize("r", [512, 166])
def test_large_radius_few_origins(r):
  rng = np.random.default_rng(r)
  b, n, H, W = 2, 3, 60, 45
  blocking = rng.random((b, H, W)) < 0.05
  targets = rng.random((b, 1, H, W)) < 0.5
  origins = np.array([[[0, 0], [44, 59], [20, 30]], [[-1, 3], [22, 0], [44, 10]]], np.int64)
  _check(blocking, targets, origins, r)
  open_ = np.zeros((1, H, W), bool)
  _check(open_, targets[:1], origins[:1], r)


def test_origins_on_blocking_cells_and_3d_targets():
  rng = np.random.default_rng(4)
  b, n, H, W, r = 3, 6, 50, 61, 12
  blocking = rng.random((b, H, W)) < 0.3
  origins = _origins(rng, b, n, H, W)
  for i in range(b):
    blocking[i, origins[i, 2, 1], origins[i, 2, 0]] = True
  targets = rng.random((b, H, W)) < 0.3
  got = dmap.count_visible(torch.from_numpy(blocking).cuda(), torch.from_numpy(targets).cuda(),
                           torch.from_numpy(origins[:, 2]), r)           # (b, 2): n = 1 kept
  assert got.shape == (b, 1)
  want = count_visible(blocking, targets[:, None], origins[:, 2:3], r)[:, 0]
  assert np.array_equal(got.cpu().numpy(), want)
  vis = dmap.visible_cells(torch.from_numpy(blocking).cuda(), origins[:, 2], r)
  assert vis.shape == (b, 1, 2 * r + 1, 2 * r + 1) and vis[:, 0, r, r].all()   # an origin on a blocking cell


def _world(b=4, T=8, fixed=None):
  poses = _walk(b, T, seed=31)
  nb = _builder(True, fixed=fixed)
  for t in range(T):
    nb.step(_depth(b, poses[t], 31), cam_pose=poses[t], **LOCAL)
  return nb.world_map


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_builder_world_maps(fixed):
  world = _world(fixed=fixed)
  seen = world.mask[:, 0]
  obstacle = seen & (world.height_map[:, 0] > 0.2)
  cam = world.get_camera()
  r = 40
  vis = world.visible_cells(obstacle, r)
  assert torch.equal(vis, dmap.visible_cells(obstacle, cam, r))
  cnt = world.count_visible(obstacle, ~seen, r)
  assert torch.equal(cnt, dmap.count_visible(obstacle, ~seen, cam, r))
  o = cam.cpu().numpy()[:, None]
  want = visible_cells(obstacle.cpu().numpy(), o, r)
  assert np.array_equal(vis.cpu().numpy(), want)
  assert np.array_equal(cnt.cpu().numpy(), count_visible(obstacle.cpu().numpy(), (~seen).cpu().numpy()[:, None], o,
                                                         r)[:, 0])
  assert want.any() and obstacle.any()


def test_window_output_above_2_31_elements():
  """b * n * (2r + 1)^2 > 2^31 on an all-blocking map: lines stop at once; the far end of the output is checked."""
  r = 512
  side = 2 * r + 1
  b, n = 1, 2100                          # 2100 * 1025^2 = 2.206e9 bytes
  assert b * n * side * side > 2 ** 31
  H, W = 64, 64
  blocking = torch.ones((b, H, W), dtype=torch.bool, device="cuda")
  origins = torch.tensor([[[(k * 7) % W, (k * 3) % H] for k in range(n)]], dtype=torch.int64)
  origins[0, -1] = torch.tensor([W - 1, H - 1])
  origins[0, -2] = torch.tensor([W, 0])                  # outside
  vis = dmap.visible_cells(blocking, origins, r)
  # on an all-blocking map only the origin and its orthogonal neighbours inside the map are visible: a diagonal
  # neighbour is behind two blocking side cells, and every longer line has a blocking intermediate cell
  corner = torch.tensor([[0, 1, 0], [1, 1, 0], [0, 0, 0]], dtype=torch.bool)
  last = vis[0, -1]                                      # the corner (W - 1, H - 1)
  assert torch.equal(last[r - 1:r + 2, r - 1:r + 2].cpu(), corner)
  assert int(last.sum()) == 3
  assert not vis[0, -2].any()
  mid = vis[0, n // 2]                                   # an origin inside
  x, z = origins[0, n // 2].tolist()
  inside = sum(1 for dx, dz in ((0, 0), (1, 0), (-1, 0), (0, 1), (0, -1)) if 0 <= x + dx < W and 0 <= z + dz < H)
  assert int(mid.sum()) == inside
  del vis, last, mid
  torch.cuda.empty_cache()


def test_no_sync_one_launch_current_stream_inputs_untouched():
  rng = np.random.default_rng(5)
  b, H, W, r = 4, 300, 260, 33
  blocking = torch.from_numpy(rng.random((b, 1, H, W)) < 0.1).cuda()
  targets = torch.from_numpy(rng.random((b, 3, H, W)) < 0.5).cuda()
  o_dev = torch.tensor(rng.integers(0, 260, size=(b, 5, 2)), device="cuda")
  o_host = rng.integers(0, 260, size=(b, 5, 2))
  o_big = np.stack([rng.integers(0, W, size=(b, 3000)), rng.integers(0, H, size=(b, 3000))], -1)  # pinned copy
  keep = [blocking.clone(), targets.clone(), o_dev.clone()]
  world = _world(b=2, T=3)
  obstacle = world.mask[:, 0] & (world.height_map[:, 0] > 0.2)

  def calls():
    return [dmap.visible_cells(blocking, o_dev, r), dmap.visible_cells(blocking, o_host, r),
            dmap.count_visible(blocking, targets, o_dev, r), dmap.count_visible(blocking, targets[:, 0], o_host, r),
            dmap.count_visible(blocking, targets, o_big, 7),
            world.visible_cells(obstacle, r), world.count_visible(obstacle, ~world.mask[:, 0], r)]

  want = calls()
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    with torch.cuda.stream(side):
      outs = calls()
  finally:
    torch.cuda.set_sync_debug_mode(0)
  assert nat.launch_count() - before == len(want)
  torch.cuda.current_stream().wait_stream(side)
  for o, w in zip(outs, want):
    assert torch.equal(o, w)
  assert torch.equal(blocking, keep[0]) and torch.equal(targets, keep[1]) and torch.equal(o_dev, keep[2])
  nat.device_status()


def test_device_mismatch_is_a_value_error():
  blocking = torch.zeros((2, 5, 6), dtype=torch.bool, device="cuda")
  with pytest.raises(ValueError, match="targets must be on"):
    dmap.count_visible(blocking, torch.zeros((2, 5, 6), dtype=torch.bool), [[1, 1], [2, 2]], 3)
  if torch.cuda.device_count() > 1:
    with pytest.raises(ValueError, match="origins must be on"):
      dmap.visible_cells(blocking, torch.zeros((2, 2), dtype=torch.int64, device="cuda:1"), 3)
