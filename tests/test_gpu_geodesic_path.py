"""geodesic_path (dm_geodesic_path_i32) against the plain-Python oracle of tests/_geodesic_path.py, bit for bit, with
dist from geodesic_distance on the device: random grids at several densities, rooms and a spiral maze, shapes from 1 x 1
to 400 x 400 with H != W, b from 1 to 32 and n from 1 to 64, starts at corners, on borders, on obstacles, on goals and
outside the map, max_cells of 1, small values, exactly the path length and H * W, (b, 1, H, W) inputs, non-contiguous
views and a dist that is not a distance field.  Also: the certificate on 2400 x 2400 grids and MapBuilder world maps
(growing and fixed canvas), TopdownMap's default start, the waypoint recipe against a numpy restatement, an output
above 2^31 elements, no host sync, one launch per call on the current stream, inputs never written, CUDA-graph replay
and a device mismatch."""
import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._geodesic import spiral_maze
from tests._geodesic_path import certificate, oracle
from tests._visibility import visible_window
from tests.test_gpu_semantic_builder import LOCAL, _builder, _depth, _walk

pytestmark = pytest.mark.gpu


def _grid(kind, b, H, W, rng):
  if kind.startswith("random"):
    return rng.random((b, H, W)) >= float(kind.split()[1])
  if kind == "rooms":      # walls every 37 rows / 29 columns with doors
    t = np.ones((b, H, W), bool)
    t[:, 36::37, :] = False
    t[:, :, 28::29] = False
    t[:, 36::37, 5::29] = True
    t[:, 10::37, 28::29] = True
    return t
  if kind == "spiral":
    return np.broadcast_to(spiral_maze(H, W), (b, H, W)).copy()
  raise ValueError(kind)


def _starts(rng, trav, goals, n):
  """(b, n, 2) int64: random cells, then corners, border cells, cells outside the map, a goal and an obstacle."""
  b, H, W = trav.shape
  s = np.stack([rng.integers(0, W, size=(b, n)), rng.integers(0, H, size=(b, n))], axis=-1)
  special = [(0, 0), (W - 1, H - 1), (W - 1, 0), (0, H - 1), (W // 2, 0), (0, H // 2), (-1, H // 2), (W, 0),
             (W // 2, H), (-5, -5)]
  for k in range(min(n, len(special))):
    s[:, (k * 3 + 1) % n] = special[k]
  for i in range(b):
    for k, where in ((n - 1, goals[i]), (n - 2, ~trav[i])):
      zs, xs = np.nonzero(where)
      if n > len(special) + 2 and len(zs):
        j = rng.integers(len(zs))
        s[i, k] = (xs[j], zs[j])
  return s.astype(np.int64)


def _run(trav, dist, starts, max_cells):
  """The call with device and with host starts (they must agree), against the oracle; returns the host results."""
  t = torch.from_numpy(trav).cuda() if isinstance(trav, np.ndarray) else trav
  cells, lengths = dmap.geodesic_path(t, dist, torch.from_numpy(starts).cuda(), max_cells)
  c2, l2 = dmap.geodesic_path(t, dist, starts, max_cells)
  assert torch.equal(cells, c2) and torch.equal(lengths, l2)
  assert cells.dtype == torch.int32 and lengths.dtype == torch.int32
  assert cells.shape == (*starts.shape[:2], max_cells, 2) and lengths.shape == starts.shape[:2]
  b, H, W = t.shape[0], t.shape[-2], t.shape[-1]
  th, dh = t.reshape(b, H, W).cpu().numpy(), dist.reshape(b, H, W).cpu().numpy()
  want_c, want_l = oracle(th, dh, starts, max_cells)
  got_c, got_l = cells.cpu().numpy(), lengths.cpu().numpy()
  assert np.array_equal(got_l, want_l)
  assert np.array_equal(got_c, want_c)
  return th, dh, got_c, got_l


def _certify(trav, dist, starts, cells, lengths, full=True):
  """Every non-empty path is a certified shortest path (full: max_cells was never the limit)."""
  n_ok = 0
  for i in range(cells.shape[0]):
    for k in range(cells.shape[1]):
      x, z = starts[i, k]
      inside = 0 <= x < trav.shape[2] and 0 <= z < trav.shape[1]
      if not inside or dist[i, z, x] < 0:
        assert lengths[i, k] == 0
        continue
      if full:
        assert certificate(trav[i], dist[i], (x, z), cells[i, k, :lengths[i, k]])
        n_ok += 1
  return n_ok


SHAPES = [(1, 1), (1, 57), (45, 1), (33, 65), (97, 40), (128, 200)]
KINDS = ["random 0.0", "random 0.2", "random 0.45", "rooms", "spiral"]


@pytest.mark.parametrize("H,W", SHAPES)
@pytest.mark.parametrize("kind", KINDS)
def test_matches_oracle(kind, H, W):
  rng = np.random.default_rng(H * 1000 + W + len(kind))
  b, n = 3, 16
  trav = _grid(kind, b, H, W, rng)
  goals = rng.random((b, H, W)) < 0.002
  goals[:, 0, 0] = True
  dist = dmap.geodesic_distance(torch.from_numpy(trav).cuda(), torch.from_numpy(goals).cuda())
  starts = _starts(rng, trav, goals, n)
  th, dh, cells, lengths = _run(trav, dist, starts, H * W)
  _certify(th, dh, starts, cells, lengths)


@pytest.mark.parametrize("b,n,H,W,kind", [(32, 64, 61, 47, "random 0.2"), (1, 64, 400, 400, "rooms"),
                                          (2, 1, 400, 311, "spiral"), (32, 1, 20, 90, "random 0.45"),
                                          (1, 3, 1, 1, "random 0.0")])
def test_batch_starts_and_400(b, n, H, W, kind):
  rng = np.random.default_rng(b * 100 + n + H)
  trav = _grid(kind, b, H, W, rng)
  goals = np.zeros((b, H, W), bool)
  goals[:, H - 1, W - 1] = goals[:, 0, 0] = True
  t = torch.from_numpy(trav).cuda()
  dist = dmap.geodesic_distance(t, torch.from_numpy(goals).cuda())
  starts = _starts(rng, trav, goals, n)
  th, dh, cells, lengths = _run(t, dist, starts, H * W)
  _certify(th, dh, starts, cells, lengths)
  if kind == "spiral":          # the inner end of the one-cell corridor: a path of thousands of cells
    far = dh.reshape(b, -1).argmax(1)
    long = _run(t, dist, np.stack([far % W, far // W], -1)[:, None].astype(np.int64), H * W)[3]
    assert long.min() > 5000


def test_max_cells_one_small_exact_and_full():
  rng = np.random.default_rng(7)
  b, n, H, W = 4, 12, 70, 90
  trav = _grid("rooms", b, H, W, rng)
  goals = np.zeros((b, H, W), bool)
  goals[:, 5, 80] = True
  t = torch.from_numpy(trav).cuda()
  dist = dmap.geodesic_distance(t, torch.from_numpy(goals).cuda())
  starts = _starts(rng, trav, goals, n)
  full = _run(t, dist, starts, H * W)[3]
  assert full.max() > 20
  for m in (1, 2, 3, 17, int(full.max()), int(full.max()) - 1):
    lengths = _run(t, dist, starts, m)[3]
    assert np.array_equal(lengths, np.minimum(full, m))


def test_views_and_4d_inputs():
  rng = np.random.default_rng(8)
  b, n, H, W = 3, 9, 50, 66
  trav = _grid("random 0.2", b, H, W, rng)
  goals = rng.random((b, H, W)) < 0.003
  t = torch.from_numpy(trav).cuda()
  dist = dmap.geodesic_distance(t, torch.from_numpy(goals).cuda())
  starts = _starts(rng, trav, goals, n)
  want = dmap.geodesic_path(t, dist, torch.from_numpy(starts).cuda(), 300)
  t_view = torch.stack([~t, t], dim=1)[:, 1]              # channel-strided views
  d_view = torch.stack([dist, dist + 1], dim=-1)[..., 0]
  s_view = torch.stack([torch.from_numpy(starts).cuda()] * 2, dim=1)[:, 0]
  assert not t_view.is_contiguous() and not d_view.is_contiguous() and not s_view.is_contiguous()
  for tt, dd, ss in ((t_view, d_view, s_view), (t[:, None], dist[:, None], s_view), (t[:, None], dist, starts),
                     (t, dist[:, None], starts.astype(np.int32))):
    got = dmap.geodesic_path(tt, dd, ss, 300)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
  one = dmap.geodesic_path(t, dist, starts[:, 4], 300)    # (b, 2): n = 1 kept
  assert one[0].shape == (b, 1, 300, 2) and torch.equal(one[0][:, 0], want[0][:, 4])


def test_a_dist_that_is_not_a_field():
  rng = np.random.default_rng(9)
  b, n, H, W = 4, 40, 30, 37
  trav = rng.random((b, H, W)) > 0.15
  dist = rng.integers(-1, 20, size=(b, H, W)).astype(np.int32)
  dist[:, 0, :3] = [np.iinfo(np.int32).max, np.iinfo(np.int32).min, 0]
  dist[:, 1, 0] = np.iinfo(np.int32).max - 5
  trav[:, :2, 0] = True
  starts = _starts(rng, trav, dist == 0, n)
  starts[:, 0] = (0, 0)
  _, _, cells, lengths = _run(trav, torch.from_numpy(dist).cuda(), starts, H * W)
  assert lengths[:, 0].min() >= 2 and (lengths > 1).sum() > 10


def test_certificate_2400():
  rng = np.random.default_rng(11)
  H = W = 2400
  trav = np.concatenate([_grid("rooms", 1, H, W, rng), _grid("random 0.25", 1, H, W, rng)])
  goals = np.zeros_like(trav)
  goals[0, 1200, 1200] = goals[1, 5, 7] = goals[1, 2000, 300] = True
  t = torch.from_numpy(trav).cuda()
  dist = dmap.geodesic_distance(t, torch.from_numpy(goals).cuda())
  starts = _starts(rng, trav, goals, 14)
  starts[:, 2] = (2399, 2399)
  max_cells = int(dist.max()) // 5 + 1
  th, dh, cells, lengths = _run(t, dist, starts, max_cells)
  assert _certify(th, dh, starts, cells, lengths) >= 10 and lengths.max() > 1000


def _world(b=6, T=10, fixed=None):
  poses = _walk(b, T, seed=41)
  nb = _builder(True, fixed=fixed)
  for t in range(T):
    nb.step(_depth(b, poses[t], 41), cam_pose=poses[t], **LOCAL)
  return nb.world_map


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_builder_world_maps_and_default_start(fixed):
  world = _world(fixed=fixed)
  hm, mask = world.height_map[:, 0], world.mask[:, 0]
  # unknown cells count as free: on these short walks the seen free cells around the agent do not connect to it
  free = (mask & (hm <= 0.2)) | ~mask
  b, H, W = free.shape
  cam = world.get_camera()
  free[torch.arange(b), cam[:, 1], cam[:, 0]] = True     # the agent stands on a free cell
  to_agent = world.geodesic_distance(free)
  # the goal of each environment: its free cell farthest from the agent, so the path spans the explored area
  far = to_agent.flatten(1).argmax(1)
  goals = torch.stack([far % W, far // W], dim=-1)
  dist = dmap.geodesic_distance(free, goals)
  max_cells = int(dist.max()) // 5 + 1
  cells, lengths = world.geodesic_path(free, dist, max_cells)
  want = dmap.geodesic_path(free, dist, cam, max_cells)
  assert torch.equal(cells, want[0]) and torch.equal(lengths, want[1])
  assert cells.shape == (b, 1, max_cells, 2)
  fh, dh = free.cpu().numpy(), dist.cpu().numpy()
  rng = np.random.default_rng(12)
  starts = np.concatenate([cam.cpu().numpy()[:, None], _starts(rng, fh, dh == 0, 15)], axis=1)
  _, _, c, l = _run(free, dist, starts, max_cells)
  assert _certify(fh, dh, starts, c, l) >= b and (l[:, 0] >= 1).all() and (l[:, 0] > 1).any()
  assert np.array_equal(c[:, :1], cells.cpu().numpy())


def test_waypoint_recipe():
  """The docstring's recipe, run as written, against the same quantity restated with numpy and the visibility
  oracle: the farthest path index whose cells from the start on all lie in the window and are visible."""
  rng = np.random.default_rng(13)
  b, n, H, W, r, max_cells = 3, 10, 80, 70, 12, 400
  trav_np = _grid("random 0.2", b, H, W, rng)
  trav_np[:, 30:50, 33] = False                           # a wall the paths bend around
  traversable = torch.from_numpy(trav_np).cuda()
  goals = np.zeros((b, H, W), bool)
  goals[:, 40, 60] = True
  dist = dmap.geodesic_distance(traversable, torch.from_numpy(goals).cuda())
  starts = torch.from_numpy(_starts(rng, trav_np, goals, n)).cuda()
  cells, lengths = dmap.geodesic_path(traversable, dist, starts, max_cells)
  side = 2 * r + 1
  vis = dmap.visible_cells(~traversable, starts, r).flatten(2)
  rel = cells.long() - starts[:, :, None, :] + r
  ok = ((rel >= 0) & (rel < side)).all(-1)
  ok &= torch.arange(max_cells, device=cells.device) < lengths[..., None]
  seen = vis.gather(2, (rel[..., 1] * side + rel[..., 0]).clamp(0, side * side - 1)) & ok
  j = seen.int().cumprod(-1).sum(-1) - 1
  waypoint = cells.gather(2, j.clamp(min=0).long()[..., None, None].expand(-1, -1, 1, 2))[:, :, 0]
  c, l, s = cells.cpu().numpy(), lengths.cpu().numpy(), starts.cpu().numpy()
  want_j = np.full((b, n), -1)
  for i in range(b):
    for k in range(n):
      sx, sz = s[i, k]
      win = visible_window(~trav_np[i], sx, sz, r)
      for q in range(l[i, k]):
        dx, dz = c[i, k, q] - (sx, sz)
        if max(abs(dx), abs(dz)) > r or not win[r + dz, r + dx]:
          break
        want_j[i, k] = q
  assert np.array_equal(j.cpu().numpy(), want_j)
  assert (want_j > 0).sum() >= b and (want_j[l > 0] < l[l > 0] - 1).any()   # some waypoints short of the goal
  has = want_j >= 0
  assert np.array_equal(waypoint.cpu().numpy()[has], c[has, want_j[has]])


def test_output_above_2_31_elements():
  """b * n * max_cells * 2 > 2^31 int32: the last paths lie past element 2^31; their far end is checked."""
  H = W = 1024
  b, n, max_cells = 1, 1025, H * W
  assert b * n * max_cells * 2 > 2 ** 31
  trav = torch.ones((b, H, W), dtype=torch.bool, device="cuda")
  trav[0, 500, 100:900] = False
  dist = dmap.geodesic_distance(trav, torch.tensor([[[0, 0]]]))
  starts = torch.tensor([[[(k * 37) % W, (k * 11) % H] for k in range(n)]], dtype=torch.int64)
  starts[0, -1] = torch.tensor([W - 1, H - 1])
  starts[0, -2] = torch.tensor([W, 0])                    # outside
  cells, lengths = dmap.geodesic_path(trav, dist, starts, max_cells)
  th, dh = trav.cpu().numpy(), dist.cpu().numpy()
  want_c, want_l = oracle(th, dh, starts[:, -3:].numpy(), 2048)
  got_l = lengths[0, -3:].cpu().numpy()
  assert np.array_equal(got_l, want_l[0]) and got_l[-1] > 1000 and got_l[-2] == 0
  tail = cells[0, -3:, :2048].cpu().numpy()
  assert np.array_equal(tail, want_c[0])
  assert (cells[0, -3:, 2048:] == -1).all() and int(cells[0, -1, -1, 1]) == -1
  assert certificate(th[0], dh[0], (W - 1, H - 1), tail[-1, :got_l[-1]])
  del cells, lengths
  torch.cuda.empty_cache()


def test_no_sync_one_launch_current_stream_inputs_untouched():
  rng = np.random.default_rng(5)
  b, H, W = 4, 300, 260
  trav_np = _grid("rooms", b, H, W, rng)
  trav = torch.from_numpy(trav_np).cuda()[:, None]
  dist = dmap.geodesic_distance(trav, torch.from_numpy(rng.random((b, H, W)) < 0.001).cuda()[:, None])
  s_dev = torch.tensor(rng.integers(0, 260, size=(b, 5, 2)), device="cuda")
  s_host = rng.integers(0, 260, size=(b, 5, 2))
  s_big = np.stack([rng.integers(0, W, size=(b, 3000)), rng.integers(0, H, size=(b, 3000))], -1)  # pinned copy
  keep = [trav.clone(), dist.clone(), s_dev.clone()]
  world = _world(b=2, T=3)
  free = world.mask[:, 0] | True
  world_dist = dmap.geodesic_distance(free, torch.tensor([[[3, 4]], [[5, 6]]]))

  def calls():
    return [dmap.geodesic_path(trav, dist, s_dev, 2000), dmap.geodesic_path(trav, dist, s_host, 7),
            dmap.geodesic_path(trav, dist, s_big, 64), world.geodesic_path(free, world_dist, 500)]

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
    assert torch.equal(o[0], w[0]) and torch.equal(o[1], w[1])
  assert torch.equal(trav, keep[0]) and torch.equal(dist, keep[1]) and torch.equal(s_dev, keep[2])
  nat.device_status()


def test_cuda_graph_replay_sees_new_contents():
  rng = np.random.default_rng(14)
  b, n, H, W, max_cells = 2, 6, 60, 75, 900
  contents = []
  for _ in range(2):
    trav_np = _grid("random 0.2", b, H, W, rng)
    goals = rng.random((b, H, W)) < 0.002
    goals[:, 30, 30] = True
    contents.append((trav_np, goals, _starts(rng, trav_np, goals, n)))
  trav = torch.from_numpy(contents[0][0]).cuda()
  dist = dmap.geodesic_distance(trav, torch.from_numpy(contents[0][1]).cuda())
  starts = torch.from_numpy(contents[0][2]).cuda()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    dmap.geodesic_path(trav, dist, starts, max_cells)     # warm up off the capture
  torch.cuda.current_stream().wait_stream(side)
  torch.cuda.synchronize()
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    cells, lengths = dmap.geodesic_path(trav, dist, starts, max_cells)
  for trav_np, goals, s in (contents[1], contents[0]):
    trav.copy_(torch.from_numpy(trav_np))
    dist.copy_(dmap.geodesic_distance(trav, torch.from_numpy(goals).cuda()))
    starts.copy_(torch.from_numpy(s))
    graph.replay()
    torch.cuda.synchronize()
    want_c, want_l = oracle(trav_np, dist.cpu().numpy(), s, max_cells)
    assert np.array_equal(lengths.cpu().numpy(), want_l) and np.array_equal(cells.cpu().numpy(), want_c)
  nat.device_status()


def test_device_mismatch_is_a_value_error():
  t = torch.ones((2, 5, 6), dtype=torch.bool, device="cuda")
  d = torch.zeros((2, 5, 6), dtype=torch.int32)
  with pytest.raises(ValueError, match="dist must be on"):
    dmap.geodesic_path(t, d, [[1, 1], [2, 2]], 3)
  if torch.cuda.device_count() > 1:
    with pytest.raises(ValueError, match="dist must be on"):
      dmap.geodesic_path(t, d.to("cuda:1"), [[1, 1], [2, 2]], 3)
    with pytest.raises(ValueError, match="starts must be on"):
      dmap.geodesic_path(t, d.cuda(), torch.zeros((2, 2), dtype=torch.int64, device="cuda:1"), 3)
