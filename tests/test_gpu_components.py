"""connected_components (dm_connected_components_i32) against scipy.ndimage.label, bit for bit: labels, counts and
sizes under 4- and 8-connectivity, on shapes around the kernel's 32 x 32 tiles (1 x 1 to 400 x 400, b = 1 and 32, and
2400 x 2400), random masks at low, high and percolation-threshold densities, a one-cell spiral, checkerboards, one-cell
stripes, full and empty masks, (b, C, H, W) input, and MapBuilder world maps (seen, free and frontier masks, the class
planes of a semantic map).  Also: no host sync, one launch per call on a side stream, inputs never written, and capture
in a CUDA graph."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._components import PERCOLATION, oracle, pattern
from tests.test_gpu_semantic_builder import LOCAL, _builder, _depth, _inputs, _walk

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (1, 57), (45, 1), (31, 33), (32, 32), (33, 65), (97, 40), (128, 200)]
KINDS = ["random 0.1", "random 0.9", "random percolation", "spiral", "checkerboard", "vertical stripes",
         "horizontal stripes", "all true", "all false"]


def _check(mask: torch.Tensor, connectivity: int):
  """Runs both forms of the call and compares them with the oracle."""
  labels, counts, sizes = dmap.connected_components(mask, connectivity, return_sizes=True)
  labels2, counts2 = dmap.connected_components(mask, connectivity)
  assert labels.dtype == counts.dtype == sizes.dtype == torch.int32
  assert labels.shape == sizes.shape == mask.shape and counts.shape == mask.shape[:-2] and counts.is_cuda
  assert torch.equal(labels, labels2) and torch.equal(counts, counts2)
  want = oracle(mask.cpu().numpy(), connectivity)
  for got, w, what in zip((labels, counts, sizes), want, ("labels", "counts", "sizes")):
    assert np.array_equal(got.cpu().numpy(), w), f"{what} differ from scipy.ndimage.label"
  return labels, counts, sizes


@pytest.mark.parametrize("connectivity", [4, 8])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("H,W", SHAPES)
def test_matches_oracle(H, W, kind, connectivity):
  rng = np.random.default_rng(H * 1000 + W + 7 * len(kind) + connectivity)
  mask = np.stack([pattern(kind, H, W, rng, connectivity) for _ in range(3)])
  _check(torch.from_numpy(mask).cuda(), connectivity)


@pytest.mark.parametrize("b", [1, 32])
@pytest.mark.parametrize("connectivity", [4, 8])
def test_400(b, connectivity):
  rng = np.random.default_rng(b + connectivity)
  mask = np.stack([pattern((KINDS * 4)[i], 400, 400, rng, connectivity) for i in range(b)])
  if b == 1:
    mask[0] = pattern("random percolation", 400, 400, rng, connectivity)
  _check(torch.from_numpy(mask).cuda(), connectivity)


def test_known_counts():
  cb = torch.from_numpy(pattern("checkerboard", 97, 40, None)).cuda()[None]
  assert dmap.connected_components(cb, 8)[1].tolist() == [1]
  assert dmap.connected_components(cb, 4)[1].tolist() == [97 * 40 // 2]   # the largest possible count
  spiral = torch.from_numpy(pattern("spiral", 300, 300, None)).cuda()[None]
  labels, counts, sizes = dmap.connected_components(spiral, 4, return_sizes=True)
  assert counts.tolist() == [1] and int(sizes.max()) == int(spiral.sum())


@pytest.mark.parametrize("connectivity", [4, 8])
def test_4d_equals_planes(connectivity):
  rng = np.random.default_rng(connectivity)
  mask = torch.from_numpy(rng.random((3, 5, 70, 90)) < PERCOLATION[connectivity]).cuda()
  labels, counts, sizes = _check(mask, connectivity)
  for c in range(5):
    l, k, s = dmap.connected_components(mask[:, c], connectivity, return_sizes=True)   # a non-contiguous view
    assert torch.equal(l, labels[:, c]) and torch.equal(k, counts[:, c]) and torch.equal(s, sizes[:, c])
  expanded = mask[:, :1].expand(3, 4, 70, 90)
  l, k = dmap.connected_components(expanded, connectivity)
  assert torch.equal(l, labels[:, :1].expand(3, 4, 70, 90)) and torch.equal(k, counts[:, :1].expand(3, 4))


@pytest.mark.parametrize("connectivity", [4, 8])
def test_2400(connectivity):
  rng = np.random.default_rng(40 + connectivity)
  mask = np.stack([pattern("rooms", 2400, 2400, rng), pattern("random percolation", 2400, 2400, rng, connectivity)])
  labels, counts, _ = _check(torch.from_numpy(mask).cuda(), connectivity)
  assert counts[0] == 1 and counts[1] > 1000     # the doors join all rooms


def _world(fixed=None, kind=None, b=6, T=10, C=8):
  poses = _walk(b, T, seed=31)
  nb = _builder(True, fixed=fixed)
  for t in range(T):
    nb.step(_depth(b, poses[t], 31), cam_pose=poses[t], **LOCAL, **(_inputs(kind, b, C, t) if kind else {}))
  return nb.world_map


def frontier(seen: torch.Tensor, free: torch.Tensor) -> torch.Tensor:
  """connected_components' docstring recipe: seen free cells next to an unseen cell."""
  return free & (F.max_pool2d((~seen).float()[:, None], 3, 1, 1)[:, 0] > 0)


@pytest.mark.parametrize("fixed", [None, (600, 640)])
def test_builder_world_maps(fixed):
  world = _world(fixed)
  seen = world.mask[:, 0]
  free = seen & (world.height_map[:, 0] <= 0.2)
  front = frontier(seen, free)
  assert front.any() and (front & ~free).sum() == 0
  for mask in (seen, free, front):
    for connectivity in (4, 8):
      _check(mask, connectivity)
  labels, counts, sizes = dmap.connected_components(front, return_sizes=True)
  kept = labels * (sizes >= 5)
  assert ((kept > 0) == (front & (sizes >= 5))).all()


def test_semantic_class_planes():
  world = _world(kind="labels", C=16, b=4)
  planes = world.topdown_map > 0.5          # (b, C, H, W): the cells each class was seen on
  assert planes.dim() == 4 and planes.shape[1] == 16 and planes.any()
  for connectivity in (4, 8):
    _check(planes, connectivity)
  _check(world.mask, 8)


def test_no_sync_one_launch_side_stream_inputs_untouched():
  rng = np.random.default_rng(5)
  mask = torch.from_numpy(rng.random((4, 3, 300, 260)) < 0.45).cuda()
  view = mask[:, 1]
  keep = mask.clone()
  want = [dmap.connected_components(m, c, return_sizes=s) for m, c, s in ((mask, 8, True), (view, 4, False))]
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    with torch.cuda.stream(side):
      got = [dmap.connected_components(mask, 8, return_sizes=True)]
      assert nat.launch_count() - before == 1
      got.append(dmap.connected_components(view, 4))
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
  first, second = (rng.random((2, 2, 150, 170)) < PERCOLATION[8] for _ in range(2))
  mask = torch.from_numpy(first).cuda()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    dmap.connected_components(mask, 8, return_sizes=True)   # warm up off the capture
  torch.cuda.current_stream().wait_stream(side)
  torch.cuda.synchronize()
  graph = torch.cuda.CUDAGraph()
  with torch.cuda.graph(graph):
    labels, counts, sizes = dmap.connected_components(mask, 8, return_sizes=True)
  for contents in (second, first):
    mask.copy_(torch.from_numpy(contents))
    graph.replay()
    torch.cuda.synchronize()
    for got, w in zip((labels, counts, sizes), oracle(contents, 8)):
      assert np.array_equal(got.cpu().numpy(), w)
  nat.device_status()
