"""score_poses (dm_score_poses_i32) against its definition, bit for bit: the oracle composition (tests/_match.py) over
source shapes from 1 x 1 to 300 x 257, windows from 1 x 1 to 129 x 200 (5 x 8 takes the naive rotation), flip_h on and
off, random / k * pi / 2 / near-zero yaws, off-grid translations, candidates inside, straddling and outside the source,
b = 1, 3, 32 and n = 1, 7, ~300, shared and per-environment candidates, per-environment source offsets, 3-D planes and
C = 3 with a shared window and with per-plane windows, all-False and all-True inputs.  Then the config-4 composition
(a crop_egocentric_map loop) on builder world maps, the noisy-odometry recipe of the docstring on a walk, no host sync
(with a parameter block above 64 KiB), one launch on a side stream, CUDA candidates, and inputs never written."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from dungeon_maps_b200 import synth
from tests._match import lattice, random_planes, score_poses
from tests.test_gpu_parity import npy
from tests.test_gpu_semantic_builder import HFOV, LOCAL, PITCH, _builder, _depth, _inputs, _walk

pytestmark = pytest.mark.gpu

RES = 0.05


def _source(b, Hs, Ws, flip_h=True, woff=None, hoff=None):
  """A global-frame map of b x Hs x Ws; offsets default to the centre, or 1 or b values."""
  woff = Ws / 2. + 0.5 if woff is None else woff
  hoff = Hs / 2. - 1. if hoff is None else hoff
  top = torch.zeros((b, 1, Hs, Ws), device="cuda")
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=RES, map_width=Ws, map_height=Hs,
                           width_offset=woff, height_offset=hoff, to_global=True, flip_h=flip_h, device="cuda")
  return dmap.TopdownMap(topdown_map=top, mask=top > 0, height_map=top, map_projector=proj, is_height_map=True)


def _candidates(rng, b, n, Hs, Ws, woff, hoff, shared):
  """(n, 3) or (b, n, 3) float32: off-grid inside at a random yaw, straddling a corner at |yaw| <= ANGLE_EPS, far
  outside, k * pi / 2, -pi, near the left edge just above ANGLE_EPS, yaw 0 on the grid, then random around the
  centre; each environment takes them in its own order."""
  woff, hoff = float(np.mean(woff)), float(np.mean(hoff))
  cx, cz = (Ws / 2 - woff) * RES, (Hs / 2 - hoff) * RES
  span = max(Hs, Ws) * RES / 2
  fixed = [(cx + 0.013, cz - 0.021, rng.uniform(-math.pi, math.pi)), ((Ws - woff) * RES, -hoff * RES, 0.0009),
           (cx + 400., cz - 300., 0.7), (cx - 0.3 * span, cz + 0.2 * span, math.pi / 2),
           (cx + 0.5 * span, cz, -math.pi),
           (-woff * RES + 0.0123, cz + 0.0311, 0.0011), (cx + 2 * RES, cz - 3 * RES, 0.), (cx, cz, 3 * math.pi / 2),
           (cx + 0.0004, cz - 0.0007, -0.0009)]

  def one():
    rows = [fixed[i] if i < len(fixed) else (cx + rng.uniform(-span, span), cz + rng.uniform(-span, span),
                                             rng.uniform(-math.pi, math.pi)) for i in range(max(n, len(fixed)))]
    order = rng.permutation(len(rows))[:n]
    return np.array([rows[i] for i in order], np.float32)

  return one() if shared else np.stack([one() for _ in range(b)])


def _check(src, planes, window, poses, u=None, v=None):
  """Kernel == oracle, bit for bit; returns the kernel's scores."""
  got = dmap.score_poses(src, planes, window, poses, width_offset=u, height_offset=v)
  p = src.proj
  h, w = window.shape[-2:]
  u_ = dmap.get(u, w / 2.)
  v_ = dmap.get(v, h / 2.)
  pl = npy(planes) if planes.dim() == 4 else npy(planes)[:, None]
  win = npy(window) if window.dim() == 4 else npy(window)[:, None]
  pose_np = poses.cpu().numpy() if torch.is_tensor(poses) else poses
  want = score_poses(pl, win, p.width_offset, p.height_offset, p.map_res, p.flip_h, pose_np, u_, v_)
  b, C, n = want.shape
  assert got.dtype is torch.int32 and got.is_cuda
  assert tuple(got.shape) == ((b, C, n) if planes.dim() == 4 else (b, n))
  assert np.array_equal(npy(got).reshape(b, C, n), want), "scores differ from the oracle"
  return got


WINDOWS = [(1, 1), (5, 8), (6, 7), (64, 64), (129, 200)]      # (h, w); 5 x 8: 9 * 40 < 400, the naive rotation
SOURCES = [(1, 1), (37, 53), (300, 257)]


@pytest.mark.parametrize("h,w", WINDOWS, ids=[f"{h}x{w}" for h, w in WINDOWS])
@pytest.mark.parametrize("flip_h", [True, False], ids=["flip", "noflip"])
@pytest.mark.parametrize("mode", ["3d", "shared", "per_plane"])
def test_matches_oracle(h, w, flip_h, mode):
  rng = np.random.default_rng(h * 1000 + w + 7 * flip_h + len(mode))
  b = 3
  for Hs, Ws in SOURCES:
    src = _source(b, Hs, Ws, flip_h)
    C = 1 if mode == "3d" else 3
    planes = torch.from_numpy(random_planes(rng, (b, C, Hs, Ws), 0.45)).cuda()
    window = torch.from_numpy(random_planes(rng, (b, C if mode == "per_plane" else 1, h, w), 0.3)).cuda()
    if mode == "3d":
      planes, window = planes[:, 0], window[:, 0]
    elif mode == "shared":
      window = window[:, 0]
    p = src.proj
    _check(src, planes, window, _candidates(rng, b, 7, Hs, Ws, p.width_offset, p.height_offset, shared=False))
    _check(src, planes, window, _candidates(rng, b, 1, Hs, Ws, p.width_offset, p.height_offset, shared=True))
    # per-environment window offsets (one at the bottom row), shared candidates
    u = torch.tensor([w / 2., 0., w - 1.5])
    v = torch.tensor([0., h / 2., 3.])
    _check(src, planes, window, _candidates(rng, b, 7, Hs, Ws, p.width_offset, p.height_offset, shared=True), u, v)


@pytest.mark.parametrize("b,n,h,w", [(32, 300, 6, 7), (1, 300, 64, 64), (32, 7, 129, 200)])
def test_batch_and_candidate_counts(b, n, h, w):
  rng = np.random.default_rng(b * n + h)
  Hs, Ws = 90, 110
  woff = rng.uniform(20, 90, size=b).astype(np.float32)          # per-environment source offsets
  hoff = rng.uniform(10, 80, size=b).astype(np.float32)
  src = _source(b, Hs, Ws, woff=torch.from_numpy(woff), hoff=torch.from_numpy(hoff))
  planes = torch.from_numpy(random_planes(rng, (b, 2, Hs, Ws), 0.4)).cuda()
  window = torch.from_numpy(random_planes(rng, (b, 2, h, w), 0.25)).cuda()
  _check(src, planes, window, _candidates(rng, b, n, Hs, Ws, woff, hoff, shared=False))
  _check(src, planes, window[:, 0], _candidates(rng, b, n, Hs, Ws, woff, hoff, shared=True), u=w / 2., v=0.)


@pytest.mark.parametrize("mode", ["3d", "shared", "per_plane"])
def test_all_false_all_true_and_outside(mode):
  rng = np.random.default_rng(5)
  b, Hs, Ws, h, w = 3, 40, 50, 9, 11
  src = _source(b, Hs, Ws)
  p = src.proj
  C = 1 if mode == "3d" else 3
  for pd, wd in ((0., 1.), (1., 0.), (1., 1.), (0.5, 1.), (1., 0.5)):
    planes = torch.from_numpy(random_planes(rng, (b, C, Hs, Ws), pd)).cuda()
    window = torch.from_numpy(random_planes(rng, (b, C if mode == "per_plane" else 1, h, w), wd)).cuda()
    if mode == "3d":
      planes, window = planes[:, 0], window[:, 0]
    elif mode == "shared":
      window = window[:, 0]
    got = _check(src, planes, window, _candidates(rng, b, 9, Hs, Ws, p.width_offset, p.height_offset, shared=False))
    if pd == 0. or wd == 0.:
      assert not bool(got.any())
  # candidates fully outside the source score 0, all-True inputs included
  planes = torch.ones((b, C, Hs, Ws), dtype=torch.bool, device="cuda")
  window = torch.ones((b, C, h, w) if mode == "per_plane" else (b, h, w), dtype=torch.bool, device="cuda")
  if mode == "3d":
    planes = planes[:, 0]
  far = np.array([[400., -300., 0.3], [-500., 2., 0.], [0., 900., math.pi / 2]], np.float32)
  got = _check(src, planes, window, far)
  assert not bool(got.any())
  # the agent in the middle of an all-True source at yaw 0: every window cell counts
  mid = np.array([[(Ws / 2 - float(p.width_offset)) * RES, (Hs / 2 - float(p.height_offset)) * RES, 0.]], np.float32)
  assert bool((_check(src, planes, window, mid) == h * w).all())


def _run_builder(kind, C, fixed=None, T=6, seed=71, b=3):
  """A builder walk; returns the builder, the poses, and the local map of the last step."""
  poses = _walk(b, T, seed=seed)
  nb = _builder(True, fixed=fixed)
  local = None
  for t in range(T):
    kw = dict(LOCAL) if kind == "height" else dict(LOCAL, **_inputs(kind, b, C, t))
    local = nb.step(_depth(b, poses[t], seed), cam_pose=poses[t], **kw)
  return nb, poses, local


def _composed(src, planes, window, cands, u, v):
  """The definition with crop_egocentric_map: one crop per candidate, ANDed with the window and counted."""
  b, C = planes.shape[:2]
  h, w = window.shape[-2:]
  m = dmap.TopdownMap(topdown_map=planes.float(), mask=planes, height_map=planes.float(), map_projector=src.proj,
                      is_height_map=True)
  win = window if window.dim() == 4 else window[:, None]
  out = []
  for k in range(cands.shape[1]):
    crop = dmap.crop_egocentric_map(m, w, h, cam_pose=cands[:, k], width_offset=u, height_offset=v)
    out.append((crop.mask & win).sum(dim=(2, 3), dtype=torch.int32))
  return torch.stack(out, dim=-1)


def _lattice_around(pose, steps, dxz=RES, dyaw=math.radians(1.)):
  return torch.from_numpy(lattice(pose.numpy(), steps, dxz, dyaw))


@pytest.mark.parametrize("fixed", [None, (300, 320)], ids=["growing", "fixed"])
def test_builder_obstacle_planes_match_the_crop_loop(fixed):
  nb, poses, local = _run_builder("height", 1, fixed)
  world = nb.world_map
  seen = world.mask[:, 0]
  obstacle = seen & (world.height_map[:, 0] > 0.2)
  planes = torch.stack((obstacle, seen & ~obstacle), dim=1)
  window = local.mask[:, 0] & (local.height_map[:, 0] > 0.2)
  assert bool(window.any())
  u, v = LOCAL["width_offset"], LOCAL["height_offset"]
  cands = _lattice_around(poses[-1], 2)                                  # (b, 125, 3)
  got = dmap.score_poses(world, planes, window, cands, width_offset=u, height_offset=v)
  assert torch.equal(got, _composed(world, planes, window, cands, u, v))
  assert bool((got[:, 0] > 0).any())
  one = dmap.score_poses(world, obstacle, window, cands, width_offset=u, height_offset=v)
  assert torch.equal(one, got[:, 0])


def test_class_planes_with_per_plane_windows_match_the_crop_loop():
  nb, poses, local = _run_builder("labels", 16)
  world = nb.world_map
  planes = world.topdown_map > 0.5                                       # (b, 16, Hs, Ws)
  window = local.topdown_map > 0.5                                       # (b, 16, 120, 120)
  assert planes.shape[1] == 16 and window.shape[1] == 16 and bool(window.any())
  u, v = LOCAL["width_offset"], LOCAL["height_offset"]
  cands = _lattice_around(poses[-1], 2)
  got = dmap.score_poses(world, planes, window, cands, width_offset=u, height_offset=v)
  assert torch.equal(got, _composed(world, planes, window, cands, u, v))
  assert bool((got > 0).any())


def _room_depth(b, pose, seed):
  """A 6 x 6 m room: from anywhere inside it the walls are within the 5.05 m depth truncation."""
  return synth.room_depth(b, 120, 160, HFOV, PITCH, 0.88, pose.cuda(), seed=seed, half=3.0, device="cuda")


def _recipe():
  """The docstring's recipe on a walk: the world holds steps 0..T-2 at their true poses; step T-1's local map is
  matched on a 7 x 7 x 7 lattice (1 cell, 1 degree) around its odometry pose, the true pose perturbed by (2, -2, 2)
  lattice steps.  The walk stays in a room whose walls every frame sees, so that each local map has obstacle cells to
  match (asserted): a window without obstacles scores 0 everywhere and has no best pose.  Returns the winner's
  absolute error (x, z, yaw) per environment, the lattice steps, and a report of the scores."""
  b, T, steps = 3, 8, 3
  dxz, dyaw = RES, math.radians(1.)
  poses = _walk(b, T, seed=23, half=1.5)
  nb = _builder(True)
  for t in range(T - 1):
    nb.step(_room_depth(b, poses[t], 23), cam_pose=poses[t], **LOCAL)
  true = poses[T - 1]
  odom = (true + torch.tensor([2 * dxz, -2 * dxz, 2 * dyaw], dtype=torch.float32)).to(torch.float32)
  depth = _room_depth(b, true, 23)
  world = nb.world_map
  seen = world.mask[:, 0]
  obstacle = seen & (world.height_map[:, 0] > 0.2)
  planes = torch.stack((obstacle, seen & ~obstacle), dim=1)
  local = nb.plot(depth, cam_pose=odom, **LOCAL)
  window = local.mask[:, 0] & (local.height_map[:, 0] > 0.2)
  assert bool((window.sum(dim=(1, 2)) >= 50).all()), f"too few obstacle cells: {window.sum(dim=(1, 2)).tolist()}"
  cands = _lattice_around(odom, steps, dxz, dyaw)
  s = dmap.score_poses(world, planes, window, cands, width_offset=LOCAL["width_offset"],
                       height_offset=LOCAL["height_offset"])
  score = (s[:, 0] - s[:, 1]).cpu()
  best = score.argmax(-1)
  pose = cands[torch.arange(b), best]
  err = (pose - true).abs()
  top2 = score.float().topk(2, dim=-1).values
  near = ((cands - true[:, None]) / torch.tensor([dxz, dxz, dyaw])).abs().amax(-1).argmin(-1)
  report = [dict(env=i, window_cells=int(window[i].sum()), best=score[i].max().item(), at_true=score[i, near[i]].item(),
                 at_odom=score[i, cands.shape[1] // 2].item(), margin=(top2[i, 0] - top2[i, 1]).item(),
                 err=[round(x, 4) for x in err[i].tolist()]) for i in range(b)]
  print("recipe:", report)
  nb.step(depth, cam_pose=pose, **LOCAL)
  assert nb.world_map.mask.any()
  return err, (dxz, dyaw), report


@pytest.mark.xfail(strict=True, reason="environments 0 and 2 land 4 and 2 cells off in x with z and yaw exact, as "
                   "when the window holds one straight wall: sliding along it keeps or adds obstacle hits")
def test_recipe_recovers_the_true_pose():
  """The recipe's argmax lies within one lattice step of the true pose in x, z and yaw for every environment."""
  err, (dxz, dyaw), report = _recipe()
  ok = (err[:, 0] <= dxz * 1.01) & (err[:, 1] <= dxz * 1.01) & (err[:, 2] <= dyaw * 1.01)
  assert bool(ok.all()), f"the recipe missed the true pose: {report}"


def test_recipe_recovers_heading_and_offset_across_the_walls():
  """What the recipe does recover on the same walk: the heading and z within one lattice step for every environment,
  and the whole pose for at least one (environment 1 sees enough structure)."""
  err, (dxz, dyaw), report = _recipe()
  assert bool(((err[:, 1] <= dxz * 1.01) & (err[:, 2] <= dyaw * 1.01)).all()), report
  full = (err[:, 0] <= dxz * 1.01) & (err[:, 1] <= dxz * 1.01) & (err[:, 2] <= dyaw * 1.01)
  assert bool(full.any()), report


def _random_case(b, n, seed=3):
  rng = np.random.default_rng(seed)
  Hs, Ws, h, w = 120, 130, 60, 50
  src = _source(b, Hs, Ws)
  p = src.proj
  planes = torch.from_numpy(random_planes(rng, (b, 2, Hs, Ws), 0.4)).cuda()
  window = torch.from_numpy(random_planes(rng, (b, h, w), 0.2)).cuda()
  cands = torch.from_numpy(_candidates(rng, b, n, Hs, Ws, p.width_offset, p.height_offset, shared=False))
  return src, planes, window, cands


def test_no_host_sync_one_launch_on_a_side_stream():
  small = _random_case(3, 7)
  large = _random_case(32, 1331, seed=4)                 # 32 * 1331 blocks of 80 B: above the 64 KiB ring slot
  assert large[3].numel() // 3 * nat.EGO_SAMPLE_WORDS * 4 > 64 * 1024
  want = [dmap.score_poses(*case) for case in (small, large)]
  torch.cuda.synchronize()
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    with torch.cuda.stream(side):
      outs = [dmap.score_poses(*small)]
      assert nat.launch_count() - before == 1
      outs.append(dmap.score_poses(*large))
      assert nat.launch_count() - before == 2
  finally:
    torch.cuda.set_sync_debug_mode(0)
  torch.cuda.current_stream().wait_stream(side)
  for o, w in zip(outs, want):
    assert torch.equal(o, w)
  # behind a long sleep and an overwrite of the planes on the side stream: the scores see the new planes
  src, planes, window, cands = small
  with torch.cuda.stream(side):
    torch.cuda._sleep(20_000_000)
    planes.logical_not_()
    late = dmap.score_poses(src, planes, window, cands)
  side.synchronize()
  _check(src, planes, window, cands.numpy())
  assert torch.equal(late, dmap.score_poses(src, planes, window, cands))


def test_cuda_candidates_and_inputs_untouched():
  src, planes, window, cands = _random_case(3, 40, seed=8)
  keep = [planes.clone(), window.clone()]
  host = dmap.score_poses(src, planes, window, cands)
  dev = dmap.score_poses(src, planes, window, cands.cuda())
  per_plane = dmap.score_poses(src, planes, window[:, None].expand(3, 2, *window.shape[1:]), cands.cuda())
  torch.cuda.synchronize()
  assert torch.equal(host, dev) and torch.equal(host, per_plane)
  assert torch.equal(planes, keep[0]) and torch.equal(window, keep[1])
  _check(src, planes, window, cands)
  # views are read as views: a plane of a (b, C, Hs, Ws) stack, a transposed window
  _check(src, planes[:, 1], window.transpose(1, 2).contiguous().transpose(1, 2), cands[:, :5])


def test_device_mismatch_is_a_value_error():
  src, planes, window, cands = _random_case(3, 4)
  with pytest.raises(ValueError, match="window must be on"):
    dmap.score_poses(src, planes, window.cpu(), cands)
  with pytest.raises(ValueError, match="CUDA"):
    dmap.score_poses(src, planes.cpu(), window.cpu(), cands)
