"""TopdownMap.select_egocentric (dm_crop_egocentric_f32) against its definition, bit for bit: the GPU composition of
this library's public functions (map_dequantize -> local_to_global_space -> map_quantize -> torch gather) and the
oracle's (tests/_egocentric.py).  Height maps, 16-plane float maps with their own or shared height planes, and the
world maps of native, fixed-canvas and reset builders; flip_h on and off; random yaws, |yaw| <= ANGLE_EPS and
k * pi / 2; off-grid poses; windows inside, straddling and outside the source.  Also: the returned projector, no host
sync, one launch on the current stream, and the source never written."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from dungeon_maps_b200 import _params as prm
from tests._egocentric import crop_egocentric
from tests.test_gpu_parity import npy
from tests.test_gpu_semantic_builder import LOCAL, _builder, _depth, _inputs, _walk

pytestmark = pytest.mark.gpu

RES = 0.05
HS, WS = 90, 110          # source map
SRC_WOFF, SRC_HOFF = 50.5, 40.


def _source(kind, flip_h=True, b=6, fill=dmap.NINF, seed=0):
  """kind: "height" (C = 1), "values" (16 planes with 16 height planes), "shared" (4 planes, one height plane expanded
  over them with stride 0, as a value map's local map carries it)."""
  g = torch.Generator(device="cuda").manual_seed(seed)
  C = {"height": 1, "values": 16, "shared": 4}[kind]
  top = torch.rand((b, C, HS, WS), generator=g, device="cuda") * 4 - 2
  mask = torch.rand((b, C, HS, WS), generator=g, device="cuda") > 0.4
  hm = top
  if kind == "values":
    hm = torch.rand((b, C, HS, WS), generator=g, device="cuda")
  elif kind == "shared":
    hm = torch.rand((b, 1, HS, WS), generator=g, device="cuda").expand(b, C, HS, WS)
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=RES, map_width=WS, map_height=HS,
                           width_offset=SRC_WOFF, height_offset=SRC_HOFF, to_global=True, flip_h=flip_h,
                           fill_value=fill, device="cuda")
  return dmap.TopdownMap(topdown_map=top, mask=mask, height_map=hm, map_projector=proj,
                         is_height_map=kind == "height")


def _poses(b, seed):
  """(b, 3): inside the source at a random yaw, straddling its corner at |yaw| <= ANGLE_EPS, far outside, at k pi / 2,
  at -pi, and off-grid near the edge at a yaw just above ANGLE_EPS; then random."""
  rng = np.random.default_rng(seed)
  cx, cz = (WS / 2 - SRC_WOFF) * RES, (HS / 2 - SRC_HOFF) * RES     # global x, z of the source's centre cell
  fixed = [(cx + 0.013, cz - 0.021, rng.uniform(-math.pi, math.pi)),
           ((WS - SRC_WOFF) * RES, -SRC_HOFF * RES, 0.0009),
           (cx + 400., cz - 300., 0.7),
           (cx - 0.3, cz + 0.2, math.pi / 2),
           (cx + 0.5, cz, -math.pi),
           (-SRC_WOFF * RES + 0.0123, cz + 0.0311, 0.0011)]
  out = [fixed[i] if i < len(fixed) else (cx + rng.uniform(-3, 3), cz + rng.uniform(-3, 3),
                                          rng.uniform(-math.pi, math.pi)) for i in range(b)]
  return torch.tensor(out, dtype=torch.float32)


def _composed(src, crop_w, crop_h, pose, u, v, fill):
  """The definition with this library's public functions on the GPU."""
  top = src.topdown_map
  b, C, Hs, Ws = top.shape
  p = src.proj
  n = crop_h * crop_w
  idx = torch.arange(n, device="cuda")
  xb = (idx % crop_w).to(torch.float32).expand(b, n)
  zb = (idx // crop_w).to(torch.float32).expand(b, n)
  lx, lz = dmap.map_dequantize(xb, zb, u, v, p.map_res, crop_h, p.flip_h)
  pts = torch.stack((lx, torch.zeros_like(lx), lz), dim=-1)
  g = dmap.local_to_global_space(pts, pose)
  X, Z = dmap.map_quantize(g[..., 0], g[..., 2], p.width_offset, p.height_offset, p.map_res, Hs, p.flip_h)
  inside = (X >= 0) & (X < Ws) & (Z >= 0) & (Z < Hs)
  cell = torch.where(inside, Z * Ws + X, torch.zeros_like(X))

  def gather(t, fill_):
    k = t.shape[1]
    got = t.reshape(b, k, -1).gather(2, cell[:, None, :].expand(b, k, n))
    return torch.where(inside[:, None, :], got, torch.tensor(fill_, dtype=t.dtype, device="cuda")).view(
      b, k, crop_h, crop_w)

  hm = None if src.is_height_map else gather(src.height_map.to(torch.float32), -math.inf)
  return gather(top, fill), gather(src.mask, False), hm


def _bits(t):
  t = t.contiguous()
  return t.view(torch.int32) if t.dtype is torch.float32 else t


def _check(src, crop_w, crop_h, pose=None, u=None, v=None, fill=None):
  """Kernel == GPU composition == oracle, bit for bit; returns the kernel's map."""
  m = src.select_egocentric(crop_w, crop_h, cam_pose=pose, width_offset=u, height_offset=v, fill_value=fill)
  p = src.proj
  pose_ = prm.host_f32(dmap.get(pose, p.cam_pose, [0., 0., 0.]), (3,))
  u_ = dmap.get(u, crop_w / 2.)
  v_ = dmap.get(v, crop_h / 2.)
  fill_ = dmap.get(fill, p.fill_value, dmap.NINF)
  b, C = src.topdown_map.shape[:2]
  assert tuple(m.topdown_map.shape) == (b, C, crop_h, crop_w) and m.mask.dtype is torch.bool
  assert m.is_height_map == src.is_height_map
  want = _composed(src, crop_w, crop_h, pose_, u_, v_, fill_)
  assert torch.equal(_bits(m.topdown_map), _bits(want[0])), "topdown differs from the composition"
  assert torch.equal(m.mask, want[1]), "mask differs from the composition"
  if src.is_height_map:
    assert m.height_map is m.topdown_map
  else:
    assert torch.equal(_bits(m.height_map), _bits(want[2])), "heights differ from the composition"
  hs = None if src.is_height_map else npy(src.height_map)
  orc = crop_egocentric(npy(src.topdown_map), npy(src.mask), hs, p.width_offset, p.height_offset, p.map_res,
                        p.flip_h, pose_.numpy(), crop_w, crop_h, u_, v_, fill_)
  assert npy(m.topdown_map).tobytes() == orc[0].tobytes(), "topdown differs from the oracle"
  assert np.array_equal(npy(m.mask), orc[1]), "mask differs from the oracle"
  if not src.is_height_map:
    assert npy(m.height_map).tobytes() == orc[2].tobytes(), "heights differ from the oracle"
  return m


SIZES = [(4, 5), (5, 4), (7, 8), (64, 48), (256, 256)]   # (crop_h, crop_w); 4 x 5: 9 * 20 < 400, the naive rotation


@pytest.mark.parametrize("crop_h,crop_w", SIZES, ids=[f"{h}x{w}" for h, w in SIZES])
@pytest.mark.parametrize("flip_h", [True, False], ids=["flip", "noflip"])
@pytest.mark.parametrize("kind", ["height", "values", "shared"])
def test_matches_composition_and_oracle(kind, flip_h, crop_h, crop_w):
  src = _source(kind, flip_h)
  b = src.topdown_map.shape[0]
  pose = _poses(b, seed=crop_h * 1000 + crop_w)
  m = _check(src, crop_w, crop_h, pose)
  # sample 2 stands 400 m away: all fill, mask all False
  assert not m.mask[2].any() and bool((m.topdown_map[2] == dmap.NINF).all())
  if kind == "shared":
    assert m.height_map.stride(1) == 0
  # per-sample window offsets (bottom-centre for some), one shared pose, another fill
  u = torch.tensor([crop_w / 2., 0., 1.5, crop_w / 2., -3., crop_w - 1.])
  v = torch.tensor([0., crop_h / 2., 0., 2.5, 0., crop_h + 7.])
  _check(src, crop_w, crop_h, pose[3:4], u, v, fill=-7.5)
  # bottom-centre for every sample
  _check(src, crop_w, crop_h, pose, crop_w / 2., 0.)


@pytest.mark.parametrize("kind", ["height", "values"])
def test_per_sample_source_offsets(kind):
  """A source that crop_topdown_map produced carries one pair of offsets per sample."""
  src = _source(kind)
  b = src.topdown_map.shape[0]
  centers = torch.tensor([[55., 45.], [10., 80.], [100., 3.], [60., 60.], [0., 0.], [33., 21.]])
  crop = src.select(centers, 70, 50)
  assert crop.proj.width_offset.shape == (b,)
  _check(crop, 33, 40, _poses(b, seed=3))
  _check(crop, 4, 5, _poses(b, seed=4)[:1], fill=0.)


def test_default_offsets_and_projector():
  src = _source("values")
  b = src.topdown_map.shape[0]
  pose = _poses(b, seed=9)
  crop_h, crop_w = 32, 40
  m = _check(src, crop_w, crop_h, pose)
  p = m.proj
  assert p is not src.proj and p.to_global is False and src.proj.to_global is True
  assert (p.map_width, p.map_height, p.map_res, p.flip_h) == (crop_w, crop_h, src.proj.map_res, src.proj.flip_h)
  assert torch.equal(prm.host_f32(p.cam_pose, (3,)), pose)
  assert float(p.width_offset) == crop_w / 2. and float(p.height_offset) == crop_h / 2.
  assert p.fill_value == src.proj.fill_value and p.width == src.proj.width
  # the agent's cell: get_camera() of the window, and the window holds there what the source holds at the agent
  cam = m.get_camera().cpu()
  assert cam.tolist() == [[crop_w // 2, crop_h - 1 - crop_h // 2]]
  X, Z = cam[0].tolist()
  at = src.get_coords(torch.cat((pose[:, :1], torch.zeros(b, 1), pose[:, 1:2]), 1).view(b, 1, 3)).view(b, 2).cpu()
  for i in range(b):
    xs, zs = at[i].tolist()
    if 0 <= xs < WS and 0 <= zs < HS:
      assert torch.equal(_bits(m.topdown_map[i, :, Z, X]), _bits(src.topdown_map[i, :, zs, xs]))
  # per-sample offsets: get_coords of each sample's local origin is its agent cell
  v = torch.tensor([0., 3., 5., 7., 11., 13.])
  m2 = src.select_egocentric(crop_w, crop_h, cam_pose=pose, height_offset=v)
  cells = m2.get_coords(torch.zeros((b, 1, 3)), is_global=False).view(b, 2).cpu()
  assert cells[:, 0].tolist() == [crop_w // 2] * b
  assert cells[:, 1].tolist() == [crop_h - 1 - int(x) for x in v.tolist()]


def _run_builder(kind, C, fixed=None, T=5, seed=71):
  b = 3
  poses = _walk(b, T, seed=seed)
  nb = _builder(True, fixed=fixed)
  for t in range(T):
    kw = dict(LOCAL) if kind == "height" else dict(LOCAL, **_inputs(kind, b, C, t))
    nb.step(_depth(b, poses[t], seed), cam_pose=poses[t], **kw)
  return nb, poses[T - 1]


@pytest.mark.parametrize("fixed", [None, (300, 320)], ids=["growing", "fixed"])
@pytest.mark.parametrize("kind,C", [("height", 1), ("labels", 16)])
def test_builder_world_maps(kind, C, fixed):
  nb, last = _run_builder(kind, C, fixed)
  world = nb.world_map
  assert torch.equal(prm.host_f32(world.proj.cam_pose, (3,)), last)   # the pose of the latest step
  m = _check(world, 64, 64)                                          # default pose and offsets
  assert m.mask.any()
  _check(world, 96, 80, v=0.)
  nb.reset_envs([False, True, False])
  after = _check(nb.world_map, 64, 64)
  assert not after.mask[1].any() and bool((after.topdown_map[1] == dmap.NINF).all())
  if not after.is_height_map:
    assert bool((after.height_map[1] == -math.inf).all())
  assert torch.equal(after.mask[0], m.mask[0]) and torch.equal(_bits(after.topdown_map[2]), _bits(m.topdown_map[2]))


@pytest.mark.parametrize("kind,C", [("height", 1), ("labels", 16)])
def test_no_host_sync_and_one_launch(kind, C):
  nb, last = _run_builder(kind, C)
  world = nb.world_map
  poses = [last, last + torch.tensor([0.1, -0.2, 0.3])]
  torch.cuda.synchronize()
  before = nat.launch_count()
  torch.cuda.set_sync_debug_mode("error")
  try:
    outs = [world.select_egocentric(128, 96, cam_pose=p) for p in poses]
    outs.append(world.select_egocentric(64, 64, height_offset=0.))
  finally:
    torch.cuda.set_sync_debug_mode(0)
  assert nat.launch_count() - before == 3
  for p, m in zip(poses, outs):
    want = _check(world, 128, 96, p)
    assert torch.equal(_bits(m.topdown_map), _bits(want.topdown_map)) and torch.equal(m.mask, want.mask)


def test_source_untouched_no_alias_current_stream():
  src = _source("values")
  b = src.topdown_map.shape[0]
  pose = _poses(b, seed=5)
  snap = [t.clone() for t in (src.topdown_map, src.mask, src.height_map)]
  m = src.select_egocentric(50, 40, cam_pose=pose)
  torch.cuda.synchronize()
  for old, new in zip(snap, (src.topdown_map, src.mask, src.height_map)):
    assert torch.equal(_bits(old), _bits(new))
  spans = lambda ts: [(t.untyped_storage().data_ptr(), t.untyped_storage().data_ptr() + t.untyped_storage().nbytes())
                      for t in ts]
  for a0, a1 in spans((m.topdown_map, m.mask, m.height_map)):
    for s0, s1 in spans((src.topdown_map, src.mask, src.height_map)):
      assert a1 <= s0 or s1 <= a0, "an output aliases the source"
  # on a side stream, behind a long sleep and an overwrite of the source: the window must see the new values
  side = torch.cuda.Stream()
  side.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(side):
    torch.cuda._sleep(20_000_000)
    src.topdown_map.mul_(-1.0)
    late = src.select_egocentric(50, 40, cam_pose=pose)
  side.synchronize()
  want = _check(src, 50, 40, pose)
  assert torch.equal(_bits(late.topdown_map), _bits(want.topdown_map))
  assert not torch.equal(_bits(late.topdown_map), _bits(m.topdown_map))


def test_cuda_pose_tensor():
  src = _source("height")
  pose = _poses(src.topdown_map.shape[0], seed=12)
  m = src.select_egocentric(20, 24, cam_pose=pose.cuda())
  want = _check(src, 20, 24, pose)
  assert torch.equal(_bits(m.topdown_map), _bits(want.topdown_map))
