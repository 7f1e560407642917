"""MapBuilder.reset_envs (dm_fuse_clear_envs_f32) against the hand-edited workaround it replaces, a general-path builder
whose world planes of the finished environments are overwritten with fill / -inf / False: same maps, offsets and shapes
after every reset and every step, tracked rectangles and box kept, the C step still taken, no host sync, and the
caller's tensors never written."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from dungeon_maps_b200 import maps as dmaps
from oracle import dm_oracle as orc
from tests._golden import assert_same
from tests.test_gpu_parity import assert_workspaces_clean, npy
from tests.test_gpu_semantic_builder import LOCAL, PITCH, _box, _depth, _inputs, _plane_box, _same_map, _walk

pytestmark = pytest.mark.gpu

HFOV = math.radians(70)
GLOBAL = dict(width_offset=60., height_offset=60.)
EMPTY_BOX = [0x7fffffff, -1, 0x7fffffff, -1]


def _builder(native, fixed=None, fill=dmap.NINF, reduction=None, to_global=True):
  proj = dmap.MapProjector(width=160, height=120, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0., height_offset=0.,
                           cam_pitch=PITCH, cam_height=0.88, map_res=0.05, map_width=120, map_height=120,
                           trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=3, fill_value=fill,
                           reduction=reduction, to_global=to_global, device="cuda")
  return dmap.MapBuilder(map_projector=proj, fixed_canvas=fixed, native_step=native)


def _kw(kind, b, C, t, plot_kw=LOCAL):
  return dict(plot_kw) if kind == "height" else dict(plot_kw, **_inputs(kind, b, C, t))


def _workaround(builder, done, fill):
  """What a user writes without reset_envs: the done planes overwritten by hand, which drops the tracked box."""
  wm = builder.world_map
  if wm is None or wm.is_empty:
    return
  d = done.to(wm.mask.device).view(-1, 1, 1, 1)
  top = torch.where(d, torch.tensor(fill, dtype=torch.float32, device=d.device), wm.topdown_map)
  hm = top if wm.is_height_map else torch.where(d, torch.tensor(-math.inf, device=d.device), wm.height_map)
  builder._world_map = dmap.TopdownMap(topdown_map=top, mask=wm.mask & ~d, height_map=hm, map_projector=wm.proj,
                                       is_height_map=wm.is_height_map)


def _fill_of(fill):
  return dmap.NINF if fill is None else fill


def _assert_rectangles_are_mask_extents(world, what):
  boxes = _plane_box(world)
  mask = npy(world.mask)
  b, C = mask.shape[:2]
  for p in range(b * C):
    rows, cols = np.nonzero(mask[p // C, p % C])
    want = EMPTY_BOX if rows.size == 0 else [rows.min(), rows.max(), cols.min(), cols.max()]
    assert list(boxes[p]) == list(want), f"{what}: plane {p}"


def _scan_box(world):
  """What an unseeded dm_fuse_bbox_i64 finds for the world map, whole planes scanned."""
  keep = []
  b, C, h, w = world.mask.shape
  src = dmaps._fuse_source(world, world.proj, b, C, C * h * w, world.mask.device, keep)
  src.plane_box = None
  out = torch.empty((5,), dtype=torch.int64, device=world.mask.device)
  nat.check(nat.lib().dm_fuse_bbox_i64((nat.DmFuseSource * 1)(src), 1, b, C, world.proj.map_res, out.data_ptr(),
                                       nat.stream_ptr(world.mask.device)), "dm_fuse_bbox_i64")
  return npy(out)


RESETS = {1: [False, True, False], 3: [True, False, True], 5: [True, True, True]}   # after step t: done flags


@pytest.mark.parametrize("plot_kw", [LOCAL, GLOBAL], ids=["local", "global"])
@pytest.mark.parametrize("fill,reduction", [(dmap.NINF, None), (0., None), (50., "min"), (float("nan"), None),
                                            (0., "sum")], ids=["ninf", "zero", "min50", "nan", "sum"])
@pytest.mark.parametrize("kind,C", [("height", 1), ("uniform", 3), ("labels", 16)])
def test_reset_envs_equals_the_workaround(kind, C, fill, reduction, plot_kw):
  b, T = 3, 7
  poses = _walk(b, T, seed=31)
  nb, gb = _builder(True, fill=fill, reduction=reduction), _builder(False, fill=fill, reduction=reduction)
  for t in range(T):
    depth = _depth(b, poses[t], 31)
    kw = _kw(kind, b, C, t, plot_kw)
    nb.step(depth, cam_pose=poses[t], **kw)
    gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} world", boxes=False)
    if t in RESETS:
      done = torch.tensor(RESETS[t], device="cuda")
      nb.reset_envs(done)
      _workaround(gb, done, _fill_of(fill))
      _same_map(nb.world_map, gb.world_map, f"reset after step {t}", boxes=False)
      if _plane_box(nb.world_map) is not None:
        _assert_rectangles_are_mask_extents(nb.world_map, f"reset after step {t}")
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("labels", 16)])
def test_tracking_survives_and_the_c_step_is_taken(kind, C):
  b, T = 3, 6
  poses = _walk(b, T, seed=37)
  nb, gb = _builder(True), _builder(False)
  taken = []
  c_step = nb._native_step
  def spy(*args, **kwargs):
    world = nb.world_map
    out = c_step(*args, **kwargs)
    taken.append(out is not None and (world.is_empty or nb._native_world_ok(world, b, world.mask.device,
                                                                             0 if kind == "height" else C)))
    return out
  nb._native_step = spy
  for t in range(T):
    depth = _depth(b, poses[t], 37)
    kw = _kw(kind, b, C, t)
    nb.step(depth, cam_pose=poses[t], **kw)
    gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} world", boxes=False)
    if t in (1, 3):
      done = torch.tensor([t == 1, True, False], device="cuda")
      nb.reset_envs(done)
      _workaround(gb, done, dmap.NINF)
      wm = nb.world_map
      assert dmaps._tracked_box_valid(wm, nb.proj, wm.mask.device), "the tracked box was dropped"
      _assert_rectangles_are_mask_extents(wm, f"reset after step {t}")
      box, scan = _box(wm), _scan_box(wm)
      assert list(box[:4]) == list(scan[:4]) and (box[4] > 0) == (scan[4] > 0), f"box {box} != scan {scan}"
  assert all(taken) and len(taken) == T, f"the C step was not taken at every step: {taken}"
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("uniform", 3)])
def test_resetting_the_extreme_environment_shrinks_the_map(kind, C):
  b, T = 3, 4
  poses = _walk(b, T, seed=41, half=8.0)
  nb, keep, gb = _builder(True), _builder(True), _builder(False)
  for t in range(T):
    depth = _depth(b, poses[t], 41)
    kw = _kw(kind, b, C, t)
    for bld in (nb, keep, gb):
      bld.step(depth, cam_pose=poses[t], **kw)
  # the environment whose cells alone reach furthest in some direction
  mask = npy(nb.world_map.mask).any(axis=1)
  ext = []
  for e in range(b):
    rows, cols = np.nonzero(mask[e])
    ext.append((rows.min(), -rows.max(), cols.min(), -cols.max()))
  ext = np.array(ext)
  unique = [(e, k) for k in range(4) for e in range(b) if all(ext[e, k] < ext[o, k] for o in range(b) if o != e)]
  assert unique, "no environment holds an extreme of the map alone"
  e = unique[0][0]
  done = torch.zeros(b, dtype=torch.bool, device="cuda")
  done[e] = True
  nb.reset_envs(done)
  _workaround(gb, done, dmap.NINF)
  # the last frame again (the others add no new cells), with nothing valid for the reset environment
  depth = _depth(b, poses[T - 1], 41)
  depth[e] = 0.
  kw = _kw(kind, b, C, T - 1)
  for bld in (nb, keep, gb):
    bld.step(depth, cam_pose=poses[T - 1], **kw)
  _same_map(nb.world_map, gb.world_map, "after the reset", boxes=False)
  assert nb.world_map.mask.shape[-2] * nb.world_map.mask.shape[-1] < keep.world_map.mask.shape[-2] * \
      keep.world_map.mask.shape[-1], "the world map did not shrink"
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("labels", 16)])
def test_all_envs_equals_reset(kind, C):
  b, T = 3, 4
  poses = _walk(b, T + 1, seed=43)
  x, y = _builder(True), _builder(True)
  for t in range(T):
    depth = _depth(b, poses[t], 43)
    for bld in (x, y):
      bld.step(depth, cam_pose=poses[t], **_kw(kind, b, C, t))
  x.reset_envs(torch.ones(b, dtype=torch.bool, device="cuda"))
  assert int(x.world_map.mask.sum()) == 0 and _box(x.world_map)[4] == 0
  y.reset()
  depth = _depth(b, poses[T], 43)
  for bld in (x, y):
    bld.step(depth, cam_pose=poses[T], **_kw(kind, b, C, T))
  _same_map(x.world_map, y.world_map, "reset_envs(all) vs reset()", boxes=False)
  assert np.array_equal(_plane_box(x.world_map), _plane_box(y.world_map))
  assert list(_box(x.world_map)[:4]) == list(_box(y.world_map)[:4])
  assert_workspaces_clean()


@pytest.mark.parametrize("native", [True, False], ids=["native", "general"])
@pytest.mark.parametrize("kind,C", [("height", 1), ("onehot", 4)])
def test_fixed_canvas(native, kind, C):
  b, T = 3, 5
  poses = _walk(b, T, seed=47)
  nb, gb = _builder(native, fixed=(400, 380), fill=0.), _builder(False, fixed=(400, 380), fill=0.)
  for t in range(T):
    depth = _depth(b, poses[t], 47)
    kw = _kw(kind, b, C, t)
    nb.step(depth, cam_pose=poses[t], **kw)
    gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} canvas", boxes=False)
    if t in (1, 3):
      wm = nb.world_map
      before = [t_.clone() for t_ in (wm.topdown_map, wm.mask, wm.height_map)]
      ptrs = [t_.data_ptr() for t_ in (wm.topdown_map, wm.mask, wm.height_map)]
      done = [False, True, t == 3]
      nb.reset_envs(done)   # a host list: uploaded
      _workaround(gb, torch.tensor(done), 0.)
      wm = nb.world_map
      assert [t_.data_ptr() for t_ in (wm.topdown_map, wm.mask, wm.height_map)] == ptrs, "the clear is not in place"
      for old, new in zip(before, (wm.topdown_map, wm.mask, wm.height_map)):
        assert torch.equal(old[0], new[0]), "environment 0 was touched"
      assert int(wm.mask[1].sum()) == 0
      _same_map(wm, gb.world_map, f"reset after step {t}", boxes=False)
  assert bool(nb._handles) == native
  assert_workspaces_clean()


def test_local_frame_builder_keeps_rectangles_only():
  b, C, T = 3, 3, 5
  poses = _walk(b, T, seed=53)
  nb, gb = _builder(True, to_global=False), _builder(False, to_global=False)
  for t in range(T):
    depth = _depth(b, poses[t], 53)
    kw = _kw("uniform", b, C, t)
    nb.step(depth, cam_pose=poses[t], **kw)
    gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} world", boxes=False)
    if t in (1, 3):
      done = torch.tensor([True, False, t == 3])
      nb.reset_envs(done)   # a CPU tensor: uploaded
      _workaround(gb, done, dmap.NINF)
      assert _box(nb.world_map) is None and _plane_box(nb.world_map) is not None
      _assert_rectangles_are_mask_extents(nb.world_map, f"reset after step {t}")
      _same_map(nb.world_map, gb.world_map, f"reset after step {t}", boxes=False)
  assert not nb._handles
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("uniform", 3)])
def test_no_host_sync_and_all_false_changes_nothing(kind, C):
  b = 3
  poses = _walk(b, 3, seed=59)
  nb = _builder(True)
  for t in range(3):
    nb.step(_depth(b, poses[t], 59), cam_pose=poses[t], **_kw(kind, b, C, t))
  wm = nb.world_map
  snap = [t_.clone() for t_ in (wm.topdown_map, wm.mask, wm.height_map, wm._tracked_box.box, wm._tracked_box.plane_box)]
  none = torch.zeros(b, dtype=torch.bool, device="cuda")
  some = torch.tensor([False, True, False], device="cuda")
  torch.cuda.synchronize()
  torch.cuda.set_sync_debug_mode("error")
  try:
    nb.reset_envs(none)
    after = nb.world_map
    # copies: the reset below clears environment 1 of these very tensors in place
    now = [t_.clone() for t_ in (after.topdown_map, after.mask, after.height_map, after._tracked_box.box,
                                 after._tracked_box.plane_box)]
    nb.reset_envs(some)
  finally:
    torch.cuda.set_sync_debug_mode(0)
  assert after is wm
  for old, new in zip(snap, now):
    assert torch.equal(old.view(torch.uint8) if old.dtype is torch.float32 else old,
                       new.view(torch.uint8) if new.dtype is torch.float32 else new), "an all-False reset changed bits"
  assert int(nb.world_map.mask[1].sum()) == 0 and int(nb.world_map.mask[0].sum()) > 0
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("uniform", 3)])
def test_caller_tensors_are_never_written(kind, C):
  b = 3
  poses = _walk(b, 4, seed=61)
  # 1. a step with nothing valid: the world map is the local map the step returned
  nb, gb = _builder(True), _builder(False)
  depth = torch.zeros((b, 1, 120, 160), device="cuda")
  local = nb.step(depth, cam_pose=poses[0], **_kw(kind, b, C, 0))
  gb.step(depth, cam_pose=poses[0], **_kw(kind, b, C, 0))
  assert nb.world_map.mask is local.mask
  snap = [t_.clone() for t_ in (local.topdown_map, local.mask, local.height_map)]
  done = torch.tensor([True, False, False], device="cuda")
  nb.reset_envs(done)
  _workaround(gb, done, dmap.NINF)
  for old, new in zip(snap, (local.topdown_map, local.mask, local.height_map)):
    assert torch.equal(old, new), "the local map was written"
  assert nb.world_map.mask is not local.mask
  _same_map(nb.world_map, gb.world_map, "reset of an adopted local map", boxes=False)
  for t in (1, 2):
    depth = _depth(b, poses[t], 61)
    nb.step(depth, cam_pose=poses[t], **_kw(kind, b, C, t))
    gb.step(depth, cam_pose=poses[t], **_kw(kind, b, C, t))
    _same_map(nb.world_map, gb.world_map, f"step {t} world", boxes=False)
  # 2. a world map handed to the constructor
  given = nb.world_map
  snap = [t_.clone() for t_ in (given.topdown_map, given.mask, given.height_map)]
  cb = dmap.MapBuilder(map_projector=nb.proj, world_map=given)
  gb2 = dmap.MapBuilder(map_projector=nb.proj, world_map=given, native_step=False)
  done = torch.tensor([False, True, True], device="cuda")
  cb.reset_envs(done)
  _workaround(gb2, done, dmap.NINF)
  for old, new in zip(snap, (given.topdown_map, given.mask, given.height_map)):
    assert torch.equal(old, new), "the constructor's world map was written"
  assert dmaps._tracked_box_valid(cb.world_map, cb.proj, cb.world_map.mask.device), "the copy lost its tracked box"
  _assert_rectangles_are_mask_extents(cb.world_map, "cleared copy")
  depth = _depth(b, poses[3], 61)
  for bld in (cb, gb2):
    bld.step(depth, cam_pose=poses[3], **_kw(kind, b, C, 3))
  _same_map(cb.world_map, gb2.world_map, "constructor world map, next step", boxes=False)
  assert_workspaces_clean()


@pytest.mark.parametrize("kind,C", [("height", 1), ("uniform", 2)])
def test_dense_copy_on_and_off(kind, C):
  b, T = 3, 6
  poses = _walk(b, T, seed=67)
  runs = []
  try:
    for dense in (1, 0):
      nat.lib().dm_debug_set_dense_shift(dense)
      bld = _builder(True)
      worlds = []
      for t in range(T):
        bld.step(_depth(b, poses[t], 67), cam_pose=poses[t], **_kw(kind, b, C, t))
        if t in (1, 3):
          bld.reset_envs(torch.tensor([t == 3, True, False], device="cuda"))
        worlds.append((bld.world_map, _plane_box(bld.world_map)))
      runs.append(worlds)
  finally:
    nat.lib().dm_debug_set_dense_shift(1)
  for t, ((wa, ba), (wb, bb)) in enumerate(zip(*runs)):
    _same_map(wa, wb, f"step {t} world (dense vs per-cell)", boxes=False)
    assert np.array_equal(ba, bb), f"step {t}: tracked rectangles differ"
  assert_workspaces_clean()


@pytest.mark.parametrize("kind", ["height", "labels"])
def test_reset_envs_vs_oracle(kind):
  b, T, C = 2, 4, 4
  poses = _walk(b, T, seed=71)
  nb = _builder(True)
  k = nb.proj.cam_params
  world = None
  for t in range(T):
    depth = _depth(b, poses[t], 71)
    kw = {} if kind == "height" else _inputs(kind, b, C, t)
    local = nb.step(depth, cam_pose=poses[t], **LOCAL, **kw)
    p = poses[t].numpy()
    values = None
    if kind != "height":
      ids = kw["label_map"].to(torch.int64)
      values = npy((torch.arange(C, device="cuda").view(1, -1, 1, 1) == ids).float())
    top, mask, hgt = orc.orth_project(npy(depth), values, None, p, 60., 0., PITCH, 0.88, 0.05, 120, 120, k.fx, k.fy,
                                      k.cx, k.cy, 0.15, 5.05, None, 3, False, True, -np.inf, None, True)
    assert_same(npy(local.topdown_map), top, f"step {t} local")
    src = [orc.FuseSource(top if kind == "height" else hgt, mask, None if kind == "height" else top, 60., 0., 0.05,
                          True, False, p)]
    if world is not None:
      src.insert(0, orc.FuseSource(world["height"], world["mask"], None if kind == "height" else world["topdown"],
                                   world["width_offset"], world["height_offset"], 0.05, True, True, p))
    world = orc.fuse(src, True, p, 0.05, True)
    if t == 1:
      nb.reset_envs(torch.tensor([False, True], device="cuda"))
      for name, v in (("topdown", -np.inf), ("height", -np.inf), ("mask", False)):
        world[name] = world[name].copy()
        world[name][1] = v
    wm = nb.world_map
    assert [wm.proj.map_height, wm.proj.map_width] == [world["map_height"], world["map_width"]], f"step {t} shape"
    assert_same(npy(wm.topdown_map), world["topdown"], f"step {t} world")
    assert_same(npy(wm.mask), world["mask"], f"step {t} world mask")
    if kind != "height":
      assert_same(npy(wm.height_map), world["height"], f"step {t} world height")
  assert nb._handles
  assert_workspaces_clean()


def test_argument_errors_and_no_world_map():
  b = 3
  poses = _walk(b, 1, seed=73)
  nb = _builder(True)
  nb.reset_envs(torch.ones(b, dtype=torch.bool, device="cuda"))   # nothing to clear yet
  assert nb.world_map.is_empty
  nb.step(_depth(b, poses[0], 73), cam_pose=poses[0], **LOCAL)
  snap = nb.world_map.topdown_map.clone()
  bad = [torch.ones(b + 1, dtype=torch.bool, device="cuda"), torch.ones(b, dtype=torch.uint8, device="cuda"),
         torch.ones(b, device="cuda"), [1, 0, 1], np.ones(b - 1, dtype=bool), torch.ones((b, 1), dtype=torch.bool)]
  if torch.cuda.device_count() > 1:
    bad.append(torch.ones(b, dtype=torch.bool, device="cuda:1"))
  for d in bad:
    with pytest.raises(ValueError):
      nb.reset_envs(d)
  assert torch.equal(snap, nb.world_map.topdown_map)
  assert_workspaces_clean()
