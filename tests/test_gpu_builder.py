"""MapBuilder.step with its host side in C (dm_builder_*, csrc/dm_builder.cu) against the general Python path and
the oracle: same local maps, same world-map shapes / offsets / tensors, step after step."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import synth
from oracle import dm_oracle as orc
from tests._golden import assert_same
from tests.test_gpu_parity import assert_workspaces_clean, npy

pytestmark = pytest.mark.gpu

HFOV = math.radians(70)
PITCH = math.radians(-10)


def _walk(b, T, seed, half=4.0):
  import sys
  sys.path.insert(0, str(__import__("pathlib").Path(__file__).resolve().parents[1]))
  from bench import BuilderWorkload
  return BuilderWorkload.walk(b, T, seed=seed, half=half)


def _builder(native, fixed=None, fill=dmap.NINF, reduction=None, H=120, W=160):
  proj = dmap.MapProjector(width=W, height=H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0., height_offset=0.,
                           cam_pitch=PITCH, cam_height=0.88, map_res=0.05, map_width=120, map_height=120,
                           trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=3, fill_value=fill,
                           reduction=reduction, to_global=True, device="cuda")
  return dmap.MapBuilder(map_projector=proj, fixed_canvas=fixed, native_step=native)


def _same_map(a, b_, what):
  assert [a.proj.map_height, a.proj.map_width] == [b_.proj.map_height, b_.proj.map_width], f"{what} shape"
  assert_same(np.asarray(a.proj.width_offset, np.float32).reshape(-1), np.asarray(b_.proj.width_offset, np.float32).reshape(-1), f"{what} woff")
  assert_same(np.asarray(a.proj.height_offset, np.float32).reshape(-1), np.asarray(b_.proj.height_offset, np.float32).reshape(-1), f"{what} hoff")
  assert_same(npy(a.topdown_map), npy(b_.topdown_map), f"{what} topdown")
  assert_same(npy(a.mask), npy(b_.mask), f"{what} mask")
  assert_same(npy(a.height_map), npy(b_.height_map), f"{what} height")
  assert a.is_height_map == b_.is_height_map


@pytest.mark.parametrize("plot_kw", [
  dict(to_global=False, width_offset=60., height_offset=0., map_width=120, map_height=120),   # local maps (config 4)
  dict(),                                                                                     # plotted in the global frame
  dict(to_global=False, width_offset=40.5, height_offset=3., map_width=90, map_height=70),
])
@pytest.mark.parametrize("fill,reduction", [(dmap.NINF, None), (None, None), (50., "min")])
def test_native_step_equals_general_path(plot_kw, fill, reduction):
  b, T, H, W = 3, 5, 120, 160
  poses = _walk(b, T, seed=5)
  nb, gb = _builder(True, fill=fill, reduction=reduction), _builder(False, fill=fill, reduction=reduction)
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=5, half=6.0, device="cuda")
    kw = dict(plot_kw)
    if not plot_kw:  # global-frame local maps need room around the origin
      kw = dict(width_offset=60., height_offset=60.)
    ln = nb.step(depth, cam_pose=poses[t], **kw)
    lg = gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(ln, lg, f"step {t} local")
    _same_map(nb.world_map, gb.world_map, f"step {t} world")
    assert_same(npy(nb.world_map.get_camera()), npy(gb.world_map.get_camera()), "get_camera")
  assert nb._handles and not gb._handles, "the native path was not taken"
  # a later general merge accepts what the native path left behind (tracked box included)
  depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[0].cuda(), seed=6, half=6.0, device="cuda")
  kw = dict(plot_kw) or dict(width_offset=60., height_offset=60.)
  nb.step(depth, cam_pose=poses[0], center_mode=dmap.CenterMode.none, valid_map=torch.ones((b, 1, H, W), dtype=torch.bool), **kw)
  gb.step(depth, cam_pose=poses[0], **kw)
  _same_map(nb.world_map, gb.world_map, "mixed paths world")
  assert_workspaces_clean()


def test_native_step_fixed_canvas_equals_general_path():
  b, T, H, W = 3, 6, 120, 160
  poses = _walk(b, T, seed=9)
  nb, gb = _builder(True, fixed=(400, 380)), _builder(False, fixed=(400, 380))
  kw = dict(to_global=False, width_offset=60., height_offset=0., map_width=120, map_height=120)
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=9, half=6.0, device="cuda")
    ln, lg = nb.step(depth, cam_pose=poses[t], **kw), gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(ln, lg, f"step {t} local")
    _same_map(nb.world_map, gb.world_map, f"step {t} canvas")
  assert nb._handles and not gb._handles
  assert 0 < int(nb.world_map.mask.sum()) < nb.world_map.mask.numel()
  nb.reset(); gb.reset()
  assert nb.world_map.is_empty
  assert_workspaces_clean()


def test_native_step_vs_oracle_and_fallbacks():
  """The native step against the oracle's restatement of fuse_topdown_maps, plus the cases that must fall back to
  the general path (numpy depth, value maps, a centre mode, tensor-valued offsets)."""
  b, T, H, W = 2, 3, 120, 160
  poses = _walk(b, T, seed=3)
  nb = _builder(True)
  k = nb.proj.cam_params
  world = None
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=3, half=6.0, device="cuda")
    local = nb.step(depth, cam_pose=poses[t], to_global=False, width_offset=60., height_offset=0.)
    p = poses[t].numpy()
    want = orc.orth_project(npy(depth), None, None, p, 60., 0., PITCH, 0.88, 0.05, 120, 120, k.fx, k.fy, k.cx, k.cy,
                            0.15, 5.05, None, 3, False, True, -np.inf, None, True)
    assert_same(npy(local.topdown_map), want[0], f"step {t} local")
    src = [orc.FuseSource(npy(local.height_map), npy(local.mask), None, 60., 0., 0.05, True, False, p)]
    if world is not None:
      src.insert(0, orc.FuseSource(world["height"], world["mask"], None, world["width_offset"], world["height_offset"],
                                   0.05, True, True, p))
    world = orc.fuse(src, True, p, 0.05, True)
    wm = nb.world_map
    assert [wm.proj.map_height, wm.proj.map_width] == [world["map_height"], world["map_width"]]
    assert_same(npy(wm.topdown_map), world["topdown"], f"step {t} world")
    assert_same(npy(wm.mask), world["mask"], f"step {t} world mask")
  n_handles = len(nb._handles)
  depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[0].cuda(), seed=3, half=6.0, device="cuda")
  base = dict(to_global=False, width_offset=60., height_offset=0.)
  nb.step(npy(depth), cam_pose=poses[0], **base)                                        # host depth
  nb.step(depth, cam_pose=poses[0], center_mode="camera", **base)                       # a centre mode
  nb.step(depth, cam_pose=poses[0], **dict(base, width_offset=torch.full((b,), 60.)))   # per-sample offsets
  nb.step(depth, cam_pose=poses[0], merge=False, **base)                                # plot only
  assert len(nb._handles) == n_handles, "a fallback case created a native handle"
  assert_workspaces_clean()


def test_plane_boxes_equal_the_mask_extents_and_a_full_scan():
  """The per-plane rectangles the scatter pass leaves next to a map it wrote (DmFuseSource.plane_box) are exactly the
  extents of that plane's valid cells, a merge that scans only those rectangles equals a merge that scans whole
  planes, and an in-place edit of the mask drops them."""
  b, T, H, W = 3, 4, 120, 160
  poses = _walk(b, T + 1, seed=11)
  gb = _builder(False)   # general path: fuse_topdown_maps
  kw = dict(to_global=False, width_offset=60., height_offset=0., map_width=120, map_height=120)
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=11, half=6.0, device="cuda")
    gb.step(depth, cam_pose=poses[t], **kw)
  wm = gb.world_map
  tb = wm._tracked_box
  assert tb.plane_box is not None and tuple(tb.plane_box.shape) == (b, 4)
  boxes = tb.plane_box.cpu().numpy()
  mask = npy(wm.mask)
  for p in range(b):
    rows, cols = np.nonzero(mask[p, 0])
    assert list(boxes[p]) == [rows.min(), rows.max(), cols.min(), cols.max()], f"plane {p}"
  depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[T].cuda(), seed=11, half=6.0, device="cuda")
  local = gb.plot(depth, cam_pose=poses[T], **kw)
  target = gb.proj.clone(cam_pose=poses[T])
  boxed = dmap.fuse_topdown_maps(wm, local, map_projector=target)
  planes, tb.plane_box = tb.plane_box, None
  full = dmap.fuse_topdown_maps(wm, local, map_projector=target)
  tb.plane_box = planes
  _same_map(boxed, full, "boxed scan vs full scan")
  wm.mask[0, 0, 0, 0] = True          # in-place edit: the rectangles no longer describe the mask
  edited = dmap.fuse_topdown_maps(wm, local, map_projector=target)
  assert bool(edited.mask.any()) and edited.mask.sum() >= full.mask.sum()
  # the same through the C step object: world maps of the native path carry the rectangles too
  nb = _builder(True)
  for t in range(T):
    depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=11, half=6.0, device="cuda")
    nb.step(depth, cam_pose=poses[t], **kw)
  assert_same(npy(nb.world_map._tracked_box.plane_box), boxes, "native path plane boxes")
  assert_workspaces_clean()


@pytest.mark.parametrize("native", [True, False])
@pytest.mark.parametrize("fill,reduction,values", [(dmap.NINF, None, False), (None, None, False), (50., "min", False),
                                                   (dmap.NINF, None, True)])
def test_dense_world_copy_equals_the_per_cell_scatter(native, fill, reduction, values):
  """A merge copies the old world map into the new canvas densely when every cell of a plane moves by one whole
  (dx, dz) (dm_fuse.cu: plane_shift) and cell by cell otherwise: the same maps, offsets and tracked rectangles,
  step after step (dm_debug_set_dense_shift switches the dense path off), and the oracle's bits."""
  from dungeon_maps_b200 import _native as nat
  if values and native:
    pytest.skip("the C step covers height maps only")
  b, T, H, W = 3, 7, 120, 160
  poses = _walk(b, T, seed=11)
  kw = dict(to_global=False, width_offset=60., height_offset=0., map_width=120, map_height=120)
  runs = []
  try:
    for dense in (1, 0):
      nat.lib().dm_debug_set_dense_shift(dense)
      bld = _builder(native, fill=fill, reduction=reduction)
      worlds = []
      for t in range(T):
        depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=11, half=6.0, device="cuda")
        vm = synth.uniform((b, 2, H, W), 100 + t, -1., 1., device="cuda") if values else None
        bld.step(depth, cam_pose=poses[t], value_map=vm, **kw)
        wm = bld.world_map
        tb = getattr(wm, "_tracked_box", None)
        worlds.append((wm, None if tb is None or tb.plane_box is None else tb.plane_box.cpu().numpy().copy()))
      runs.append(worlds)
  finally:
    nat.lib().dm_debug_set_dense_shift(1)
  for t, ((wa, ba), (wb, bb)) in enumerate(zip(*runs)):
    _same_map(wa, wb, f"step {t} world (dense vs per-cell)")
    assert (ba is None) == (bb is None)
    if ba is not None:
      assert np.array_equal(ba, bb), f"step {t}: tracked rectangles differ"
  assert_workspaces_clean()


def test_prefilled_canvases_and_their_tail(monkeypatch):
  """The C step fills canvases of the old map's size class before the bounding box is known (the old map's cells + 2 %)
  and dm_builder_merge fills whatever tail the new map has beyond that.  With a generous size class (patched to 2 x) and
  a fast walk the new map regularly lands between the guess and the class: same world maps as the general path, which
  never speculates.  Height maps, then class ids of a few classes (values, heights and mask canvases)."""
  from dungeon_maps_b200 import maps as dmaps
  monkeypatch.setattr(dmaps, "_canvas_cap", lambda n: 2 * n)
  b, T, H, W, C = 8, 8, 120, 160, 3
  poses = _walk(b, T, seed=23, half=12.0)
  def make(native):
    proj = dmap.MapProjector(width=W, height=H, hfov=HFOV, cam_pose=[0., 0., 0.], width_offset=0., height_offset=0.,
                             cam_pitch=PITCH, cam_height=0.88, map_res=0.03, map_width=200, map_height=200,
                             trunc_depth_min=0.15, trunc_depth_max=5.05, clip_border=3, fill_value=dmap.NINF,
                             to_global=True, device="cuda")
    return dmap.MapBuilder(map_projector=proj, native_step=native)
  for labels in (False, True):
    nb, gb = make(True), make(False)
    grew = 0
    for t in range(T):
      depth = synth.room_depth(b, H, W, HFOV, PITCH, 0.88, poses[t].cuda(), seed=23, half=14.0, device="cuda")
      kw = dict(to_global=False, width_offset=100., height_offset=0., map_width=200, map_height=200)
      if labels:
        kw.update(label_map=synth.block_labels(b, C, H, W, seed=300 + t, device="cuda"), num_classes=C)
      before = 0 if nb.world_map is None or nb.world_map.is_empty else nb.world_map.mask.numel()
      nb.step(depth, cam_pose=poses[t], **kw)
      gb.step(depth, cam_pose=poses[t], **kw)
      after = nb.world_map.mask.numel()
      if before >= (1 << 18) and before + before // 50 + 4096 < after <= 2 * before:
        grew += 1
      _same_map(nb.world_map, gb.world_map, f"labels={labels} step {t} world")
    assert nb._handles, "the native path was not taken"
    assert nb.world_map.is_height_map != labels
    assert grew > 0, f"labels={labels}: no step exercised the tail fill: make the walk faster"
  assert_workspaces_clean()
