"""MapBuilder.step for value maps with its host side in C (dm_builder_create_values / _plot_values / _merge_values /
_step_fixed_values) against the general Python path and the oracle: same maps, offsets, tracked boxes, step by step."""
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
LOCAL = dict(to_global=False, width_offset=60., height_offset=0., map_width=120, map_height=120)  # config-4 kwargs


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


def _depth(b, pose, seed, H=120, W=160):
  return synth.room_depth(b, H, W, HFOV, PITCH, 0.88, pose.cuda(), seed=seed, half=6.0, device="cuda")


def _inputs(kind, b, C, t, H=120, W=160):
  """Step keyword arguments of one frame: float planes (uniform or one-hot) or class ids (some of them >= C or 255)."""
  if kind == "uniform":
    return dict(value_map=synth.uniform((b, C, H, W), 100 + t, -1., 1., device="cuda"))
  if kind == "onehot":
    return dict(value_map=synth.block_onehot(b, C, H, W, seed=200 + t, device="cuda"))
  ids = synth.block_labels(b, C + 3, H, W, seed=300 + t, device="cuda")   # ids C..C+2 are "no class"
  ids[:, :, :8] = 255
  return dict(label_map=ids, num_classes=C)


def _plane_box(m):
  tb = getattr(m, "_tracked_box", None)
  return None if tb is None or tb.plane_box is None else npy(tb.plane_box)


def _box(m):
  tb = getattr(m, "_tracked_box", None)
  return None if tb is None or tb.box is None else npy(tb.box)


def _same_map(a, b_, what, boxes=True):
  assert [a.proj.map_height, a.proj.map_width] == [b_.proj.map_height, b_.proj.map_width], f"{what} shape"
  for name in ("width_offset", "height_offset"):
    x, y = getattr(a.proj, name), getattr(b_.proj, name)
    if torch.is_tensor(y):
      assert torch.is_tensor(x) and x.shape == y.shape and x.dtype == y.dtype, f"{what} {name} type"
    assert_same(np.asarray(x, np.float32).reshape(-1), np.asarray(y, np.float32).reshape(-1), f"{what} {name}")
  assert tuple(a.topdown_map.shape) == tuple(b_.topdown_map.shape), f"{what} topdown shape"
  assert_same(npy(a.topdown_map), npy(b_.topdown_map), f"{what} topdown")
  assert_same(npy(a.mask), npy(b_.mask), f"{what} mask")
  assert_same(npy(a.height_map), npy(b_.height_map), f"{what} height")
  assert a.is_height_map == b_.is_height_map, f"{what} is_height_map"
  if boxes:
    for get in (_box, _plane_box):
      x, y = get(a), get(b_)
      assert (x is None) == (y is None), f"{what}: tracked box presence"
      if x is not None:
        assert np.array_equal(x, y), f"{what}: tracked boxes differ"


@pytest.mark.parametrize("plot_kw", [LOCAL, dict(width_offset=60., height_offset=60.),
                                     dict(to_global=False, width_offset=40.5, height_offset=3., map_width=90,
                                          map_height=70)], ids=["local", "global", "odd"])
@pytest.mark.parametrize("fill,reduction", [(dmap.NINF, None), (None, None), (0., None), (50., "min"),
                                            (float("nan"), None)], ids=["ninf", "none", "zero", "min50", "nan"])
@pytest.mark.parametrize("kind,C", [("uniform", 3), ("onehot", 16), ("labels", 16)])
def test_value_step_equals_general_path(kind, C, fill, reduction, plot_kw):
  b, T = 3, 8
  poses = _walk(b, T, seed=5)
  nb, gb = _builder(True, fill=fill, reduction=reduction), _builder(False, fill=fill, reduction=reduction)
  for t in range(T):
    depth = _depth(b, poses[t], 5)
    kw = dict(plot_kw, **_inputs(kind, b, C, t))
    ln = nb.step(depth, cam_pose=poses[t], **kw)
    lg = gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(ln, lg, f"step {t} local", boxes=False)
    assert ln.height_map.stride(1) == 0 and tuple(ln.height_map.shape) == tuple(ln.topdown_map.shape)
    _same_map(nb.world_map, gb.world_map, f"step {t} world")
    assert_same(npy(nb.world_map.get_camera()), npy(gb.world_map.get_camera()), "get_camera")
    if fill != fill:
      assert _box(nb.world_map) is None and _plane_box(nb.world_map) is None, "a NaN fill tracks no box"
    elif _plane_box(nb.world_map) is not None:
      assert _plane_box(nb.world_map).shape == (b * C, 4)
  assert nb._handles and not gb._handles, "the C step was not taken"
  assert_workspaces_clean()


@pytest.mark.parametrize("kind", ["uniform", "labels"])
def test_value_step_vs_oracle(kind):
  b, T, C, H, W = 2, 3, 4, 120, 160
  poses = _walk(b, T, seed=3)
  nb = _builder(True)
  k = nb.proj.cam_params
  world = None
  for t in range(T):
    depth = _depth(b, poses[t], 3)
    kw = _inputs(kind, b, C, t)
    local = nb.step(depth, cam_pose=poses[t], **LOCAL, **kw)
    p = poses[t].numpy()
    values = kw.get("value_map")
    if values is None:
      ids = kw["label_map"].to(torch.int64)
      values = (torch.arange(C, device="cuda").view(1, -1, 1, 1) == ids).float()
    top, mask, hgt = orc.orth_project(npy(depth), npy(values), None, p, 60., 0., PITCH, 0.88, 0.05, 120, 120, k.fx, k.fy,
                                      k.cx, k.cy, 0.15, 5.05, None, 3, False, True, -np.inf, None, True)
    assert_same(npy(local.topdown_map), top, f"step {t} local")
    assert_same(npy(local.height_map[:, :1]), hgt, f"step {t} local height")
    src = [orc.FuseSource(hgt, mask, top, 60., 0., 0.05, True, False, p)]
    if world is not None:
      src.insert(0, orc.FuseSource(world["height"], world["mask"], world["topdown"], world["width_offset"],
                                   world["height_offset"], 0.05, True, True, p))
    world = orc.fuse(src, True, p, 0.05, True)
    wm = nb.world_map
    assert [wm.proj.map_height, wm.proj.map_width] == [world["map_height"], world["map_width"]]
    assert_same(npy(wm.topdown_map), world["topdown"], f"step {t} world")
    assert_same(npy(wm.mask), world["mask"], f"step {t} world mask")
    assert_same(npy(wm.height_map), world["height"], f"step {t} world height")
  assert nb._handles
  assert_workspaces_clean()


@pytest.mark.parametrize("kind", ["onehot", "labels"])
def test_fixed_canvas_value_step_equals_general_path(kind):
  b, T, C = 3, 6, 5
  poses = _walk(b, T, seed=9)
  nb, gb = _builder(True, fixed=(400, 380), fill=0.), _builder(False, fixed=(400, 380), fill=0.)
  first = None
  for t in range(T):
    depth = _depth(b, poses[t], 9)
    kw = dict(LOCAL, **_inputs(kind, b, C, t))
    ln, lg = nb.step(depth, cam_pose=poses[t], **kw), gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(ln, lg, f"step {t} local", boxes=False)
    _same_map(nb.world_map, gb.world_map, f"step {t} canvas", boxes=False)
    first = first or nb.world_map.topdown_map.data_ptr()
    assert nb.world_map.topdown_map.data_ptr() == first, "the canvas is updated in place"
  assert nb._handles and not gb._handles
  assert 0 < int(nb.world_map.mask.sum()) < nb.world_map.mask.numel()
  nb.reset(); gb.reset()
  assert nb.world_map.is_empty
  assert_workspaces_clean()


def test_long_walk_crosses_size_classes():
  from dungeon_maps_b200 import maps as dmaps
  b, T, C = 4, 40, 8
  # walkers start near the origin and head out diagonally without turning: the world map grows every step
  start = _walk(b, 1, seed=13, half=1.0)[0]
  poses = torch.stack([start + torch.tensor([0.25 * t, 0.125 * t, 0.]) for t in range(T)])
  nb, gb = _builder(True), _builder(False)
  classes = set()
  for t in range(T):
    depth = synth.room_depth(b, 120, 160, HFOV, PITCH, 0.88, poses[t].cuda(), seed=13, half=20.0, device="cuda")
    kw = dict(LOCAL, **_inputs("labels", b, C, t))
    nb.step(depth, cam_pose=poses[t], **kw)
    gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} world")
    n = nb.world_map.mask.numel()
    if n >= (1 << 18):
      classes.add(dmaps._canvas_cap(n))
  assert len(classes) >= 3, f"the world canvas crossed only {len(classes)} size classes"
  assert nb._handles and not gb._handles
  assert_workspaces_clean()


def test_fallbacks_create_no_handle():
  b, C, H, W = 2, 3, 120, 160
  poses = _walk(b, 2, seed=17)
  depth = _depth(b, poses[0], 17)
  v = synth.uniform((b, C, H, W), 1, -1., 1., device="cuda")
  cases = [
    dict(value_map=v.cpu()),                                                  # host values
    dict(value_map=v.double()),                                               # float64
    dict(value_map=v.transpose(2, 3).contiguous().transpose(2, 3)),           # non-contiguous
    dict(value_map=v, valid_map=torch.ones((b, 1, H, W), dtype=torch.bool, device="cuda")),
    dict(value_map=v, center_mode=dmap.CenterMode.camera),
  ]
  for i, extra in enumerate(cases):
    nb, gb = _builder(True), _builder(False)
    for t in range(2):
      ln = nb.step(_depth(b, poses[t], 17), cam_pose=poses[t], **LOCAL, **extra)
      lg = gb.step(_depth(b, poses[t], 17), cam_pose=poses[t], **LOCAL, **extra)
      _same_map(ln, lg, f"case {i} local", boxes=False)
      _same_map(nb.world_map, gb.world_map, f"case {i} world")
    assert not nb._handles, f"case {i} created a native handle"
  nb, gb = _builder(True, fill=0., reduction="sum"), _builder(False, fill=0., reduction="sum")
  _same_map(nb.step(depth, cam_pose=poses[0], value_map=v, **LOCAL), gb.step(depth, cam_pose=poses[0], value_map=v, **LOCAL),
            "sum local", boxes=False)
  _same_map(nb.world_map, gb.world_map, "sum world")
  assert not nb._handles
  ids = synth.block_labels(b, C, H, W, seed=1, device="cuda")
  nb = _builder(True)
  with pytest.raises(ValueError):
    nb.step(depth, cam_pose=poses[0], label_map=ids, **LOCAL)
  with pytest.raises(ValueError):
    nb.step(depth, cam_pose=poses[0], value_map=v, label_map=ids, num_classes=C, **LOCAL)
  assert not nb._handles
  assert_workspaces_clean()


def test_mixed_paths():
  b, T, C = 3, 4, 4
  poses = _walk(b, T, seed=19)
  nb, gb = _builder(True, fill=0.), _builder(False, fill=0.)
  c_steps = []   # (step, world map the C step started from) of every step the C step took
  c_step = nb._native_step
  def spy(*args, **kwargs):
    started_from = nb.world_map
    local = c_step(*args, **kwargs)
    if local is not None:
      c_steps.append((t, started_from))
    return local
  nb._native_step = spy
  for t in range(T):
    depth = _depth(b, poses[t], 19)
    kw = dict(LOCAL, **_inputs("onehot", b, C, t))
    before = nb.world_map
    if t == 1:   # a C-step world map continued by the general path (a valid_map forces it)
      valid = torch.ones((b, 1, 120, 160), dtype=torch.bool, device="cuda")
      nb.step(depth, cam_pose=poses[t], valid_map=valid, **kw)
      gb.step(depth, cam_pose=poses[t], valid_map=valid, **kw)
    else:        # t == 2: the general path's world map of step 1 continued by the C step
      nb.step(depth, cam_pose=poses[t], **kw)
      gb.step(depth, cam_pose=poses[t], **kw)
    _same_map(nb.world_map, gb.world_map, f"step {t} world")
    if t == 2:
      assert c_steps[-1] == (2, before) and not before.is_empty, "step 2 did not continue the general world map in C"
  assert [s for s, _ in c_steps] == [0, 2, 3], "the C step was not taken where it should be, or taken at step 1"
  hb = _builder(True)
  hb.step(_depth(b, poses[0], 19), cam_pose=poses[0], **LOCAL)   # height world map
  assert hb.world_map.is_height_map
  with pytest.raises(AssertionError):
    hb.step(_depth(b, poses[1], 19), cam_pose=poses[1], **LOCAL, **_inputs("onehot", b, C, 1))
  assert_workspaces_clean()


def test_handle_cache_is_bounded():
  b, C = 2, 3
  poses = _walk(b, 10, seed=21)
  nb = _builder(True)
  seen = []
  for t in range(10):
    nb.step(_depth(b, poses[t], 21), cam_pose=poses[t], **dict(LOCAL, width_offset=50. + t),
            **_inputs("uniform", b, C, t))
    seen.extend(h for h in nb._handles.values() if h not in seen)
    assert len(nb._handles) <= nb._MAX_HANDLES
  assert len(seen) == 10
  live = list(nb._handles.values())
  assert all(h.handle for h in live)
  assert all(not h.handle for h in seen if h not in live), "an evicted handle was not destroyed"
  assert_workspaces_clean()
