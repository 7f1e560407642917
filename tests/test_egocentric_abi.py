"""TopdownMap.select_egocentric without a device: dm_crop_egocentric_f32 refuses bad arguments before any CUDA call,
dm_pack_ego_samples packs what _params.local_to_global packs, the Python layer refuses bad calls before any device
work, and the definition (tests/_egocentric.py, composed from the oracle) is a plain slice of the source at yaw 0 and
its rotation by 90 degrees at yaw pi/2."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from dungeon_maps_b200 import _params as prm
from tests._egocentric import crop_egocentric

# never dereferenced: every call below is refused before the first launch
TOP, HEIGHT, MASK, SAMPLES, OUT_TOP, OUT_HEIGHT, OUT_MASK = (0x10000, 0x20000, 0x30000, 0x40000, 0x50000, 0x60000,
                                                             0x70000)
REFUSALS = ["topdown", "mask", "samples", "out_topdown", "out_mask", "b=0", "C=0", "Hs=0", "Ws=0", "crop_h=0",
            "crop_w=-1", "map_res=0", "map_res=nan", "height without out_height", "out_height without height",
            "plane stride", "unaligned samples", "window of 2^31 cells"]


@pytest.mark.parametrize("case", REFUSALS)
def test_crop_egocentric_refuses_bad_arguments(case):
  a = dict(topdown=TOP, height=HEIGHT, plane=40 * 30, mask=MASK, b=2, C=3, Hs=40, Ws=30, res=0.05, flip_h=1,
           samples=SAMPLES, crop_h=8, crop_w=6, fill=float("-inf"), out_topdown=OUT_TOP, out_height=OUT_HEIGHT,
           out_mask=OUT_MASK)
  if case in ("topdown", "mask", "samples", "out_topdown", "out_mask"):
    a[case] = None
  elif "=" in case and not case.startswith("window"):
    name, value = case.split("=")
    a[{"map_res": "res"}.get(name, name)] = float(value) if name == "map_res" else int(value)
  elif case == "height without out_height":
    a["out_height"] = None
  elif case == "out_height without height":
    a["height"] = None
  elif case == "plane stride":
    a["plane"] = 40 * 30 - 1
  elif case == "unaligned samples":
    a["samples"] = SAMPLES + 2
  elif case == "window of 2^31 cells":
    a["crop_h"], a["crop_w"] = 1 << 16, 1 << 15
  rc = nat.lib().dm_crop_egocentric_f32(a["topdown"], a["height"], a["plane"], a["mask"], a["b"], a["C"], a["Hs"],
                                        a["Ws"], a["res"], a["flip_h"], a["samples"], a["crop_h"], a["crop_w"],
                                        a["fill"], a["out_topdown"], a["out_height"], a["out_mask"], None)
  assert rc == -1


def test_pack_ego_samples_refuses_null_arguments():
  cfg = nat.DmPoseCfg()
  buf = torch.zeros(64)
  p = buf.data_ptr()
  assert nat.lib().dm_pack_ego_samples(cfg, p, p, p, p, p, p, None, 1, p) == -1
  assert nat.lib().dm_pack_ego_samples(None, p, p, p, p, p, p, p, 1, p) == -1
  assert nat.lib().dm_pack_ego_samples(cfg, p, p, p, p, p, p, p, -1, p) == -1


@pytest.mark.parametrize("n", [20, 45, 65536])
def test_pack_ego_samples_matches_local_to_global(n):
  yaws = [0., 0.0009, -0.0009, math.pi, -math.pi, math.pi / 2, 0.3, -2.1, 1e-3, 0.0011]
  b = len(yaws)
  g = torch.Generator().manual_seed(n)
  pose = torch.cat((torch.rand((b, 2), generator=g) * 20 - 10, torch.tensor(yaws, dtype=torch.float32)[:, None]), 1)
  offsets = [torch.rand((b,), generator=g) * 400 - 200 for _ in range(4)]
  got = prm.ego_samples(pose, *offsets, n)
  want = torch.cat((prm.local_to_global(pose, n), torch.stack(offsets, dim=1)), dim=1)
  assert got.shape == (b, nat.EGO_SAMPLE_WORDS)
  assert got.numpy().tobytes() == want.numpy().tobytes()
  assert (got.view(torch.int32)[:, 13] == int(9 * n >= 400)).all()


def _source(b=3, C=2, Hs=11, Ws=13, to_global=True, height_map=False, woff=6., hoff=5.):
  g = torch.Generator().manual_seed(7)
  top = torch.rand((b, C, Hs, Ws), generator=g)
  mask = torch.rand((b, C, Hs, Ws), generator=g) > 0.3
  hm = top if height_map else torch.rand((b, C, Hs, Ws), generator=g)
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=0.25, map_width=Ws, map_height=Hs,
                           width_offset=woff, height_offset=hoff, to_global=to_global)
  return dmap.TopdownMap(topdown_map=top, mask=mask, height_map=hm, map_projector=proj, is_height_map=height_map)


@pytest.mark.parametrize("case", ["empty", "local frame", "width 0", "height 0", "poses", "width offsets",
                                  "height offsets"])
def test_value_errors_before_any_device_work(case):
  src = _source()
  kw = dict(crop_width=4, crop_height=5, cam_pose=[[0., 0., 0.]])
  if case == "empty":
    src = dmap.TopdownMap(map_projector=src.proj)
  elif case == "local frame":
    src = _source(to_global=False)
  elif case == "width 0":
    kw["crop_width"] = 0
  elif case == "height 0":
    kw["crop_height"] = 0
  elif case == "poses":
    kw["cam_pose"] = torch.zeros((2, 3))
  elif case == "width offsets":
    kw["width_offset"] = [1., 2.]
  elif case == "height offsets":
    kw["height_offset"] = np.zeros(4, np.float32)
  with pytest.raises(ValueError):
    src.select_egocentric(**kw)
  with pytest.raises(ValueError):
    dmap.crop_egocentric_map(src, **kw)


RES = 0.25


def _oracle(src, pose, crop_w, crop_h, u, v, fill=-np.inf):
  p = src.proj
  return crop_egocentric(src.topdown_map.numpy(), src.mask.numpy(), src.height_map.numpy(), p.width_offset,
                         p.height_offset, p.map_res, p.flip_h, pose, crop_w, crop_h, u, v, fill)


def _padded(a, pad, fill):
  return np.pad(a, ((0, 0), (0, 0), (pad, pad), (pad, pad)), constant_values=fill)


# integer-cell poses (multiples of map_res): inside, straddling the corners, and entirely outside the 11 x 13 source
CELLS = [(0, 0), (3, -2), (-7, 6), (9, 9), (-40, 3)]


@pytest.mark.parametrize("crop_h,crop_w", [(5, 4), (7, 9), (6, 6)])
def test_yaw_zero_is_a_slice(crop_h, crop_w):
  src = _source()
  b, C, Hs, Ws = src.topdown_map.shape
  W, H = 6, 5     # the source's offsets
  u, v = crop_w // 2, crop_h // 2
  pad = 64
  want_top, want_mask, want_h = (_padded(t.numpy(), pad, f) for t, f in
                                 ((src.topdown_map, -np.inf), (src.mask, False), (src.height_map, -np.inf)))
  for px, pz in CELLS:
    pose = np.array([[px * RES, pz * RES, 0.]], np.float32)
    top, mask, hgt = _oracle(src, pose, crop_w, crop_h, u, v)
    # yaw 0: (X, Z) = (c - u + px + W, r + Hs - crop_h - H + v - pz) with flip_h
    c0, r0 = W - u + px + pad, Hs - crop_h - H + v - pz + pad
    sl = np.s_[:, :, r0:r0 + crop_h, c0:c0 + crop_w]
    assert np.array_equal(top, want_top[sl]) and np.array_equal(mask, want_mask[sl])
    assert np.array_equal(hgt, want_h[sl])


@pytest.mark.parametrize("crop_h,crop_w", [(5, 4), (7, 9)])
def test_yaw_half_pi_is_rot90_of_a_slice(crop_h, crop_w):
  src = _source()
  b, C, Hs, Ws = src.topdown_map.shape
  W, H = 6, 5
  u, v = crop_w // 2, crop_h // 2
  pad = 64
  want_top = _padded(src.topdown_map.numpy(), pad, -np.inf)
  want_mask = _padded(src.mask.numpy(), pad, False)
  # float32 gives R exactly: sin(pi/2) = 1, 1 - cos(pi/2) = 1, so R = (0, 0, 1, 0, 1, 0, -1, 0, 0) and
  # local_to_global_space (rot then add) maps (lx, 0, lz) to (x - lz, 0, z + lx): the camera's forward direction (+z
  # local, up in the window) is global -x.  With flip_h, lz = (crop_h - 1 - r - v) * res and lx = (c - u) * res, so
  #   X = r + (px - crop_h + 1 + v + W),  Z = -c + (Hs - 1 - pz + u - H):
  # window row r reads source column X0 + r, window column c reads source row Z0 - c.  The source slice S of rows
  # Z0 - crop_w + 1 .. Z0 and columns X0 .. X0 + crop_h - 1 is the window turned by 90 degrees: window = rot90(S, -1).
  for px, pz in CELLS:
    pose = np.array([[px * RES, pz * RES, math.pi / 2]], np.float32)
    top, mask, _ = _oracle(src, pose, crop_w, crop_h, u, v)
    X0, Z0 = px - crop_h + 1 + v + W + pad, Hs - 1 - pz + u - H + pad
    sl = np.s_[:, :, Z0 - crop_w + 1:Z0 + 1, X0:X0 + crop_h]
    assert np.array_equal(top, np.rot90(want_top[sl], -1, axes=(2, 3)))
    assert np.array_equal(mask, np.rot90(want_mask[sl], -1, axes=(2, 3)))
