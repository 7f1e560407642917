"""The point primitives without a device: compute_center_offsets against the reference's values in
tests/golden/primitives.npz, and the C entries behind the point kernels (csrc/dm_points.cu) refusing bad arguments
before any CUDA call, among them the sizes their kernels would index with a 32-bit int."""

import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._golden import Golden, assert_same

# never dereferenced: every call below is refused before the first launch
IN, AUX, OUT, OUT2 = 0x10000, 0x20000, 0x30000, 0x40000


@pytest.mark.parametrize("to_global", [True, False])
@pytest.mark.parametrize("mode", ["none", "origin", "camera"])
def test_compute_center_offsets_matches_reference(mode, to_global):
  g = Golden("primitives")
  wo, ho = dmap.compute_center_offsets(torch.from_numpy(g["cco_pose"]), torch.tensor([1.5]), torch.tensor([-2.0]),
                                       0.03, 400, 400, to_global, mode)
  assert_same(wo.numpy(), g[f"cco_w_{mode}_{int(to_global)}"], f"{mode} to_global={to_global} width_offset")
  assert_same(ho.numpy(), g[f"cco_h_{mode}_{int(to_global)}"], f"{mode} to_global={to_global} height_offset")


CROP_REFUSALS = ["image", "center", "out", "b=-1", "c=-1", "h=0", "w=0", "crop_h=-1", "crop_w=-1",
                 "crop of 2^31 cells", "image plane of 2^31 cells"]


def _crop_args(case):
  a = dict(image=IN, center=AUX, b=2, c=3, h=40, w=30, crop_h=8, crop_w=6, out=OUT)
  if case in ("image", "center", "out"):
    a[case] = None
  elif "=" in case:
    name, value = case.split("=")
    a[name] = int(value)
  elif case == "crop of 2^31 cells":
    a["crop_h"], a["crop_w"] = 1 << 16, 1 << 15
  elif case == "image plane of 2^31 cells":
    a["h"], a["w"] = 1 << 15, 1 << 16
  return a


@pytest.mark.parametrize("case", CROP_REFUSALS)
def test_crop_nearest_f32_refuses_bad_arguments(case):
  a = _crop_args(case)
  rc = nat.lib().dm_crop_nearest_f32(a["image"], a["center"], a["b"], a["c"], a["h"], a["w"], a["crop_h"],
                                     a["crop_w"], 1, float("-inf"), a["out"], None)
  assert rc == -1


@pytest.mark.parametrize("case", CROP_REFUSALS)
def test_crop_nearest_u8_refuses_bad_arguments(case):
  a = _crop_args(case)
  rc = nat.lib().dm_crop_nearest_u8(a["image"], a["center"], a["b"], a["c"], a["h"], a["w"], a["crop_h"],
                                    a["crop_w"], a["out"], None)
  assert rc == -1


@pytest.mark.parametrize("case", ["depth", "points", "valid_out", "frames=-1", "H=0", "W=-2",
                                  "frame of 2^31 pixels"])
def test_depth_to_points_refuses_bad_arguments(case):
  a = dict(depth=IN, frames=2, H=24, W=32, points=OUT, valid_out=OUT2)
  if case in ("depth", "points", "valid_out"):
    a[case] = None
  elif "=" in case:
    name, value = case.split("=")
    a[name] = int(value)
  else:
    a["frames"], a["H"], a["W"] = 1, 1 << 16, 1 << 15
  rc = nat.lib().dm_depth_to_points_f32(a["depth"], None, a["frames"], a["H"], a["W"], 20., 20., 16., 12., 1, 1, 0.1,
                                        1, 5., a["points"], a["valid_out"], None)
  assert rc == -1


@pytest.mark.parametrize("case", ["points", "steps", "out", "b=-1", "n=-1", "n_steps=-1"])
def test_transform_points_refuses_bad_arguments(case):
  a = dict(points=IN, steps=AUX, n_steps=2, b=3, n=45, out=OUT)
  if case in ("points", "steps", "out"):
    a[case] = None
  else:
    name, value = case.split("=")
    a[name] = int(value)
  rc = nat.lib().dm_transform_points_f32(a["points"], a["steps"], a["n_steps"], a["b"], a["n"], a["out"], None)
  assert rc == -1


@pytest.mark.parametrize("case", ["points", "out", "n=-1"])
def test_image_camera_refuses_bad_arguments(case):
  a = dict(points=IN, n=45, out=OUT)
  if case == "n=-1":
    a["n"] = -1
  else:
    a[case] = None
  rc = nat.lib().dm_image_camera_f32(a["points"], a["n"], 20., 20., 16., 12., 1, 24, 0, a["out"], None)
  assert rc == -1


@pytest.mark.parametrize("entry", ["dm_map_quantize_f32", "dm_map_dequantize_f32"])
@pytest.mark.parametrize("case", ["x", "z", "width_offset", "height_offset", "x_out", "z_out", "b=-1", "n=-1"])
def test_map_quantize_refuses_bad_arguments(entry, case):
  a = dict(x=IN, z=IN + 256, width_offset=AUX, height_offset=AUX + 64, b=3, n=7, x_out=OUT, z_out=OUT2)
  if "=" in case:
    name, value = case.split("=")
    a[name] = int(value)
  else:
    a[case] = None
  rc = getattr(nat.lib(), entry)(a["x"], a["z"], a["width_offset"], a["height_offset"], a["b"], a["n"], 0.05, 40, 1,
                                 a["x_out"], a["z_out"], None)
  assert rc == -1
