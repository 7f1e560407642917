"""score_poses without a device: dm_score_poses_i32 refuses bad arguments before any CUDA call, the Python function
refuses bad calls before any device work, it is exported, and the definition (tests/_match.py, composed from the
oracle) is the overlap count of a shifted numpy slice at yaw 0 and of its rotation by 90 degrees at yaw pi/2."""
import math

import numpy as np
import pytest
import torch

import dungeon_maps_b200 as dmap
from dungeon_maps_b200 import _native as nat
from tests._match import random_planes, score_poses

# never dereferenced: every call below is refused before the first launch
PLANES, WINDOW, SAMPLES, SCORES = 0x10000, 0x20000, 0x30000, 0x40000
REFUSALS = ["planes", "window", "samples", "scores", "b=0", "C=0", "Hs=0", "Ws=-1", "h=0", "w=-1", "n=0",
            "window_planes=0", "window_planes=2", "map_res=0", "map_res=nan", "map_res=-1", "b * n of 2^31",
            "h * w of 2^31", "Hs * Ws of 2^31", "unaligned samples"]


@pytest.mark.parametrize("case", REFUSALS)
def test_score_poses_refuses_bad_arguments(case):
  a = dict(planes=PLANES, b=2, C=3, Hs=40, Ws=30, map_res=0.05, flip_h=1, window=WINDOW, window_planes=3, h=8, w=6,
           samples=SAMPLES, n=5, scores=SCORES)
  if case in ("planes", "window", "samples", "scores"):
    a[case] = None
  elif "=" in case:
    name, value = case.split("=")
    a[name] = float(value) if name == "map_res" else int(value)
  elif case == "b * n of 2^31":
    a["b"], a["n"] = 1 << 16, 1 << 15
  elif case == "h * w of 2^31":
    a["h"], a["w"] = 1 << 16, 1 << 15
  elif case == "Hs * Ws of 2^31":
    a["Hs"], a["Ws"] = 1 << 15, 1 << 16
  elif case == "unaligned samples":
    a["samples"] = SAMPLES + 2
  rc = nat.lib().dm_score_poses_i32(a["planes"], a["b"], a["C"], a["Hs"], a["Ws"], a["map_res"], a["flip_h"],
                                    a["window"], a["window_planes"], a["h"], a["w"], a["samples"], a["n"],
                                    a["scores"], None)
  assert rc == -1


def test_score_poses_limits_are_exclusive():
  """One cell below each 2^31 limit is not refused for its size (the null scores pointer is what refuses it)."""
  for b, n, h, w, Hs, Ws in ((1 << 16, (1 << 15) - 1, 8, 6, 40, 30), (2, 5, (1 << 16) - 1, 1 << 15, 40, 30)):
    assert nat.lib().dm_score_poses_i32(PLANES, b, 1, Hs, Ws, 0.05, 1, WINDOW, 1, h, w, SAMPLES, n, None, None) == -1


def test_exported():
  assert dmap.score_poses is dmap.maps.score_poses
  assert "score_poses" in dmap.maps.__all__


def _source(b=2, Hs=11, Ws=13, to_global=True, woff=6., hoff=5., flip_h=True, res=0.25):
  top = torch.zeros((1, 1, 1, 1)).expand(b, 1, Hs, Ws)     # only the shape and the projector are read
  proj = dmap.MapProjector(width=16, height=12, hfov=1.2, map_res=res, map_width=Ws, map_height=Hs,
                           width_offset=woff, height_offset=hoff, to_global=to_global, flip_h=flip_h)
  mask = torch.zeros((1, 1, 1, 1), dtype=torch.bool).expand(b, 1, Hs, Ws)
  return dmap.TopdownMap(topdown_map=top, mask=mask, height_map=top, map_projector=proj, is_height_map=True)


def _big(shape):
  return torch.ones((1,) * len(shape), dtype=torch.bool).expand(*shape)


VALUE_ERRORS = {
  "empty source": "needs a map", "local-frame source": "global-frame", "planes not a tensor": "bool tensor",
  "planes uint8": "bool tensor", "window float": "bool tensor", "planes 2-D": r"\(b, Hs, Ws\)",
  "planes 5-D": r"\(b, Hs, Ws\)", "planes batch": "like the source", "planes height": "like the source",
  "planes width": "like the source", "planes no channel": "like the source", "window 2-D": "window must be",
  "window 4-D with 3-D planes": "window must be", "window planes count": "window must be",
  "window batch": "window must be", "window empty": "not be empty", "poses 1-D": "cam_poses",
  "poses 4 columns": "cam_poses", "poses n=0": "cam_poses", "poses batch": "cam_poses", "poses 4-D": "cam_poses",
  "width offsets": "width_offset", "height offsets": "height_offset", "b * n": "2\\^31", "h * w": "2\\^31",
  "Hs * Ws": "2\\^31", "planes on the host": "CUDA",
}


@pytest.mark.parametrize("case", list(VALUE_ERRORS))
def test_value_errors_before_any_device_work(case):
  b = 2
  src = _source(b)
  planes = torch.ones((b, 3, 11, 13), dtype=torch.bool)
  window = torch.ones((b, 4, 5), dtype=torch.bool)
  kw = dict(cam_poses=np.zeros((7, 3), np.float32))
  if case == "empty source":
    src = dmap.TopdownMap(map_projector=src.proj)
  elif case == "local-frame source":
    src = _source(b, to_global=False)
  elif case == "planes not a tensor":
    planes = planes.numpy()
  elif case == "planes uint8":
    planes = planes.to(torch.uint8)
  elif case == "window float":
    window = window.float()
  elif case == "planes 2-D":
    planes = planes[0, 0]
  elif case == "planes 5-D":
    planes = planes[None]
  elif case == "planes batch":
    planes = planes[:1]
  elif case == "planes height":
    planes = planes[:, :, :10]
  elif case == "planes width":
    planes = planes[:, :, :, 1:]
  elif case == "planes no channel":
    planes = planes[:, :0]
  elif case == "window 2-D":
    window = window[0]
  elif case == "window 4-D with 3-D planes":
    planes, window = planes[:, 0], window[:, None]
  elif case == "window planes count":
    window = window[:, None].expand(b, 2, 4, 5)
  elif case == "window batch":
    window = torch.ones((3, 4, 5), dtype=torch.bool)
  elif case == "window empty":
    window = window[:, :, :0]
  elif case == "poses 1-D":
    kw["cam_poses"] = [0., 0., 0.]
  elif case == "poses 4 columns":
    kw["cam_poses"] = torch.zeros((7, 4))
  elif case == "poses n=0":
    kw["cam_poses"] = torch.zeros((0, 3))
  elif case == "poses batch":
    kw["cam_poses"] = torch.zeros((3, 7, 3))
  elif case == "poses 4-D":
    kw["cam_poses"] = torch.zeros((1, b, 7, 3))
  elif case == "width offsets":
    kw["width_offset"] = [1., 2., 3.]
  elif case == "height offsets":
    kw["height_offset"] = np.zeros(4, np.float32)
  elif case == "b * n":
    kw["cam_poses"] = torch.zeros((1, 3)).expand(2 ** 30, 3)
  elif case == "h * w":
    window = _big((b, 1 << 16, 1 << 15))
  elif case == "Hs * Ws":
    src = _source(b, Hs=1 << 15, Ws=1 << 16)
    planes = _big((b, 1 << 15, 1 << 16))
  with pytest.raises(ValueError, match=VALUE_ERRORS[case]):
    dmap.score_poses(src, planes, window, **kw)


RES = 0.25


def _oracle(src, planes, window, poses, u, v):
  p = src.proj
  return score_poses(planes, window, p.width_offset, p.height_offset, p.map_res, p.flip_h, poses, u, v)


def _padded(a, pad):
  return np.pad(a, ((0, 0), (0, 0), (pad, pad), (pad, pad)), constant_values=False)


# integer-cell poses (multiples of map_res): inside, straddling the corners, and entirely outside the 11 x 13 source
CELLS = [(0, 0), (3, -2), (-7, 6), (9, 9), (-40, 3)]


@pytest.mark.parametrize("h,w", [(5, 4), (7, 9), (6, 6)])
def test_yaw_zero_is_a_shifted_overlap(h, w):
  b, Hs, Ws, W, H = 2, 11, 13, 6, 5
  src = _source(b)
  rng = np.random.default_rng(h * 100 + w)
  planes = random_planes(rng, (b, 2, Hs, Ws), 0.5)
  window = random_planes(rng, (b, 1, h, w), 0.6)
  u, v = w // 2, h // 2
  pad = 64
  padded = _padded(planes, pad)
  poses = np.array([[px * RES, pz * RES, 0.] for px, pz in CELLS], np.float32)
  got = _oracle(src, planes, window, poses, u, v)
  for k, (px, pz) in enumerate(CELLS):
    # yaw 0: (X, Z) = (c - u + px + W, r + Hs - h - H + v - pz) with flip_h
    c0, r0 = W - u + px + pad, Hs - h - H + v - pz + pad
    want = (padded[:, :, r0:r0 + h, c0:c0 + w] & window).sum(axis=(2, 3))
    assert np.array_equal(got[:, :, k], want)
  assert not got[:, :, -1].any()      # the last pose is entirely outside


@pytest.mark.parametrize("h,w", [(5, 4), (7, 9)])
def test_yaw_half_pi_is_a_rot90_overlap(h, w):
  b, Hs, Ws, W, H = 2, 11, 13, 6, 5
  src = _source(b)
  rng = np.random.default_rng(h * 100 + w + 1)
  planes = random_planes(rng, (b, 2, Hs, Ws), 0.5)
  window = random_planes(rng, (b, 2, h, w), 0.6)     # one window per plane
  u, v = w // 2, h // 2
  pad = 64
  padded = _padded(planes, pad)
  poses = np.array([[[px * RES, pz * RES, math.pi / 2] for px, pz in CELLS]] * b, np.float32)
  got = _oracle(src, planes, window, poses, u, v)
  for k, (px, pz) in enumerate(CELLS):
    # as in test_egocentric_abi: window row r reads source column X0 + r, window column c reads source row Z0 - c,
    # so the window sees rot90(S, -1) of the slice S of rows Z0 - w + 1 .. Z0 and columns X0 .. X0 + h - 1
    X0, Z0 = px - h + 1 + v + W + pad, Hs - 1 - pz + u - H + pad
    seen = np.rot90(padded[:, :, Z0 - w + 1:Z0 + 1, X0:X0 + h], -1, axes=(2, 3))
    assert np.array_equal(got[:, :, k], (seen & window).sum(axis=(2, 3)))
